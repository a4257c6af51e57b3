// mc_kernels.cu -- Lewiner marching cubes on the GPU, order-exact with the reference's sequential
// implementation (SdfKit/MarchingCubes.cs:39-546, SdfKit/Cell.cs:130-549).  Compiled for sm_100a with
// -fmad=false: every FP64/FP32 decision and interpolation is the IEEE operation the CPU path performs.
//
// The reference numbers vertices by "first touch" while visiting cells z-outer / y / x-inner and walking
// each cell's tiling row left to right, de-duplicating through two rolling face layers.  Every tiling row
// references exactly the sign-changing edges of its cube (+ optionally the centre vertex), so first touch
// is a pure function of geometry (DESIGN.md "order-exact formulation"):
//   * the creator ("owner") of a grid-edge vertex is the sharing cell smallest in (k, j, i);
//   * its id is  vbase[owner] + rank of the edge among the owner's created vertices in row order,
//     vbase = exclusive prefix sum of per-cell created-vertex counts in visiting order;
//   * triangle t of a cell is row entries 3t..3t+2 at  tbase[cell] + t.
// Pipeline (one pass over the distance field, everything else is O(active cells)):
//   K2 mc_classify  dist -> active cells per 128-cell chunk of a cell row
//   K3 mc_scan      warp-shuffle + decoupled look-back exclusive scan of the chunk counts (run twice: record slots
//                   after K2, vertex / triangle prefixes after K4a)
//   K4a mc_compact  active chunks -> one McRecord per active cell, in visiting order, + full per-chunk counts
//   K4b mc_emit     per record: triangle indices, created vertices (position, colour), normals gathered
//                   in the reference's accumulation order, -normalize, Mesh.Transform, AABB
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "mc_kernels.cuh"
#include "mc_luts.h"

#define MC_EPS 0.0000001                       // FLT_EPSILON of MarchingCubes.cs:37 / Cell.cs:65
#define MC_AMBIG 0x80000000u
// leaf = the tiling row a cell uses: dense row id [0:10) | triangles [10:14) | uses the centre vertex [14]
#define MC_LEAF(row, nt, center) ((unsigned)(row) | ((unsigned)(nt) << 10) | ((unsigned)(center) << 14))
#define MC_LEAF_ROW(l) ((l) & 0x3FFu)
#define MC_LEAF_NT(l) (((l) >> 10) & 0xFu)
#define MC_LEAF_CENTER(l) (((l) >> 14) & 1u)
#define FULL 0xFFFFFFFFu

// Static facts about one tiling row, precomputed on the host so that no kernel scans a row to answer them.
struct McRowMeta {
    unsigned short off;          // offset of the row's first entry in the LUT blob
    unsigned char nt;            // triangles
    unsigned char pad;
    unsigned short refmask;      // slots (edges 0..11, centre 12) the row references
    unsigned short before[13];   // before[e] = slots first referenced earlier in the row than e
    unsigned char occ[13];       // how many times the row references slot e
    unsigned char pad2[3];
    unsigned long long occ_packed;   // occ[0..11], 3 bits each, pre-shifted into McRecord::aux position
};

static const signed char h_lut[MCL_BLOB_SIZE] = MCL_BLOB_INIT;
__device__ const signed char d_lut[MCL_BLOB_SIZE] = MCL_BLOB_INIT;
__device__ unsigned d_leaf[256];               // unambiguous cube index -> leaf, else MC_AMBIG
__device__ unsigned short d_cross[256];        // cube index -> 12-bit mask of sign-changing edges
__device__ McRowMeta d_meta[MCR_NROWS];
// cube index -> leaf [0:15) | ambiguous [15] | vertices an INTERIOR cell creates (edges 5, 6, 10) [16:19)
__device__ unsigned d_quick[256];
#define MC_QUICK_AMBIG 0x8000u

// edge -> corner pair (Luts.cs:26-28 in corner numbering; MarchingCubes.cs:70-71)
__host__ __device__ static inline void mc_edge_corners(int e, int& a, int& b)
{
    const int A[12] = {0, 1, 2, 3, 4, 5, 6, 7, 0, 1, 2, 3};
    const int B[12] = {1, 2, 3, 0, 5, 6, 7, 4, 4, 5, 6, 7};
    a = A[e];
    b = B[e];
}

cudaError_t mc_init_tables()
{
    static unsigned leaf[256];
    static unsigned short cross[256];
    static McRowMeta meta[MCR_NROWS];
    static unsigned quick[256];
    const struct { int off, rows, len; } tables[] = MCR_TABLES;
    int rid = 0;
    for (auto& t : tables) {
        for (int r = 0; r < t.rows; r++, rid++) {
            McRowMeta& m = meta[rid];
            memset(&m, 0, sizeof(m));
            m.off = (unsigned short)(t.off + r * t.len);
            m.nt = (unsigned char)(t.len / 3);
            unsigned seen = 0;
            for (int k = 0; k < t.len; k++) {
                const int e = h_lut[m.off + k];
                if (e < 0 || e > 12) return cudaErrorInvalidValue;
                if (!((seen >> e) & 1u)) m.before[e] = (unsigned short)seen;
                seen |= 1u << e;
                m.occ[e]++;
            }
            m.refmask = (unsigned short)seen;
            for (int e = 0; e < 12; e++) {
                if (m.occ[e] > 7) return cudaErrorInvalidValue;
                m.occ_packed |= (unsigned long long)m.occ[e] << (16 + 3 * e);
            }
        }
    }
    if (rid != MCR_NROWS) return cudaErrorInvalidValue;
    // unambiguous Lewiner cases: first row id of the tiling table, triangle count (MarchingCubes.cs:98-372)
    const struct { int cas, row0, nt; } simple[] = {
        {1, MCR_tiling1, 1}, {2, MCR_tiling2, 2}, {5, MCR_tiling5, 3}, {8, MCR_tiling8, 2},
        {9, MCR_tiling9, 4}, {11, MCR_tiling11, 4}, {14, MCR_tiling14, 4}};
    for (int idx = 0; idx < 256; idx++) {
        int cas = h_lut[MCL_cases + idx * 2], cfg = h_lut[MCL_cases + idx * 2 + 1];
        leaf[idx] = (cas == 0) ? 0u : MC_AMBIG;
        for (auto& s : simple)
            if (s.cas == cas) leaf[idx] = MC_LEAF(s.row0 + cfg, s.nt, 0);
        unsigned m = 0;
        for (int e = 0; e < 12; e++) {
            int a, b;
            mc_edge_corners(e, a, b);
            if (((idx >> a) ^ (idx >> b)) & 1) m |= 1u << e;
        }
        cross[idx] = (unsigned short)m;
        quick[idx] = ((leaf[idx] & MC_AMBIG) ? MC_QUICK_AMBIG : (leaf[idx] & 0x7FFFu)) | ((unsigned)__builtin_popcount(m & 0x460u) << 16);
    }
    cudaError_t err = cudaMemcpyToSymbol(d_leaf, leaf, sizeof(leaf));
    if (err == cudaSuccess) err = cudaMemcpyToSymbol(d_cross, cross, sizeof(cross));
    if (err == cudaSuccess) err = cudaMemcpyToSymbol(d_meta, meta, sizeof(meta));
    if (err == cudaSuccess) err = cudaMemcpyToSymbol(d_quick, quick, sizeof(quick));
    return err;
}

// ---------------------------------------------------------------------------------------------------
// Lewiner disambiguation (FP64, no contraction)
// ---------------------------------------------------------------------------------------------------

// MarchingCubes.TestFace (MarchingCubes.cs:376-407)
__device__ static bool mc_test_face(const double* v, int face)
{
    const int af = face < 0 ? -face : face;
    double A = 0.0, B = 0.0, C = 0.0, D = 0.0;
    switch (af) {
    case 1: A = v[0]; B = v[4]; C = v[5]; D = v[1]; break;
    case 2: A = v[1]; B = v[5]; C = v[6]; D = v[2]; break;
    case 3: A = v[2]; B = v[6]; C = v[7]; D = v[3]; break;
    case 4: A = v[3]; B = v[7]; C = v[4]; D = v[0]; break;
    case 5: A = v[0]; B = v[3]; C = v[2]; D = v[1]; break;
    case 6: A = v[4]; B = v[7]; C = v[6]; D = v[5]; break;
    }
    const double acbd = A * C - B * D;
    if (acbd > -MC_EPS && acbd < MC_EPS) return face >= 0;
    return (double)face * A * acbd >= 0;
}

// MarchingCubes.TestInternal (MarchingCubes.cs:412-546)
__device__ static bool mc_test_internal(const double* v, int cas, int cfg, int sub, int s)
{
    double t, At = 0.0, Bt = 0.0, Ct = 0.0, Dt = 0.0;
    if (cas == 4 || cas == 10) {
        const double a = (v[4] - v[0]) * (v[6] - v[2]) - (v[7] - v[3]) * (v[5] - v[1]);
        const double b = v[2] * (v[4] - v[0]) + v[0] * (v[6] - v[2]) - v[1] * (v[7] - v[3]) - v[3] * (v[5] - v[1]);
        t = -b / (2 * a + MC_EPS);
        if (t < 0 || t > 1) return s > 0;
        At = v[0] + (v[4] - v[0]) * t;
        Bt = v[3] + (v[7] - v[3]) * t;
        Ct = v[2] + (v[6] - v[2]) * t;
        Dt = v[1] + (v[5] - v[1]) * t;
    } else {
        int edge;
        if (cas == 6) edge = d_lut[MCL_test6 + cfg * 3 + 2];
        else if (cas == 7) edge = d_lut[MCL_test7 + cfg * 5 + 4];
        else if (cas == 12) edge = d_lut[MCL_test12 + cfg * 4 + 3];
        else edge = d_lut[MCL_tiling13_5_1 + (cfg * 4 + sub) * 18];
        if (edge >= 0 && edge < 12) {
            // reference edge e runs a->b; the three opposite edges, interpolated at the same parameter,
            // are given as (from,to) corner pairs for Bt, Ct, Dt (MarchingCubes.cs:440-511), 3 bits each
            const unsigned tab[12] = {
                // a | b<<3 | B0<<6 | B1<<9 | C0<<12 | C1<<15 | D0<<18 | D1<<21
                0u | 1u << 3 | 3u << 6 | 2u << 9 | 7u << 12 | 6u << 15 | 4u << 18 | 5u << 21,
                1u | 2u << 3 | 0u << 6 | 3u << 9 | 4u << 12 | 7u << 15 | 5u << 18 | 6u << 21,
                2u | 3u << 3 | 1u << 6 | 0u << 9 | 5u << 12 | 4u << 15 | 6u << 18 | 7u << 21,
                3u | 0u << 3 | 2u << 6 | 1u << 9 | 6u << 12 | 5u << 15 | 7u << 18 | 4u << 21,
                4u | 5u << 3 | 7u << 6 | 6u << 9 | 3u << 12 | 2u << 15 | 0u << 18 | 1u << 21,
                5u | 6u << 3 | 4u << 6 | 7u << 9 | 0u << 12 | 3u << 15 | 1u << 18 | 2u << 21,
                6u | 7u << 3 | 5u << 6 | 4u << 9 | 1u << 12 | 0u << 15 | 2u << 18 | 3u << 21,
                7u | 4u << 3 | 6u << 6 | 5u << 9 | 2u << 12 | 1u << 15 | 3u << 18 | 0u << 21,
                0u | 4u << 3 | 3u << 6 | 7u << 9 | 2u << 12 | 6u << 15 | 1u << 18 | 5u << 21,
                1u | 5u << 3 | 0u << 6 | 4u << 9 | 3u << 12 | 7u << 15 | 2u << 18 | 6u << 21,
                2u | 6u << 3 | 1u << 6 | 5u << 9 | 0u << 12 | 4u << 15 | 3u << 18 | 7u << 21,
                3u | 7u << 3 | 2u << 6 | 6u << 9 | 1u << 12 | 5u << 15 | 0u << 18 | 4u << 21};
            const unsigned r = tab[edge];
#define TC(n) v[(r >> (3 * (n))) & 7u]
            t = TC(0) / (TC(0) - TC(1) + MC_EPS);
            At = 0;
            Bt = TC(2) + (TC(3) - TC(2)) * t;
            Ct = TC(4) + (TC(5) - TC(4)) * t;
            Dt = TC(6) + (TC(7) - TC(6)) * t;
#undef TC
        }
    }
    int test = 0;
    if (At >= 0) test += 1;
    if (Bt >= 0) test += 2;
    if (Ct >= 0) test += 4;
    if (Dt >= 0) test += 8;
    switch (test) {
    case 5: if (At * Ct - Bt * Dt < MC_EPS) return s > 0; break;
    case 10: if (At * Ct - Bt * Dt >= MC_EPS) return s > 0; break;
    case 7: case 11: case 13: case 14: case 15: return s < 0;
    default: return s > 0;
    }
    return s < 0;
}

#define LEAF2(name, cfg, nt, center) MC_LEAF(MCR_##name + (cfg), nt, center)
#define LEAF3(name, cfg, sub, nt, center) MC_LEAF(MCR_##name + (cfg) * MCL_##name##_D1 + (sub), nt, center)

// MarchingCubes.TheBigSwitch for the ambiguous cases (MarchingCubes.cs:105-366): chooses the tiling row.
// v[k] = (double)value_k - (double)iso in the reference's corner numbering.
__device__ __noinline__ static unsigned mc_resolve(int idx, const double* v)
{
    const int cas = d_lut[MCL_cases + idx * 2];
    const int cfg = d_lut[MCL_cases + idx * 2 + 1];
    int sub = 0;
    switch (cas) {
    case 3:
        return mc_test_face(v, d_lut[MCL_test3 + cfg]) ? LEAF2(tiling3_2, cfg, 4, 0) : LEAF2(tiling3_1, cfg, 2, 0);
    case 4:
        return mc_test_internal(v, cas, cfg, 0, d_lut[MCL_test4 + cfg]) ? LEAF2(tiling4_1, cfg, 2, 0) : LEAF2(tiling4_2, cfg, 6, 0);
    case 6:
        if (mc_test_face(v, d_lut[MCL_test6 + cfg * 3])) return LEAF2(tiling6_2, cfg, 5, 0);
        return mc_test_internal(v, cas, cfg, 0, d_lut[MCL_test6 + cfg * 3 + 1]) ? LEAF2(tiling6_1_1, cfg, 3, 0) : LEAF2(tiling6_1_2, cfg, 9, 1);
    case 7:
        if (mc_test_face(v, d_lut[MCL_test7 + cfg * 5 + 0])) sub += 1;
        if (mc_test_face(v, d_lut[MCL_test7 + cfg * 5 + 1])) sub += 2;
        if (mc_test_face(v, d_lut[MCL_test7 + cfg * 5 + 2])) sub += 4;
        switch (sub) {
        case 0: return LEAF2(tiling7_1, cfg, 3, 0);
        case 1: return LEAF3(tiling7_2, cfg, 0, 5, 0);
        case 2: return LEAF3(tiling7_2, cfg, 1, 5, 0);
        case 3: return LEAF3(tiling7_3, cfg, 0, 9, 1);
        case 4: return LEAF3(tiling7_2, cfg, 2, 5, 0);
        case 5: return LEAF3(tiling7_3, cfg, 1, 9, 1);
        case 6: return LEAF3(tiling7_3, cfg, 2, 9, 1);
        default:
            return mc_test_internal(v, cas, cfg, sub, d_lut[MCL_test7 + cfg * 5 + 3]) ? LEAF2(tiling7_4_2, cfg, 9, 0) : LEAF2(tiling7_4_1, cfg, 5, 0);
        }
    case 10:
    case 12: {
        const int tst = (cas == 10) ? MCL_test10 + cfg * 3 : MCL_test12 + cfg * 4;
        const bool f0 = mc_test_face(v, d_lut[tst]);
        const bool f1 = mc_test_face(v, d_lut[tst + 1]);
        if (cas == 10) {
            if (f0) return f1 ? LEAF2(tiling10_1_1_, cfg, 4, 0) : LEAF2(tiling10_2, cfg, 8, 1);
            if (f1) return LEAF2(tiling10_2_, cfg, 8, 1);
            return mc_test_internal(v, cas, cfg, 0, d_lut[tst + 2]) ? LEAF2(tiling10_1_1, cfg, 4, 0) : LEAF2(tiling10_1_2, cfg, 8, 0);
        }
        if (f0) return f1 ? LEAF2(tiling12_1_1_, cfg, 4, 0) : LEAF2(tiling12_2, cfg, 8, 1);
        if (f1) return LEAF2(tiling12_2_, cfg, 8, 1);
        return mc_test_internal(v, cas, cfg, 0, d_lut[tst + 2]) ? LEAF2(tiling12_1_1, cfg, 4, 0) : LEAF2(tiling12_1_2, cfg, 8, 0);
    }
    case 13: {
        for (int k = 0; k < 6; k++)
            if (mc_test_face(v, d_lut[MCL_test13 + cfg * 7 + k])) sub += 1 << k;
        sub = d_lut[MCL_subconfig13 + sub];
        if (sub < 0) return MC_LEAF(0, 0, 0);   // "Impossible case 13?" (MarchingCubes.cs:364-366): no triangles
        if (sub == 0) return LEAF2(tiling13_1, cfg, 4, 0);
        if (sub <= 6) return LEAF3(tiling13_2, cfg, sub - 1, 6, 0);
        if (sub <= 18) return LEAF3(tiling13_3, cfg, sub - 7, 10, 1);
        if (sub <= 22) return LEAF3(tiling13_4, cfg, sub - 19, 12, 1);
        if (sub <= 26) {
            const int s5 = sub - 23;
            return mc_test_internal(v, cas, cfg, s5, d_lut[MCL_test13 + cfg * 7 + 6]) ? LEAF3(tiling13_5_1, cfg, s5, 6, 0)
                                                                                      : LEAF3(tiling13_5_2, cfg, s5, 10, 0);
        }
        if (sub <= 38) return LEAF3(tiling13_3_, cfg, sub - 27, 10, 1);
        if (sub <= 44) return LEAF3(tiling13_2_, cfg, sub - 39, 6, 0);
        if (sub == 45) return LEAF2(tiling13_1_, cfg, 4, 0);
        return MC_LEAF(0, 0, 0);   // "Impossible case 13?" (MarchingCubes.cs:365): no triangles
    }
    }
    return MC_LEAF(0, 0, 0);
}

// ---------------------------------------------------------------------------------------------------
// geometry helpers
// ---------------------------------------------------------------------------------------------------

// Which of a cell's 13 vertex slots it creates itself (first touch in visiting order); kg = GLOBAL layer.
__device__ static inline unsigned mc_owned_mask(int i, int j, int kg)
{
    unsigned m = (1u << 5) | (1u << 6) | (1u << 10) | (1u << 12);
    if (j == 0) m |= (1u << 4) | (1u << 9);
    if (i == 0) m |= (1u << 7) | (1u << 11);
    if (i == 0 && j == 0) m |= 1u << 8;
    if (kg == 0) {
        m |= (1u << 1) | (1u << 2);
        if (j == 0) m |= 1u << 0;
        if (i == 0) m |= 1u << 3;
    }
    return m;
}

__device__ static inline size_t mc_vox(const McGrid& g, int i, int j, int kg, int dx, int dy, int dz)
{
    const int x = (i + dx) * g.step, y = (j + dy) * g.step, zl = (kg + dz) * g.step - g.z0;
    return ((size_t)zl * g.ny + y) * (size_t)g.nx + x;
}

// values of the 8 cube corners minus iso, as doubles, reference corner numbering (Cell.cs:206-213): one base address,
// then constant strides (x: step, y: step*nx, z: step*nx*ny)
__device__ static inline void mc_load_cell(const McGrid& g, const float* __restrict__ dist, int i, int j, int kg, double* v)
{
    const double iso = (double)g.iso;
    const size_t sx = (size_t)g.step, sy = (size_t)g.step * (size_t)g.nx, sz = (size_t)g.step * (size_t)g.nx * (size_t)g.ny;
    const float* p = dist + mc_vox(g, i, j, kg, 0, 0, 0);
    const float f0 = __ldg(p), f1 = __ldg(p + sx), f2 = __ldg(p + sx + sy), f3 = __ldg(p + sy);
    const float f4 = __ldg(p + sz), f5 = __ldg(p + sz + sx), f6 = __ldg(p + sz + sx + sy), f7 = __ldg(p + sz + sy);
    v[0] = (double)f0 - iso; v[1] = (double)f1 - iso; v[2] = (double)f2 - iso; v[3] = (double)f3 - iso;
    v[4] = (double)f4 - iso; v[5] = (double)f5 - iso; v[6] = (double)f6 - iso; v[7] = (double)f7 - iso;
}


// leaf + created-vertex count of an active cell
__device__ __noinline__ static unsigned mc_resolve_cell(const McGrid& g, const float* __restrict__ dist, int idx, int i, int j, int kg)
{
    double v[8];
    mc_load_cell(g, dist, i, j, kg, v);
    return mc_resolve(idx, v);
}

__device__ static inline unsigned mc_cell_leaf(const McGrid& g, const float* __restrict__ dist, int idx, int i, int j, int kg)
{
    unsigned leaf = d_leaf[idx];
    if (leaf & MC_AMBIG) leaf = mc_resolve_cell(g, dist, idx, i, j, kg);
    return leaf;
}

// leaf + packed counts of an active cell: interior unambiguous cells (nearly all) need one 256-entry table lookup,
// cells on the i/j/k = 0 faces or with an ambiguous cube index take the out-of-line path
__device__ __noinline__ static unsigned mc_cell_info_slow(const McGrid& g, const float* __restrict__ dist, int idx, int i, int j, int kg, unsigned* leaf_out);

// quick = s_quick[idx] (the 256-entry table staged in shared memory: streaming loads evict it from L1 otherwise)
__device__ static inline unsigned mc_cell_info(const McGrid& g, const float* __restrict__ dist, unsigned quick, int idx, int i, int j, int kg,
                                               unsigned* leaf_out)
{
    if (!(quick & MC_QUICK_AMBIG) && i > 0 && j > 0 && kg > 0) {
        *leaf_out = quick & 0x7FFFu;
        return MC_LEAF_NT(quick) ? MC_CNT_PACK(1, (quick >> 16) & 7u, MC_LEAF_NT(quick)) : 0u;   // nt == 0 only for idx 0 / 255
    }
    if (idx == 0 || idx == 255) { *leaf_out = 0; return 0u; }
    return mc_cell_info_slow(g, dist, idx, i, j, kg, leaf_out);
}

// packed (active, created vertices, triangles) of an active cell; a cell whose leaf has no triangles (the
// reference's "impossible" case 13) is recorded but emits nothing
__device__ static inline unsigned mc_cell_counts(unsigned leaf, int idx, int i, int j, int kg)
{
    if (MC_LEAF_NT(leaf) == 0u) return MC_CNT_PACK(1, 0, 0);
    const unsigned nv = __popc((unsigned)d_cross[idx] & mc_owned_mask(i, j, kg)) + MC_LEAF_CENTER(leaf);
    return MC_CNT_PACK(1, nv, MC_LEAF_NT(leaf));
}

__device__ __noinline__ static unsigned mc_cell_info_slow(const McGrid& g, const float* __restrict__ dist, int idx, int i, int j, int kg, unsigned* leaf_out)
{
    const unsigned leaf = mc_cell_leaf(g, dist, idx, i, j, kg);
    *leaf_out = leaf;
    return mc_cell_counts(leaf, idx, i, j, kg);
}

// ---------------------------------------------------------------------------------------------------
// sign rows: 5 sign bits for voxels (i0..i0+4)*step of one voxel row: bit t = value > iso (strict, Cell.cs:221-228;
// the float compare is exact for (double)value - (double)iso > 0).  Loads are issued branch-free (addresses
// clamped into the row) so that a whole batch of rows is in flight before the first compare.
// ---------------------------------------------------------------------------------------------------
struct McRowLoad {
    float4 q;      // VEC: voxels i0..i0+3 ; generic: t = 0..3
    float e;       // VEC: voxel i0+4 for lane 31 (own voxel i0+3 for the other lanes: same sector) ; generic: t = 4
};

template <bool VEC>
__device__ static inline McRowLoad mc_row_load(const float* __restrict__ row, int nx, int step, int i0, unsigned lane)
{
    McRowLoad r;
    if (VEC) {   // step == 1, nx % 4 == 0: one 16-byte load per lane (+ the right neighbour for lane 31)
        const int ic = min(i0, nx - 4);
        r.q = __ldg(reinterpret_cast<const float4*>(row + ic));
        r.e = __ldg(row + ic + ((lane == 31u && i0 + 4 < nx) ? 4 : 3));
    } else {
        const long long last = nx - 1;
        r.q.x = __ldg(row + min((long long)(i0 + 0) * step, last));
        r.q.y = __ldg(row + min((long long)(i0 + 1) * step, last));
        r.q.z = __ldg(row + min((long long)(i0 + 2) * step, last));
        r.q.w = __ldg(row + min((long long)(i0 + 3) * step, last));
        r.e = __ldg(row + min((long long)(i0 + 4) * step, last));
    }
    return r;
}

template <bool VEC>
__device__ static inline unsigned mc_row_bits(const McRowLoad& r, float iso, int nx, int step, int i0, unsigned lane)
{
    unsigned s = (r.q.x > iso ? 1u : 0u) | (r.q.y > iso ? 2u : 0u) | (r.q.z > iso ? 4u : 0u) | (r.q.w > iso ? 8u : 0u);
    if (VEC) {
        if (i0 >= nx) s = 0u;
        unsigned nb = __shfl_down_sync(FULL, s, 1) & 1u;
        if (lane == 31u) nb = (i0 + 4 < nx && r.e > iso) ? 1u : 0u;
        s |= nb << 4;
    } else {
        s |= (r.e > iso ? 16u : 0u);
        unsigned valid = 0;
#pragma unroll
        for (int t = 0; t < 5; t++)
            if ((long long)(i0 + t) * step < nx) valid |= 1u << t;
        s &= valid;
    }
    return s;
}


// ---------------------------------------------------------------------------------------------------
// K2 mc_classify: one warp marches a 128-cell x-chunk by MC_R rows through MC_K layers; every voxel's
// sign is computed once per march (x/y/z halos aside).  Output: the number of ACTIVE CELLS of every chunk -- pure
// streaming + bit tricks; everything that needs a cube index (leaf, vertex / triangle counts) is left to K4a, which
// only visits the active chunks, and a second run of the scan.
// ---------------------------------------------------------------------------------------------------
#define MC_K 16
#define MC_CLASSIFY_WARPS 8

template <bool VEC, int MC_R>
__device__ static inline void mc_plane_signs(const float* __restrict__ plane, size_t row_stride, int nrows, int nx, int step,
                                             float iso, int i0, unsigned lane, unsigned* out)
{
    McRowLoad ld[MC_R + 1];
#pragma unroll
    for (int r = 0; r <= MC_R; r++) ld[r] = mc_row_load<VEC>(plane + (size_t)min(r, nrows) * row_stride, nx, step, i0, lane);
#pragma unroll
    for (int r = 0; r <= MC_R; r++) out[r] = mc_row_bits<VEC>(ld[r], iso, nx, step, i0, lane);
}

// 0xFFFFFFFF if a > b (ordered: false for NaN) else 0 -- one FSET, no predicate/select pair
__device__ static inline unsigned mc_gt_mask(float a, float b)
{
    unsigned m;
    asm("set.gt.u32.f32 %0, %1, %2;" : "=r"(m) : "f"(a), "f"(b));
    return m;
}

// Vector path (step 1, nx % 4 == 0) of one plane: the voxel arrays are padded, so every lane loads unconditionally
// (MC_R + 1) x (LDG.128 + the right-neighbour LDG.32) back to back, then turns them into 5-bit sign words.
// lp = this lane's pointer to voxel (i0, row 0) of the plane; vm = 0xF for lanes inside the row, else 0.
template <int MC_R>
__device__ static inline void mc_plane_signs_vec(const float* __restrict__ lp, unsigned row_stride, int eoff, bool e_ok, unsigned vm,
                                                 float iso, unsigned lane, unsigned* out)
{
    float4 q[MC_R + 1];
    float e[MC_R + 1];
#pragma unroll
    for (int r = 0; r <= MC_R; r++) {
        const float* rp = lp + (size_t)r * row_stride;
        q[r] = __ldg(reinterpret_cast<const float4*>(rp));
        e[r] = __ldg(rp + eoff);
    }
#pragma unroll
    for (int r = 0; r <= MC_R; r++) {
        const unsigned m0 = mc_gt_mask(q[r].x, iso), m1 = mc_gt_mask(q[r].y, iso), m2 = mc_gt_mask(q[r].z, iso), m3 = mc_gt_mask(q[r].w, iso);
        unsigned s = (m0 & 1u) | (m1 & ~1u);
        s = (s & 3u) | (m2 & ~3u);
        s = (s & 7u) | (m3 & ~7u);
        s &= vm;
        unsigned nb = __shfl_down_sync(FULL, s, 1);
        if (lane == 31u) nb = (e_ok && e[r] > iso) ? 1u : 0u;
        out[r] = s | ((nb & 1u) << 4);
    }
}

template <bool VEC, int MC_R, int MINB>
__global__ void __launch_bounds__(MC_CLASSIFY_WARPS * 32, MINB)
mc_classify_kernel(const McGrid g, const float* __restrict__ dist, unsigned* __restrict__ counts, uint4* __restrict__ masks,
                   unsigned njb, unsigned nkb, unsigned ntiles)
{
    const unsigned lane = threadIdx.x & 31u;
    const unsigned gw = blockIdx.x * MC_CLASSIFY_WARPS + (threadIdx.x >> 5);
    const unsigned nw = gridDim.x * MC_CLASSIFY_WARPS;
    const int nx = g.nx, step = g.step, ncy = g.ncy, cpr = g.cpr;
    const float iso = g.iso;
    const size_t row_stride = (size_t)step * (size_t)nx;                // floats between voxel rows y and y+step
    const size_t plane_stride = (size_t)g.ny * (size_t)nx;              // floats per z slice
    for (unsigned tile = gw; tile < ntiles; tile += nw) {
        // tile -> (xc fastest, then row block, then layer block): neighbouring warps read neighbouring segments
        const unsigned xc = tile % (unsigned)cpr;
        const unsigned t2 = tile / (unsigned)cpr;
        const unsigned jb = t2 % njb;
        const unsigned kb = t2 / njb;
        const int i0 = (int)(xc * 128u + lane * 4u);
        const int j0 = (int)(jb * MC_R);
        const int kl0 = (int)(kb * MC_K);                               // local layer index
        const int nrows = min(MC_R, ncy - j0);
        const int nlay = min(MC_K, g.nk - kl0);
        const float* plane = dist + (size_t)((g.k0 + kl0) * step - g.z0) * plane_stride + (size_t)j0 * row_stride;
        unsigned* cnt_out = counts + ((size_t)kl0 * ncy + j0) * cpr + xc;
        uint4* mask_out = masks + ((size_t)kl0 * ncy + j0) * cpr + xc;
        // vector path constants
        const int eoff = (lane == 31u) ? 4 : 3;
        const bool e_ok = i0 + 4 < nx;
        const unsigned vm = (i0 < nx) ? 0xFu : 0u;
        // cells of this lane that exist (i0 + c < ncx), replicated into the 5-bit row fields 0..MC_R-1
        const unsigned c4 = (i0 + 3 < g.ncx) ? 15u : (i0 < g.ncx ? ((1u << (g.ncx - i0)) - 1u) : 0u);
        const unsigned long long cellmask = (unsigned long long)c4 * (0x10842108421ull & ((1ull << (5 * nrows)) - 1ull));

        unsigned prev[MC_R + 1], cur[MC_R + 1];
        if (VEC) mc_plane_signs_vec<MC_R>(plane + i0, (unsigned)nx, eoff, e_ok, vm, iso, lane, prev);
        else mc_plane_signs<false, MC_R>(plane, row_stride, nrows, nx, step, iso, i0, lane, prev);
        unsigned por = 0u, pand = 31u;                                  // OR / AND over the lane's sign words of the lower plane
#pragma unroll
        for (int r = 0; r <= MC_R; r++) { por |= prev[r]; pand &= prev[r]; }
#pragma unroll 1
        for (int kk = 0; kk < nlay; kk++) {
            plane += (size_t)step * plane_stride;
            if (VEC) mc_plane_signs_vec<MC_R>(plane + i0, (unsigned)nx, eoff, e_ok, vm, iso, lane, cur);
            else mc_plane_signs<false, MC_R>(plane, row_stride, nrows, nx, step, iso, i0, lane, cur);
            unsigned cor = 0u, cand = 31u;
#pragma unroll
            for (int r = 0; r <= MC_R; r++) { cor |= cur[r]; cand &= cur[r]; }
            // no lane of the warp sees a sign change in its 4 x 8 cells of this layer (the common case): 8 zero counts
            const bool quiet = ((por | cor) == 0u) || ((pand & cand) == 31u);
            if (__all_sync(FULL, quiet)) {
                if ((int)lane < nrows) cnt_out[(size_t)lane * cpr] = 0u;
            } else {
                // count the ACTIVE CELLS of every row, all rows at once on packed words (field r = 5 bits of row r):
                // cell c of row r is active unless its 8 corner signs are all 0 or all 1
                unsigned long long prevp = 0ull, curp = 0ull;
#pragma unroll
                for (int r = 0; r <= MC_R; r++) { prevp |= (unsigned long long)prev[r] << (5 * r); curp |= (unsigned long long)cur[r] << (5 * r); }
                unsigned long long anyp = prevp | curp, allp = prevp & curp;
                anyp |= anyp >> 5;                                       // rows r, r+1 x both planes
                allp &= allp >> 5;
                anyp |= anyp >> 1;                                       // voxels c, c+1
                allp &= allp >> 1;
                const unsigned long long actp = anyp & ~allp & cellmask;
                // per row: the count, and the chunk's 128-bit activity mask in natural cell order (bit 4*lane + c):
                // word w = OR of the nibbles of lanes 8w .. 8w+7 (xor-shuffle tree inside each group of 8 lanes)
                unsigned mine = 0;
                const unsigned sh = 4u * (lane & 7u);
                unsigned* mw = reinterpret_cast<unsigned*>(mask_out) + (lane >> 3);
#pragma unroll
                for (int r = 0; r < MC_R; r++) {
                    const unsigned nib = (unsigned)(actp >> (5 * r)) & 15u;
                    const unsigned t = __reduce_add_sync(FULL, __popc(nib));
                    if (lane == (unsigned)r) mine = t;
                    unsigned w = nib << sh;
                    w |= __shfl_xor_sync(FULL, w, 1);
                    w |= __shfl_xor_sync(FULL, w, 2);
                    w |= __shfl_xor_sync(FULL, w, 4);
                    if ((lane & 7u) == 0u && r < nrows) mw[(size_t)r * cpr * 4] = w;
                }
                if ((int)lane < nrows) cnt_out[(size_t)lane * cpr] = MC_CNT_FIRST(mine);
            }
            cnt_out += (size_t)ncy * cpr;
            mask_out += (size_t)ncy * cpr;
#pragma unroll
            for (int r = 0; r <= MC_R; r++) prev[r] = cur[r];
            por = cor;
            pand = cand;
        }
    }
}

template <bool VEC, int R, int MINB>
static cudaError_t mc_launch_classify_t(const McGrid& g, const float* dist, unsigned* counts, uint4* masks, cudaStream_t s)
{
    const unsigned njb = (g.ncy + R - 1) / R, nkb = (g.nk + MC_K - 1) / MC_K;
    const unsigned long long nt = (unsigned long long)g.cpr * njb * nkb;
    if (nt > 0xFFFFFFFFull) return cudaErrorInvalidValue;
    const unsigned ntiles = (unsigned)nt;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    unsigned blocks = (ntiles + MC_CLASSIFY_WARPS - 1) / MC_CLASSIFY_WARPS;
    const unsigned maxb = (unsigned)sms * 8u;
    if (blocks > maxb) blocks = maxb;
    mc_classify_kernel<VEC, R, MINB><<<blocks, MC_CLASSIFY_WARPS * 32, 0, s>>>(g, dist, counts, masks, njb, nkb, ntiles);
    return cudaGetLastError();
}

cudaError_t mc_launch_classify(const McGrid& g, const float* dist, unsigned* counts, uint4* masks, cudaStream_t s)
{
    if (g.nchunks == 0) return cudaSuccess;
    const bool vec = g.step == 1 && (g.nx & 3) == 0 && g.nx >= 4;
    if (!vec) return mc_launch_classify_t<false, 8, 1>(g, dist, counts, masks, s);
    return mc_launch_classify_t<true, 8, 2>(g, dist, counts, masks, s);
}

// ---------------------------------------------------------------------------------------------------
// K2' mc_classify_signs: the outputs of mc_classify (active cells + 128-bit activity mask per chunk) from the SIGN
// BLOCKS the sampling kernels write as a by-product (csrc/jit_kernels.cuh) -- 1 bit per voxel instead of the 4-byte
// distance, so the distance field is never re-read to find the surface.  step == 1 only (voxel tiles == cell chunks).
// Layout: uint4 signs[((y*tpr + xc)*nzg + zg)*32 + L]; word zb%4 of group zg = zb/4, bit 4p + k <-> voxel
// (xc*128 + 4L + k, y, 8*zb + p) has value > iso.
// A warp takes one (row j, chunk xc) column and MC_SZB z-blocks (all loads issued up front): per block two coalesced 128-byte loads
// (rows j, j+1) give every lane the signs of its 4 x 2 x 8 voxels; the x neighbour comes from lane L+1 (lane 31: the
// next tile), the z neighbour from the next bit plane (plane 7: the next block).
// ---------------------------------------------------------------------------------------------------
#define MC_SZB 8

__global__ void __launch_bounds__(256)
mc_classify_signs_kernel(const McGrid g, const uint4* __restrict__ signs, unsigned tpr, unsigned nzg, unsigned* __restrict__ counts,
                         uint4* __restrict__ masks, unsigned ncols, unsigned nwork, int zg_first, int zb_last)
{
    const unsigned lane = threadIdx.x & 31u;
    const unsigned gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const int off = g.k0 - g.z0;                                          // plane zl = local layer kl + off  (step == 1)
    const size_t colwords = (size_t)nzg * 32u;                            // uint4s per (row, tile) column
    const unsigned sh = 4u * (lane & 7u);
    for (unsigned w = gw; w < nwork; w += nw) {
        const unsigned seg = w / ncols, col = w - seg * ncols;
        const unsigned j = col / (unsigned)g.cpr, xc = col - j * (unsigned)g.cpr;
        const int zg0 = zg_first + (int)(seg * (MC_SZB / 4)), zb0 = zg0 * 4;
        const uint4* rowA = signs + ((size_t)j * tpr + xc) * colwords + (size_t)zg0 * 32u + lane;
        const uint4* rowB = rowA + (size_t)tpr * colwords;
        const bool edge = lane == 31u && xc + 1u < tpr;                   // lane 31's x neighbour: lane 0's word of the next tile
        // cells of this lane that exist (i = xc*128 + 4L + k < ncx), replicated over the 8 planes
        const int left = g.ncx - (int)(xc * 128u + lane * 4u);
        const unsigned cellmask = (left >= 4 ? 15u : (left <= 0 ? 0u : ((1u << left) - 1u))) * 0x11111111u;
        // all loads of the item first: two groups of 4 blocks per row as uint4, + the first block of the next group (only its
        // first plane is needed); lane 31 also fetches lane 0's words of the next tile
        unsigned a[MC_SZB + 1], b[MC_SZB + 1], an[MC_SZB + 1], bn[MC_SZB + 1];
        {
            const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
            const bool in0 = zg0 < (int)nzg, in1 = zg0 + 1 < (int)nzg, in2 = zg0 + 2 < (int)nzg;
            const uint4 a0 = in0 ? __ldg(rowA) : z4, a1 = in1 ? __ldg(rowA + 32) : z4;
            const uint4 b0 = in0 ? __ldg(rowB) : z4, b1 = in1 ? __ldg(rowB + 32) : z4;
            a[8] = in2 ? __ldg(reinterpret_cast<const unsigned*>(rowA + 64)) : 0u;
            b[8] = in2 ? __ldg(reinterpret_cast<const unsigned*>(rowB + 64)) : 0u;
            const uint4* nA = rowA + colwords - 31;
            const uint4* nB = rowB + colwords - 31;
            const uint4 c0 = (in0 && edge) ? __ldg(nA) : z4, c1 = (in1 && edge) ? __ldg(nA + 32) : z4;
            const uint4 d0 = (in0 && edge) ? __ldg(nB) : z4, d1 = (in1 && edge) ? __ldg(nB + 32) : z4;
            an[8] = (in2 && edge) ? __ldg(reinterpret_cast<const unsigned*>(nA + 64)) : 0u;
            bn[8] = (in2 && edge) ? __ldg(reinterpret_cast<const unsigned*>(nB + 64)) : 0u;
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
            b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w; b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
            an[0] = c0.x; an[1] = c0.y; an[2] = c0.z; an[3] = c0.w; an[4] = c1.x; an[5] = c1.y; an[6] = c1.z; an[7] = c1.w;
            bn[0] = d0.x; bn[1] = d0.y; bn[2] = d0.z; bn[3] = d0.w; bn[4] = d1.x; bn[5] = d1.y; bn[6] = d1.z; bn[7] = d1.w;
        }
        // An item whose words are all 0 or all 1 in every lane -- both rows, the next tile's first lane, the first plane of the
        // next group -- has no sign change: nothing to count (`counts` is zeroed before the launch).  Most items of a scene are
        // like that (0.4 % of the README scene's cells are active), and this test replaces ~250 instructions by ~30.
        {
            unsigned o = 0u, n = 0xFFFFFFFFu;
#pragma unroll
            for (int q = 0; q < MC_SZB; q++) { o |= a[q] | b[q]; n &= a[q] & b[q]; }
            const unsigned t8 = a[MC_SZB] | b[MC_SZB], u8 = a[MC_SZB] & b[MC_SZB];      // next group: only its first plane (low nibble bits)
            o |= t8 & 0x0000000Fu; n &= u8 | 0xFFFFFFF0u;
            if (edge) {
#pragma unroll
                for (int q = 0; q < MC_SZB; q++) { o |= (an[q] | bn[q]) & 0x11111111u; n &= (an[q] & bn[q]) | 0xEEEEEEEEu; }   // voxel k = 0 of the next tile
                o |= (an[MC_SZB] | bn[MC_SZB]) & 1u; n &= (an[MC_SZB] & bn[MC_SZB]) | 0xFFFFFFFEu;
            }
            if (__all_sync(FULL, o == 0u) || __all_sync(FULL, n == 0xFFFFFFFFu)) continue;
        }
        unsigned any[MC_SZB + 1], all[MC_SZB + 1];                        // OR / AND over rows j, j+1 and voxels c, c+1; bit 4p + k
#pragma unroll
        for (int q = 0; q <= MC_SZB; q++) {
            const unsigned sa = __shfl_down_sync(FULL, a[q], 1), sb = __shfl_down_sync(FULL, b[q], 1);
            const unsigned na = lane == 31u ? an[q] : sa, nb = lane == 31u ? bn[q] : sb;
            const unsigned ax = ((a[q] >> 1) & 0x77777777u) | ((na << 3) & 0x88888888u);   // voxel c+1: k+1 of this lane, k = 0 of the next
            const unsigned bx = ((b[q] >> 1) & 0x77777777u) | ((nb << 3) & 0x88888888u);
            any[q] = a[q] | ax | b[q] | bx;
            all[q] = a[q] & ax & b[q] & bx;
        }
#pragma unroll
        for (int q = 0; q < MC_SZB; q++) {
            const int zb = zb0 + q;
            if (zb > zb_last) break;                                       // warp-uniform
            const unsigned anyz = (any[q] >> 4) | (any[q + 1] << 28), allz = (all[q] >> 4) | (all[q + 1] << 28);
            const unsigned act = (any[q] | anyz) & ~(all[q] & allz) & cellmask;   // bit 4p + k: cell (4L + k) of layer 8zb + p - off
            const int kl_base = zb * 8 - off;
            const int klane = kl_base + (int)lane;                         // lane p < 8 stores the count of layer p
            const bool cnt_lane = lane < 8u && klane >= 0 && klane < g.nk;
            unsigned* const cnt_out = counts + ((size_t)(cnt_lane ? klane : 0) * g.ncy + j) * g.cpr + xc;
            if (!__any_sync(FULL, act != 0u)) {
                if (cnt_lane) *cnt_out = 0u;
                continue;
            }
            // active cells of all 8 layers at once: nibble-wise popcount, summed over the warp in byte fields (<= 128 each)
            unsigned t = act - ((act >> 1) & 0x55555555u);
            t = (t & 0x33333333u) + ((t >> 2) & 0x33333333u);                           // nibble p = active cells of layer p in this lane
            const unsigned ce = __reduce_add_sync(FULL, t & 0x0F0F0F0Fu);               // byte q = layer 2q
            const unsigned co = __reduce_add_sync(FULL, (t >> 4) & 0x0F0F0F0Fu);        // byte q = layer 2q + 1
            if (cnt_lane) { const unsigned nc = (((lane & 1u) ? co : ce) >> (8u * ((lane >> 1) & 3u))) & 0xFFu; *cnt_out = MC_CNT_FIRST(nc); }
#pragma unroll
            for (int p = 0; p < 8; p++) {
                const int kl = kl_base + p;
                const unsigned n = (((p & 1) ? co : ce) >> (8 * (p >> 1))) & 0xFFu;
                if (n == 0u || kl < 0 || kl >= g.nk) continue;                          // warp-uniform
                // the chunk's 128-bit activity mask in natural cell order (bit 4L + k): word w = OR of the nibbles of lanes 8w..8w+7
                unsigned wd = ((act >> (4 * p)) & 15u) << sh;
                wd |= __shfl_xor_sync(FULL, wd, 1);
                wd |= __shfl_xor_sync(FULL, wd, 2);
                wd |= __shfl_xor_sync(FULL, wd, 4);
                if ((lane & 7u) == 0u) reinterpret_cast<unsigned*>(masks + ((size_t)kl * g.ncy + j) * g.cpr + xc)[lane >> 3] = wd;
            }
        }
    }
}

cudaError_t mc_launch_classify_signs(const McGrid& g, const uint4* signs, unsigned tiles_per_row, unsigned nzg, unsigned* counts,
                                     uint4* masks, cudaStream_t s)
{
    if (g.nchunks == 0) return cudaSuccess;
    if (g.step != 1 || g.k0 < g.z0) return cudaErrorInvalidValue;
    const int off = g.k0 - g.z0;
    const int zg_first = off >> 5, zb_last = (off + g.nk - 1) >> 3;        // z-groups / z-blocks holding the lower plane of a classified layer
    const unsigned ncols = (unsigned)g.ncy * (unsigned)g.cpr, nseg = (unsigned)(zb_last - zg_first * 4 + MC_SZB) / MC_SZB;
    const unsigned long long nwork = (unsigned long long)ncols * nseg;   // <= nchunks < 2^32
    if (nwork > 0xFFFFFFFFull) return cudaErrorInvalidValue;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    unsigned long long blocks = (nwork + 7) / 8;
    if (blocks > (unsigned long long)sms * 8u) blocks = (unsigned long long)sms * 8u;
    mc_classify_signs_kernel<<<(unsigned)blocks, 256, 0, s>>>(g, signs, tiles_per_row, nzg, counts, masks, ncols, (unsigned)nwork, zg_first, zb_last);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// K3 mc_scan: exclusive prefix sums (records, vertices, triangles) over the chunk counts, in visiting
// order.  Single pass: warp-shuffle scans inside a tile, decoupled look-back between tiles.
// ---------------------------------------------------------------------------------------------------
// (Measured and dropped: 16384-item tiles -- 64 items per thread in four rounds, read twice -- so that the 8.4 M chunks of a
// 1024^3 grid are 512 tiles in one wave instead of 2048 in two: 0.095 -> 0.125 ms for the two scans.)
#define SCAN_THREADS 256
#define SCAN_ITEMS 16
#define SCAN_ROUNDS 1
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS * SCAN_ROUNDS)

struct ScanWs {
    unsigned ticket;
    unsigned pad[3];
    uint4 desc[1];   // status (0 none, 1 aggregate, 2 inclusive), act, verts, tris -- one 16-byte word per tile
};

size_t mc_scan_workspace_bytes(unsigned nchunks)
{
    const size_t ntiles = ((size_t)nchunks + SCAN_TILE - 1) / SCAN_TILE;
    return 16 + (ntiles + 1) * sizeof(uint4);
}

__device__ static inline uint4 ld_desc(const uint4* p)
{
    uint4 r;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}
__device__ static inline void st_desc(uint4* p, uint4 v)
{
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__global__ void __launch_bounds__(SCAN_THREADS)
mc_scan_kernel(const unsigned* __restrict__ counts, uint4* __restrict__ base, unsigned n, ScanWs* ws, McTotals* totals, unsigned write_every,
               unsigned* __restrict__ alist)
{
    __shared__ unsigned s_tile;
    __shared__ uint3 s_warp[SCAN_THREADS / 32];
    __shared__ uint3 s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ws->ticket, 1u);   // tiles start in order: look-back cannot deadlock
    __syncthreads();
    const unsigned tile = s_tile;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const unsigned first = tile * SCAN_TILE + threadIdx.x * (SCAN_ITEMS * SCAN_ROUNDS);   // (n <= 0xFFFFFFF0: no overflow below)

    unsigned c[SCAN_ITEMS];
    uint3 sum = make_uint3(0, 0, 0);
#pragma unroll 1
    for (int r = 0; r < SCAN_ROUNDS; r++) {
        const unsigned f = first + (unsigned)r * SCAN_ITEMS;
        if (f >= n) break;
        if (f + SCAN_ITEMS <= n) {                             // (rounds start at multiples of 16 items: 64-byte aligned)
#pragma unroll
            for (int q = 0; q < SCAN_ITEMS / 4; q++) {
                const uint4 v = *reinterpret_cast<const uint4*>(counts + f + 4 * q);
                c[4 * q] = v.x; c[4 * q + 1] = v.y; c[4 * q + 2] = v.z; c[4 * q + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < SCAN_ITEMS; k++) c[k] = (f + k < n) ? counts[f + k] : 0u;
        }
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) { sum.x += MC_CNT_ACT(c[k]); sum.y += MC_CNT_V(c[k]); sum.z += MC_CNT_T(c[k]); }
    }
    // inclusive warp scan
    uint3 inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned x = __shfl_up_sync(FULL, inc.x, d), y = __shfl_up_sync(FULL, inc.y, d), z = __shfl_up_sync(FULL, inc.z, d);
        if (lane >= (unsigned)d) { inc.x += x; inc.y += y; inc.z += z; }
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint3 woff = make_uint3(0, 0, 0), agg = make_uint3(0, 0, 0);
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; w++) {
        const uint3 t = s_warp[w];
        if ((unsigned)w < warp) { woff.x += t.x; woff.y += t.y; woff.z += t.z; }
        agg.x += t.x; agg.y += t.y; agg.z += t.z;
    }
    // decoupled look-back by warp 0
    if (warp == 0) {
        uint3 excl = make_uint3(0, 0, 0);
        if (tile > 0) {
            if (lane == 0) st_desc(&ws->desc[tile], make_uint4(1u, agg.x, agg.y, agg.z));
            int pred = (int)tile - 1;
            for (;;) {
                const int t = pred - (int)lane;
                uint4 d = make_uint4(2u, 0, 0, 0);           // tiles before the first: inclusive prefix 0
                if (t >= 0) {
                    do { d = ld_desc(&ws->desc[t]); } while (d.x == 0u);
                }
                const unsigned incl_mask = __ballot_sync(FULL, d.x == 2u);
                const int stop = incl_mask ? (__ffs(incl_mask) - 1) : 32;
                uint3 part = ((int)lane <= stop) ? make_uint3(d.y, d.z, d.w) : make_uint3(0, 0, 0);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    part.x += __shfl_xor_sync(FULL, part.x, o);
                    part.y += __shfl_xor_sync(FULL, part.y, o);
                    part.z += __shfl_xor_sync(FULL, part.z, o);
                }
                excl.x += part.x; excl.y += part.y; excl.z += part.z;
                if (incl_mask) break;
                pred -= 32;
            }
        }
        if (lane == 0) {
            st_desc(&ws->desc[tile], make_uint4(2u, excl.x + agg.x, excl.y + agg.y, excl.z + agg.z));
            s_excl = excl;
            // totals in 64 bits, accumulated per tile: the 32-bit prefixes above wrap silently for a slab with more than 2^32
            // records / vertices / triangles, the totals do not -- the host checks them before anything is emitted
            atomicAdd(&totals->nact, (unsigned long long)agg.x);
            atomicAdd(&totals->nverts, (unsigned long long)agg.y);
            atomicAdd(&totals->ntris, (unsigned long long)agg.z);
        }
    }
    __syncthreads();
    const uint3 te = s_excl;
    uint3 run = make_uint3(te.x + woff.x + inc.x - sum.x, te.y + woff.y + inc.y - sum.y, te.z + woff.z + inc.z - sum.z);
#pragma unroll 1
    for (int r = 0; r < SCAN_ROUNDS; r++) {
        const unsigned f = first + (unsigned)r * SCAN_ITEMS;
        if (f >= n) break;
        if (SCAN_ROUNDS > 1) {
#pragma unroll
            for (int k = 0; k < SCAN_ITEMS; k++) c[k] = (f + k < n) ? counts[f + k] : 0u;      // second read: L1 / L2
        }
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) {
            // prefixes are only ever looked up for non-empty items (the lookups test the count first) and at multiples of
            // write_every (cell-layer boundaries): 99 % of the 16-byte stores of the first scan are skipped
            if (f + k < n && (c[k] != 0u || (f + k) % write_every == 0u)) base[f + k] = make_uint4(run.x, run.y, run.z, c[k]);
            // first scan: the active chunks by rank (run.y counts them), so that K4a visits those only
            if (alist && f + k < n && c[k] != 0u) alist[run.y] = f + k;
            run.x += MC_CNT_ACT(c[k]); run.y += MC_CNT_V(c[k]); run.z += MC_CNT_T(c[k]);
        }
    }
}

cudaError_t mc_launch_scan(const unsigned* counts, uint4* base, unsigned nchunks, void* scan_ws, size_t ws_bytes,
                           McTotals* totals, unsigned write_every, unsigned* alist, cudaStream_t s)
{
    if (nchunks == 0) return cudaSuccess;                     // (the last tile always writes the totals otherwise)
    if (ws_bytes < mc_scan_workspace_bytes(nchunks)) return cudaErrorInvalidValue;
    cudaError_t err = cudaMemsetAsync(scan_ws, 0, mc_scan_workspace_bytes(nchunks), s);
    if (err == cudaSuccess) err = cudaMemsetAsync(totals, 0, sizeof(McTotals), s);
    if (err != cudaSuccess) return err;
    const unsigned ntiles = (nchunks + SCAN_TILE - 1) / SCAN_TILE;
    mc_scan_kernel<<<ntiles, SCAN_THREADS, 0, s>>>(counts, base, nchunks, (ScanWs*)scan_ws, totals, write_every ? write_every : 1u, alist);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// K4a mc_compact: one LANE per active cell.  A warp takes `ch` consecutive ACTIVE chunks (the list the first scan wrote:
// 1 % of the chunks in the README scene -- walking all chunks cost 0.1 ms of dependent count loads), lists their active
// cells (chunk by chunk, cell order inside a chunk -- i.e. visiting order) from the activity masks K2 wrote, and hands
// one cell to every lane: 8 corner loads (scalar: fetching each row pair as one aligned 16-byte load + selects was
// measured 50 % slower, 0.16 -> 0.25 ms), cube index, leaf (256-entry table; FP64 tests for the ambiguous cases), created
// vertices / triangles, and a segmented warp scan that yields the cell's offsets inside its chunk.  Writes the
// 32-byte record at base[chunk].x + (rank in chunk) and, per chunk, the full packed counts for the second scan.
// ---------------------------------------------------------------------------------------------------
__device__ static inline int mc_nth_set_bit(uint4 m, unsigned n)   // position (0..127) of the n-th (0-based) set bit
{
    unsigned c = __popc(m.x);
    if (n < c) return (int)__fns(m.x, 0, (int)n + 1);
    n -= c; c = __popc(m.y);
    if (n < c) return 32 + (int)__fns(m.y, 0, (int)n + 1);
    n -= c; c = __popc(m.z);
    if (n < c) return 64 + (int)__fns(m.z, 0, (int)n + 1);
    n -= c;
    return 96 + (int)__fns(m.w, 0, (int)n + 1);
}

__device__ static inline unsigned long long mc_record_aux(unsigned leaf, int i, int j, int kg)
{
    const McRowMeta* mt = d_meta + MC_LEAF_ROW(leaf);
    const unsigned own = mc_owned_mask(i, j, kg) & mt->refmask;
    return mt->occ_packed | (unsigned long long)(__popc(mt->before[5] & own) | (__popc(mt->before[6] & own) << 4) |
                                                 (__popc(mt->before[10] & own) << 8) | (__popc(mt->before[12] & own) << 12));
}

#ifndef MC_COMPACT_MINB
#define MC_COMPACT_MINB 4
#endif
__global__ void __launch_bounds__(256, MC_COMPACT_MINB)
mc_compact_kernel(const McGrid g, const float* __restrict__ dist, const unsigned* __restrict__ alist, unsigned nactive, unsigned ch,
                  const uint4* __restrict__ base, McRecord* __restrict__ recs, const uint4* __restrict__ masks,
                  unsigned* __restrict__ acounts)
{
    __shared__ unsigned s_quick[256];
    s_quick[threadIdx.x & 255u] = d_quick[threadIdx.x & 255u];
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u;
    const unsigned gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned nw = (gridDim.x * blockDim.x) >> 5;
    const float iso = g.iso;
    for (unsigned r0 = gw * ch; r0 < nactive; r0 += nw * ch) {
        // lane L < ch looks after the active chunk of rank r0 + L
        const unsigned myr = r0 + lane;
        unsigned myc = 0, nact = 0, myslot = 0;
        uint4 mymask = make_uint4(0, 0, 0, 0);
        if (lane < ch && myr < nactive) {
            myc = alist[myr];
            const uint4 b4 = base[myc];                           // x: first record slot, w: what the classifier counted
            myslot = b4.x;
            nact = MC_CNT_ACT(b4.w);
            mymask = masks[myc];
        }
        unsigned incl = nact;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned t = __shfl_up_sync(FULL, incl, d);
            if (lane >= (unsigned)d) incl += t;
        }
        const unsigned total = __shfl_sync(FULL, incl, 31);
        const unsigned pre = incl - nact;                         // items of the chunks before mine
        unsigned carry = 0;                                       // packed counts of the leading chunk's items in earlier batches
        for (unsigned b = 0; b < total; b += 32u) {
            const unsigned t = b + lane;
            const bool valid = t < total;
            // owner lane: the last L with pre_L <= t and nact_L > 0  ==  (number of lanes with incl_L <= t)
            unsigned lo = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const unsigned probe = lo + (unsigned)step - 1u;   // lanes [lo, probe] all have incl <= t ?
                const unsigned v = __shfl_sync(FULL, incl, probe & 31u);
                if (probe < 32u && v <= t) lo += (unsigned)step;
            }
            const unsigned src = valid ? min(lo, 31u) : 0u;
            const unsigned spre = __shfl_sync(FULL, pre, src), snact = __shfl_sync(FULL, nact, src), sslot = __shfl_sync(FULL, myslot, src);
            const unsigned chunk = __shfl_sync(FULL, myc, src), srank = r0 + src;
            uint4 sm;
            sm.x = __shfl_sync(FULL, mymask.x, src); sm.y = __shfl_sync(FULL, mymask.y, src);
            sm.z = __shfl_sync(FULL, mymask.z, src); sm.w = __shfl_sync(FULL, mymask.w, src);
            unsigned cnt = 0, leaf = 0, q = 0;
            int i = 0, j = 0, kl = 0;
            if (valid) {
                q = t - spre;                                     // rank of my cell among the chunk's active cells
                const unsigned xc = chunk % (unsigned)g.cpr, row = chunk / (unsigned)g.cpr;
                j = (int)(row % (unsigned)g.ncy);
                kl = (int)(row / (unsigned)g.ncy);
                i = (int)(xc * 128u) + mc_nth_set_bit(sm, q);
                const int kg = g.k0 + kl;
                float f[8];
                {
                    const size_t sx = (size_t)g.step, sy = (size_t)g.step * (size_t)g.nx, sz = (size_t)g.step * (size_t)g.nx * (size_t)g.ny;
                    const float* p = dist + mc_vox(g, i, j, kg, 0, 0, 0);
                    f[0] = __ldg(p); f[1] = __ldg(p + sx); f[2] = __ldg(p + sx + sy); f[3] = __ldg(p + sy);
                    f[4] = __ldg(p + sz); f[5] = __ldg(p + sz + sx); f[6] = __ldg(p + sz + sx + sy); f[7] = __ldg(p + sz + sy);
                }
                int idx = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) idx |= (f[k] > iso ? 1 : 0) << k;
                cnt = mc_cell_info(g, dist, s_quick[idx], idx, i, j, kg, &leaf);
            }
            // segmented scan: exclusive sum of cnt over the earlier items of the same chunk
            unsigned sc = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned v = __shfl_up_sync(FULL, sc, d);
                if (lane >= (unsigned)d) sc += v;
            }
            const unsigned excl = sc - cnt;                        // exclusive over the whole batch
            const int seg0 = (int)spre - (int)b;                   // lane of my chunk's first item (< 0: it started in an earlier batch)
            const unsigned at0 = __shfl_sync(FULL, excl, seg0 > 0 ? seg0 : 0);
            const unsigned within = excl - at0 + (seg0 < 0 ? carry : 0u);   // packed (act | verts | tris) before me in my chunk
            if (valid) {
                const int kg = g.k0 + kl;
                McRecord r;
                r.cell = (unsigned)i + (unsigned)g.ncx * ((unsigned)j + (unsigned)g.ncy * (unsigned)kl);
                r.info = leaf;
                r.vbase = MC_CNT_V(within);
                r.tbase = MC_CNT_T(within);
                r.aux = mc_record_aux(leaf, i, j, kg);
                r.pad = 0;
                recs[sslot + q] = r;
                if (q + 1u == snact) acounts[srank] = within + cnt;     // last cell of the chunk: its full packed counts, by active-chunk rank
            }
            // carry for a chunk that continues into the next batch: totals of its items seen so far
            const unsigned last_within = __shfl_sync(FULL, within + cnt, 31);
            carry = last_within;
        }
    }
}

cudaError_t mc_launch_compact(const McGrid& g, const float* dist, const unsigned* alist, unsigned nactive, const uint4* base,
                              McRecord* recs, const uint4* masks, unsigned* acounts, cudaStream_t s)
{
    if (g.nchunks == 0 || nactive == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // chunks per warp: enough warp items to fill the machine twice over (a README chunk holds ~24 active cells)
    unsigned ch = nactive / ((unsigned)sms * 128u);
    ch = ch < 1u ? 1u : (ch > 32u ? 32u : ch);
    const unsigned groups = (nactive + ch - 1u) / ch;
    unsigned blocks = (groups + 7u) / 8u;
    if (blocks > (unsigned)sms * 8u) blocks = (unsigned)sms * 8u;
    mc_compact_kernel<<<blocks, 256, 0, s>>>(g, dist, alist, nactive, ch, base, recs, masks, acounts);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// K4b mc_emit: one thread per active cell.  Everything is unrolled over the edge id so that corner / gradient
// selections are static (registers, no local memory) and a warp whose cells have similar cube indices walks
// the same code; the only dynamically indexed table, the cell's 13 vertex ids, lives in shared memory.
// ---------------------------------------------------------------------------------------------------
#define MC_EMIT_THREADS 128

// index of the record of cell (i, j, kl), -1 if that cell is not active
__device__ static inline int mc_find_record(const McEmitParams& p, int i, int j, int kl, unsigned* chunk_vbase = nullptr)
{
    const McGrid& g = p.g;
    const unsigned chunk = ((unsigned)kl * (unsigned)g.ncy + (unsigned)j) * (unsigned)g.cpr + ((unsigned)i >> 7);
    if (MC_CNT_ACT(__ldg(p.counts + chunk)) == 0u) return -1;      // base / masks are only written for active chunks
    const uint4 b = __ldg(p.base + chunk);
    const uint4 m = __ldg(p.masks + chunk);
    const unsigned q = (unsigned)i & 127u, w = q >> 5, bit = q & 31u;      // natural order: bit q of the 128-bit mask
    const unsigned ww = w == 0 ? m.x : (w == 1 ? m.y : (w == 2 ? m.z : m.w));
    if (!((ww >> bit) & 1u)) return -1;
    unsigned rank = __popc(ww & ((1u << bit) - 1u));
    if (w > 0) rank += __popc(m.x);
    if (w > 1) rank += __popc(m.y);
    if (w > 2) rank += __popc(m.z);
    if (chunk_vbase) *chunk_vbase = __ldg(&p.abase[b.y].y);      // vertex prefix of the chunk, by its rank among the active chunks
    return (int)(b.x + rank);
}

struct McF3 { float x, y, z; };

// gradient row R (ORIGINAL corner numbering, Cell.cs:491-498): component differences v[p] - v[q]
template <int R>
__device__ static inline void mc_vg_row(const double* v, double& gx, double& gy, double& gz)
{
    constexpr int PX[8] = {0, 0, 3, 3, 4, 4, 7, 7}, QX[8] = {1, 1, 2, 2, 5, 5, 6, 6};
    constexpr int PY[8] = {0, 1, 1, 0, 4, 5, 5, 4}, QY[8] = {3, 2, 2, 3, 7, 6, 6, 7};
    constexpr int PZ[8] = {0, 1, 2, 3, 0, 1, 2, 3}, QZ[8] = {4, 5, 6, 7, 4, 5, 6, 7};
    gx = v[PX[R]] - v[QX[R]];
    gy = v[PY[R]] - v[QY[R]];
    gz = v[PZ[R]] - v[QZ[R]];
}

// end corners of edge E as positional indices dz*4 + dy*2 + dx (Luts.cs:26-28, Cell.cs:303-308)
__host__ __device__ constexpr int mc_end1(int e) { return e == 0 ? 0 : e == 1 ? 1 : e == 2 ? 3 : e == 3 ? 2 : e == 4 ? 4 : e == 5 ? 5 : e == 6 ? 7 : e == 7 ? 6 : e == 8 ? 0 : e == 9 ? 1 : e == 10 ? 3 : 2; }
__host__ __device__ constexpr int mc_end2(int e) { return e == 0 ? 1 : e == 1 ? 3 : e == 2 ? 2 : e == 3 ? 0 : e == 4 ? 5 : e == 5 ? 7 : e == 6 ? 6 : e == 7 ? 4 : e == 8 ? 4 : e == 9 ? 5 : e == 10 ? 7 : 6; }
__host__ __device__ constexpr int mc_reorder(int i) { return i == 2 ? 3 : i == 3 ? 2 : i == 6 ? 7 : i == 7 ? 6 : i; }   // vv[] (Cell.cs:453-460)

// adds, for `times` references of local edge E in a sharing cell, the two end-corner gradient contributions
// exactly like Cell.AddGradientFromIndex (Cell.cs:154-158,331-333): note vg is indexed with the dz*4+dy*2+dx
// corner index although its rows are in the v0..v7 numbering -- a quirk of the reference that is preserved.
template <int E>
__device__ static inline void mc_add_edge_gradients(const double* v, int times, McF3& n)
{
    constexpr int I1 = mc_end1(E), I2 = mc_end2(E);
    const double w1 = __drcp_rn(MC_EPS + fabs(v[mc_reorder(I1)]));   // == 1.0 / x, correctly rounded
    const double w2 = __drcp_rn(MC_EPS + fabs(v[mc_reorder(I2)]));
    double ax, ay, az, bx, by, bz;
    mc_vg_row<I1>(v, ax, ay, az);
    mc_vg_row<I2>(v, bx, by, bz);
    const float g1x = (float)(ax * w1), g1y = (float)(ay * w1), g1z = (float)(az * w1);
    const float g2x = (float)(bx * w2), g2y = (float)(by * w2), g2z = (float)(bz * w2);
    for (int t = 0; t < times; t++) {
        n.x = n.x + g1x; n.y = n.y + g1y; n.z = n.z + g1z;
        n.x = n.x + g2x; n.y = n.y + g2y; n.z = n.z + g2z;
    }
}

__device__ static inline unsigned mc_float_key(float f)   // monotonic float -> uint
{
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// where a block's vertices go: the output arrays at the block's first slot, indexed by the local vertex index
struct McStage {
    float* v;      // positions, 3 floats per local vertex
    float* c;      // colours (3 floats) -- or, for distance-only voxels, the (cell, edge) recipe (2 words)
    float* n;      // normals
};

__device__ static inline void mc_store_vertex(const McEmitParams& p, const McStage& st, unsigned loc, McF3 pos, McF3 col, McF3 nsum, unsigned* lo, unsigned* hi,
                                             unsigned cell, unsigned edge)
{
    // Cell.NegativeNormals (Cell.cs:97-109): -Vector3.Normalize(sum)
    const float len = sqrtf((nsum.x * nsum.x + nsum.y * nsum.y) + nsum.z * nsum.z);
    McF3 n = {-(nsum.x / len), -(nsum.y / len), -(nsum.z / len)};
    if (p.has_xf) {   // Mesh.Transform (Mesh.cs:57-62)
        const float* M = p.M;
        const float* N = p.N;
        const McF3 tp = {pos.x * M[0] + pos.y * M[4] + pos.z * M[8] + M[12], pos.x * M[1] + pos.y * M[5] + pos.z * M[9] + M[13],
                         pos.x * M[2] + pos.y * M[6] + pos.z * M[10] + M[14]};
        const McF3 tn = {n.x * N[0] + n.y * N[4] + n.z * N[8], n.x * N[1] + n.y * N[5] + n.z * N[9],
                         n.x * N[2] + n.y * N[6] + n.z * N[10]};
        const float l2 = sqrtf((tn.x * tn.x + tn.y * tn.y) + tn.z * tn.z);
        pos = tp;
        n.x = tn.x / l2; n.y = tn.y / l2; n.z = tn.z / l2;
    }
    float* vo = st.v + loc * 3u;
    float* no = st.n + loc * 3u;
    vo[0] = pos.x; vo[1] = pos.y; vo[2] = pos.z;
    if (p.rgb) { float* co = st.c + loc * 3u; co[0] = col.x; co[1] = col.y; co[2] = col.z; }
    else { st.c[loc * 2u] = __uint_as_float(cell); st.c[loc * 2u + 1u] = __uint_as_float(edge); }   // colours follow from sdfk_k_vertex_colors
    no[0] = n.x; no[1] = n.y; no[2] = n.z;
    // Mesh.Measure (Mesh.cs:30-45), reduced per thread -> per warp -> one atomic per warp
    lo[0] = min(lo[0], mc_float_key(pos.x)); lo[1] = min(lo[1], mc_float_key(pos.y)); lo[2] = min(lo[2], mc_float_key(pos.z));
    hi[0] = max(hi[0], mc_float_key(pos.x)); hi[1] = max(hi[1], mc_float_key(pos.y)); hi[2] = max(hi[2], mc_float_key(pos.z));
}

// who creates the vertex on edge E of cell (i, j, kg) when the cell itself does not: offset of the creating cell
// (the sharing cell smallest in (k, j, i)) and the edge's id there
template <int E>
__device__ static inline void mc_creator_of(int i, int j, int kg, int& di, int& dj, int& dk, int& e2)
{
    di = dj = dk = 0;
    e2 = E;
    if (E == 0) { dk = kg > 0 ? -1 : 0; dj = j > 0 ? -1 : 0; e2 = dk ? (dj ? 6 : 4) : (dj ? 2 : 0); }
    else if (E == 1) { dk = -1; e2 = 5; }
    else if (E == 2) { dk = -1; e2 = 6; }
    else if (E == 3) { dk = kg > 0 ? -1 : 0; di = i > 0 ? -1 : 0; e2 = dk ? (di ? 5 : 7) : (di ? 1 : 3); }
    else if (E == 4) { dj = -1; e2 = 6; }
    else if (E == 7) { di = -1; e2 = 5; }
    else if (E == 8) { if (j > 0) { dj = -1; if (i > 0) { di = -1; e2 = 10; } else e2 = 11; } else { di = -1; e2 = 9; } }
    else if (E == 9) { dj = -1; e2 = 10; }
    else if (E == 11) { di = -1; e2 = 10; }
}

// vertex id (slab-local) of slot E referenced by this cell
template <int E>
__device__ static inline int mc_vertex_id(const McEmitParams& p, const McRecord& rec, const McRowMeta* meta, unsigned owned,
                                          int i, int j, int kl, int kg)
{
    if ((owned >> E) & 1u) return (int)(rec.vbase + (unsigned)__popc((unsigned)meta->before[E] & owned));
    int di, dj, dk, e2;
    mc_creator_of<E>(i, j, kg, di, dj, dk, e2);
    const int oi = i + di, oj = j + dj, okl = kl + dk;
    unsigned cvb = 0;
    const int orr = (okl >= 0) ? mc_find_record(p, oi, oj, okl, &cvb) : -1;
    if (orr < 0) { atomicExch(p.error_flag, 1); return 0; }
    const McRecord* orp = p.recs + orr;
    uint4 oa = __ldg(reinterpret_cast<const uint4*>(orp));                  // cell, info, vbase (chunk-local), tbase
    oa.z += cvb;
    if (MC_LEAF_NT(oa.y) == 0u) { atomicExch(p.error_flag, 5); return 0; }   // creator is an "impossible case 13" cell
    const unsigned long long aux = __ldg(&orp->aux);
    if (e2 == 5) return (int)(oa.z + MC_AUX_RANK(aux, 0));
    if (e2 == 6) return (int)(oa.z + MC_AUX_RANK(aux, 1));
    if (e2 == 10) return (int)(oa.z + MC_AUX_RANK(aux, 2));
    // creator on the grid boundary (i, j or k == 0): it also creates edges other than 5, 6, 10
    const McRowMeta* om = d_meta + MC_LEAF_ROW(oa.y);
    if (!((om->refmask >> e2) & 1u)) { atomicExch(p.error_flag, 2); return 0; }
    return (int)(oa.z + (unsigned)__popc((unsigned)om->before[e2] & mc_owned_mask(oi, oj, kg + dk) & om->refmask));
}

// contribution of one sharing cell (ci, cj, ck), which sees the grid edge as its local edge ES, to a vertex normal
template <int ES>
__device__ static inline void mc_gather_from(const McEmitParams& p, int ci, int cj, int ck, McF3& nsum)
{
    const McGrid& g = p.g;
    if (ci < 0 || cj < 0 || ck < 0 || ci >= g.ncx || cj >= g.ncy || ck >= g.ncz) return;
    const int ckl = ck - g.k0;
    if (ckl < 0 || ckl >= g.nk) { atomicExch(p.error_flag, 3); return; }
    double sv[8];
    mc_load_cell(g, p.dist, ci, cj, ck, sv);
    // how often the sharing cell's tiling row references the edge: for an unambiguous cube index (nearly always) straight from
    // the tables (no record lookup: the corners are needed anyway), else from the cell's record
    int idx = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) idx |= (sv[k] > 0.0 ? 1 : 0) << k;
    const unsigned quick = __ldg(&d_quick[idx]);
    int times;
    if (!(quick & MC_QUICK_AMBIG)) {
        times = (int)d_meta[MC_LEAF_ROW(quick & 0x7FFFu)].occ[ES];
    } else {
        const int sr = mc_find_record(p, ci, cj, ckl);
        if (sr < 0) { atomicExch(p.error_flag, 4); return; }
        times = (int)MC_AUX_OCC(__ldg(&p.recs[sr].aux), ES);
    }
    mc_add_edge_gradients<ES>(sv, times, nsum);
}

// position + colour of the vertex the cell creates on its edge E (Cell.AddFaceFromEdgeIndex, new-vertex branch,
// Cell.cs:313-357), then the gradient contributions of every sharing cell in visiting order (the accumulation order
// of the reference's normals[]): the grid edge starts at lattice point (X, Y, Z) and runs along AXIS; sharing cells
// in (k, j, i) order are  x: (Y-1,Z-1) e6, (Y,Z-1) e4, (Y-1,Z) e2, (Y,Z) e0;  y: (X-1,Z-1) e5, (X,Z-1) e7, (X-1,Z) e1,
// (X,Z) e3;  z: (X-1,Y-1) e10, (X,Y-1) e11, (X-1,Y) e9, (X,Y) e8.
template <int E>
__device__ static inline void mc_create_edge_vertex(const McEmitParams& p, const double* v, int occ_self, int i, int j, int kg,
                                                    const McStage& st, unsigned loc, unsigned* lo, unsigned* hi, unsigned cell)
{
    const McGrid& g = p.g;
    constexpr int I1 = mc_end1(E), I2 = mc_end2(E);
    constexpr int dx1 = I1 & 1, dy1 = (I1 >> 1) & 1, dz1 = I1 >> 2, dx2 = I2 & 1, dy2 = (I2 >> 1) & 1, dz2 = I2 >> 2;
    const double stp = (double)g.step;
    const int X0 = i * g.step, Y0 = j * g.step, Z0 = kg * g.step;           // Cell.x/y/z are voxel coordinates
    const double w1 = __drcp_rn(MC_EPS + fabs(v[mc_reorder(I1)]));   // == 1.0 / x, correctly rounded
    const double w2 = __drcp_rn(MC_EPS + fabs(v[mc_reorder(I2)]));
    double fx = 0.0, fy = 0.0, fz = 0.0, ff = 0.0;
    fx += dx1 * w1; fy += dy1 * w1; fz += dz1 * w1; ff += w1;
    fx += dx2 * w2; fy += dy2 * w2; fz += dz2 * w2; ff += w2;
    McF3 pos, col = {0.f, 0.f, 0.f}, nsum = {0.f, 0.f, 0.f};
    pos.x = (float)(X0 + stp * fx / ff); pos.y = (float)(Y0 + stp * fy / ff); pos.z = (float)(Z0 + stp * fz / ff);
    if (p.rgb) {
        const float* c1 = p.rgb + mc_vox(g, i, j, kg, dx1, dy1, dz1) * 3;
        const float* c2 = p.rgb + mc_vox(g, i, j, kg, dx2, dy2, dz2) * 3;
        const float f1 = (float)w1, f2 = (float)w2;
        const McF3 cm = {__ldg(c1) * f1 + __ldg(c2) * f2, __ldg(c1 + 1) * f1 + __ldg(c2 + 1) * f2, __ldg(c1 + 2) * f1 + __ldg(c2 + 2) * f2};
        col.x = (float)(cm.x / ff); col.y = (float)(cm.y / ff); col.z = (float)(cm.z / ff);
    }
    constexpr int AXIS = (dx1 != dx2) ? 0 : ((dy1 != dy2) ? 1 : 2);
    const int X = i + (dx1 < dx2 ? dx1 : dx2), Y = j + (dy1 < dy2 ? dy1 : dy2), Z = kg + (dz1 < dz2 ? dz1 : dz2);
    // the creating cell is the first sharing cell in visiting order; it sees the edge as E
    mc_add_edge_gradients<E>(v, occ_self, nsum);
    if (AXIS == 0) {          // this cell is one of (X, Y-1|Y, Z-1|Z); skip itself, keep the order
        if (E == 6) { mc_gather_from<4>(p, X, Y, Z - 1, nsum); mc_gather_from<2>(p, X, Y - 1, Z, nsum); mc_gather_from<0>(p, X, Y, Z, nsum); }
        if (E == 4) { mc_gather_from<2>(p, X, Y - 1, Z, nsum); mc_gather_from<0>(p, X, Y, Z, nsum); }
        if (E == 2) { mc_gather_from<0>(p, X, Y, Z, nsum); }
    } else if (AXIS == 1) {
        if (E == 5) { mc_gather_from<7>(p, X, Y, Z - 1, nsum); mc_gather_from<1>(p, X - 1, Y, Z, nsum); mc_gather_from<3>(p, X, Y, Z, nsum); }
        if (E == 7) { mc_gather_from<1>(p, X - 1, Y, Z, nsum); mc_gather_from<3>(p, X, Y, Z, nsum); }
        if (E == 1) { mc_gather_from<3>(p, X, Y, Z, nsum); }
    } else {
        if (E == 10) { mc_gather_from<11>(p, X, Y - 1, Z, nsum); mc_gather_from<9>(p, X - 1, Y, Z, nsum); mc_gather_from<8>(p, X, Y, Z, nsum); }
        if (E == 11) { mc_gather_from<9>(p, X - 1, Y, Z, nsum); mc_gather_from<8>(p, X, Y, Z, nsum); }
        if (E == 9) { mc_gather_from<8>(p, X, Y, Z, nsum); }
    }
    mc_store_vertex(p, st, loc, pos, col, nsum, lo, hi, cell, (unsigned)E);
}


// ---- vertices an interior cell creates (edges 5, 6, 10): one neighbourhood load instead of four cell loads -----------------
// The grid edge of slot E runs along AXIS from lattice point (X, Y, Z); the up to four cells around it -- in visiting order
// (p, q) = (0,0) [the creating cell itself], (1,0), (0,1), (1,1) in the two perpendicular axes, lower axis fastest -- see
// it as their local edge ES (AXIS x: 6, 4, 2, 0;  y: 5, 7, 1, 3;  z: 10, 11, 9, 8) and jointly touch only a 3 x 3 x 2 block
// of voxels (2 along the edge).  The former code loaded 8 corners per sharing cell one cell after the other (32 scattered
// 4-byte loads per vertex, each cell's loads issued only after the previous cell's table look-ups: 21 sectors per request,
// latency-bound at 33 % issue utilisation).  Here the 18 values are loaded once, up front and independently of each other,
// every cell's corners are static selections from them, the occurrence counts come from tables staged in shared memory, and
// the two end-corner weights -- the same two voxels for all four cells -- are computed once.  The arithmetic per cell is
// exactly mc_add_edge_gradients' (same operations in the same order), so the result is bit-identical.
template <int E>
struct McEdgeGeom {
    static constexpr int I1 = mc_end1(E), I2 = mc_end2(E);
    static constexpr int dx1 = I1 & 1, dy1 = (I1 >> 1) & 1, dz1 = I1 >> 2, dx2 = I2 & 1, dy2 = (I2 >> 1) & 1, dz2 = I2 >> 2;
    static constexpr int AXIS = (dx1 != dx2) ? 0 : ((dy1 != dy2) ? 1 : 2);
};

// corners (reference numbering v0..v7) of the sharing cell (P, Q) out of the neighbourhood nb[oz][oy][ox]
template <int AXIS, int P, int Q>
__device__ static inline void mc_cell_from_nb(const double (&nb)[3][3][3], double* v)
{
    constexpr int bx = AXIS == 0 ? 0 : P, by = AXIS == 0 ? P : (AXIS == 1 ? 0 : Q), bz = AXIS == 2 ? 0 : Q;
    v[0] = nb[bz][by][bx];         v[1] = nb[bz][by][bx + 1];         v[2] = nb[bz][by + 1][bx + 1];         v[3] = nb[bz][by + 1][bx];
    v[4] = nb[bz + 1][by][bx];     v[5] = nb[bz + 1][by][bx + 1];     v[6] = nb[bz + 1][by + 1][bx + 1];     v[7] = nb[bz + 1][by + 1][bx];
}

template <int AXIS, int P, int Q, int ES>
__device__ static inline void mc_gather_from_nb(const McEmitParams& p, const double (&nb)[3][3][3], int ci, int cj, int ck,
                                                const unsigned* s_quick, const unsigned long long* s_occ, McF3& nsum)
{
    const McGrid& g = p.g;
    if (ci >= g.ncx || cj >= g.ncy || ck >= g.ncz) return;            // (ci, cj, ck >= 0 always: the creator is the (0,0) cell)
    const int ckl = ck - g.k0;
    if (ckl < 0 || ckl >= g.nk) { atomicExch(p.error_flag, 3); return; }
    double sv[8];
    mc_cell_from_nb<AXIS, P, Q>(nb, sv);
    int idx = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) idx |= (sv[k] > 0.0 ? 1 : 0) << k;
    const unsigned quick = s_quick[idx];
    int times;
    if (!(quick & MC_QUICK_AMBIG)) {
        times = (int)MC_AUX_OCC(s_occ[MC_LEAF_ROW(quick & 0x7FFFu)], ES);
    } else {
        const int sr = mc_find_record(p, ci, cj, ckl);
        if (sr < 0) { atomicExch(p.error_flag, 4); return; }
        times = (int)MC_AUX_OCC(__ldg(&p.recs[sr].aux), ES);
    }
    mc_add_edge_gradients<ES>(sv, times, nsum);
}

template <int E>
__device__ static inline void mc_create_interior_vertex(const McEmitParams& p, int occ_self, int i, int j, int kg, const McStage& st,
                                                        unsigned loc, unsigned* lo, unsigned* hi, unsigned cell, const unsigned* s_quick,
                                                        const unsigned long long* s_occ)
{
    typedef McEdgeGeom<E> G;
    constexpr int AXIS = G::AXIS;
    const McGrid& g = p.g;
    // lattice point where the edge starts, and the first voxel of the neighbourhood (one cell back in the perpendicular axes)
    const int X = i + (G::dx1 < G::dx2 ? G::dx1 : G::dx2), Y = j + (G::dy1 < G::dy2 ? G::dy1 : G::dy2), Z = kg + (G::dz1 < G::dz2 ? G::dz1 : G::dz2);
    const int cx0 = X - (AXIS != 0), cy0 = Y - (AXIS != 1), cz0 = Z - (AXIS != 2);      // == (i, j, kg): the creating cell
    constexpr int EX = AXIS == 0 ? 2 : 3, EY = AXIS == 1 ? 2 : 3, EZ = AXIS == 2 ? 2 : 3;
    const double iso = (double)g.iso;
    double nb[3][3][3];
    {
        // 18 independent loads; lattice points beyond the grid / the slab are clamped (their cells do not contribute)
        size_t ox[3], oy[3], oz[3];
#pragma unroll
        for (int a = 0; a < 3; a++) {
            ox[a] = (size_t)min((cx0 + a) * g.step, g.nx - 1);
            oy[a] = (size_t)min((cy0 + a) * g.step, g.ny - 1) * (size_t)g.nx;
            oz[a] = (size_t)min(max((cz0 + a) * g.step - g.z0, 0), g.nzl - 1) * (size_t)g.nx * (size_t)g.ny;
        }
        float f[3][3][3];
#pragma unroll
        for (int c = 0; c < EZ; c++)
#pragma unroll
            for (int b = 0; b < EY; b++)
#pragma unroll
                for (int a = 0; a < EX; a++) f[c][b][a] = __ldg(p.dist + oz[c] + oy[b] + ox[a]);
#pragma unroll
        for (int c = 0; c < EZ; c++)
#pragma unroll
            for (int b = 0; b < EY; b++)
#pragma unroll
                for (int a = 0; a < EX; a++) nb[c][b][a] = (double)f[c][b][a] - iso;
    }
    double v[8];
    mc_cell_from_nb<AXIS, 0, 0>(nb, v);
    // position + colour: Cell.AddFaceFromEdgeIndex, new-vertex branch (Cell.cs:313-357) -- as mc_create_edge_vertex
    constexpr int I1 = G::I1, I2 = G::I2;
    const double stp = (double)g.step;
    const int X0 = i * g.step, Y0 = j * g.step, Z0 = kg * g.step;
    const double w1 = __drcp_rn(MC_EPS + fabs(v[mc_reorder(I1)]));
    const double w2 = __drcp_rn(MC_EPS + fabs(v[mc_reorder(I2)]));
    double fx = 0.0, fy = 0.0, fz = 0.0, ff = 0.0;
    fx += G::dx1 * w1; fy += G::dy1 * w1; fz += G::dz1 * w1; ff += w1;
    fx += G::dx2 * w2; fy += G::dy2 * w2; fz += G::dz2 * w2; ff += w2;
    McF3 pos, col = {0.f, 0.f, 0.f}, nsum = {0.f, 0.f, 0.f};
    pos.x = (float)(X0 + stp * fx / ff); pos.y = (float)(Y0 + stp * fy / ff); pos.z = (float)(Z0 + stp * fz / ff);
    if (p.rgb) {
        const float* c1 = p.rgb + mc_vox(g, i, j, kg, G::dx1, G::dy1, G::dz1) * 3;
        const float* c2 = p.rgb + mc_vox(g, i, j, kg, G::dx2, G::dy2, G::dz2) * 3;
        const float f1 = (float)w1, f2 = (float)w2;
        const McF3 cm = {__ldg(c1) * f1 + __ldg(c2) * f2, __ldg(c1 + 1) * f1 + __ldg(c2 + 1) * f2, __ldg(c1 + 2) * f1 + __ldg(c2 + 2) * f2};
        col.x = (float)(cm.x / ff); col.y = (float)(cm.y / ff); col.z = (float)(cm.z / ff);
    }
    // normals: the creating cell first, then the other sharing cells in visiting order
    mc_add_edge_gradients<E>(v, occ_self, nsum);
    constexpr int ES1 = AXIS == 0 ? 4 : (AXIS == 1 ? 7 : 11), ES2 = AXIS == 0 ? 2 : (AXIS == 1 ? 1 : 9), ES3 = AXIS == 0 ? 0 : (AXIS == 1 ? 3 : 8);
    // cell (P, Q): +P in the lower perpendicular axis, +Q in the higher one
    const int pi = AXIS == 0 ? 0 : 1, pj = AXIS == 0 ? 1 : 0;                    // what +P adds to (ci, cj)
    const int qj = AXIS == 2 ? 1 : 0, qk = AXIS == 2 ? 0 : 1;                    // what +Q adds to (cj, ck)
    mc_gather_from_nb<AXIS, 1, 0, ES1>(p, nb, i + pi, j + pj, kg, s_quick, s_occ, nsum);
    mc_gather_from_nb<AXIS, 0, 1, ES2>(p, nb, i, j + qj, kg + qk, s_quick, s_occ, nsum);
    mc_gather_from_nb<AXIS, 1, 1, ES3>(p, nb, i + pi, j + pj + qj, kg + qk, s_quick, s_occ, nsum);
    mc_store_vertex(p, st, loc, pos, col, nsum, lo, hi, cell, (unsigned)E);
}

// Cell.CalculateCenterVertex (Cell.cs:501-549) + its accumulated gradient
__device__ static inline void mc_create_center_vertex(const McEmitParams& p, const double* v, int times, int i, int j, int kg,
                                                      const McStage& st, unsigned loc, unsigned* lo, unsigned* hi, unsigned cell)
{
    const McGrid& g = p.g;
    const double stp = (double)g.step;
    const int X0 = i * g.step, Y0 = j * g.step, Z0 = kg * g.step;
    double w[8];
#pragma unroll
    for (int q = 0; q < 8; q++) w[q] = __drcp_rn(MC_EPS + fabs(v[q]));
    double fx = 0.0, fy = 0.0, fz = 0.0, ff = 0.0;
    McF3 fc = {0.f, 0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const int cdx = (0x66 >> q) & 1, cdy = (0xCC >> q) & 1, cdz = (0xF0 >> q) & 1;   // corner q -> (dx,dy,dz)
        fx += (double)cdx * w[q]; fy += (double)cdy * w[q]; fz += (double)cdz * w[q]; ff += w[q];
        if (p.rgb) {
            const float* cp = p.rgb + mc_vox(g, i, j, kg, cdx, cdy, cdz) * 3;
            const float wq = (float)w[q];
            const float cx = __ldg(cp) * wq, cy = __ldg(cp + 1) * wq, cz = __ldg(cp + 2) * wq;
            if (q == 0) { fc.x = cx; fc.y = cy; fc.z = cz; }
            else { fc.x = fc.x + cx; fc.y = fc.y + cy; fc.z = fc.z + cz; }
        }
    }
    McF3 pos, col, nsum = {0.f, 0.f, 0.f};
    pos.x = (float)(X0 + stp * fx / ff); pos.y = (float)(Y0 + stp * fy / ff); pos.z = (float)(Z0 + stp * fz / ff);
    col.x = (float)(fc.x / ff); col.y = (float)(fc.y / ff); col.z = (float)(fc.z / ff);
    double gs[3] = {0.0, 0.0, 0.0};
    {
        double gx, gy, gz;
        mc_vg_row<0>(v, gx, gy, gz); gs[0] = w[0] * gx; gs[1] = w[0] * gy; gs[2] = w[0] * gz;
        mc_vg_row<1>(v, gx, gy, gz); gs[0] = gs[0] + w[1] * gx; gs[1] = gs[1] + w[1] * gy; gs[2] = gs[2] + w[1] * gz;
        mc_vg_row<2>(v, gx, gy, gz); gs[0] = gs[0] + w[2] * gx; gs[1] = gs[1] + w[2] * gy; gs[2] = gs[2] + w[2] * gz;
        mc_vg_row<3>(v, gx, gy, gz); gs[0] = gs[0] + w[3] * gx; gs[1] = gs[1] + w[3] * gy; gs[2] = gs[2] + w[3] * gz;
        mc_vg_row<4>(v, gx, gy, gz); gs[0] = gs[0] + w[4] * gx; gs[1] = gs[1] + w[4] * gy; gs[2] = gs[2] + w[4] * gz;
        mc_vg_row<5>(v, gx, gy, gz); gs[0] = gs[0] + w[5] * gx; gs[1] = gs[1] + w[5] * gy; gs[2] = gs[2] + w[5] * gz;
        mc_vg_row<6>(v, gx, gy, gz); gs[0] = gs[0] + w[6] * gx; gs[1] = gs[1] + w[6] * gy; gs[2] = gs[2] + w[6] * gz;
        mc_vg_row<7>(v, gx, gy, gz); gs[0] = gs[0] + w[7] * gx; gs[1] = gs[1] + w[7] * gy; gs[2] = gs[2] + w[7] * gz;
    }
    const float gx = (float)gs[0], gy = (float)gs[1], gz = (float)gs[2];
    for (int t = 0; t < times; t++) { nsum.x = nsum.x + gx; nsum.y = nsum.y + gy; nsum.z = nsum.z + gz; }
    mc_store_vertex(p, st, loc, pos, col, nsum, lo, hi, cell, 12u);
}

#define MC_FOR_EDGES(M) M(0) M(1) M(2) M(3) M(4) M(5) M(6) M(7) M(8) M(9) M(10) M(11)

// K4b runs as two kernels.
//   mc_emit_tris_kernel   one thread per record: the vertex id of every slot the cell references, its triangles, and one
//                         TASK (record, slot) per vertex the cell creates, stored at the vertex' own index.
//   mc_emit_verts_kernel  one thread per created VERTEX.  Creating a vertex is the expensive part (FP64 interpolation, the
//                         ordered gather of up to four cells' gradients) and its code depends on the edge the vertex sits on;
//                         inside the per-record kernel the three interior kinds (edges 5, 6, 10) each ran with a third of
//                         the lanes (12 of 32 lanes active on average, 5.6e8 warp instructions).  Here a block first sorts
//                         its 1024 tasks by kind in shared memory and then works through one kind at a time with full warps.
#ifndef MC_VERT_THREADS
#define MC_VERT_THREADS 256
#endif
#ifndef MC_VERT_PER_BLOCK
#define MC_VERT_PER_BLOCK 1024
#endif

__global__ void __launch_bounds__(MC_EMIT_THREADS, 12)
mc_emit_tris_kernel(const McEmitParams p)
{
    __shared__ int s_vid[MC_EMIT_THREADS][13];
    const McGrid& g = p.g;
    const unsigned r = p.rec_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= p.rec_end) return;
    McRecord rec = p.recs[r];
    const int i = (int)(rec.cell % (unsigned)g.ncx);
    const unsigned t2 = rec.cell / (unsigned)g.ncx;
    const int j = (int)(t2 % (unsigned)g.ncy);
    const int kl = (int)(t2 / (unsigned)g.ncy);
    const int kg = g.k0 + kl;
    {   // records carry chunk-local offsets
        const unsigned arank = __ldg(&p.base[t2 * (unsigned)g.cpr + ((unsigned)i >> 7)].y);
        const uint4 cb = __ldg(p.abase + arank);
        rec.vbase += cb.y;
        rec.tbase += cb.z;
    }
    const McRowMeta* meta = d_meta + MC_LEAF_ROW(rec.info);
    const signed char* row = d_lut + meta->off;
    const int nent = 3 * (int)MC_LEAF_NT(rec.info);
    const unsigned owned = mc_owned_mask(i, j, kg);
    const unsigned refd = nent ? meta->refmask : 0u;                // nent == 0: "impossible case 13", emits nothing
    int* vid = s_vid[threadIdx.x];
    // ---- vertex id of every slot this cell references
    if (i > 0 && j > 0 && kg > 0) {
        // interior cell (nearly all): it creates slots 5, 6, 10, 12 itself, and the creator of every other edge is a fixed
        // neighbour whose record carries the rank of that edge -- one generic loop over the referenced edges (a warp runs
        // max-edges-per-cell iterations instead of walking 12 specialised blocks)
        unsigned own = refd & owned;
        while (own) {
            const int e = __ffs((int)own) - 1;
            own &= own - 1u;
            vid[e] = (int)(rec.vbase + (unsigned)__popc((unsigned)meta->before[e] & owned));
        }
        // Every other edge is created by one of SIX neighbours (offsets -1 in i / j / k), each answering for up to two edges
        // with the rank fields of its record (0: e5, 1: e6, 2: e10):
        //   (0,0,-1): e1 <- its e5, e2 <- its e6     (-1,0,-1): e3 <- e5     (0,-1,-1): e0 <- e6
        //   (0,-1,0): e4 <- its e6, e9 <- its e10    (-1,-1,0): e8 <- e10    (-1,0,0):  e7 <- e5, e11 <- e10
        // One look-up per NEIGHBOUR (round 2: one per edge, 9 instead of 6), the chunk words (count, first record, mask) of
        // neighbours in the same chunk fetched once, and the three chunk words / the three record words requested together
        // instead of one after the other (4 dependent round trips -> 2).
        const unsigned need = refd & ~owned;
        unsigned cchunk = 0xFFFFFFFFu, ccnt = 0u;
        uint4 cb = make_uint4(0, 0, 0, 0), cm = make_uint4(0, 0, 0, 0);
#define MC_NEIGHBOUR(DI, DJ, DK, EA, RA, EB, RB)                                                                       \
        if (need & ((1u << EA) | (EB >= 0 ? (1u << (EB >= 0 ? EB : 0)) : 0u))) {                                         \
            const int oi = i - DI, oj = j - DJ, okl = kl - DK;                                                           \
            int id_a = 0, id_b = 0;                                                                                      \
            if (okl < 0) atomicExch(p.error_flag, 1);                                                                    \
            else {                                                                                                       \
                const unsigned chunk = ((unsigned)okl * (unsigned)g.ncy + (unsigned)oj) * (unsigned)g.cpr + ((unsigned)oi >> 7); \
                if (chunk != cchunk) {                                                                                   \
                    cchunk = chunk;                                                                                      \
                    ccnt = __ldg(p.counts + chunk);                /* base / masks hold data only for active chunks: */  \
                    cb = __ldg(p.base + chunk);                    /* requested together, used only if the count says so */ \
                    cm = __ldg(p.masks + chunk);                                                                         \
                }                                                                                                        \
                const unsigned q = (unsigned)oi & 127u, w = q >> 5, bit = q & 31u;                                       \
                const unsigned ww = w == 0 ? cm.x : (w == 1 ? cm.y : (w == 2 ? cm.z : cm.w));                            \
                if (MC_CNT_ACT(ccnt) == 0u || !((ww >> bit) & 1u)) atomicExch(p.error_flag, 1);                          \
                else {                                                                                                   \
                    unsigned rank = __popc(ww & ((1u << bit) - 1u));                                                     \
                    if (w > 0) rank += __popc(cm.x);                                                                     \
                    if (w > 1) rank += __popc(cm.y);                                                                     \
                    if (w > 2) rank += __popc(cm.z);                                                                     \
                    const McRecord* orp = p.recs + (cb.x + rank);                                                        \
                    const unsigned cvb = __ldg(&p.abase[cb.y].y);                    /* vertex prefix of the chunk */     \
                    const uint4 oa = __ldg(reinterpret_cast<const uint4*>(orp));     /* cell, info, vbase (chunk-local), tbase */ \
                    const unsigned long long oaux = __ldg(&orp->aux);                                                    \
                    if (MC_LEAF_NT(oa.y) == 0u) atomicExch(p.error_flag, 5);         /* creator is an "impossible case 13" cell */ \
                    else { id_a = (int)(oa.z + cvb + MC_AUX_RANK(oaux, RA)); id_b = (int)(oa.z + cvb + MC_AUX_RANK(oaux, RB)); } \
                }                                                                                                        \
            }                                                                                                            \
            if ((need >> EA) & 1u) vid[EA] = id_a;                                                                       \
            if (EB >= 0 && ((need >> (EB >= 0 ? EB : 0)) & 1u)) vid[EB >= 0 ? EB : 0] = id_b;                            \
        }
        MC_NEIGHBOUR(0, 0, 1, 1, 0, 2, 1)
        MC_NEIGHBOUR(1, 0, 1, 3, 0, -1, 0)
        MC_NEIGHBOUR(0, 1, 1, 0, 1, -1, 0)
        MC_NEIGHBOUR(0, 1, 0, 4, 1, 9, 2)
        MC_NEIGHBOUR(1, 1, 0, 8, 2, -1, 0)
        MC_NEIGHBOUR(1, 0, 0, 7, 0, 11, 2)
#undef MC_NEIGHBOUR
    } else {
#define VID(E) if ((refd >> E) & 1u) vid[E] = mc_vertex_id<E>(p, rec, meta, owned, i, j, kl, kg);
        MC_FOR_EDGES(VID)
#undef VID
        if ((refd >> 12) & 1u) vid[12] = (int)(rec.vbase + (unsigned)__popc((unsigned)meta->before[12] & owned));
    }
    // ---- triangles (Cell.AddFace order): global index = id - vlocal0 + vglobal0
    {
        int* out = p.tris + ((long long)(rec.tbase - p.tlocal0)) * 3;
        const int shift = (int)(p.vglobal0 - (long long)p.vlocal0);
        for (int k = 0; k < nent; k++) out[k] = vid[row[k]] + shift;
    }
    // ---- one task per vertex this cell creates, at the vertex' slot (= id - vlocal0)
    unsigned mine = refd & owned;
    while (mine) {
        const int e = __ffs((int)mine) - 1;
        mine &= mine - 1u;
        // edges 5, 6, 10 (what mc_emit_verts creates from the voxel neighbourhood alone): the task carries the CELL and how often
        // the cell's own row references the edge, so that the vertex kernel starts its gathers without waiting for the record
        const bool nb = e == 5 || e == 6 || e == 10;
        p.tasks[(long long)vid[e] - (long long)p.vlocal0] = nb ? make_uint2(rec.cell, (unsigned)e | ((unsigned)meta->occ[e] << 4)) : make_uint2(r, (unsigned)e);
    }
}

// creates the vertex of task (record r, slot E) at vertex slot `slot`
template <int E>
__device__ static inline void mc_run_vertex_task(const McEmitParams& p, unsigned r, const McStage& st, unsigned loc, unsigned* lo, unsigned* hi)
{
    const McGrid& g = p.g;
    const uint4 ra = __ldg(reinterpret_cast<const uint4*>(p.recs + r));      // cell, info, vbase, tbase
    const unsigned long long aux = __ldg(&p.recs[r].aux);
    const int i = (int)(ra.x % (unsigned)g.ncx);
    const unsigned t2 = ra.x / (unsigned)g.ncx;
    const int j = (int)(t2 % (unsigned)g.ncy);
    const int kg = g.k0 + (int)(t2 / (unsigned)g.ncy);
    double v[8];
    mc_load_cell(g, p.dist, i, j, kg, v);
    if (E == 12) mc_create_center_vertex(p, v, d_meta[MC_LEAF_ROW(ra.y)].occ[12], i, j, kg, st, loc, lo, hi, ra.x);
    else mc_create_edge_vertex<(E == 12 ? 0 : E)>(p, v, (int)MC_AUX_OCC(aux, (E == 12 ? 0 : E)), i, j, kg, st, loc, lo, hi, ra.x);
}

#ifndef MC_VERT_MINB
#define MC_VERT_MINB 4    // measured at 1024^3: 3 (80 regs) 0.683 ms, 4 (64 regs) 0.655 ms, 6 (40 regs) 0.731 ms
#endif
__global__ void __launch_bounds__(MC_VERT_THREADS, MC_VERT_MINB)
mc_emit_verts_kernel(const McEmitParams p)
{
    __shared__ uint2 s_item[MC_VERT_PER_BLOCK];      // (record, slot E | local vertex index << 8), grouped by kind
    __shared__ unsigned s_cnt[4], s_base[4];
    __shared__ unsigned s_quick[256];                // cube index -> leaf of an unambiguous cell
    __shared__ unsigned long long s_occ[MCR_NROWS];  // tiling row -> how often it references each edge (McRecord::aux layout)
    const unsigned tid = threadIdx.x;
    for (unsigned t = tid; t < 256u; t += MC_VERT_THREADS) s_quick[t] = d_quick[t];
    for (unsigned t = tid; t < (unsigned)MCR_NROWS; t += MC_VERT_THREADS) s_occ[t] = d_meta[t].occ_packed;
    const unsigned first = p.vert_begin + blockIdx.x * MC_VERT_PER_BLOCK;
    if (tid < 4) s_cnt[tid] = 0u;
    __syncthreads();
    // kind: 0 = edge 5, 1 = edge 6, 2 = edge 10 (what an interior cell creates), 3 = everything else (grid boundary, centre)
    uint2 task[MC_VERT_PER_BLOCK / MC_VERT_THREADS];
    unsigned kind[MC_VERT_PER_BLOCK / MC_VERT_THREADS], pos[MC_VERT_PER_BLOCK / MC_VERT_THREADS];
#pragma unroll
    for (int q = 0; q < MC_VERT_PER_BLOCK / MC_VERT_THREADS; q++) {
        const unsigned loc = (unsigned)q * MC_VERT_THREADS + tid, vtx = first + loc;
        kind[q] = 4u;
        if (vtx < p.vert_end) {
            task[q] = __ldg(p.tasks + vtx);
            const unsigned e = task[q].y & 15u;
            kind[q] = e == 5u ? 0u : (e == 6u ? 1u : (e == 10u ? 2u : 3u));
            task[q].y = (task[q].y & 0xFFu) | (loc << 8);         // slot E [0:4) | own occurrence count [4:8) | local vertex index
            pos[q] = atomicAdd(&s_cnt[kind[q]], 1u);
        }
    }
    __syncthreads();
    if (tid == 0) { s_base[0] = 0u; s_base[1] = s_cnt[0]; s_base[2] = s_cnt[0] + s_cnt[1]; s_base[3] = s_cnt[0] + s_cnt[1] + s_cnt[2]; }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < MC_VERT_PER_BLOCK / MC_VERT_THREADS; q++)
        if (kind[q] < 4u) s_item[s_base[kind[q]] + pos[q]] = task[q];
    __syncthreads();
    // (Measured and dropped: an L2 prefetch pass over all of the block's tasks before the work loops -- 0.39 -> 0.50 ms: the
    // prefetches need the same dependent record load first and then saturate the load/store queue.  Round 2, second session,
    // all bit-exact and all slower than this kernel's 0.39 ms at 1024^3 (DESIGN.md section 4): the rows of the 3 x 3 x 2
    // neighbourhood / the two corners' colours as aligned 16-byte loads + selects (0.51 ms at 80 registers; divergent
    // LDG.128 cost more than three LDG.32 -- the same change made K4a 50 % slower); a block's rows staged in shared memory
    // and stored coalesced (0.39 ms at 3 CTAs / SM, 0.69 ms at 4: the stage takes the L1 the gathers live on; the scattered
    // stores themselves are 0.06 ms of the kernel); one launch per kind of vertex so that the hot code fits the 32 KB
    // instruction cache (3 x 0.32 ms: every launch re-reads the block's sectors and writes partial sectors of the outputs);
    // fewer vertices in flight for L2 reuse across layers (256..512 per block: 0.48..0.55 ms); the sharing cells' corners from
    // dense 32-byte "corner blocks" that K4a wrote next to the records instead of the voxel gathers (0.39 -> 0.46 ms, K4a
    // +0.025 ms: one more dependent look-up per vertex outweighs 14 fewer scattered loads -- the kernel is bound by the
    // LATENCY of its dependent loads at 32 resident warps, which is why the tasks now carry the cell id); an L1 prefetch of
    // the thread's vertex of the next kind (one address per voxel row + the two colours, from the task alone) issued before
    // the current kind's vertex is created (0.36 -> 0.40 ms: the extra L1 traffic costs more than the overlap gains).  The kernel moves 0.84 GB
    // from DRAM for a 0.16 GB footprint of touched sectors and runs at the ~3 TB/s this box sustains for scattered sectors.)
    const McStage st = {p.verts + (size_t)first * 3, p.rgb ? p.cols + (size_t)first * 3 : reinterpret_cast<float*>(p.recipes + first),
                        p.nrms + (size_t)first * 3};
    unsigned lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
#define MC_KIND(K, E)                                                                                          \
    for (unsigned idx = tid; idx < s_cnt[K]; idx += MC_VERT_THREADS) {                                         \
        const uint2 it = s_item[s_base[K] + idx];                     /* cell, E | own occurrences << 4 | local index << 8 */ \
        const int ci = (int)(it.x % (unsigned)p.g.ncx);                                                        \
        const unsigned t2 = it.x / (unsigned)p.g.ncx;                                                          \
        mc_create_interior_vertex<E>(p, (int)((it.y >> 4) & 15u), ci, (int)(t2 % (unsigned)p.g.ncy), p.g.k0 + (int)(t2 / (unsigned)p.g.ncy), \
                                     st, it.y >> 8, lo, hi, it.x, s_quick, s_occ);                             \
    }
    MC_KIND(0, 5) MC_KIND(1, 6) MC_KIND(2, 10)
#undef MC_KIND
    for (unsigned idx = tid; idx < s_cnt[3]; idx += MC_VERT_THREADS) {
        const uint2 it = s_item[s_base[3] + idx];
        const unsigned loc = it.y >> 8;
        switch (it.y & 15u) {
#define MC_CASE(E) case E: mc_run_vertex_task<E>(p, it.x, st, loc, lo, hi); break;
        MC_CASE(0) MC_CASE(1) MC_CASE(2) MC_CASE(3) MC_CASE(4) MC_CASE(7) MC_CASE(8) MC_CASE(9) MC_CASE(11) MC_CASE(12)
#undef MC_CASE
        default: break;
        }
    }
    // AABB: warp min/max, then one atomic per warp and component
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const unsigned l = __reduce_min_sync(FULL, lo[a]), h = __reduce_max_sync(FULL, hi[a]);
        if ((threadIdx.x & 31u) == 0) {
            if (l != 0xFFFFFFFFu) atomicMin(p.aabb_keys + a, l);
            if (h != 0u) atomicMax(p.aabb_keys + 3 + a, h);
        }
    }
}

cudaError_t mc_launch_emit(const McEmitParams& p, cudaStream_t s)
{
    const unsigned n = p.rec_end - p.rec_begin;
    if (n == 0) return cudaSuccess;
    mc_emit_tris_kernel<<<(n + MC_EMIT_THREADS - 1u) / MC_EMIT_THREADS, MC_EMIT_THREADS, 0, s>>>(p);
    cudaError_t e = cudaGetLastError();
    const unsigned nv = p.vert_end - p.vert_begin;
    if (e != cudaSuccess || nv == 0) return e;
    mc_emit_verts_kernel<<<(nv + MC_VERT_PER_BLOCK - 1u) / MC_VERT_PER_BLOCK, MC_VERT_THREADS, 0, s>>>(p);
    return cudaGetLastError();
}

__global__ void mc_offset_ids_kernel(int* __restrict__ ids, size_t n, int delta)
{
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) ids[k] += delta;
}

cudaError_t mc_launch_offset_ids(int* ids, size_t n, int delta, cudaStream_t s)
{
    if (n == 0 || delta == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const size_t blocks = std::min<size_t>((n + 255) / 256, (size_t)sms * 8);
    mc_offset_ids_kernel<<<(unsigned)blocks, 256, 0, s>>>(ids, n, delta);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// A few words device -> mapped page-locked host memory, written by a kernel: the small read-backs between the stages
// must not queue behind a large mesh download in the device-to-host copy engine (cudaMemcpyAsync would).
// ---------------------------------------------------------------------------------------------------
__global__ void mc_readback_kernel(const unsigned* __restrict__ src, unsigned* __restrict__ dst, unsigned nwords)
{
    for (unsigned k = threadIdx.x; k < nwords; k += blockDim.x) dst[k] = src[k];
    __threadfence_system();
}

// (records, vertices, triangles) before chunk `idx` in visiting order, to mapped host memory: the record prefix is per
// chunk (base), the vertex / triangle prefixes per ACTIVE chunk (abase, indexed by the number of active chunks before idx)
__global__ void mc_boundary_kernel(const uint4* __restrict__ base, const uint4* __restrict__ abase, size_t idx, uint4* __restrict__ dst)
{
    const uint4 b = base[idx];
    const uint4 a = abase[b.y];
    *dst = make_uint4(b.x, a.y, a.z, 0u);
    __threadfence_system();
}

cudaError_t mc_launch_boundary(const uint4* base, const uint4* abase, size_t idx, void* dst_host_mapped, cudaStream_t s)
{
    mc_boundary_kernel<<<1, 1, 0, s>>>(base, abase, idx, (uint4*)dst_host_mapped);
    return cudaGetLastError();
}

cudaError_t mc_launch_readback(const void* src_dev, void* dst_host_mapped, unsigned nwords, cudaStream_t s)
{
    if (nwords == 0) return cudaSuccess;
    mc_readback_kernel<<<1, 32, 0, s>>>((const unsigned*)src_dev, (unsigned*)dst_host_mapped, nwords);
    return cudaGetLastError();
}

// (records, vertices, triangles) before the first chunk of every cell layer l = 0..nlayers-1, to mapped host memory
// (the slab planner reads per-layer triangle counts of its coarse probe pass from these)
__global__ void mc_layer_prefix_kernel(const uint4* __restrict__ base, const uint4* __restrict__ abase, size_t per_layer, unsigned nlayers,
                                       uint4* __restrict__ dst)
{
    for (unsigned l = blockIdx.x * blockDim.x + threadIdx.x; l < nlayers; l += gridDim.x * blockDim.x) {
        const uint4 b = base[per_layer * l];
        const uint4 a = abase[b.y];
        dst[l] = make_uint4(b.x, a.y, a.z, 0u);
    }
    __threadfence_system();
}

cudaError_t mc_launch_layer_prefixes(const uint4* base, const uint4* abase, size_t per_layer, unsigned nlayers, void* dst_host_mapped, cudaStream_t s)
{
    if (nlayers == 0) return cudaSuccess;
    mc_layer_prefix_kernel<<<1, 128, 0, s>>>(base, abase, per_layer, nlayers, (uint4*)dst_host_mapped);
    return cudaGetLastError();
}
