// mc_kernels.cuh -- shared declarations of the marching-cubes stage (host + device).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

// Geometry of one meshing job (a whole grid, or one z-slab of it).  Voxel layout: x fastest,
// dist[(zl*ny + y)*nx + x], rgb[...*3]; zl = z - z0 (DESIGN.md "data layout").
struct McGrid {
    int nx, ny;            // voxel dims in x, y (never partitioned)
    int nzl;               // slices held locally
    int z0;                // global z of local slice 0
    int nz;                // global slice count
    int step;              // MarchingCubes step (MarchingCubes.cs:49-68)
    int ncx, ncy, ncz;     // GLOBAL cell counts per axis: cells at x = i*step, i < ncx
    int k0;                // first GLOBAL cell layer classified locally
    int nk;                // number of cell layers classified locally (incl. ghost layers)
    int kown0, kown1;      // GLOBAL cell layers [kown0, kown1) this slab emits
    int cpr;               // 128-cell chunks per cell row = ceil(ncx/128)
    float iso;
    unsigned nchunks;      // nk * ncy * cpr
};

// One record per active cell, in the reference's visiting order (z outer, y, x inner).
struct __align__(32) McRecord {
    unsigned cell;         // local linear cell id: i + ncx*(j + ncy*(k - k0))
    unsigned info;         // leaf: tiling row id [0:10) | ntris [10:14) | uses centre vertex [14]
    unsigned vbase;        // created vertices before this cell INSIDE ITS CHUNK (+ base[chunk].y = slab-local prefix)
    unsigned tbase;        // triangles before this cell inside its chunk (+ base[chunk].z)
    unsigned long long aux;   // what neighbours ask of this cell, so that a lookup is one 32-byte read:
                              //   [0:16)  creation rank of slots 5, 6, 10, 12 (4 bits each) -> vertex id = vbase + rank
                              //   [16:52) how often the row references edge e = 0..11 (3 bits each)
    unsigned long long pad;
};
#define MC_AUX_RANK(aux, q) ((unsigned)((aux) >> (4 * (q))) & 0xFu)           /* q: 0 -> e5, 1 -> e6, 2 -> e10, 3 -> centre */
#define MC_AUX_OCC(aux, e) ((unsigned)((aux) >> (16 + 3 * (e))) & 0x7u)

// per-chunk packed counts: nactive [0:8) | nverts [8:19) | ntris [19:30)
#define MC_CNT_ACT(c) ((c) & 0xFFu)
#define MC_CNT_V(c) (((c) >> 8) & 0x7FFu)
#define MC_CNT_T(c) (((c) >> 19) & 0x7FFu)
#define MC_CNT_PACK(a, v, t) ((unsigned)(a) | ((unsigned)(v) << 8) | ((unsigned)(t) << 19))
/* what the classifiers write: n active cells, and 1 in the vertex field of an active chunk -- the first scan then yields, per
 * chunk, its first record slot (x) and its rank among the ACTIVE chunks (y), which indexes the second, much shorter scan */
#define MC_CNT_FIRST(n) ((n) ? ((unsigned)(n) | 0x100u) : 0u)

struct McTotals {          // written by the scan
    unsigned long long nact, nverts, ntris;
};

struct McEmitParams {
    McGrid g;
    const float* dist;
    const float* rgb;
    const unsigned* counts;        // per chunk packed counts
    const uint4* base;             // per chunk (first scan): x = records before it, y = ACTIVE chunks before it, w = packed counts
    const uint4* abase;            // per active chunk (second scan): y = vertices, z = triangles before it
    const McRecord* recs;
    const uint4* masks;            // per active chunk: 128-bit activity mask, bit q <-> cell q of the chunk
    unsigned rec_begin, rec_end;   // records emitted by this slab (owned layers)
    unsigned vlocal0, tlocal0;     // slab-local prefix at the first owned layer
    long long vglobal0, tglobal0;  // global ids of the slab's first owned vertex / triangle
    float* verts;                  // outputs, indexed by (id - vglobal0) / (tri - tglobal0)
    float* cols;
    float* nrms;
    int* tris;
    uint2* recipes;                // distance-only voxels (rgb == NULL): per vertex (cell, edge) for the deferred colours
    uint2* tasks;                  // per vertex slot, tris kernel -> verts kernel: (record, slot E) of the cell that creates it; for
                                   // slots 5, 6, 10: (cell id, E | the cell's own reference count of the edge << 4)
    unsigned vert_begin, vert_end; // slab-local vertex slots created by records [rec_begin, rec_end)
    unsigned* aabb_keys;           // 6 ordered-uint keys: min xyz, max xyz
    int has_xf;
    float M[16];                   // Mesh.Transform matrix (row-major, row-vector convention)
    float N[16];                   // its normal transform
    int* error_flag;
};

// The vector path of mc_classify reads up to MC_PAD_ROWS voxel rows (+ a few floats) past the rows it needs;
// voxel arrays are allocated with that much padding so those loads need no clamping.
#define MC_PAD_ROWS 10

// host-side launchers (mc_kernels.cu)
cudaError_t mc_init_tables();
cudaError_t mc_launch_classify(const McGrid& g, const float* dist, unsigned* counts, uint4* masks, cudaStream_t s);
// same outputs from the sign planes written by the sampling kernels (step == 1): no pass over the distance field
cudaError_t mc_launch_classify_signs(const McGrid& g, const uint4* signs, unsigned tiles_per_row, unsigned nzg, unsigned* counts,
                                     uint4* masks, cudaStream_t s);
// base[i] is written only for items with a non-zero count and at multiples of write_every (1 = everywhere);
// alist (optional, first scan): alist[rank among the non-empty items] = item, i.e. the list of active chunks
cudaError_t mc_launch_scan(const unsigned* counts, uint4* base, unsigned nchunks, void* scan_ws, size_t ws_bytes,
                           McTotals* totals, unsigned write_every, unsigned* alist, cudaStream_t s);
size_t mc_scan_workspace_bytes(unsigned nchunks);
// visits the nactive active chunks listed in alist (by rank)
cudaError_t mc_launch_compact(const McGrid& g, const float* dist, const unsigned* alist, unsigned nactive, const uint4* base,
                              McRecord* recs, const uint4* masks, unsigned* acounts, cudaStream_t s);
cudaError_t mc_launch_boundary(const uint4* base, const uint4* abase, size_t idx, void* dst_host_mapped, cudaStream_t s);
// the same prefixes at the first chunk of each of nlayers cell layers (per_layer chunks apart): nlayers uint4 to mapped host memory
cudaError_t mc_launch_layer_prefixes(const uint4* base, const uint4* abase, size_t per_layer, unsigned nlayers, void* dst_host_mapped, cudaStream_t s);
cudaError_t mc_launch_emit(const McEmitParams& p, cudaStream_t s);
// ids[k] += delta for k < n: the triangles of a mesh part emitted with vertex ids from 0 moved to its global vertex base
cudaError_t mc_launch_offset_ids(int* ids, size_t n, int delta, cudaStream_t s);
// nwords 32-bit words from device memory to MAPPED page-locked host memory, by a kernel (no copy engine involved)
cudaError_t mc_launch_readback(const void* src_dev, void* dst_host_mapped, unsigned nwords, cudaStream_t s);
