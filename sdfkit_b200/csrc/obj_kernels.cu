// obj_kernels.cu -- Mesh.WriteObj (Mesh.cs:66-97) on the device: the OBJ text of a mesh, byte for byte what the host writer
// prints, in three kernels.
//   obj_line_bytes_kernel  bytes of every line, summed per block of OBJ_LINES_PER_BLOCK lines
//   obj_scan_kernel        64-bit exclusive scan of the block sums (one CTA; the host reads the result once to cut chunks)
//   obj_format_kernel      the lines of a range of blocks at their offsets: each warp lays its 32 lines out in shared memory
//                          at the alignment of their destination and stores the span with 16-byte stores (bytes only at
//                          the two ends)
// The format pass recomputes the digits instead of reading them from the length pass: storing them would cost more memory
// traffic (~50 B per line written and read back) than the arithmetic, and both passes are far below the PCIe copy of the text.
#include "obj_kernels.cuh"
#include "obj_text.cuh"

#define OBJ_WARP_BUF (16 + 32 * OBJ_LINE_MAX)   // one warp's lines + the head alignment pad (a multiple of 16)

struct ObjLine {
    int kind;              // 0 "v", 1 "vn", 2 "f", -1 past the end
    int len;
    NetFloat f[3];
    ObjIndex ix[3];
};

__device__ __forceinline__ void line_decode(const ObjMesh& m, int64_t line, ObjLine& L)
{
    const int64_t nvn = m.nv + m.nn;
    if (line < nvn) {
        const bool vert = line < m.nv;
        const float* p = vert ? m.v + 3 * line : m.n + 3 * (line - m.nv);
        L.kind = vert ? 0 : 1;
        L.len = vert ? 5 : 6;                                        // "v " / "vn ", two spaces, '\n'
#pragma unroll
        for (int k = 0; k < 3; k++) {
            L.f[k] = net_float(__float_as_uint(p[k]));
            L.len += L.f[k].len;
        }
    } else if (line < nvn + m.nt) {
        const int32_t* p = m.t + 3 * (line - nvn);
        L.kind = 2;
        L.len = 11;                                                  // "f ", three "//", two spaces, '\n'
#pragma unroll
        for (int k = 0; k < 3; k++) {
            L.ix[k] = obj_index(p[k]);
            L.len += 2 * L.ix[k].len;
        }
    } else {
        L.kind = -1;
        L.len = 0;
    }
}

__device__ __forceinline__ void line_write(const ObjLine& L, char* p)
{
    if (L.kind == 2) {
        *p++ = 'f';
        *p++ = ' ';
#pragma unroll
        for (int k = 0; k < 3; k++) {
            p = obj_index_write(L.ix[k], p);
            *p++ = '/';
            *p++ = '/';
            p = obj_index_write(L.ix[k], p);
            *p++ = k < 2 ? ' ' : '\n';
        }
    } else {
        *p++ = 'v';
        if (L.kind == 1) *p++ = 'n';
        *p++ = ' ';
#pragma unroll
        for (int k = 0; k < 3; k++) {
            net_float_write(L.f[k], p);
            p += L.f[k].len;
            *p++ = k < 2 ? ' ' : '\n';
        }
    }
}

__global__ void __launch_bounds__(OBJ_LINES_PER_BLOCK) obj_line_bytes_kernel(ObjMesh m, uint32_t* __restrict__ block_bytes)
{
    __shared__ uint32_t wsum[OBJ_LINES_PER_BLOCK / 32];
    ObjLine L;
    line_decode(m, (int64_t)blockIdx.x * OBJ_LINES_PER_BLOCK + threadIdx.x, L);
    uint32_t s = (uint32_t)L.len;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < OBJ_LINES_PER_BLOCK / 32; w++) t += wsum[w];
        block_bytes[blockIdx.x] = t;
    }
}

// out[i] = sum of in[0 .. i), out[n] = the total; one CTA of 1024 threads, each scanning a contiguous run of the input
__global__ void __launch_bounds__(1024) obj_scan_kernel(const uint32_t* __restrict__ in, uint64_t* __restrict__ out, int64_t n)
{
    __shared__ uint64_t wsum[32];
    const int64_t per = (n + 1023) / 1024, beg = min(n, (int64_t)threadIdx.x * per), end = min(n, beg + per);
    uint64_t local = 0;
    for (int64_t i = beg; i < end; i++) local += in[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t x = local;
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = wsum[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        wsum[lane] = w;                                              // inclusive over warps
    }
    __syncthreads();
    uint64_t run = x - local + (warp > 0 ? wsum[warp - 1] : 0);
    for (int64_t i = beg; i < end; i++) { out[i] = run; run += in[i]; }
    if (threadIdx.x == 0) out[n] = wsum[31];
}

__global__ void __launch_bounds__(OBJ_LINES_PER_BLOCK) obj_format_kernel(ObjMesh m, const uint64_t* __restrict__ block_off, int64_t b0,
                                                                           uint64_t base, char* __restrict__ out)
{
    __shared__ __align__(16) char buf[OBJ_LINES_PER_BLOCK / 32][OBJ_WARP_BUF];
    __shared__ uint32_t wsum[OBJ_LINES_PER_BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b = b0 + blockIdx.x;
    ObjLine L;
    line_decode(m, b * OBJ_LINES_PER_BLOCK + threadIdx.x, L);

    uint32_t incl = (uint32_t)L.len;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    const uint32_t wtot = __shfl_sync(0xffffffffu, incl, 31);
    if (lane == 31) wsum[warp] = wtot;
    __syncthreads();
    uint32_t wbase = 0;
    for (int w = 0; w < warp; w++) wbase += wsum[w];

    // the warp's lines occupy [d0, d1) of the chunk; in shared memory they start at d0 % 16 so that the 16-byte-aligned
    // part of the destination maps to 16-byte-aligned shared words
    const uint64_t d0 = block_off[b] - base + wbase, d1 = d0 + wtot;
    const int pad = (int)(d0 & 15);
    char* s = buf[warp];
    if (L.len) line_write(L, s + pad + (incl - L.len));
    __syncwarp();
    const uint64_t a0 = (d0 + 15) & ~(uint64_t)15, a1 = d1 & ~(uint64_t)15;
    if (a0 >= a1) {
        for (uint32_t i = lane; i < wtot; i += 32) out[d0 + i] = s[pad + i];
    } else {
        if (lane < (int)(a0 - d0)) out[d0 + lane] = s[pad + lane];
        if (lane < (int)(d1 - a1)) out[a1 + lane] = s[pad + (a1 - d0) + lane];
        const uint4* src = reinterpret_cast<const uint4*>(s + pad + (a0 - d0));
        uint4* dst = reinterpret_cast<uint4*>(out + a0);
        for (int v = lane; v < (int)((a1 - a0) >> 4); v += 32) dst[v] = src[v];
    }
}

// one warp per 2^20 bit patterns: the lanes format 32 consecutive floats, lane 0 hashes their text in order
__global__ void __launch_bounds__(256) obj_selftest_kernel(uint32_t first, uint32_t nblocks, uint64_t* __restrict__ digests)
{
    __shared__ char txt[8][32][16];
    __shared__ int len[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t w = blockIdx.x * 8 + warp;
    if (w >= nblocks) return;
    const uint32_t base = (first + w) << 20;
    uint64_t h = 14695981039346656037ull;
    for (uint32_t it = 0; it < (1u << 15); it++) {
        const NetFloat f = net_float(base + it * 32 + lane);
        net_float_write(f, txt[warp][lane]);
        txt[warp][lane][f.len] = '\n';
        len[warp][lane] = f.len + 1;
        __syncwarp();
        if (lane == 0)
            for (int j = 0; j < 32; j++)
                for (int k = 0; k < len[warp][j]; k++) { h ^= (unsigned char)txt[warp][j][k]; h *= 1099511628211ull; }
        __syncwarp();
    }
    if (lane == 0) digests[w] = h;
}

cudaError_t obj_offsets(const ObjMesh& m, uint32_t* block_bytes, uint64_t* block_off, cudaStream_t s)
{
    const int64_t nb = obj_line_blocks(m);
    if (nb > 0x7fffffff) return cudaErrorInvalidValue;
    if (nb > 0) obj_line_bytes_kernel<<<(unsigned)nb, OBJ_LINES_PER_BLOCK, 0, s>>>(m, block_bytes);
    obj_scan_kernel<<<1, 1024, 0, s>>>(block_bytes, block_off, nb);
    return cudaGetLastError();
}

cudaError_t obj_format(const ObjMesh& m, const uint64_t* block_off, int64_t b0, int64_t b1, uint64_t base, char* out, cudaStream_t s)
{
    if (b1 <= b0) return cudaSuccess;
    obj_format_kernel<<<(unsigned)(b1 - b0), OBJ_LINES_PER_BLOCK, 0, s>>>(m, block_off, b0, base, out);
    return cudaGetLastError();
}

cudaError_t obj_selftest(uint32_t first, uint32_t nblocks, uint64_t* digests, cudaStream_t s)
{
    if (nblocks == 0) return cudaSuccess;
    obj_selftest_kernel<<<(nblocks + 7) / 8, 256, 0, s>>>(first, nblocks, digests);
    return cudaGetLastError();
}
