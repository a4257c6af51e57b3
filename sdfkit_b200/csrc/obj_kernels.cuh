// obj_kernels.cuh -- Mesh.WriteObj (Mesh.cs:66-97) on the device: launchers of the kernels in obj_kernels.cu.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define OBJ_LINES_PER_BLOCK 256   // lines per CTA of the length and format passes (one per thread); the unit of chunking

// the mesh on the device; the file's lines are nv "v", then nn "vn", then nt "f" lines
struct ObjMesh {
    const float* v;
    const float* n;
    const int32_t* t;
    int64_t nv, nn, nt;
};

inline int64_t obj_lines(const ObjMesh& m) { return m.nv + m.nn + m.nt; }
inline int64_t obj_line_blocks(const ObjMesh& m) { return (obj_lines(m) + OBJ_LINES_PER_BLOCK - 1) / OBJ_LINES_PER_BLOCK; }

// block_off[b] = bytes of the text before line block b (b = 0 .. obj_line_blocks), the last entry is the total.
// block_bytes: obj_line_blocks(m) words of scratch.
cudaError_t obj_offsets(const ObjMesh& m, uint32_t* block_bytes, uint64_t* block_off, cudaStream_t s);
// the text of line blocks [b0, b1) at out[block_off[b] - base ...]; base = block_off[b0] (the host has read the offsets)
cudaError_t obj_format(const ObjMesh& m, const uint64_t* block_off, int64_t b0, int64_t b1, uint64_t base, char* out, cudaStream_t s);
// digests[i] = FNV-1a-64 of the text + '\n' of every float with bit pattern in [(first + i) << 20, (first + i + 1) << 20)
cudaError_t obj_selftest(uint32_t first, uint32_t nblocks, uint64_t* digests, cudaStream_t s);
