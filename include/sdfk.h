/* sdfk.h -- C ABI of libsdfk.so: the B200-native replacement for SdfKit's data-parallel hot path.
 *
 * The reference (praeclarum/SdfKit, pure C#) has no FFI; the seam it offers is managed: the `Sdf`
 * delegate produced by SdfExprEx.ToSdf and consumed by Voxels.SampleSdf / SdfEx.ToVoxels / ToMesh /
 * ToImage / RayMarcher, plus the data-only entry MarchingCubes.CreateMesh(Voxels,...).  These are the
 * entry points a P/Invoke shim binds to put the GPU behind that seam (INTEGRATION.md shows the C# side).
 * Each function cites the reference interface it replaces (paths relative to the SdfKit repository).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on failure; sdfk_last_error() returns the message of the
 *     last failure on the calling thread.  No C++ exception crosses this boundary.
 *   - the caller owns every host buffer it passes; the library never keeps a host pointer after return.
 *   - handles are released only by their *_destroy function.
 *   - all entry points taking a ctx are serialised per ctx (internal mutex).  sdfk_ctx_create drives one GPU;
 *     sdfk_ctx_create_multi drives N GPUs from one process: sampling / meshing shard by z-slab, rendering by row band,
 *     behind the same entry points (see "multi-GPU" below and DESIGN.md section 5).
 *   - matrices are 16 floats, row-major System.Numerics.Matrix4x4 (M11 M12 M13 M14 M21 ...), row-vector
 *     convention; the caller computes them (the C# shim with System.Numerics itself).
 *   - device layout of voxels is x-fastest; the C# `[x,y,z]` layout appears only in import/export.
 */
#ifndef SDFK_H
#define SDFK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDFK_OK 0
#define SDFK_ERR_INVALID (-1)      /* bad argument */
#define SDFK_ERR_CUDA (-2)         /* CUDA runtime / driver failure */
#define SDFK_ERR_COMPILE (-3)      /* NVRTC rejected the SDF source (the log is in sdfk_last_error) */
#define SDFK_ERR_UNSUPPORTED (-4)  /* e.g. an opaque (non-SdfExpr) SDF, grid too large for 32-bit cell ids */
#define SDFK_ERR_INTERNAL (-5)

typedef struct sdfk_ctx sdfk_ctx;
typedef struct sdfk_sdf sdfk_sdf;
typedef struct sdfk_voxels sdfk_voxels;
typedef struct sdfk_mesh sdfk_mesh;

/* IProgress<float>.Report (MarchingCubes.cs:81): called on the calling thread with z/nz_bound per layer. */
typedef void (*sdfk_progress_fn)(float fraction, void* user);

const char* sdfk_last_error(void);
int sdfk_version(void);

/* ---- context: one GPU, one stream --------------------------------------------------------------- */
int sdfk_ctx_create(int device, sdfk_ctx** out);
/* same, launching on a caller-owned cudaStream_t (e.g. the host framework's current stream) */
int sdfk_ctx_create_on_stream(int device, void* cuda_stream, sdfk_ctx** out);
/* ---- multi-GPU context: N devices of one box behind ONE handle (SURVEY.md section 8b/8e) -------------------------
 * devices = NULL means 0..ndev-1; a device may be listed more than once (every entry gets its own stream, pools and
 * worker thread -- used by the single-GPU tests of this layer).  On such a context
 *   sdfk_sdf_compile        loads the module on every device;
 *   sdfk_voxels_sample      returns voxels SHARDED by z-slab (cost-balanced cuts, one halo slice per side, recomputed
 *                           rather than exchanged); sdfk_voxels_resample / _clip / _export / _destroy understand them;
 *   sdfk_mesh_create        on sharded voxels (step 1) classifies every slab on its device, exchanges the per-slab
 *                           (vertices, triangles) counts in host memory and emits at global ids: a device-resident mesh
 *                           in one part per device; sdfk_mesh_counts / _export / _stats / _destroy understand it,
 *                           sdfk_mesh_export moves every part over its own PCIe link;
 *   sdfk_sdf_to_mesh_host   (SdfEx.ToMesh, Sdf.cs:59-63) lands ONE host mesh, every device copying its share to its
 *                           global offset;
 *   sdfk_render*            render row bands (RayMarcher.cs:50-61), one per device, into the one host image;
 *   the timers / marks      report the slowest device, sdfk_ctx_launch_count the sum.
 * Slab-level calls (sdfk_voxels_sample_slab / _distances, sdfk_mesh_classify / _emit, sdfk_voxels_import, sdfk_sdf_eval)
 * run on device 0 of the context.  The results are identical, bit for bit and in order, to a single-GPU context's. */
int sdfk_ctx_create_multi(int ndev, const int* devices, sdfk_ctx** out);
int sdfk_ctx_device_count(sdfk_ctx* ctx, int* ndev);
/* host wall clock (ms) of the last multi-GPU call on this context, from entry until every device had finished */
int sdfk_ctx_last_wall_ms(sdfk_ctx* ctx, double* milliseconds);
/* The z-slab plan: cuts the cell layers of an nx*ny*nz grid (MarchingCubes.cs:49-68) into `parts` contiguous ranges of
 * near-equal cost = voxels + active_cell_cost * active cells, the active cells estimated by a coarse (<= 128^3) meshing
 * pass of the same SDF (0 = default cost).  kb_ke receives 2*parts ints: [kb, ke) per part.  Deterministic. */
int sdfk_plan_layers(sdfk_ctx* ctx, sdfk_sdf* sdf, const float min[3], const float max[3], int nx, int ny, int nz, int step,
                     int clip, int parts, double active_cell_cost, int* kb_ke);
int sdfk_ctx_destroy(sdfk_ctx* ctx);
int sdfk_ctx_synchronize(sdfk_ctx* ctx);
int sdfk_ctx_stream(sdfk_ctx* ctx, void** cuda_stream);
/* CUDA-event stopwatch on the ctx stream (device time between the two calls) */
int sdfk_ctx_timer_start(sdfk_ctx* ctx);
int sdfk_ctx_timer_stop(sdfk_ctx* ctx, float* milliseconds);
/* event marks on the ctx stream: record mark `slot` (0..63) without synchronising; elapsed = device ms between
 * two recorded marks (synchronises on the later one) */
int sdfk_ctx_mark(sdfk_ctx* ctx, int slot);
int sdfk_ctx_elapsed(sdfk_ctx* ctx, int slot_a, int slot_b, float* milliseconds);
/* how many kernels this ctx has launched so far */
int sdfk_ctx_launch_count(sdfk_ctx* ctx, int64_t* launches);
/* tuning switches (results never depend on them).  SDFK_OPT_SIGN_PLANES (default 1): the sampling kernels also write
 * 1 sign bit per voxel (value > 0), from which marching cubes at iso 0 / step 1 finds the active cells without
 * re-reading the distances; 0 = always classify from the distances. */
#define SDFK_OPT_SIGN_PLANES 1
int sdfk_ctx_set_option(sdfk_ctx* ctx, int option, int value);

/* Measurement aid: the rate (GB/s) at which a store-only kernel -- one CTA per 16 KiB in memory order, the order the sampling
 * kernels hand their work out in -- fills `bytes` of device memory on device 0 of the context (best of `reps` runs, CUDA events).
 * The ceiling of Voxels.SampleSdf (SdfKit/Voxels.cs:72-125), which writes 16 B per voxel and reads nothing; a copy (the usual
 * "HBM bandwidth" figure) is slower than a pure store stream on B200. */
int sdfk_ctx_store_bandwidth(sdfk_ctx* ctx, size_t bytes, int reps, double* gb_per_s);

/* page-locked host buffers: results exported into them travel at full PCIe speed (a pageable destination is staged
 * by the driver at a fraction of it).  Optional -- every export accepts any host pointer. */
int sdfk_host_alloc(size_t bytes, void** out);
int sdfk_host_free(void* p);

/* ---- SdfExpr.ToSdf(): SdfExprCompiler.Compile (SdfExpr.cs:208-211,234-271) ------------------------
 * body = statements of `sk_float4 sdf_eval(sk_float3 p)` in the SDF source dialect (csrc/sdfk_prelude.h),
 * produced by lowering the expression tree.  NVRTC-compiled for sm_100a without FMA contraction.       */
int sdfk_sdf_compile(sdfk_ctx* ctx, const char* body, size_t len, sdfk_sdf** out);
int sdfk_sdf_destroy(sdfk_sdf* sdf);
/* NVRTC-compile only (needs no GPU): validates a body and reports the cubin size. */
int sdfk_sdf_check(const char* body, size_t len, size_t* cubin_bytes);
/* The packed (two points per instruction, add/mul/fma.rn.f32x2) form of an SDF body may divide by a constant with a
 * 3-instruction correctly rounded sequence instead of the generic IEEE division.  Before emitting it for a constant the
 * host side asks the device to compare it with div.rn.f32 for ALL 2^32 dividends (a few ms, cached by the caller);
 * mismatches != 0 means: keep the generic division for this constant.  sdfk_selftest_sqrt does the same for the packed
 * square root (all 2^32 arguments against sqrt.rn.f32). */
int sdfk_constdiv_verify(sdfk_ctx* ctx, float divisor, int64_t* mismatches);
int sdfk_selftest_sqrt(sdfk_ctx* ctx, int64_t* mismatches);
/* the Sdf delegate itself (Sdf.cs:8): rgbd[i] = sdf(xyz[i]); host pointers, n*3 floats in, n*4 out */
int sdfk_sdf_eval(sdfk_sdf* sdf, const float* xyz, float* rgbd, int64_t n);

/* ---- Voxels (Voxels.cs) ---------------------------------------------------------------------------
 * SdfEx.ToVoxels / Voxels.SampleSdf (+ ClipToBounds when clip != 0) (Sdf.cs:49-57, Voxels.cs:72-167).
 * Asynchronous on the ctx stream; the voxels stay resident in HBM.                                     */
int sdfk_voxels_sample(sdfk_ctx* ctx, sdfk_sdf* sdf, const float min[3], const float max[3],
                       int nx, int ny, int nz, int clip, sdfk_voxels** out);
/* one z-slab [z_begin, z_end) of the same nx*ny*nz grid (multi-GPU sharding; halo slices are resampled) */
int sdfk_voxels_sample_slab(sdfk_ctx* ctx, sdfk_sdf* sdf, const float min[3], const float max[3],
                            int nx, int ny, int nz, int clip, int z_begin, int z_end, sdfk_voxels** out);
/* Distance-only voxels for meshing (SdfEx.ToMesh, Sdf.cs:59-63, where the caller never sees the voxels): 4 B/voxel
 * instead of 16.  Values are identical to sdfk_voxels_sample_slab's; the colours marching cubes needs are evaluated at
 * the created vertices by a second JIT kernel, with identical results.  `sdf` must stay alive while these voxels are
 * meshed; exporting Colors from them is SDFK_ERR_UNSUPPORTED. */
int sdfk_voxels_sample_distances(sdfk_ctx* ctx, sdfk_sdf* sdf, const float min[3], const float max[3],
                                 int nx, int ny, int nz, int clip, int z_begin, int z_end, sdfk_voxels** out);
/* re-sample into an existing voxels object (same grid; no allocation) -- the steady-state hot call */
int sdfk_voxels_resample(sdfk_voxels* vox, sdfk_sdf* sdf, int clip);
/* new Voxels(values, colors, min, max) (Voxels.cs:23-35): host arrays in C# layout
 * values[nx][ny][nz], colors[nx][ny][nz][3] (colors may be NULL = zeros)                                */
int sdfk_voxels_import(sdfk_ctx* ctx, const float* values, const float* colors, const float min[3],
                       const float max[3], int nx, int ny, int nz, sdfk_voxels** out);
/* Voxels.Values / Voxels.Colors (Voxels.cs:8-9) in C# layout; either pointer may be NULL.  For a slab the
 * arrays are [nx][ny][z_end - z_begin].  The field leaves in x-chunks: a chunk is transposed to the C# layout on the
 * device while the previous one crosses PCIe (page-locked destinations -- sdfk_host_alloc -- travel at link speed).   */
int sdfk_voxels_export(sdfk_voxels* vox, float* values, float* colors);
/* Voxels.ClipToBounds (Voxels.cs:133-167) on resident voxels */
int sdfk_voxels_clip(sdfk_voxels* vox);
/* dims = {nx, ny, nz, z_begin, z_end}; device pointers to the x-fastest arrays (dist, rgb) */
int sdfk_voxels_info(sdfk_voxels* vox, int dims[5], void** dist_dev, void** rgb_dev);
/* sharded voxels (multi-GPU context): the cell layers [kb, ke) every device owns (2 ints per part), and the per-device
 * slab handle (borrowed; NULL for a device that owns nothing) */
int sdfk_voxels_layers(sdfk_voxels* vox, int* kb_ke, int max_parts, int* nparts);
int sdfk_voxels_part(sdfk_voxels* vox, int part, sdfk_voxels** out);
int sdfk_voxels_destroy(sdfk_voxels* vox);

/* ---- MarchingCubes.CreateMesh / Voxels.ToMesh (MarchingCubes.cs:39-92, Voxels.cs:67-70) -------------
 * transform / normal_transform: the matrices Mesh.Transform applies (MarchingCubes.cs:85-90, Mesh.cs:47-64),
 * computed by the caller; both NULL leaves the mesh in voxel-index space.
 * Any grid whose voxels fit in device memory is meshed: a grid with more cells or 128-cell chunks than one meshing job's
 * 32-bit ids hold (from ~1626^3 on) is meshed in consecutive sub-slabs of cell layers, one after the other, into ONE mesh
 * (the same arrays, handle and results as a one-job mesh).  The same holds per device on a multi-GPU context. */
int sdfk_mesh_create(sdfk_ctx* ctx, sdfk_voxels* vox, float iso, int step, const float transform[16],
                     const float normal_transform[16], sdfk_progress_fn progress, void* user, sdfk_mesh** out);
/* Slab meshing for multi-GPU jobs, in two phases around the caller's all-gather of counts:
 *   sdfk_mesh_classify: classify + scan the cell layers of this slab that lie in [k_begin, k_end) (global
 *                       cell-layer range this rank owns); reports how many vertices / triangles it owns.
 *                       One call is one meshing job: fewer than 2^32 cells and 128-cell chunks in the classified layers
 *                       (ghost layers included), else SDFK_ERR_UNSUPPORTED -- split the range over several calls.
 *   sdfk_mesh_emit:     write the owned vertices / triangles with global ids starting at vertex_base /
 *                       triangle_base (exclusive sums of the lower ranks' counts).                      */
int sdfk_mesh_classify(sdfk_ctx* ctx, sdfk_voxels* vox, float iso, int step, int k_begin, int k_end,
                       sdfk_mesh** out, int64_t* nverts, int64_t* ntris);
int sdfk_mesh_emit(sdfk_mesh* mesh, int64_t vertex_base, int64_t triangle_base, const float transform[16],
                   const float normal_transform[16]);
/* sdfk_mesh_emit with the result delivered to HOST memory: the owned cell layers are emitted in `nchunks` sub-ranges
 * (0 = automatic) and every finished part streams to page-locked host memory (owned by the mesh handle, see
 * sdfk_mesh_host_ptrs) on a copy stream while the next sub-range is computed -- in a multi-GPU job every rank moves its
 * share of the mesh over its own PCIe link.  Returns when the arrays are complete. */
int sdfk_mesh_emit_host(sdfk_mesh* mesh, int64_t vertex_base, int64_t triangle_base, const float transform[16],
                        const float normal_transform[16], int nchunks);
int sdfk_mesh_counts(sdfk_mesh* mesh, int64_t* nverts, int64_t* ntris);
/* SdfEx.ToMesh (Sdf.cs:59-63) in one call, with the mesh delivered to HOST memory.  The grid is cut into z-slabs
 * (nslabs; 0 = automatic: ~128 cell layers each, at most 16; a slab with a lot of surface is emitted in sub-ranges); each slab is sampled (distance-only voxels + sign blocks), classified,
 * compacted and emitted at its global vertex / triangle offsets, and its part of the mesh streams to page-locked host
 * memory on a copy stream while the following slabs are computed.  The result is identical, bit for bit and in order,
 * to sdfk_voxels_sample + sdfk_mesh_create + sdfk_mesh_export.  The arrays live in page-locked memory owned by the mesh
 * handle (recycled through the ctx) until sdfk_mesh_destroy; sdfk_mesh_export on such a mesh is a host memcpy.
 * progress is called on the calling thread, per cell layer, as slabs complete. */
int sdfk_sdf_to_mesh_host(sdfk_ctx* ctx, sdfk_sdf* sdf, const float min[3], const float max[3], int nx, int ny, int nz, int clip,
                          float iso, int step, const float transform[16], const float normal_transform[16], int nslabs,
                          sdfk_progress_fn progress, void* user, sdfk_mesh** out);
int sdfk_mesh_host_ptrs(sdfk_mesh* mesh, const float** vertices, const float** colors, const float** normals,
                        const int32_t** triangles);
/* Mesh.Vertices/Colors/Normals/Triangles + Min/Max (Mesh.cs:10-18): any pointer may be NULL.
 * aabb = {min.x, min.y, min.z, max.x, max.y, max.z}                                                     */
int sdfk_mesh_export(sdfk_mesh* mesh, float* vertices, float* colors, float* normals, int32_t* triangles,
                     float aabb[6]);
int sdfk_mesh_device_ptrs(sdfk_mesh* mesh, void** vertices, void** colors, void** normals, void** triangles);
/* sharded mesh (multi-GPU context): part r (borrowed handle on device r; NULL if empty) and the global index of its first
 * vertex / triangle */
int sdfk_mesh_part(sdfk_mesh* mesh, int part, sdfk_mesh** out, int64_t* vertex_base, int64_t* triangle_base);
/* stats[0..3] = device ms of classify, scan, compact, emit; stats[4] = active cells; stats[7] = 1 if classified from sign planes */
int sdfk_mesh_stats(sdfk_mesh* mesh, double stats[8]);
int sdfk_mesh_destroy(sdfk_mesh* mesh);

/* ---- Mesh.WriteObj (Mesh.cs:66-97) -----------------------------------------------------------------
 * The OBJ text of host arrays -- "v x y z" per vertex, "vn x y z" per normal, "f a//a b//b c//c" per triangle (indices
 * triangles[k] + 1 in 32-bit two's complement, as the reference's
 * int arithmetic wraps), '\n' line ends, floats as .NET Core float.ToString() prints them -- formatted on device 0
 * of the context and handed to `sink` in file order, in chunks, on the calling thread.  nnormals may differ from nvertices;
 * nindices must be a multiple of 3; an empty mesh makes no sink call.  sink returns 0 to continue; anything else stops the
 * call (SDFK_ERR_INVALID, the sink's value in the message).  The sink must not call into the same ctx.  bytes_written (may
 * be NULL) receives the bytes the sink accepted.  The streams are idle again when the call returns, whatever the result. */
typedef int (*sdfk_write_fn)(const void* bytes, size_t n, void* user);
int sdfk_obj_write(sdfk_ctx* ctx, const float* vertices, int64_t nvertices, const float* normals, int64_t nnormals,
                   const int32_t* triangles, int64_t nindices, sdfk_write_fn sink, void* user, int64_t* bytes_written);
/* digests[i] = FNV-1a-64 of the .NET text (+ '\n') of every float with bit pattern in block first_block + i (2^20 each,
 * in increasing order); first_block + nblocks <= 4096 */
int sdfk_selftest_float_text(sdfk_ctx* ctx, uint32_t first_block, uint32_t nblocks, uint64_t* digests);

/* ---- RayMarcher (RayMarcher.cs) ---------------------------------------------------------------------
 * cam_pos = translation of inverse(ViewTransform); inv_view_proj = inverse(ViewTransform * projection)
 * (RayMarcher.cs:95-108) -- computed by the caller.  rows [row_begin, row_end) of the w*h image are
 * rendered into rgb (host, (row_end-row_begin)*w*3 floats) -- the reference's row bands (RayMarcher.cs:50-61). */
int sdfk_render(sdfk_ctx* ctx, sdfk_sdf* sdf, int w, int h, const float cam_pos[3], const float inv_view_proj[16],
                float near_plane, float far_plane, int iterations, int row_begin, int row_end, float* rgb);
/* RayMarcher.RenderDepth (RayMarcher.cs:69-93): depth host buffer of (row_end-row_begin)*w floats */
int sdfk_render_depth(sdfk_ctx* ctx, sdfk_sdf* sdf, int w, int h, const float cam_pos[3],
                      const float inv_view_proj[16], float near_plane, int iterations, int row_begin, int row_end,
                      float* depth);
/* RayMarcher.Render followed by Vec3Data.SaveTga's pixel conversion (VectorData.cs:570-619) on the device: the rows come back
 * as the TGA payload -- 3 bytes per pixel in B, G, R order, (byte)(v * 255) with clamping -- a quarter of the float image. */
int sdfk_render_bgr8(sdfk_ctx* ctx, sdfk_sdf* sdf, int w, int h, const float cam_pos[3], const float inv_view_proj[16],
                     float near_plane, float far_plane, int iterations, int row_begin, int row_end, unsigned char* bgr);
/* RayMarcher.RenderDepth followed by FloatData.SaveDepthTga's pixel conversion (VectorData.cs:244-276) on the device: the rows
 * come back as the TGA payload, one byte per pixel: v >= tga_far -> 0, v <= tga_near -> 255, else
 * (byte)(255.0f * (tga_far - v) / (tga_far - tga_near)).  march_near = RayMarcher.NearPlaneDistance. */
int sdfk_render_depth_gray8(sdfk_ctx* ctx, sdfk_sdf* sdf, int w, int h, const float cam_pos[3], const float inv_view_proj[16],
                            float march_near, int iterations, float tga_near, float tga_far, int row_begin, int row_end,
                            unsigned char* gray);
/* same kernels writing to device memory, asynchronous on the ctx stream */
int sdfk_render_device(sdfk_ctx* ctx, sdfk_sdf* sdf, int w, int h, const float cam_pos[3],
                       const float inv_view_proj[16], float near_plane, float far_plane, int iterations,
                       int row_begin, int row_end, void* rgb_dev);

#ifdef __cplusplus
}
#endif
#endif /* SDFK_H */
