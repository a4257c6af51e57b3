// Native.cs -- P/Invoke declarations for libsdfk.so (include/sdfk.h).  SOURCE ONLY: this image has no .NET
// toolchain, so this shim is not compiled or tested here; the Python mirror (sdfkit_b200/) exercises the same ABI.
using System;
using System.Runtime.InteropServices;

namespace SdfKit.B200
{
    internal static unsafe class Native
    {
        const string Lib = "sdfk";   // libsdfk.so

        [UnmanagedFunctionPointer(CallingConvention.Cdecl)]
        public delegate void ProgressFn(float fraction, IntPtr user);

        // sdfk_write_fn: one chunk of OBJ text in file order; 0 = continue, anything else stops sdfk_obj_write
        [UnmanagedFunctionPointer(CallingConvention.Cdecl)]
        public delegate int WriteFn(IntPtr bytes, UIntPtr n, IntPtr user);

        [DllImport(Lib)] public static extern IntPtr sdfk_last_error();
        [DllImport(Lib)] public static extern int sdfk_version();

        [DllImport(Lib)] public static extern int sdfk_ctx_create(int device, out IntPtr ctx);
        // N GPUs of one box behind one handle: sampling / meshing shard by z-slab, rendering by row band, inside the library
        [DllImport(Lib)] public static extern int sdfk_ctx_create_multi(int ndev, int[]? devices, out IntPtr ctx);
        [DllImport(Lib)] public static extern int sdfk_ctx_device_count(IntPtr ctx, out int ndev);
        [DllImport(Lib)] public static extern int sdfk_ctx_destroy(IntPtr ctx);
        [DllImport(Lib)] public static extern int sdfk_ctx_synchronize(IntPtr ctx);

        [DllImport(Lib)] public static extern int sdfk_sdf_compile(IntPtr ctx, byte[] body, UIntPtr len, out IntPtr sdf);
        [DllImport(Lib)] public static extern int sdfk_sdf_destroy(IntPtr sdf);
        [DllImport(Lib)] public static extern int sdfk_sdf_eval(IntPtr sdf, float* xyz, float* rgbd, long n);

        [DllImport(Lib)] public static extern int sdfk_voxels_sample(IntPtr ctx, IntPtr sdf, float* min, float* max,
            int nx, int ny, int nz, int clip, out IntPtr voxels);
        [DllImport(Lib)] public static extern int sdfk_voxels_import(IntPtr ctx, float* values, float* colors, float* min, float* max,
            int nx, int ny, int nz, out IntPtr voxels);
        [DllImport(Lib)] public static extern int sdfk_voxels_export(IntPtr voxels, float* values, float* colors);
        [DllImport(Lib)] public static extern int sdfk_voxels_clip(IntPtr voxels);
        [DllImport(Lib)] public static extern int sdfk_voxels_destroy(IntPtr voxels);

        [DllImport(Lib)] public static extern int sdfk_mesh_create(IntPtr ctx, IntPtr voxels, float iso, int step,
            float* transform, float* normalTransform, ProgressFn? progress, IntPtr user, out IntPtr mesh);
        [DllImport(Lib)] public static extern int sdfk_mesh_counts(IntPtr mesh, out long nverts, out long ntris);
        [DllImport(Lib)] public static extern int sdfk_mesh_export(IntPtr mesh, float* vertices, float* colors, float* normals,
            int* triangles, float* aabb);
        [DllImport(Lib)] public static extern int sdfk_sdf_to_mesh_host(IntPtr ctx, IntPtr sdf, float* min, float* max,
            int nx, int ny, int nz, int clip, float iso, int step, float* transform, float* normalTransform, int nslabs,
            ProgressFn? progress, IntPtr user, out IntPtr mesh);
        [DllImport(Lib)] public static extern int sdfk_mesh_host_ptrs(IntPtr mesh, out float* vertices, out float* colors,
            out float* normals, out int* triangles);
        [DllImport(Lib)] public static extern int sdfk_ctx_set_option(IntPtr ctx, int option, int value);
        [DllImport(Lib)] public static extern int sdfk_ctx_store_bandwidth(IntPtr ctx, UIntPtr bytes, int reps, out double gbPerS);
        [DllImport(Lib)] public static extern int sdfk_mesh_destroy(IntPtr mesh);
        // Mesh.WriteObj (Mesh.cs:66-97): the OBJ text formatted on the device, handed to `sink` chunk by chunk on the calling thread
        [DllImport(Lib)] public static extern int sdfk_obj_write(IntPtr ctx, float* vertices, long nvertices, float* normals, long nnormals,
            int* triangles, long nindices, WriteFn sink, IntPtr user, out long bytesWritten);

        // Not bound here (not needed by the drop-in; see include/sdfk.h): instrumentation (sdfk_ctx_mark / _elapsed / _timer_* /
        // _launch_count / _last_wall_ms / _stream / _create_on_stream, sdfk_mesh_stats, sdfk_sdf_check), the per-process slab API of
        // the torchrun path (sdfk_voxels_sample_slab / _sample_distances / _resample / _info / _layers / _part, sdfk_mesh_classify /
        // _emit / _emit_host / _device_ptrs / _part, sdfk_plan_layers, sdfk_render_device), pinned-buffer helpers (sdfk_host_alloc /
        // _free) and the exhaustive self-tests (sdfk_constdiv_verify, sdfk_selftest_sqrt, sdfk_selftest_float_text).
        // Vec3Data.SaveTga / FloatData.SaveDepthTga payloads packed on the device (a quarter of the float image over PCIe):
        [DllImport(Lib)] public static extern int sdfk_render_bgr8(IntPtr ctx, IntPtr sdf, int w, int h, float* camPos, float* invViewProj,
            float near, float far, int iterations, int rowBegin, int rowEnd, byte* bgr);
        [DllImport(Lib)] public static extern int sdfk_render_depth_gray8(IntPtr ctx, IntPtr sdf, int w, int h, float* camPos,
            float* invViewProj, float marchNear, int iterations, float tgaNear, float tgaFar, int rowBegin, int rowEnd, byte* gray);
        [DllImport(Lib)] public static extern int sdfk_render(IntPtr ctx, IntPtr sdf, int w, int h, float* camPos, float* invViewProj,
            float near, float far, int iterations, int rowBegin, int rowEnd, float* rgb);
        [DllImport(Lib)] public static extern int sdfk_render_depth(IntPtr ctx, IntPtr sdf, int w, int h, float* camPos,
            float* invViewProj, float near, int iterations, int rowBegin, int rowEnd, float* depth);

        public static void Check(int status)
        {
            if (status == 0) return;
            var msg = Marshal.PtrToStringUTF8(sdfk_last_error()) ?? "unknown error";
            if (status == -4) throw new NotSupportedException(msg);
            throw new InvalidOperationException($"libsdfk error {status}: {msg}");
        }
    }

    /// <summary>The GPU(s) behind every GpuSdf of the process: one device, or -- SDFK_DEVICES=0,1,2,3 / new GpuContext(new[]{..}) --
    /// several devices of one box behind one handle (sdfk_ctx_create_multi).  ToVoxels / ToMesh / ToImage then shard inside the
    /// library (z-slabs, row bands) and land ONE result; nothing else in the managed code changes.</summary>
    public sealed class GpuContext : SafeHandle
    {
        static readonly Lazy<GpuContext> shared = new(() => {
            var list = Environment.GetEnvironmentVariable("SDFK_DEVICES");
            if (!string.IsNullOrWhiteSpace(list))
                return new GpuContext(Array.ConvertAll(list.Split(','), x => int.Parse(x.Trim())));
            return new GpuContext(int.TryParse(Environment.GetEnvironmentVariable("LOCAL_RANK"), out var r) ? r : 0);
        });
        public static GpuContext Shared => shared.Value;

        public GpuContext(int device) : base(IntPtr.Zero, true)
        {
            Native.Check(Native.sdfk_ctx_create(device, out var h));
            SetHandle(h);
        }

        public GpuContext(int[] devices) : base(IntPtr.Zero, true)
        {
            Native.Check(Native.sdfk_ctx_create_multi(devices.Length, devices, out var h));
            SetHandle(h);
        }

        public int DeviceCount { get { Native.Check(Native.sdfk_ctx_device_count(handle, out var n)); return n; } }
        public override bool IsInvalid => handle == IntPtr.Zero;
        protected override bool ReleaseHandle() => Native.sdfk_ctx_destroy(handle) == 0;
        internal IntPtr Ptr => handle;
    }
}
