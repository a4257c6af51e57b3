// GpuSdf.cs -- what SdfExprEx.ToSdf() returns in the drop-in: an `Sdf` delegate whose Target is a GpuSdf holding
// the native handle.  Consumers (Voxels.SampleSdf, SdfEx.ToVoxels/ToMesh/ToImage, RayMarcher) test
// `sdf.Target is GpuSdf` and take the native path; any other delegate (an opaque lambda, Sdfs.*, SdfFuncs.*) is
// rejected with NotSupportedException -- there is no CPU fallback.  SOURCE ONLY (no .NET toolchain in this image).
using System;
using System.IO;
using System.Numerics;
using System.Runtime.ExceptionServices;
using System.Runtime.InteropServices;
using System.Text;

namespace SdfKit.B200
{
    public sealed unsafe class GpuSdf : SafeHandle
    {
        public GpuContext Context { get; }
        public string Body { get; }
        /// <summary>The tree this SDF was compiled from (WithColor re-compiles a modified tree).</summary>
        public System.Linq.Expressions.Expression<SdfFunc>? Expression { get; private set; }

        GpuSdf(GpuContext ctx, string body) : base(IntPtr.Zero, true)
        {
            Context = ctx;
            Body = body;
            var utf8 = Encoding.UTF8.GetBytes(body);
            Native.Check(Native.sdfk_sdf_compile(ctx.Ptr, utf8, (UIntPtr)utf8.Length, out var h));
            SetHandle(h);
        }

        public override bool IsInvalid => handle == IntPtr.Zero;
        protected override bool ReleaseHandle() => Native.sdfk_sdf_destroy(handle) == 0;
        internal IntPtr Ptr => handle;

        /// <summary>Replacement body of SdfExprCompiler.Compile (SdfKit/SdfExpr.cs:234-238).</summary>
        public static Sdf Compile(System.Linq.Expressions.Expression<SdfFunc> expression, GpuContext? ctx = null)
        {
            var gpu = new GpuSdf(ctx ?? GpuContext.Shared, SdfExprLowering.Lower(expression)) { Expression = expression };
            return gpu.Invoke;   // delegate.Target == gpu
        }

        /// <summary>SdfEx.WithColor (SdfKit/Sdf.cs:101-115) for a compiled SDF.  The reference wraps the delegate in an opaque
        /// lambda that overwrites the colour of every output; the same values come from the tree with a constant colour
        /// (SdfExprEx.Color, SdfKit/SdfExpr.cs:143-147), which stays on the GPU path -- the Python mirror does the same
        /// (sdfkit_b200/sdf.py: WithColor; tests/test_gpu_multi.py::test_with_color_matches_oracle).</summary>
        public Sdf WithColor(Vector3 color) =>
            Compile((Expression ?? throw new NotSupportedException("this GpuSdf was not built from an SdfExpr")).Color(color), Context);

        /// <summary>The delegate body: colorsAndDistances[i] = sdf(points[i]) (SdfKit/Sdf.cs:8).</summary>
        public void Invoke(Memory<Vector3> points, Memory<Vector4> colorsAndDistances)
        {
            if (colorsAndDistances.Length < points.Length) throw new ArgumentException("output shorter than input");
            using var pin = points.Pin();
            using var pout = colorsAndDistances.Pin();
            Native.Check(Native.sdfk_sdf_eval(handle, (float*)pin.Pointer, (float*)pout.Pointer, points.Length));
        }

        /// <summary>Native handle behind an Sdf delegate, or NotSupportedException for opaque delegates.</summary>
        public static GpuSdf Require(Sdf sdf) =>
            sdf.Target as GpuSdf ?? throw new NotSupportedException(
                "Only SDFs built from SdfExprs (SdfExpr.ToSdf()) run on the GPU path; opaque Sdf delegates are rejected " +
                "rather than run on a CPU fallback.");
    }

    /// <summary>GPU bodies for the reference's consumers; each cites the method whose body it replaces.</summary>
    public static unsafe class GpuPath
    {
        /// SdfEx.ToVoxels (SdfKit/Sdf.cs:49-57) / Voxels.SampleSdf (SdfKit/Voxels.cs:169-174)
        public static Voxels ToVoxels(Sdf sdf, Vector3 min, Vector3 max, int nx, int ny, int nz, bool clipToBounds)
        {
            var g = GpuSdf.Require(sdf);
            var voxels = new Voxels(min, max, nx, ny, nz);            // allocates Values / Colors like the reference
            Native.Check(Native.sdfk_voxels_sample(g.Context.Ptr, g.Ptr, (float*)&min, (float*)&max, nx, ny, nz,
                clipToBounds ? 1 : 0, out var h));
            try {
                fixed (float* pv = voxels.Values) fixed (Vector3* pc = voxels.Colors)
                    Native.Check(Native.sdfk_voxels_export(h, pv, (float*)pc));    // C# [x,y,z] layout
            } finally { Native.sdfk_voxels_destroy(h); }
            return voxels;
        }

        /// SdfEx.ToMesh (SdfKit/Sdf.cs:59-63): one native call.  The grid is sampled (distances only) and meshed in z-slabs on
        /// the device while the finished parts of the mesh stream to page-locked host memory owned by the native handle;
        /// the managed arrays are filled from there (Buffer.MemoryCopy, one pass per array).
        public static Mesh ToMesh(Sdf sdf, Vector3 min, Vector3 max, int nx, int ny, int nz, bool clipToBounds,
                                  float isoValue, int step, IProgress<float>? progress)
        {
            var g = GpuSdf.Require(sdf);
            MeshTransforms(min, max, nx, ny, nz, out var transform, out var normalTransform);
            Native.ProgressFn? cb = progress is null ? null : (f, _) => progress.Report(f);
            Native.Check(Native.sdfk_sdf_to_mesh_host(g.Context.Ptr, g.Ptr, (float*)&min, (float*)&max, nx, ny, nz,
                clipToBounds ? 1 : 0, isoValue, step, (float*)&transform, (float*)&normalTransform, 0, cb, IntPtr.Zero, out var mesh));
            GC.KeepAlive(cb);
            try {
                Native.Check(Native.sdfk_mesh_counts(mesh, out var nv, out var ntri));
                Native.Check(Native.sdfk_mesh_host_ptrs(mesh, out var hv, out var hc, out var hn, out var ht));
                var v = new Vector3[nv]; var c = new Vector3[nv]; var n = new Vector3[nv]; var t = new int[ntri * 3];
                fixed (Vector3* pv = v) fixed (Vector3* pc = c) fixed (Vector3* pn = n) fixed (int* pt = t) {
                    Buffer.MemoryCopy(hv, pv, nv * 12, nv * 12);
                    Buffer.MemoryCopy(hc, pc, nv * 12, nv * 12);
                    Buffer.MemoryCopy(hn, pn, nv * 12, nv * 12);
                    Buffer.MemoryCopy(ht, pt, ntri * 12, ntri * 12);
                }
                return new Mesh(v, c, n, t);
            } finally { Native.sdfk_mesh_destroy(mesh); }
        }

        /// MarchingCubes.CreateMesh (SdfKit/MarchingCubes.cs:39-92) on host-built voxels
        public static Mesh CreateMesh(Voxels volume, float isoValue, int step, IProgress<float>? progress)
        {
            var ctx = GpuContext.Shared;
            Vector3 min = volume.Min, max = volume.Max;
            IntPtr vox;
            fixed (float* pv = volume.Values) fixed (Vector3* pc = volume.Colors)
                Native.Check(Native.sdfk_voxels_import(ctx.Ptr, pv, (float*)pc, (float*)&min, (float*)&max,
                    volume.NX, volume.NY, volume.NZ, out vox));
            try { return CreateMesh(ctx, vox, min, max, volume.NX, volume.NY, volume.NZ, isoValue, step, progress); }
            finally { Native.sdfk_voxels_destroy(vox); }
        }

        /// the very matrices of MarchingCubes.cs:85-90 and Mesh.cs:49-55, computed with System.Numerics itself
        static void MeshTransforms(Vector3 min, Vector3 max, int nx, int ny, int nz, out Matrix4x4 transform, out Matrix4x4 normalTransform)
        {
            var size = max - min;
            transform =
                Matrix4x4.CreateTranslation(-(nx - 1) / 2f, -(ny - 1) / 2f, -(nz - 1) / 2f) *
                Matrix4x4.CreateScale(size.X / (nx - 1), size.Y / (ny - 1), size.Z / (nz - 1)) *
                Matrix4x4.CreateTranslation((min + max) * 0.5f);
            var nt = transform; nt.M41 = 0; nt.M42 = 0; nt.M43 = 0; nt.M44 = 1;
            Matrix4x4.Invert(nt, out var inv);
            normalTransform = Matrix4x4.Transpose(inv);
        }

        static Mesh CreateMesh(GpuContext ctx, IntPtr vox, Vector3 min, Vector3 max, int nx, int ny, int nz,
                               float iso, int step, IProgress<float>? progress)
        {
            MeshTransforms(min, max, nx, ny, nz, out var transform, out var normalTransform);
            Native.ProgressFn? cb = progress is null ? null : (f, _) => progress.Report(f);
            Native.Check(Native.sdfk_mesh_create(ctx.Ptr, vox, iso, step, (float*)&transform, (float*)&normalTransform,
                cb, IntPtr.Zero, out var mesh));
            GC.KeepAlive(cb);
            try {
                Native.Check(Native.sdfk_mesh_counts(mesh, out var nv, out var ntri));
                var v = new Vector3[nv]; var c = new Vector3[nv]; var n = new Vector3[nv]; var t = new int[ntri * 3];
                var aabb = stackalloc float[6];
                fixed (Vector3* pv = v) fixed (Vector3* pc = c) fixed (Vector3* pn = n) fixed (int* pt = t)
                    Native.Check(Native.sdfk_mesh_export(mesh, (float*)pv, (float*)pc, (float*)pn, pt, aabb));
                return new Mesh(v, c, n, t);     // Mesh ctor re-measures Min/Max (Mesh.cs:21-28); aabb is equal
            } finally { Native.sdfk_mesh_destroy(mesh); }
        }

        /// Mesh.WriteObj (SdfKit/Mesh.cs:66-97): the OBJ text is formatted on the GPU and written to `stream` in chunks, byte for
        /// byte what the reference's StreamWriter loop prints (float.ToString() text, 1-based indices, '\n' line ends).  An
        /// exception thrown by the stream stops the native call and is rethrown here.
        public static void WriteObj(Mesh mesh, Stream stream)
        {
            var ctx = GpuContext.Shared;
            Exception? error = null;
            var chunk = new byte[0];
            Native.WriteFn sink = (bytes, n, _) => {
                try {
                    int len = checked((int)(ulong)n);
                    if (chunk.Length < len) chunk = new byte[len];
                    Marshal.Copy(bytes, chunk, 0, len);
                    stream.Write(chunk, 0, len);
                    return 0;
                } catch (Exception e) { error = e; return 1; }
            };
            int status;
            fixed (Vector3* pv = mesh.Vertices) fixed (Vector3* pn = mesh.Normals) fixed (int* pt = mesh.Triangles)
                status = Native.sdfk_obj_write(ctx.Ptr, (float*)pv, mesh.Vertices.Length, (float*)pn, mesh.Normals.Length,
                    pt, mesh.Triangles.Length, sink, IntPtr.Zero, out _);
            GC.KeepAlive(sink);                // the delegate must outlive the native call that calls it
            if (error is not null) ExceptionDispatchInfo.Capture(error).Throw();
            Native.Check(status);
        }

        /// RayMarcher.Render (SdfKit/RayMarcher.cs:45-64): camera matrices from System.Numerics as in :95-108
        public static Vec3Data Render(Sdf sdf, int width, int height, Matrix4x4 view, float fovDegrees, float near, float far,
                                      int iterations)
        {
            var g = GpuSdf.Require(sdf);
            Matrix4x4.Invert(view, out var cameraTransform);
            var cam = Vector3.Transform(Vector3.Zero, cameraTransform);
            var proj = Matrix4x4.CreatePerspectiveFieldOfView(fovDegrees * MathF.PI / 180.0f, (float)width / height, near, far);
            Matrix4x4.Invert(view * proj, out var ivp);
            var img = new Vec3Data(width, height);
            fixed (float* p = img.Values)
                Native.Check(Native.sdfk_render(g.Context.Ptr, g.Ptr, width, height, (float*)&cam, (float*)&ivp, near, far,
                    iterations, 0, height, p));
            return img;
        }

        /// RayMarcher.RenderDepth (SdfKit/RayMarcher.cs:69-93)
        public static FloatData RenderDepth(Sdf sdf, int width, int height, Matrix4x4 view, float fovDegrees, float near, float far,
                                            int iterations)
        {
            var g = GpuSdf.Require(sdf);
            Matrix4x4.Invert(view, out var cameraTransform);
            var cam = Vector3.Transform(Vector3.Zero, cameraTransform);
            var proj = Matrix4x4.CreatePerspectiveFieldOfView(fovDegrees * MathF.PI / 180.0f, (float)width / height, near, far);
            Matrix4x4.Invert(view * proj, out var ivp);
            var img = new FloatData(width, height);
            fixed (float* p = img.Values)
                Native.Check(Native.sdfk_render_depth(g.Context.Ptr, g.Ptr, width, height, (float*)&cam, (float*)&ivp, near,
                    iterations, 0, height, p));
            return img;
        }
    }
}
