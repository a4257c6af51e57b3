"""The `Sdf` delegate as a GPU object, and the SdfEx facade (ToVoxels / ToMesh / ToImage).

Reference: SdfKit/Sdf.cs:6-99.  `SdfExpr.ToSdf()` returns a GpuSdf: its expression tree has been lowered
to CUDA C++ and NVRTC-compiled for sm_100a.  It is still callable like the delegate
(`sdf(points, colorsAndDistances)`, Sdf.cs:8) -- that call runs the JIT-compiled kernel on the batch.
Opaque callables (the reference's hand-written batch lambdas, Sdfs.*, SdfFuncs.*) are rejected by every
consumer with NotSupportedError: no CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _native as N
from . import numerics
from .exprs import SdfExpr, lower


class SdfConfig:
    DefaultBatchSize = 2 * 1024        # Sdf.cs:13 (a tuning hint with no effect on results; ignored on the GPU)


def require_gpu_sdf(sdf):
    if isinstance(sdf, GpuSdf):
        return sdf
    if isinstance(sdf, SdfExpr):
        return sdf.ToSdf()
    raise N.NotSupportedError(
        "only SDFs built from SdfExprs (SdfExpr.ToSdf()) run on the GPU path; opaque callables such as %r are "
        "rejected rather than run on a CPU fallback" % (sdf,))


class GpuSdf:
    """Sdf delegate backed by sdfk_sdf (JIT-compiled sample / eval / render kernels)."""

    def __init__(self, expr, ctx=None):
        self.ctx = ctx or N.Context.default()
        self.expr = expr
        # SDFK_PACKED=1: also emit the packed two-points-per-instruction body (add/mul/fma.rn.f32x2, verified fast division by
        # constants).  Bit-identical results, 40 % fewer instructions in the ray-march loop -- and measured SLOWER on B200
        # (README ToImage 0.189 -> 0.236 ms, CSG-50 sampling 10.8 -> 16.5 ms: register pairs, per-half traffic), so it is off
        # by default; DESIGN.md section 2b.
        import os
        from .exprs import PACKED_MARKER
        packed = os.environ.get("SDFK_PACKED", "0") == "1"
        plain = os.environ.get("SDFK_PLAIN_BODY", "0") == "1"        # debugging: only the scalar body, the library's default device forms
        # Division by a constant may use the 3-instruction correctly rounded sequence once the device has compared it with
        # div.rn.f32 for all 2^32 dividends (ctx.constdiv_ok: a few ms per constant, cached per context).
        self.lowered = lower(expr, fast_div=None if plain else self.ctx.constdiv_ok, packed=packed)
        low = self.lowered
        if plain:
            text = low.body
        elif packed:
            text = low.body + PACKED_MARKER + "\n" + low.body2
        else:
            # the scalar body (what the oracle compiles) + the device forms: two-point evaluator and row-of-voxels evaluator with
            # shared range guards (exprs._emit_multi) -- same IEEE operations, bit-identical results
            text = low.device_text()
        body = text.encode()
        h = C.c_void_p()
        N.check(N.lib().sdfk_sdf_compile(self.ctx.handle, body, len(body), C.byref(h)))
        self.handle = h

    # ---- the delegate: void Sdf(Memory<Vector3> points, Memory<Vector4> colorsAndDistances)
    def __call__(self, points, colorsAndDistances=None):
        pts = N.f32c(points).reshape(-1, 3)
        out = colorsAndDistances
        if out is None:
            out = np.empty((pts.shape[0], 4), dtype=np.float32)
        if out.dtype != np.float32 or not out.flags.c_contiguous or out.size != pts.shape[0] * 4:
            raise ValueError("colorsAndDistances must be a contiguous float32 array of points.Length Vector4s")
        N.check(N.lib().sdfk_sdf_eval(self.handle, N.fptr(pts), N.fptr(out), pts.shape[0]))
        return out

    # ---- SdfEx (Sdf.cs:20-99)
    def Sample(self, points, distances, batchSize=SdfConfig.DefaultBatchSize, maxDegreeOfParallelism=-1):
        return self(points, distances)

    def ToVoxels(self, min, max, nx, ny, nz, batchSize=SdfConfig.DefaultBatchSize, maxDegreeOfParallelism=-1,
                 clipToBounds=True):
        from .voxels import Voxels
        return Voxels._sample(self, min, max, nx, ny, nz, clip=clipToBounds)

    def ToMesh(self, min, max, nx, ny, nz, batchSize=SdfConfig.DefaultBatchSize, maxDegreeOfParallelism=-1,
               clipToBounds=True, isoValue=0.0, step=1, progress=None, slabs=0):
        """SdfEx.ToMesh (Sdf.cs:59-63).  The caller never sees the voxels, so only distances are sampled (4 B/voxel instead
        of 16) and the colours of the created vertices are evaluated from the SDF afterwards; the grid is processed in
        z-slabs whose finished mesh parts stream to page-locked host memory while the next slabs are computed
        (sdfk_sdf_to_mesh_host).  Same mesh, bit for bit, as ToVoxels(...).ToMesh(...)."""
        from .voxels import GpuMesh
        vmin, vmax = numerics.vec3(min), numerics.vec3(max)
        M, Nm = numerics.mesh_transforms(vmin, vmax, int(nx), int(ny), int(nz))
        M, Nm = N.f32c(M), N.f32c(Nm)
        cb = N.PROGRESS_FN((lambda f, _u: progress(f)) if progress else (lambda f, _u: None))
        h = C.c_void_p()
        N.check(N.lib().sdfk_sdf_to_mesh_host(self.ctx.handle, self.handle, N.fptr(vmin), N.fptr(vmax), int(nx), int(ny), int(nz),
                                              1 if clipToBounds else 0, float(isoValue), int(step), N.fptr(M), N.fptr(Nm), int(slabs),
                                              cb if progress else C.cast(None, N.PROGRESS_FN), None, C.byref(h)))
        return GpuMesh(h, self.ctx).host_view()

    def ToImage(self, width, height, *camera, verticalFieldOfViewDegrees=60.0, nearPlaneDistance=1.0,
                farPlaneDistance=100.0, depthIterations=40, batchSize=SdfConfig.DefaultBatchSize,
                maxDegreeOfParallelism=-1):
        """ToImage(w, h, viewTransform) or ToImage(w, h, cameraPosition, cameraTarget, cameraUpVector)."""
        from .raymarcher import RayMarcher
        if len(camera) == 1:
            view = np.asarray(camera[0], dtype=np.float32).reshape(4, 4)
        elif len(camera) == 3:
            view = numerics.create_look_at(*camera)          # Sdf.cs:95
        else:
            raise TypeError("ToImage takes a view matrix or (position, target, up)")
        rm = RayMarcher(width, height, self, batchSize, maxDegreeOfParallelism)
        rm.ViewTransform = view
        rm.VerticalFieldOfViewDegrees = verticalFieldOfViewDegrees
        rm.NearPlaneDistance = nearPlaneDistance
        rm.FarPlaneDistance = farPlaneDistance
        rm.DepthIterations = depthIterations
        return rm.Render()

    def WithColor(self, red, green=None, blue=None):
        """SdfEx.WithColor (Sdf.cs:101-115).  The reference wraps the delegate in an opaque lambda that overwrites the
        colour; here the same effect is obtained on the expression tree (`expr.Color(c)`), which keeps the result on the
        GPU path."""
        return GpuSdf(self.expr.Color(red, green, blue), ctx=self.ctx)

    def Dispose(self):
        if self.handle:
            N.lib().sdfk_sdf_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.Dispose()
        except Exception:
            pass
