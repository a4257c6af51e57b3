"""ctypes front-end of the CPU oracle (oracle/sdfk_oracle.cpp) -- TEST INFRASTRUCTURE.

An SDF reaches the oracle in one of two ways, both presented to the C++ code as the reference's
batched `Sdf` delegate (SdfKit/Sdf.cs:8):
  * `compile_sdf(body)`  -- the lowered dialect text (the same text NVRTC compiles for the GPU) is
    compiled by g++ -O2 -ffp-contract=off against csrc/sdfk_prelude.h into a small shared object;
  * `numpy_sdf(fn)`      -- an independent numpy float32 restatement (oracle/sdf_numpy.py), or any
    opaque `fn(points[n,3]) -> out[n,4]`, wrapped as a C callback.  This is how the reference's own
    tests (opaque C# lambdas such as Sdfs.Sphere) are restated.
"""
import atexit
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PRELUDE = os.path.join(os.path.dirname(_HERE), "sdfkit_b200", "csrc", "sdfk_prelude.h")
_CACHE = None       # compiled SDFs: a temporary directory of this process (the source tree may be read-only)
_LIB = None

SDF_FN = C.CFUNCTYPE(None, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int)
PROGRESS_FN = C.CFUNCTYPE(None, C.c_float, C.c_void_p)

_fp = C.POINTER(C.c_float)


def build(force=False):
    """Compile oracle/libsdfk_oracle.so with the committed Makefile."""
    so = os.path.join(_HERE, "libsdfk_oracle.so")
    src = os.path.join(_HERE, "sdfk_oracle.cpp")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-B" if force else "-s"], check=True, capture_output=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.orc_sample.argtypes = [SDF_FN, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _fp, _fp,
                                 C.POINTER(C.c_int)]
        L.orc_clip.argtypes = [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int]
        L.orc_mc_create.restype = C.c_void_p
        L.orc_mc_create.argtypes = [_fp, _fp, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, PROGRESS_FN, C.c_void_p,
                                    C.POINTER(C.c_ubyte), C.POINTER(C.c_ubyte)]
        L.orc_mesh_transform.argtypes = [C.c_void_p, _fp, _fp]
        L.orc_mesh_counts.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int64)]
        L.orc_mesh_export.argtypes = [C.c_void_p, _fp, _fp, _fp, C.POINTER(C.c_int), _fp]
        L.orc_mesh_free.argtypes = [C.c_void_p]
        L.orc_render.argtypes = [SDF_FN, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, _fp]
        L.orc_render_depth.argtypes = [SDF_FN, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_int, C.c_int, _fp]
        _LIB = L
    return _LIB


def _f(a):
    return a.ctypes.data_as(_fp)


def _f32c(a):
    return np.ascontiguousarray(a, dtype=np.float32)


# ------------------------------------------------------------------------------------------------
# SDFs
# ------------------------------------------------------------------------------------------------

_WRAPPER = r"""
#include "%(prelude)s"
SK_FN sk_float4 sdf_eval(sk_float3 p)
{
%(body)s}
extern "C" void sdf_batch(const float* pts, float* out, int n)
{
    for (int i = 0; i < n; i++) {
        sk_float4 r = sdf_eval(sk_make3(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]));
        out[4 * i] = r.x; out[4 * i + 1] = r.y; out[4 * i + 2] = r.z; out[4 * i + 3] = r.w;
    }
}
"""


class _Sdf:
    """Holds the C callable plus whatever must stay alive with it."""

    def __init__(self, fn, keep):
        self.fn = fn
        self._keep = keep


def compile_sdf(body):
    """g++-compile lowered dialect text (a LoweredSdf or its .body string) into an oracle SDF."""
    body = getattr(body, "body", body)
    src = _WRAPPER % {"prelude": _PRELUDE, "body": body}
    key = hashlib.sha256(src.encode()).hexdigest()[:24]
    global _CACHE
    if _CACHE is None:
        _CACHE = tempfile.mkdtemp(prefix="sdfk_oracle_")
        atexit.register(shutil.rmtree, _CACHE, True)
    so = os.path.join(_CACHE, "sdf_%s.so" % key)
    if not os.path.exists(so):
        cpp = os.path.join(_CACHE, "sdf_%s.cpp" % key)
        with open(cpp, "w") as f:
            f.write(src)
        tmp = so + ".tmp%d" % os.getpid()
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-std=c++17", "-fPIC", "-shared",
                        "-o", tmp, cpp], check=True, capture_output=True)
        os.replace(tmp, so)
    dll = C.CDLL(so)
    fn = C.cast(dll.sdf_batch, SDF_FN)
    return _Sdf(fn, dll)


def numpy_sdf(fn, writes_color=True):
    """Wrap `fn(points float32[n,3]) -> float32[n,4]` (or [n] distances when writes_color=False, like the
    reference's opaque Sdfs.* lambdas that only assign .W, Sdf.cs:135,153,211) as an oracle SDF."""
    def cb(pp, op, n):
        pts = np.ctypeslib.as_array(pp, shape=(n, 3))
        out = np.ctypeslib.as_array(op, shape=(n, 4))
        r = np.asarray(fn(pts), dtype=np.float32)
        if writes_color:
            out[:, :] = r.reshape(n, 4)
        else:
            out[:, 3] = r.reshape(n)
    cfn = SDF_FN(cb)
    return _Sdf(cfn, (cb, fn))


def _as_sdf(sdf):
    if isinstance(sdf, _Sdf):
        return sdf
    if hasattr(sdf, "body") or isinstance(sdf, str):
        return compile_sdf(sdf)
    if callable(sdf):
        return numpy_sdf(sdf)
    raise TypeError("not an oracle SDF: %r" % (sdf,))


def eval_sdf(sdf, points):
    """Invoke the Sdf delegate on points[n,3] -> out[n,4]."""
    sdf = _as_sdf(sdf)
    pts = _f32c(points).reshape(-1, 3)
    out = np.zeros((pts.shape[0], 4), dtype=np.float32)
    sdf.fn(_f(pts), _f(out), pts.shape[0])
    return out


# ------------------------------------------------------------------------------------------------
# Voxels
# ------------------------------------------------------------------------------------------------

def sample(sdf, vmin, vmax, nx, ny, nz, batch_size=2048, threads=1, return_batch_sizes=False):
    """Voxels.SampleSdf -> (values[nx,ny,nz], colors[nx,ny,nz,3]) in the reference's C# layout."""
    sdf = _as_sdf(sdf)
    mn, mx = _f32c(vmin).reshape(3), _f32c(vmax).reshape(3)
    values = np.zeros((nx, ny, nz), dtype=np.float32)
    colors = np.zeros((nx, ny, nz, 3), dtype=np.float32)
    nb = (nx * ny * nz + batch_size - 1) // batch_size
    bs = np.zeros(max(nb, 1), dtype=np.int32)
    lib().orc_sample(sdf.fn, _f(mn), _f(mx), nx, ny, nz, batch_size, threads, _f(values), _f(colors),
                     bs.ctypes.data_as(C.POINTER(C.c_int)))
    if return_batch_sizes:
        return values, colors, bs[:nb]
    return values, colors


def clip(values, vmin, vmax):
    """Voxels.ClipToBounds, in place."""
    assert values.dtype == np.float32 and values.flags.c_contiguous
    mn, mx = _f32c(vmin).reshape(3), _f32c(vmax).reshape(3)
    nx, ny, nz = values.shape
    lib().orc_clip(_f(values), _f(mn), _f(mx), nx, ny, nz)
    return values


def to_voxels(sdf, vmin, vmax, nx, ny, nz, clip_to_bounds=True, **kw):
    """SdfEx.ToVoxels (Sdf.cs:49-57)."""
    values, colors = sample(sdf, vmin, vmax, nx, ny, nz, **kw)
    if clip_to_bounds:
        clip(values, vmin, vmax)
    return values, colors


# ------------------------------------------------------------------------------------------------
# Marching cubes
# ------------------------------------------------------------------------------------------------

class OracleMesh:
    def __init__(self, vertices, colors, normals, triangles, aabb, active, case_hist, cell_index=None, cell_ntris=None):
        self.vertices, self.colors, self.normals, self.triangles = vertices, colors, normals, triangles
        self.min, self.max = aabb[:3].copy(), aabb[3:].copy()
        self.active_cells = active
        self.case_hist = case_hist
        self.cell_index, self.cell_ntris = cell_index, cell_ntris

    @property
    def center(self):
        return ((self.min + self.max).astype(np.float32) * np.float32(0.5)).astype(np.float32)

    @property
    def size(self):
        return (self.max - self.min).astype(np.float32)


def marching_cubes(values, colors, vmin=None, vmax=None, iso=0.0, step=1, progress=None, transform=True, debug=False):
    """MarchingCubes.CreateMesh (MarchingCubes.cs:39-92).  With transform=False the mesh stays in index space."""
    from sdfkit_b200 import numerics   # host-side System.Numerics restatement (pure python, no native code)
    values = _f32c(values)
    nx, ny, nz = values.shape
    colors = _f32c(colors).reshape(nx, ny, nz, 3)
    ncell = 0
    if debug:
        def count(n):
            c, v = 0, -step
            while v < n - 2 * step:
                v += step
                c += 1
            return c
        ncell = count(nx) * count(ny) * count(nz)
    ci = np.zeros(max(ncell, 1), dtype=np.uint8)
    cn = np.zeros(max(ncell, 1), dtype=np.uint8)
    ub = C.POINTER(C.c_ubyte)
    cb = PROGRESS_FN((lambda f, _u: progress(f)) if progress else (lambda f, _u: None))
    L = lib()
    h = L.orc_mc_create(_f(values), _f(colors), nx, ny, nz, float(iso), int(step), cb, None,
                        ci.ctypes.data_as(ub) if debug else None, cn.ctypes.data_as(ub) if debug else None)
    try:
        if transform:
            assert vmin is not None and vmax is not None
            M, N = numerics.mesh_transforms(vmin, vmax, nx, ny, nz)
            M, N = _f32c(M), _f32c(N)
            L.orc_mesh_transform(h, _f(M), _f(N))
        nv, nt, act = C.c_int64(), C.c_int64(), C.c_int64()
        hist = np.zeros(15, dtype=np.int64)
        L.orc_mesh_counts(h, C.byref(nv), C.byref(nt), C.byref(act), hist.ctypes.data_as(C.POINTER(C.c_int64)))
        v = np.zeros((nv.value, 3), dtype=np.float32)
        c = np.zeros((nv.value, 3), dtype=np.float32)
        n = np.zeros((nv.value, 3), dtype=np.float32)
        t = np.zeros((nt.value, 3), dtype=np.int32)
        aabb = np.zeros(6, dtype=np.float32)
        L.orc_mesh_export(h, _f(v), _f(c), _f(n), t.ctypes.data_as(C.POINTER(C.c_int)), _f(aabb))
    finally:
        L.orc_mesh_free(h)
    return OracleMesh(v, c, n, t, aabb, act.value, hist, ci if debug else None, cn if debug else None)


def to_mesh(sdf, vmin, vmax, nx, ny, nz, clip_to_bounds=True, iso=0.0, step=1, progress=None, **kw):
    """SdfEx.ToMesh (Sdf.cs:59-63)."""
    values, colors = to_voxels(sdf, vmin, vmax, nx, ny, nz, clip_to_bounds, **kw)
    return marching_cubes(values, colors, vmin, vmax, iso, step, progress)


# ------------------------------------------------------------------------------------------------
# Ray marcher
# ------------------------------------------------------------------------------------------------

def _camera(view, w, h, fov, near, far):
    from sdfkit_b200 import numerics
    if view is None:
        view = numerics.create_look_at((0, 0, 5), (0, 0, 0), (0, 1, 0))   # RayMarcher.cs:22-23
    cam, ivp = numerics.camera_matrices(view, w, h, fov, near, far)
    return _f32c(cam), _f32c(ivp)


def render(sdf, w, h, view=None, fov=60.0, near=1.0, far=100.0, iters=40, batch_size=2048, bands=None):
    """RayMarcher.Render -> float32[h,w,3]."""
    sdf = _as_sdf(sdf)
    cam, ivp = _camera(view, w, h, fov, near, far)
    out = np.zeros((h, w, 3), dtype=np.float32)
    lib().orc_render(sdf.fn, w, h, _f(cam), _f(ivp), near, far, iters, batch_size, bands or os.cpu_count(), _f(out))
    return out


def render_depth(sdf, w, h, view=None, fov=60.0, near=1.0, far=100.0, iters=40, batch_size=2048):
    """RayMarcher.RenderDepth -> float32[h,w]."""
    sdf = _as_sdf(sdf)
    cam, ivp = _camera(view, w, h, fov, near, far)
    out = np.zeros((h, w), dtype=np.float32)
    lib().orc_render_depth(sdf.fn, w, h, _f(cam), _f(ivp), near, iters, batch_size, _f(out))
    return out
