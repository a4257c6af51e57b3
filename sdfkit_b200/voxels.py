"""Voxels, MarchingCubes and Mesh -- the host-side mirror of SdfKit/Voxels.cs, MarchingCubes.cs, Mesh.cs.

The voxel field lives in HBM behind an sdfk_voxels handle (device layout x-fastest); the reference's public
arrays `Values[x,y,z]` / `Colors[x,y,z]` are materialised lazily, in the C# layout, on first access.
"""
import ctypes as C
import io
import os

import numpy as np

from . import _native as N
from . import numerics


class Mesh:
    """SdfKit.Mesh (Mesh.cs): Vertices / Colors / Normals (n x 3 float32), Triangles (flat int32, 3 per triangle)."""

    def __init__(self, vertices, colors, normals, triangles, vmin=None, vmax=None, ctx=None):
        """Mesh(vertices, colors, normals, triangles) (Mesh.cs:21-28); Min/Max are measured unless the caller already has them.
        ctx: the context that produced the mesh (None for a mesh built from host arrays); WriteObj formats on its GPU."""
        self.Vertices, self.Colors, self.Normals, self.Triangles = vertices, colors, normals, triangles
        self.Min, self.Max = vmin, vmax
        self.ctx = ctx
        if vmin is None or vmax is None:
            self._measure()

    def _measure(self):
        """Mesh.Measure (Mesh.cs:30-45)."""
        if len(self.Vertices) > 0:
            v = np.asarray(self.Vertices, dtype=np.float32).reshape(-1, 3)
            self.Min, self.Max = v.min(axis=0).astype(np.float32), v.max(axis=0).astype(np.float32)
        elif self.Min is None:
            self.Min = self.Max = np.zeros(3, dtype=np.float32)

    def Transform(self, transform):
        """Mesh.Transform (Mesh.cs:47-64) on the host arrays, in the reference's float32 operation order: v' = v . M (row
        vector), n' = normalize(n . transpose(inverse(M with its translation cleared))).  (MarchingCubes.CreateMesh's own
        index -> world transform is applied on the device, inside the emit kernel.)"""
        f = np.float32
        M = np.asarray(transform, dtype=f).reshape(4, 4)
        nt = M.copy()
        nt[3, 0] = nt[3, 1] = nt[3, 2] = f(0.0)
        nt[3, 3] = f(1.0)
        inv = numerics.invert(nt)
        Nm = numerics.transpose(inv) if inv is not None else np.full((4, 4), np.nan, dtype=f)
        v = np.array(self.Vertices, dtype=f).reshape(-1, 3)
        n = np.array(self.Normals, dtype=f).reshape(-1, 3)
        with np.errstate(all="ignore"):
            tv = np.stack([((v[:, 0] * M[0, k] + v[:, 1] * M[1, k]) + v[:, 2] * M[2, k]) + M[3, k] for k in range(3)], axis=1).astype(f)
            tn = np.stack([(n[:, 0] * Nm[0, k] + n[:, 1] * Nm[1, k]) + n[:, 2] * Nm[2, k] for k in range(3)], axis=1).astype(f)
            ln = np.sqrt((tn[:, 0] * tn[:, 0] + tn[:, 1] * tn[:, 1]) + tn[:, 2] * tn[:, 2]).astype(f)
            tn = (tn / ln[:, None]).astype(f)
        self.Vertices, self.Normals = tv, tn
        self._measure()

    @property
    def Center(self):
        return ((self.Min + self.Max).astype(np.float32) * np.float32(0.5)).astype(np.float32)

    @property
    def Size(self):
        return (self.Max - self.Min).astype(np.float32)

    @property
    def Radius(self):
        return numerics.length3(self.Size) * np.float32(0.5)

    def WriteObj(self, path_or_file):
        """Mesh.WriteObj (Mesh.cs:66-97): "v x y z", "vn x y z", "f i//i j//j k//k" (1-based).  A mesh with a context is
        formatted on its GPU (sdfk_obj_write), byte for byte the text of the host writer below, which serves the others."""
        if self.ctx is not None:
            return self._write_obj_device(path_or_file)
        fmt = _net_float
        close = False
        w = path_or_file
        if isinstance(path_or_file, str):
            w = open(path_or_file, "w", newline="\n")
            close = True
        try:
            for v in self.Vertices:
                w.write("v %s %s %s\n" % (fmt(v[0]), fmt(v[1]), fmt(v[2])))
            for v in self.Normals:
                w.write("vn %s %s %s\n" % (fmt(v[0]), fmt(v[1]), fmt(v[2])))
            t = np.asarray(self.Triangles).reshape(-1, 3) + 1
            for a, b, c in t:
                w.write("f %d//%d %d//%d %d//%d\n" % (a, a, b, b, c, c))
        finally:
            if close:
                w.close()

    def _write_obj_device(self, path_or_file):
        """Paths and binary files receive the chunks as they are (a memoryview over the page-locked stage, no copy); text
        streams receive them decoded as ASCII.  An exception raised while writing (a full disk) stops the call and is
        re-raised once the library has returned."""
        v = N.f32c(self.Vertices).reshape(-1)
        n = N.f32c(self.Normals).reshape(-1)
        t = np.ascontiguousarray(self.Triangles, dtype=np.int32).reshape(-1)
        close = isinstance(path_or_file, (str, os.PathLike))
        f = open(path_or_file, "wb") if close else path_or_file
        text = isinstance(f, io.TextIOBase)
        errors = []

        def sink(ptr, nbytes, _user):
            try:
                chunk = memoryview((C.c_ubyte * nbytes).from_address(ptr))
                f.write(bytes(chunk).decode("ascii") if text else chunk)
                return 0
            except BaseException as e:          # noqa: B036 -- carried across the C frame and re-raised below
                errors.append(e)
                return 1
        cb = N.WRITE_FN(sink)
        try:
            rc = N.lib().sdfk_obj_write(self.ctx.handle, N.fptr(v), len(v) // 3, N.fptr(n), len(n) // 3,
                                        t.ctypes.data_as(C.POINTER(C.c_int32)), len(t), cb, None, None)
        finally:
            if close:
                f.close()
        if errors:
            raise errors[0]
        N.check(rc)


def _net_float(x):
    """Shortest round-trippable float32 text, as .NET Core 3.0+ `float.ToString()` prints (invariant culture)."""
    x = np.float32(x)
    if np.isnan(x):
        return "NaN"
    if np.isinf(x):
        return "Infinity" if x > 0 else "-Infinity"
    s = np.format_float_positional(x, unique=True, trim="-")
    if x != 0:
        # single precision: scientific notation when the decimal exponent is below -4 or at least max(#digits, 7)
        # (5e-5f -> "5E-05", 1e7f -> "1E+07", 12345678f -> "12345678"; double's thresholds are -5 and 15)
        sci = np.format_float_scientific(x, unique=True, trim="-", exp_digits=2)
        mant, exp = sci.split("e")
        e10, ndig = int(exp), len(mant.replace("-", "").replace(".", ""))
        if e10 < -4 or e10 >= max(ndig, 7):
            s = mant + "E" + exp
    return "-0" if (s == "0" and np.signbit(x)) else s


class GpuMesh:
    """Handle-level view of an sdfk_mesh (used by the multi-GPU driver and the benchmark)."""

    def __init__(self, handle, ctx=None):
        self.handle = handle
        self.ctx = ctx                          # handed on to the host meshes made from this one

    def counts(self):
        nv, nt = C.c_int64(), C.c_int64()
        N.check(N.lib().sdfk_mesh_counts(self.handle, C.byref(nv), C.byref(nt)))
        return nv.value, nt.value

    def stats(self):
        s = (C.c_double * 8)()
        N.check(N.lib().sdfk_mesh_stats(self.handle, s))
        return {"classify_ms": s[0], "scan_ms": s[1], "compact_ms": s[2], "emit_ms": s[3],
                "active_cells": int(s[4]), "records": int(s[5]), "chunks": int(s[6]), "from_signs": bool(s[7])}

    def download(self, pinned=True):
        """Copy the mesh to host memory (page-locked, recycled buffers by default: full PCIe speed)."""
        nv, nt = self.counts()
        alloc = N.PinnedPool.empty if pinned else np.empty
        v = alloc((nv, 3), np.float32)
        c = alloc((nv, 3), np.float32)
        n = alloc((nv, 3), np.float32)
        t = alloc((nt * 3,), np.int32)
        aabb = np.zeros(6, dtype=np.float32)
        N.check(N.lib().sdfk_mesh_export(self.handle, N.fptr(v), N.fptr(c), N.fptr(n),
                                         t.ctypes.data_as(C.POINTER(C.c_int32)), N.fptr(aabb)))
        return Mesh(v, c, n, t, aabb[:3].copy(), aabb[3:].copy(), ctx=self.ctx)

    def host_view(self):
        """Mesh over the page-locked host arrays of a mesh made by sdfk_sdf_to_mesh_host (zero copy).  The arrays keep
        this handle alive; the buffers go back to the context's pool when the last of them is garbage collected."""
        nv, nt = self.counts()
        ptrs = [C.c_void_p() for _ in range(4)]
        N.check(N.lib().sdfk_mesh_host_ptrs(self.handle, *[C.byref(p) for p in ptrs]))
        aabb = np.zeros(6, dtype=np.float32)
        N.check(N.lib().sdfk_mesh_export(self.handle, None, None, None, None, N.fptr(aabb)))

        def view(ptr, rows, dtype, shape):
            if rows == 0 or not ptr.value:
                return np.zeros(shape, dtype=dtype)
            buf = (C.c_ubyte * (rows * 12)).from_address(ptr.value)
            buf._owner = self                      # numpy keeps the ctypes buffer alive, which keeps the mesh handle alive
            return np.frombuffer(buf, dtype=dtype).reshape(shape)
        v = view(ptrs[0], nv, np.float32, (nv, 3))
        c = view(ptrs[1], nv, np.float32, (nv, 3))
        n = view(ptrs[2], nv, np.float32, (nv, 3))
        t = view(ptrs[3], nt, np.int32, (nt * 3,))
        return Mesh(v, c, n, t, aabb[:3].copy(), aabb[3:].copy(), ctx=self.ctx)

    def destroy(self):
        if self.handle:
            N.lib().sdfk_mesh_destroy(self.handle)
            self.handle = None

    __del__ = destroy


class Voxels:
    """SdfKit.Voxels (Voxels.cs).  Construct with Voxels(values, colors, min, max) from host arrays in the C#
    layout, Voxels(min, max, nx, ny, nz) for an empty grid, or Voxels.SampleSdf(sdf, min, max, nx, ny, nz)."""

    def __init__(self, *args, ctx=None):
        self.ctx = ctx or N.Context.default()
        self.handle = None
        self._values = self._colors = None
        self._dirty = False          # the host copy was written through the indexers and not yet re-imported
        if len(args) == 4:                                   # Voxels(float[,,] values, Vector3[,,] colors, min, max)
            values, colors, vmin, vmax = args
            values = N.f32c(values)
            if values.ndim != 3:
                raise ValueError("values must be float[nx, ny, nz]")
            nx, ny, nz = values.shape
            colors = None if colors is None else N.f32c(colors).reshape(nx, ny, nz, 3)
            self._set_grid(vmin, vmax, nx, ny, nz)
            h = C.c_void_p()
            N.check(N.lib().sdfk_voxels_import(self.ctx.handle, N.fptr(values), N.fptr(colors), N.fptr(self.Min),
                                               N.fptr(self.Max), nx, ny, nz, C.byref(h)))
            self.handle = h
        elif len(args) == 5:                                 # Voxels(min, max, nx, ny, nz): zero-filled
            vmin, vmax, nx, ny, nz = args
            self._set_grid(vmin, vmax, nx, ny, nz)
        else:
            raise TypeError("Voxels(values, colors, min, max) or Voxels(min, max, nx, ny, nz)")

    def _set_grid(self, vmin, vmax, nx, ny, nz):
        self.Min, self.Max = numerics.vec3(vmin), numerics.vec3(vmax)
        self.NX, self.NY, self.NZ = int(nx), int(ny), int(nz)
        f = np.float32
        self.DX = (self.Max[0] - self.Min[0]) / f(nx) if nx >= 1 else f(0)     # Voxels.cs:32-34
        self.DY = (self.Max[1] - self.Min[1]) / f(ny) if ny >= 1 else f(0)
        self.DZ = (self.Max[2] - self.Min[2]) / f(nz) if nz >= 1 else f(0)

    # ---- IBoundedVolume
    @property
    def Center(self):
        return ((self.Min + self.Max).astype(np.float32) * np.float32(0.5)).astype(np.float32)

    @property
    def Size(self):
        return (self.Max - self.Min).astype(np.float32)

    @property
    def Radius(self):
        return numerics.length3(self.Size) * np.float32(0.5)

    # ---- sampling
    @classmethod
    def _sample(cls, sdf, vmin, vmax, nx, ny, nz, clip, colors=True):
        """colors=False: distance-only voxels for meshing (4 B/voxel); vertex colours are evaluated from `sdf` when the
        mesh is created, with identical results."""
        from .sdf import require_gpu_sdf
        sdf = require_gpu_sdf(sdf)
        v = cls(vmin, vmax, nx, ny, nz, ctx=sdf.ctx)
        h = C.c_void_p()
        if colors:
            N.check(N.lib().sdfk_voxels_sample(sdf.ctx.handle, sdf.handle, N.fptr(v.Min), N.fptr(v.Max), v.NX, v.NY, v.NZ,
                                               1 if clip else 0, C.byref(h)))
        else:
            N.check(N.lib().sdfk_voxels_sample_distances(sdf.ctx.handle, sdf.handle, N.fptr(v.Min), N.fptr(v.Max), v.NX, v.NY,
                                                         v.NZ, 1 if clip else 0, 0, v.NZ, C.byref(h)))
            v._sdf = sdf                                   # keeps the SDF alive for the deferred colours
        v.handle = h
        return v

    @classmethod
    def SampleSdf(cls, sdf, min, max, nx, ny, nz, batchSize=2048, maxDegreeOfParallelism=-1):
        """Voxels.SampleSdf (static, Voxels.cs:169-174).  batchSize / maxDegreeOfParallelism: accepted, no effect."""
        return cls._sample(sdf, min, max, nx, ny, nz, clip=False)

    def Resample(self, sdf, clip=False):
        """Instance Voxels.SampleSdf (Voxels.cs:72-125): re-fill this grid in place."""
        from .sdf import require_gpu_sdf
        sdf = require_gpu_sdf(sdf)
        if self.handle is None:
            other = Voxels._sample(sdf, self.Min, self.Max, self.NX, self.NY, self.NZ, clip)
            self.handle, other.handle = other.handle, None
        else:
            N.check(N.lib().sdfk_voxels_resample(self.handle, sdf.handle, 1 if clip else 0))
        self._sdf = sdf                                    # distance-only voxels: the SDF supplies vertex colours at meshing time
        self._values = self._colors = None
        self._dirty = False

    def ClipToBounds(self):
        self._ensure()
        N.check(N.lib().sdfk_voxels_clip(self.handle))
        self._values = None

    def _ensure(self):
        """The device copy exists and is current: an empty Voxels(min, max, n..) uploads zeros, host writes made through
        the indexers (the reference's Values is live storage, Voxels.cs:42-64) are re-imported."""
        if self.handle is None:
            z = np.zeros((self.NX, self.NY, self.NZ), dtype=np.float32)
            h = C.c_void_p()
            N.check(N.lib().sdfk_voxels_import(self.ctx.handle, N.fptr(z), None, N.fptr(self.Min), N.fptr(self.Max),
                                               self.NX, self.NY, self.NZ, C.byref(h)))
            self.handle = h
        elif self._dirty:
            values, colors = self._values, self._host_colors()
            h = C.c_void_p()
            N.check(N.lib().sdfk_voxels_import(self.ctx.handle, N.fptr(values), N.fptr(colors), N.fptr(self.Min), N.fptr(self.Max),
                                               self.NX, self.NY, self.NZ, C.byref(h)))
            N.lib().sdfk_voxels_destroy(self.handle)
            self.handle = h
            self._dirty = False

    def _export(self, want_colors):
        shape = (self.NX, self.NY, self.NZ, 3) if want_colors else (self.NX, self.NY, self.NZ)
        out = N.PinnedPool.empty(shape, np.float32)        # page-locked: the chunked export runs at PCIe speed
        N.check(N.lib().sdfk_voxels_export(self.handle, None if want_colors else N.fptr(out), N.fptr(out) if want_colors else None))
        return out

    def _host_colors(self):
        if self._colors is None:
            try:
                self._colors = self._export(True)
            except N.SdfkError as e:                       # distance-only voxels hold no colours: the reference's zeros
                if e.code != -4:
                    raise
                self._colors = np.zeros((self.NX, self.NY, self.NZ, 3), dtype=np.float32)
        return self._colors

    # ---- host materialisation (C# layout).  The arrays are read-only snapshots: writes go through the indexers
    # (`voxels[ix, iy, iz] = d`), which keep the device copy in step; `voxels.Values[...] = d` raises instead of silently
    # meshing the unmodified field.
    @property
    def Values(self):
        if self._values is None:
            self._ensure()
            self._values = self._export(False)
        v = self._values.view()
        v.setflags(write=False)
        return v

    @property
    def Colors(self):
        if self._colors is None:
            self._ensure()
            self._colors = self._export(True)              # distance-only voxels: SdfkError ("hold no colours")
        c = self._colors.view()
        c.setflags(write=False)
        return c

    def _index(self, idx):
        if len(idx) == 3 and all(isinstance(k, (int, np.integer)) for k in idx):
            ix, iy, iz = (int(k) for k in idx)
        else:
            p = numerics.vec3(idx)
            ix = int((p[0] - self.Min[0]) / self.DX)
            iy = int((p[1] - self.Min[1]) / self.DY)
            iz = int((p[2] - self.Min[2]) / self.DZ)
        if not (0 <= ix < self.NX and 0 <= iy < self.NY and 0 <= iz < self.NZ):
            raise IndexError("voxel index (%d, %d, %d) outside %dx%dx%d" % (ix, iy, iz, self.NX, self.NY, self.NZ))   # IndexOutOfRangeException
        return ix, iy, iz

    def __getitem__(self, idx):
        """voxels[ix, iy, iz] (Voxels.cs:42-46) or voxels[Vector3 p] -- the voxel containing point p (Voxels.cs:48-56)."""
        ix, iy, iz = self._index(idx)
        return self.Values[ix, iy, iz]

    def __setitem__(self, idx, value):
        """The indexers' setters (Voxels.cs:44-45,57-63): writes the host copy; the device copy is refreshed before the next
        ClipToBounds / ToMesh."""
        ix, iy, iz = self._index(idx)
        self.Values                                        # materialise
        self._values[ix, iy, iz] = np.float32(value)
        self._dirty = True

    # ---- meshing
    def ToMesh(self, isoValue=0.0, step=1, progress=None):
        return MarchingCubes.CreateMesh(self, isoValue, step, progress)

    def Dispose(self):
        if self.handle:
            N.lib().sdfk_voxels_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.Dispose()
        except Exception:
            pass


class MarchingCubes:
    """SdfKit.MarchingCubes (MarchingCubes.cs:39-92)."""

    @staticmethod
    def CreateGpuMesh(volume, isoValue=0.0, step=1, progress=None, transform=True):
        volume._ensure()
        M = Nm = None
        if transform:
            M, Nm = numerics.mesh_transforms(volume.Min, volume.Max, volume.NX, volume.NY, volume.NZ)
            M, Nm = N.f32c(M), N.f32c(Nm)
        cb = N.PROGRESS_FN((lambda f, _u: progress(f)) if progress else (lambda f, _u: None))
        h = C.c_void_p()
        N.check(N.lib().sdfk_mesh_create(volume.ctx.handle, volume.handle, float(isoValue), int(step), N.fptr(M), N.fptr(Nm),
                                         cb if progress else C.cast(None, N.PROGRESS_FN), None, C.byref(h)))
        return GpuMesh(h, volume.ctx)

    @staticmethod
    def CreateMesh(volume, isoValue=0.0, step=1, progress=None):
        gm = MarchingCubes.CreateGpuMesh(volume, isoValue, step, progress)
        try:
            return gm.download()
        finally:
            gm.destroy()
