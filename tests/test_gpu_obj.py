"""Mesh.WriteObj on the device (sdfk_obj_write): the OBJ text formatted by CUDA kernels equals the host writer's, byte for
byte.  The float text itself is pinned by an independent statement of the rule (tests/obj_text_ref.cpp: std::to_chars
plus the .NET layout), checked against the host writer's _net_float on the CPU and against the device on every float."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest

from sdfkit_b200.voxels import Mesh, _net_float

HERE = os.path.dirname(os.path.abspath(__file__))
f32 = np.float32


@pytest.fixture(scope="session")
def obj_ref(tmp_path_factory):
    exe = tmp_path_factory.mktemp("obj_ref") / "obj_text_ref"
    subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-o", str(exe), os.path.join(HERE, "obj_text_ref.cpp")], check=True)
    return str(exe)


def ref_texts(obj_ref, bits):
    out = subprocess.run([obj_ref, "texts"], input=np.asarray(bits, dtype="<u4").tobytes(), capture_output=True, check=True)
    return out.stdout.decode("ascii").split("\n")[:-1]


def edge_bits():
    """+-0, the subnormal range's ends, FLT_MIN, FLT_MAX, NaNs, +-Inf, and two ulps either side of every power of ten in
    range (1e-45 .. 1e38; this includes 1e-5, 1e-4 and 1e7) and of a few integers at the layout's thresholds."""
    b = [0x00000000, 0x00000001, 0x007FFFFF, 0x00800000, 0x7F7FFFFF, 0x7F800000, 0x7FC00000, 0x7F800001, 0xFFC00000, 0x7FFFFFFF]
    centres = [f32(10.0 ** k) for k in range(-45, 39)] + [f32(v) for v in (9999999, 12345678, 16777216, 0.1, 1 / 3)]
    for c in centres:
        u = int(np.asarray(c).view(np.uint32))
        b += [u + d for d in (-2, -1, 0, 1, 2) if 0 <= u + d < 0x7F800000]
    b = np.array(b, dtype=np.uint32)
    return np.unique(np.concatenate([b, b | np.uint32(0x80000000)]))


def test_reference_checker_agrees_with_net_float(obj_ref):
    rng = np.random.default_rng(20261022)
    bits = np.concatenate([edge_bits(), rng.integers(0, 1 << 32, 200_000, dtype=np.uint64).astype(np.uint32)])
    got = ref_texts(obj_ref, bits)
    assert len(got) == len(bits)
    bad = [(hex(int(u)), g, _net_float(x)) for u, x, g in zip(bits, bits.view(np.float32), got) if g != _net_float(x)]
    assert not bad, "%d mismatches, first (bits, checker, _net_float): %s" % (len(bad), bad[:5])


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sk():
    import sdfkit_b200
    return sdfkit_b200


def host_copy(mesh):
    """The same arrays without a context: WriteObj takes the host writer."""
    return Mesh(mesh.Vertices, mesh.Colors, mesh.Normals, mesh.Triangles, mesh.Min, mesh.Max)


def host_text(mesh):
    w = io.StringIO()
    host_copy(mesh).WriteObj(w)
    return w.getvalue().encode("ascii")


def special_mesh(ctx):
    vals = np.array(edge_bits(), dtype=np.uint32)
    vals = np.concatenate([vals, np.zeros((-len(vals)) % 3, dtype=np.uint32)]).view(np.float32).reshape(-1, 3)
    normals = vals[::-1][:7].copy()                                   # fewer normals than vertices
    tris = np.array([0, -1, 2147483647, -2147483648, 5, 6, 1, 2, 3], dtype=np.int32)
    z = np.zeros(3, dtype=np.float32)
    return Mesh(vals, None, normals, tris, z, z, ctx=ctx)


def transform_matrix():
    a, s = 0.7, 1.75
    M = np.array([[np.cos(a) * s, np.sin(a) * s, 0, 0], [-np.sin(a) * s, np.cos(a) * s, 0.3, 0], [0.1, -0.2, 0.9, 0],
                  [1.5, -2.25, 0.125, 1]], dtype=np.float32)
    return M


@pytest.fixture(scope="module")
def meshes(sk):
    """name -> (mesh with a context, the host writer's bytes)"""
    from sdfkit_b200 import scenes
    ctx = sk.Context.default()
    out = {}
    for name, (expr, mn, mx), n in (("sphere64", scenes.sphere(), 64), ("readme96", scenes.readme_scene(), 96),
                                     ("csg50", scenes.csg50(), 64)):
        out[name] = expr.ToSdf().ToMesh(mn, mx, n, n, n)
    rng = np.random.default_rng(0)
    vals = rng.uniform(-1, 1, (24, 24, 24)).astype(np.float32)
    cols = rng.uniform(0, 1, (24, 24, 24, 3)).astype(np.float32)
    out["noise24"] = sk.Voxels(vals, cols, (-1, -1, -1), (1, 1, 1), ctx=ctx).ToMesh()
    expr, mn, mx = scenes.readme_scene()
    t = expr.ToSdf().ToMesh(mn, mx, 96, 96, 96)
    t.Transform(transform_matrix())
    out["readme96_transformed"] = t
    out["specials"] = special_mesh(ctx)
    out["more_normals"] = Mesh(out["sphere64"].Vertices[:100], None, out["sphere64"].Normals[:250], out["sphere64"].Triangles[:300],
                               ctx=ctx)
    e = np.zeros((0, 3), dtype=np.float32)
    out["empty"] = Mesh(e, e, e, np.zeros(0, dtype=np.int32), ctx=ctx)
    for m in out.values():
        assert m.ctx is not None
    return {k: (m, host_text(m)) for k, m in out.items()}


def write_device(mesh, target, tmp_path):
    if target == "path":
        p = tmp_path / "m.obj"
        mesh.WriteObj(str(p))
        return p.read_bytes()
    if target == "binary":
        p = tmp_path / "b.obj"
        with open(p, "wb") as f:
            mesh.WriteObj(f)
        return p.read_bytes()
    w = io.StringIO()
    mesh.WriteObj(w)
    return w.getvalue().encode("ascii")


MESHES = ["sphere64", "readme96", "csg50", "noise24", "readme96_transformed", "specials", "more_normals", "empty"]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", ["default", "1"])
@pytest.mark.parametrize("target", ["path", "binary", "text"])
@pytest.mark.parametrize("name", MESHES)
def test_device_obj_equals_host_writer(meshes, monkeypatch, tmp_path, name, target, chunk):
    if chunk != "default":
        monkeypatch.setenv("SDFK_OBJ_CHUNK_BYTES", chunk)            # one chunk per 256 lines
    mesh, want = meshes[name]
    got = write_device(mesh, target, tmp_path)
    if got != want:
        i = next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), min(len(got), len(want)))
        line = want.count(b"\n", 0, i)
        raise AssertionError("%s: %d bytes vs %d from the host writer; first difference at byte %d, line %d:\n device %r\n host   %r" % (
            name, len(got), len(want), i, line + 1, got[got.rfind(b"\n", 0, i) + 1:][:80], want[want.rfind(b"\n", 0, i) + 1:][:80]))
    if name == "empty":
        assert got == b""


class Recorder:
    """A binary writer that counts the chunks and can fail on one of them."""

    def __init__(self, fail_at=None):
        self.parts, self.fail_at = [], fail_at

    def write(self, b):
        if self.fail_at is not None and len(self.parts) + 1 == self.fail_at:
            raise OSError(28, "No space left on device")
        self.parts.append(bytes(b))
        return len(b)


@pytest.mark.gpu
def test_small_chunks_stream_in_file_order(meshes, monkeypatch):
    monkeypatch.setenv("SDFK_OBJ_CHUNK_BYTES", "4096")
    mesh, want = meshes["readme96"]
    r = Recorder()
    mesh.WriteObj(r)
    assert len(r.parts) >= 100 and b"".join(r.parts) == want


@pytest.mark.gpu
def test_sink_failure_propagates_and_the_context_stays_usable(meshes, monkeypatch):
    monkeypatch.setenv("SDFK_OBJ_CHUNK_BYTES", "1")
    mesh, want = meshes["readme96"]
    r = Recorder(fail_at=3)
    with pytest.raises(OSError, match="No space left"):
        mesh.WriteObj(r)
    assert len(r.parts) == 2 and want.startswith(b"".join(r.parts))
    r = Recorder()
    mesh.WriteObj(r)
    assert b"".join(r.parts) == want


@pytest.mark.gpu
def test_sink_status_and_partial_triangles_are_reported(sk):
    from sdfkit_b200 import _native as N
    ctx = sk.Context.default()
    v = np.zeros((4, 3), dtype=np.float32)
    t = np.array([0, 1, 2, 3], dtype=np.int32)
    written = C.c_int64(-1)
    cb = N.WRITE_FN(lambda p, n, u: 0)
    rc = N.lib().sdfk_obj_write(ctx.handle, N.fptr(v), 4, N.fptr(v), 4, t.ctypes.data_as(C.POINTER(C.c_int32)), 4, cb, None,
                                C.byref(written))
    assert rc == -1 and b"whole number of triangles" in N.lib().sdfk_last_error()
    with pytest.raises(sk.SdfkError) as e:
        Mesh(v, None, v, t, ctx=ctx).WriteObj(io.BytesIO())
    assert e.value.code == -1
    stop = N.WRITE_FN(lambda p, n, u: 7)
    rc = N.lib().sdfk_obj_write(ctx.handle, N.fptr(v), 4, N.fptr(v), 4, t.ctypes.data_as(C.POINTER(C.c_int32)), 3, stop, None,
                                C.byref(written))
    assert rc == -1 and b"returned 7" in N.lib().sdfk_last_error() and written.value == 0


@pytest.mark.gpu
def test_multi_gpu_context_writes_the_same_bytes(sk, meshes, tmp_path):
    mctx = sk.Context(devices=[0, 0])
    try:
        for name in ("readme96", "specials"):
            m, want = meshes[name]
            assert write_device(Mesh(m.Vertices, m.Colors, m.Normals, m.Triangles, m.Min, m.Max, ctx=mctx), "binary", tmp_path) == want
    finally:
        mctx.close()


@pytest.mark.gpu
def test_meshes_remember_their_context(sk):
    from sdfkit_b200 import scenes
    expr, mn, mx = scenes.sphere()
    sdf = expr.ToSdf()
    assert sdf.ToMesh(mn, mx, 16, 16, 16).ctx is sdf.ctx
    assert sdf.ToVoxels(mn, mx, 16, 16, 16).ToMesh().ctx is sdf.ctx
    gm = sk.MarchingCubes.CreateGpuMesh(sdf.ToVoxels(mn, mx, 16, 16, 16))
    assert gm.download().ctx is sdf.ctx
    gm.destroy()


def device_float_texts(ctx, bits):
    """The device's text of each bit pattern: the vertex lines of a mesh whose coordinates are those floats."""
    v = np.concatenate([bits, np.zeros((-len(bits)) % 3, dtype=np.uint32)]).view(np.float32).reshape(-1, 3)
    w = io.BytesIO()
    e = np.zeros((0, 3), dtype=np.float32)
    Mesh(v, None, e, np.zeros(0, dtype=np.int32), np.zeros(3, f32), np.zeros(3, f32), ctx=ctx).WriteObj(w)
    return [t for line in w.getvalue().decode("ascii").split("\n")[:-1] for t in line.split(" ")[1:]][:len(bits)]


@pytest.mark.gpu
def test_every_float_text_matches_the_reference(sk, obj_ref):
    from sdfkit_b200 import _native as N
    ctx = sk.Context.default()
    d = (C.c_uint64 * 4096)()
    N.check(N.lib().sdfk_selftest_float_text(ctx.handle, 0, 4096, d))
    ref = subprocess.run([obj_ref, "digests", "0", "4096"], capture_output=True, check=True, text=True).stdout.split()
    assert len(ref) == 4096
    bad = [b for b in range(4096) if int(ref[b], 16) != d[b]]
    if bad:
        bits = np.arange(bad[0] << 20, (bad[0] + 1) << 20, dtype=np.uint64).astype(np.uint32)
        dev, want = device_float_texts(ctx, bits), ref_texts(obj_ref, bits)
        k = next((i for i in range(len(bits)) if dev[i] != want[i]), None)
        where = "bit pattern 0x%08x: device %r, reference %r" % (bits[k], dev[k], want[k]) if k is not None else "texts agree (digest only)"
        raise AssertionError("%d of 4096 blocks differ; first in block %d, %s" % (len(bad), bad[0], where))
