"""MarchingCubes.CreateMesh (sdfk_mesh_create) on grids larger than one meshing job: the cell layers are meshed in sub-slabs
whose 32-bit chunk and cell ids stay in range, into ONE ordinary device-resident mesh.

  * SDFK_MESH_SUBSLAB_CAP=n forces sub-slabs of n cell layers on small grids: every mesh equals the one-job mesh and the
    CPU oracle's bit for bit, with the same progress calls and the same classifier;
  * the same inside a multi-GPU context (device 0 listed several times);
  * the real sizes on one device: 1664^3 (more than 2^32 cells) and 2048^3 (BASELINE config 4), skipped when the shared
    device does not have the memory free."""
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
f32 = np.float32
CAPS = [1, 3, 17]


@pytest.fixture(scope="module")
def sk():
    import sdfkit_b200
    return sdfkit_b200


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def scene(name):
    from sdfkit_b200 import scenes
    return {"readme": scenes.readme_scene, "perf": scenes.perf_scene, "csg50": scenes.csg50}[name]()


def create(sk, vox, iso, step, cap, monkeypatch):
    """CreateMesh with sub-slabs of `cap` cell layers (None: no cap).  Returns the host mesh, the progress values, the
    stats and the device arrays of the device-resident mesh."""
    from sdfkit_b200 import dist as skd
    from sdfkit_b200.voxels import MarchingCubes
    if cap is None:
        monkeypatch.delenv("SDFK_MESH_SUBSLAB_CAP", raising=False)
    else:
        monkeypatch.setenv("SDFK_MESH_SUBSLAB_CAP", str(cap))
    prog = []
    try:
        gm = MarchingCubes.CreateGpuMesh(vox, iso, step, prog.append)
    finally:
        monkeypatch.delenv("SDFK_MESH_SUBSLAB_CAP", raising=False)
    try:
        stats = gm.stats()
        dev = None                                  # (a multi-GPU context's mesh is one part per device: no single arrays)
        if len(vox.ctx.devices) == 1:
            dev = [t.cpu().numpy() for t in skd.mesh_device_tensors(gm, "cuda:%d" % vox.ctx.device)]
        mesh = gm.download(pinned=False)
    finally:
        gm.destroy()
    return mesh, prog, stats, dev


def same_mesh(a, b, what):
    assert len(a.Vertices) == len(b.Vertices) and len(a.Triangles) == len(b.Triangles), what + ": counts differ"
    assert np.array_equal(np.asarray(a.Triangles), np.asarray(b.Triangles)), what + ": triangles differ"
    for name in ("Vertices", "Colors", "Normals"):
        assert np.array_equal(bits(getattr(a, name)), bits(getattr(b, name))), "%s: %s differ" % (what, name)
    assert np.array_equal(bits(a.Min), bits(b.Min)) and np.array_equal(bits(a.Max), bits(b.Max)), what + ": AABB differs"


def same_as_oracle(m, om, what):
    assert np.array_equal(np.asarray(m.Triangles).reshape(-1, 3), om.triangles), what + ": triangles vs oracle"
    assert np.array_equal(bits(m.Vertices), bits(om.vertices)), what + ": vertices vs oracle"
    assert np.array_equal(bits(m.Colors), bits(om.colors)), what + ": colours vs oracle"
    assert np.array_equal(bits(m.Normals), bits(om.normals)), what + ": normals vs oracle"
    if len(m.Vertices):
        assert np.array_equal(bits(m.Min), bits(om.min)) and np.array_equal(bits(m.Max), bits(om.max)), what + ": AABB vs oracle"


def check_caps(sk, vox, iso, step, om, monkeypatch, what):
    one, prog1, st1, _ = create(sk, vox, iso, step, None, monkeypatch)
    same_as_oracle(one, om, what + ", one job")
    for cap in CAPS:
        m, prog, st, dev = create(sk, vox, iso, step, cap, monkeypatch)
        w = "%s, sub-slab cap %d" % (what, cap)
        same_mesh(m, one, w)
        same_as_oracle(m, om, w)
        assert prog == prog1, w + ": progress calls differ"
        assert st["from_signs"] == st1["from_signs"], w + ": classifier differs"
        assert st["active_cells"] == st1["active_cells"], w + ": active cells differ"
        assert dev is not None
        assert np.array_equal(dev[3].reshape(-1), np.asarray(m.Triangles)), w + ": device triangles"
        for arr, name in zip(dev[:3], ("Vertices", "Colors", "Normals")):
            assert np.array_equal(bits(arr), bits(getattr(m, name))), "%s: device %s" % (w, name)


CASES = [("readme", (70, 52, 33), 1, 0.0), ("readme", (70, 52, 33), 2, 0.1), ("perf", (96, 96, 48), 1, 0.1),
         ("perf", (70, 52, 33), 2, 0.0), ("csg50", (96, 96, 48), 1, 0.0), ("csg50", (96, 96, 48), 2, 0.0)]


@pytest.mark.parametrize("name,dims,step,iso", CASES)
def test_forced_sub_slabs_equal_one_job_and_oracle(sk, oracle, monkeypatch, name, dims, step, iso):
    expr, mn, mx = scene(name)
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    om = oracle.to_mesh(sdf.lowered, f32(mn), f32(mx), nx, ny, nz, iso=iso, step=step)
    vox = sdf.ToVoxels(mn, mx, nx, ny, nz)
    check_caps(sk, vox, iso, step, om, monkeypatch, "%s %s step %d iso %g" % (name, dims, step, iso))
    # unclipped, then ClipToBounds on the device (classified from the distances, not the sign planes)
    raw = sdf.ToVoxels(mn, mx, nx, ny, nz, clipToBounds=False)
    raw.ClipToBounds()
    check_caps(sk, raw, iso, step, om, monkeypatch, "%s %s step %d iso %g, ClipToBounds" % (name, dims, step, iso))


@pytest.mark.parametrize("name,dims", [("readme", (70, 52, 33)), ("csg50", (96, 96, 48))])
def test_forced_sub_slabs_on_distance_only_voxels(sk, oracle, monkeypatch, name, dims):
    """Distance-only voxels: the vertex colours are evaluated from the SDF per sub-slab (deferred colour kernel)."""
    from sdfkit_b200.voxels import Voxels
    expr, mn, mx = scene(name)
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    vox = Voxels._sample(sdf, mn, mx, nx, ny, nz, clip=True, colors=False)
    for step in (1, 2):
        om = oracle.to_mesh(sdf.lowered, f32(mn), f32(mx), nx, ny, nz, step=step)
        check_caps(sk, vox, 0.0, step, om, monkeypatch, "%s %s distance-only step %d" % (name, dims, step))


def test_forced_sub_slabs_on_white_noise(sk, oracle, monkeypatch):
    """Imported white noise reaches every Lewiner case, on both sides of every sub-slab boundary."""
    rng = np.random.default_rng(0)
    v = rng.uniform(-1, 1, (64, 64, 64)).astype(f32)
    c = rng.uniform(0, 1, (64, 64, 64, 3)).astype(f32)
    mn, mx = (-1, -1, -1), (1, 1, 1)
    vox = sk.Voxels(v, c, mn, mx)
    for step in (1, 2):
        om = oracle.marching_cubes(v, c, f32(mn), f32(mx), step=step)
        check_caps(sk, vox, 0.0, step, om, monkeypatch, "white noise 64^3 step %d" % step)


@pytest.mark.parametrize("ndev", [2, 3, 5])
def test_forced_sub_slabs_on_a_multi_gpu_context(sk, monkeypatch, ndev):
    """Each device meshes its layer range in sub-slabs and moves the part's vertex ids to its global base."""
    import torch
    have = torch.cuda.device_count()
    ctx1 = sk.Context(0)
    mctx = sk.Context(devices=[k % have for k in range(ndev)])
    try:
        expr, mn, mx = scene("readme")
        for dims, iso in (((80, 64, 72), 0.0), ((70, 52, 33), 0.1)):
            one = sk.GpuSdf(expr, ctx=ctx1).ToVoxels(mn, mx, *dims).ToMesh(iso)
            vm = sk.GpuSdf(expr, ctx=mctx).ToVoxels(mn, mx, *dims)
            for cap in CAPS:
                m = create(sk, vm, iso, 1, cap, monkeypatch)[0]
                same_mesh(m, one,"%s iso %g, cap %d on %d devices" % (dims, iso, cap, ndev))
            vm.Dispose()
    finally:
        mctx.close()
        ctx1.close()


# ------------------------------------------------------------------------------------------ real sizes on one device

def need_device_bytes(nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info(0)
    if free < nbytes:
        pytest.skip("needs %.1f GB of free device memory, %.1f GB free (the device is shared)" % (nbytes / 1e9, free / 1e9))


def host_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def manifold_stats(tris, nverts):
    t = np.asarray(tris, dtype=np.int64).reshape(-1, 3)
    a = np.concatenate([t[:, 0], t[:, 1], t[:, 2]])
    b = np.concatenate([t[:, 1], t[:, 2], t[:, 0]])
    directed = a * nverts + b
    assert len(np.unique(directed)) == len(directed), "a directed edge occurs twice: inconsistent orientation"
    und = np.minimum(a, b) * nverts + np.maximum(a, b)
    uniq, cnt = np.unique(und, return_counts=True)
    return len(uniq), int(cnt.min()), int(cnt.max())


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_1664_cubed_voxels_mesh_on_one_device(sk):
    """1664^3 has 4.6e9 cells, more than one job's 32-bit ids: Voxels.ToMesh equals Sdf.ToMesh of the same grid."""
    n = 1664
    need_device_bytes(n ** 3 * 16 + (12 << 30))
    expr, mn, mx = scene("readme")
    sdf = expr.ToSdf()
    ref = sdf.ToMesh(mn, mx, n, n, n)
    ref = [np.array(a) for a in (ref.Vertices, ref.Colors, ref.Normals, ref.Triangles, ref.Min, ref.Max)]
    vox = sdf.ToVoxels(mn, mx, n, n, n)
    m = vox.ToMesh()
    for a, b, name in zip((m.Vertices, m.Colors, m.Normals), ref[:3], ("vertices", "colours", "normals")):
        assert np.array_equal(bits(a), bits(b)), name
    assert np.array_equal(np.asarray(m.Triangles), ref[3]), "triangles"
    assert np.array_equal(bits(m.Min), bits(ref[4])) and np.array_equal(bits(m.Max), bits(ref[5])), "AABB"
    # Voxels.Values of more than 2^32 voxels leave the device and come back through the import transpose
    if host_available_bytes() < 2 * n ** 3 * 4:
        vox.Dispose()
        pytest.skip("the export / import round trip needs %.0f GB of free host memory" % (2 * n ** 3 * 4 / 1e9))
    values = vox.Values
    vox.Dispose()
    back = sk.Voxels(values, None, mn, mx)
    del values
    m2 = back.ToMesh()
    back.Dispose()
    assert np.array_equal(bits(m2.Vertices), bits(m.Vertices)) and np.array_equal(bits(m2.Normals), bits(m.Normals))
    assert np.array_equal(np.asarray(m2.Triangles), np.asarray(m.Triangles))


def test_2048_cubed_voxels_mesh_on_one_device(sk):
    """BASELINE config 4 from resident voxels on ONE device: the golden digests and a closed 2-manifold."""
    n = 2048
    need_device_bytes(n ** 3 * 16 + (12 << 30))
    rec = json.load(open(os.path.join(HERE, "golden", "mesh_digests.json")))["readme"][str(n)]
    expr, mn, mx = scene("readme")
    vox = expr.ToSdf().ToVoxels(mn, mx, n, n, n)
    mesh = vox.ToMesh()
    vox.Dispose()
    nv, nt = len(mesh.Vertices), len(mesh.Triangles) // 3
    assert (nv, nt) == (rec["vertices"], rec["triangles"])
    got = {"vertices": sha(mesh.Vertices), "colors": sha(mesh.Colors), "normals": sha(mesh.Normals), "triangles": sha(mesh.Triangles)}
    assert got == rec["sha256"]
    nedges, cmin, cmax = manifold_stats(mesh.Triangles, nv)
    assert (cmin, cmax) == (2, 2), "not a closed 2-manifold"
    assert nv - nedges + nt == 2 * 25                             # 5 x 5 spheres
