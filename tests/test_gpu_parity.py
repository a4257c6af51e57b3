"""GPU parity tests: the CUDA path (through the C ABI / host mirror) against the CPU oracle on the same
inputs.  Bar (BASELINE.json north star): bit-exact cube indices, triangle counts and index buffers;
distances, colours and vertex positions within 1e-5 relative -- in practice these tests assert
bit-exact equality everywhere, because both sides perform the same IEEE operations (no FMA)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

f32 = np.float32


@pytest.fixture(scope="module")
def sk():
    import sdfkit_b200
    return sdfkit_b200


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_bits_equal(a, b, what):
    a, b = np.ascontiguousarray(a, dtype=np.float32), np.ascontiguousarray(b, dtype=np.float32)
    assert a.shape == b.shape, what
    same = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))
    if not same.all():
        bad = np.argwhere(~same)
        i = tuple(bad[0])
        raise AssertionError("%s: %d of %d values differ; first at %s: gpu=%r oracle=%r (max rel err %.3g)" % (
            what, len(bad), a.size, i, a[i], b[i], float(np.nanmax(np.abs(a - b) / np.maximum(np.abs(b), 1e-30)))))


def scenes_list(sk):
    from sdfkit_b200 import scenes
    return {"sphere": scenes.sphere(), "readme": scenes.readme_scene(), "perf": scenes.perf_scene(), "csg50": scenes.csg50()}


# ---------------------------------------------------------------------------------------------- sampling

@pytest.mark.parametrize("name,dims,clip", [
    ("sphere", (64, 64, 64), True),          # BASELINE config 1
    ("readme", (64, 64, 64), True),          # config 2 scene at test scale
    ("readme", (128, 128, 128), False),
    ("perf", (50, 37, 29), True),            # ragged: nx % 4 != 0 -> scalar store path
    ("csg50", (96, 96, 48), True),           # config 3 scene
    ("sphere", (1, 1, 1), False),            # Tests/VolumeTests.cs:39-58
    ("sphere", (5, 7, 11), True),
    ("readme", (260, 4, 3), True),           # partial last 128-voxel tile on the vector path
])
def test_sample_matches_oracle(sk, oracle, name, dims, clip):
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    vox = sdf.ToVoxels(mn, mx, nx, ny, nz, clipToBounds=clip)
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), nx, ny, nz, clip_to_bounds=clip, threads=4)
    assert_bits_equal(vox.Values, ov, "%s %s distances" % (name, dims))
    assert_bits_equal(vox.Colors, oc, "%s %s colours" % (name, dims))


def test_sample_reference_test_values(sk):
    # Tests/VolumeTests.cs:82-106,134 and Tests/SdfTests.cs:12-26 through the GPU path
    sdf = sk.SdfExprs.Sphere(0.5).ToSdf()
    v5 = sk.Voxels.SampleSdf(sdf, (-1, -1, -1), (1, 1, 1), 5, 5, 5)
    assert abs(v5[2, 2, 2] + 0.5) < 1e-3
    v128 = sdf.ToVoxels((-1, -1, -1), (1, 1, 1), 128, 128, 128)
    assert abs(v128[63, 63, 63] + 0.5) < 2e-2
    assert (v128.NX, v128.NY, v128.NZ) == (128, 128, 128)
    assert abs(v128.Size[0] - 2.0) < 1e-6


def test_sdf_delegate_matches_oracle(sk, oracle):
    rng = np.random.default_rng(3)
    pts = rng.uniform(-4, 4, (10007, 3)).astype(np.float32)
    for name, (expr, _, _) in scenes_list(sk).items():
        sdf = expr.ToSdf()
        out = np.zeros((len(pts), 4), dtype=np.float32)
        sdf(pts, out)
        assert_bits_equal(out, oracle.eval_sdf(sdf.lowered, pts), name + " delegate")
    assert sdf(np.zeros((0, 3), dtype=np.float32)).shape == (0, 4)


def test_opaque_sdf_is_rejected(sk):
    opaque = lambda pts, out: None     # the reference would run this on the CPU
    with pytest.raises(sk.NotSupportedError):
        sk.Voxels.SampleSdf(opaque, (-1, -1, -1), (1, 1, 1), 8, 8, 8)
    with pytest.raises(sk.NotSupportedError):
        sk.RayMarcher(8, 8, opaque)


def test_voxels_import_export_roundtrip(sk):
    rng = np.random.default_rng(5)
    vals = rng.uniform(-1, 1, (37, 21, 45)).astype(np.float32)
    cols = rng.uniform(0, 1, (37, 21, 45, 3)).astype(np.float32)
    v = sk.Voxels(vals, cols, (-1, -1, -1), (1, 1, 1))
    assert_bits_equal(v.Values, vals, "values roundtrip")
    assert_bits_equal(v.Colors, cols, "colours roundtrip")
    v.ClipToBounds()
    exp = vals.copy()
    for sl in [np.s_[0], np.s_[-1], np.s_[:, 0], np.s_[:, -1], np.s_[:, :, 0], np.s_[:, :, -1]]:
        exp[sl] = f32(2.0) / f32(37)
    assert_bits_equal(v.Values, exp, "ClipToBounds")


# ---------------------------------------------------------------------------------------------- marching cubes

def mesh_pair(sk, oracle, values, colors, mn, mx, iso=0.0, step=1):
    vox = sk.Voxels(values, colors, mn, mx)
    gm = sk.MarchingCubes.CreateGpuMesh(vox, iso, step)
    mesh = gm.download()
    om = oracle.marching_cubes(values, colors, np.float32(mn), np.float32(mx), iso=iso, step=step)
    return mesh, om, gm


def assert_mesh_equal(mesh, om, what):
    assert len(mesh.Vertices) == len(om.vertices), "%s: vertex count %d vs %d" % (what, len(mesh.Vertices), len(om.vertices))
    assert len(mesh.Triangles) == om.triangles.size, "%s: triangle count" % what
    assert np.array_equal(mesh.Triangles.reshape(-1, 3), om.triangles), what + ": triangle indices / order"
    assert_bits_equal(mesh.Vertices, om.vertices, what + " vertex positions")
    assert_bits_equal(mesh.Colors, om.colors, what + " vertex colours")
    assert_bits_equal(mesh.Normals, om.normals, what + " normals")
    if len(om.vertices):
        assert_bits_equal(mesh.Min, om.min, what + " aabb min")
        assert_bits_equal(mesh.Max, om.max, what + " aabb max")


@pytest.mark.parametrize("name,dims,clip", [
    ("sphere", (64, 64, 64), True),          # config 1: 4,874 active cells, 4,872 vertices, 9,740 triangles
    ("readme", (64, 64, 64), True),
    ("readme", (128, 128, 128), True),
    ("perf", (50, 37, 29), True),
    ("csg50", (96, 96, 48), True),
    ("sphere", (131, 9, 6), True),           # two 128-cell chunks per row, ragged
])
def test_mesh_matches_oracle(sk, oracle, name, dims, clip):
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    vox = sdf.ToVoxels(mn, mx, nx, ny, nz, clipToBounds=clip)
    mesh = vox.ToMesh()
    om = oracle.marching_cubes(vox.Values, vox.Colors, np.float32(mn), np.float32(mx))
    assert_mesh_equal(mesh, om, "%s %s" % (name, dims))
    if name == "sphere" and dims == (64, 64, 64):
        assert (len(om.vertices), len(om.triangles), om.active_cells) == (4872, 9740, 4874)
    assert len(om.vertices) > 0


def test_reference_goldens_through_gpu(sk, oracle):
    """The reference's vertex-count goldens (SURVEY.md 8c), meshed by the GPU path."""
    from oracle import sdf_numpy as S
    E = sk.SdfExprs
    # Tests/SdfTests.cs:42-52 (the one SdfExpr -> ToSdf -> ToMesh test) and :28-39
    assert len(E.Solid(lambda p: p.Length() - 0.5).ToSdf().ToMesh((-1, -1, -1), (1, 1, 1), 32, 32, 32).Vertices) == 1248
    assert len(E.Sphere(0.5).ToSdf().ToMesh((-1, -1, -1), (1, 1, 1), 32, 32, 32).Vertices) == 1248
    # Tests/MarchingCubesTests.cs: Sphere5 54, Sphere10 312, Unclipped 0, Clipped 384, Box10 384, Cylinder50 7456, Sphere128 72240
    def count(expr, mn, mx, n, clip):
        v = sk.Voxels.SampleSdf(expr.ToSdf(), mn, mx, n, n, n)
        if clip:
            v.ClipToBounds()
        return v.ToMesh()
    m = count(E.Sphere(1.0), (-1.5,) * 3, (1.5,) * 3, 5, False)
    assert len(m.Vertices) == 54 and np.linalg.norm(m.Center) < 1e-6 and abs(m.Size[0] / 2 - 1) < 0.3
    m = count(E.Sphere(2.0), (-2.5,) * 3, (2.5,) * 3, 10, False)
    assert len(m.Vertices) == 312 and np.linalg.norm(m.Center) < 1e-6
    m = count(E.Sphere(2.0), (-1,) * 3, (1,) * 3, 10, False)
    assert len(m.Vertices) == 0 and len(m.Triangles) == 0
    m = count(E.Sphere(2.0), (-1,) * 3, (1,) * 3, 10, True)
    assert len(m.Vertices) == 384 and abs(m.Size[0] - 2.0) < 1e-1
    m = count(E.Box(2.0), (-2.5,) * 3, (2.5,) * 3, 10, False)
    assert len(m.Vertices) == 384
    seen = []
    v = sk.Voxels.SampleSdf(E.Cylinder(1, 3).ToSdf(), (-1.5, -3.5, -1.5), (1.5, 3.5, 1.5), 50, 50, 50)
    assert len(v.ToMesh().Vertices) == 7456
    v = sk.Voxels.SampleSdf(E.Sphere(3.0).ToSdf(), (f32(-3.1),) * 3, (f32(3.1),) * 3, 128, 128, 128)
    m = v.ToMesh(progress=seen.append)
    assert len(m.Vertices) == 72240
    assert min(seen) < 1e-6 and max(seen) > 1 - 1e-6 and all(0 <= f <= 1 for f in seen)
    assert abs(m.Size[0] / 2 - 3.0) < 0.1
    # ColoredSpheres (opaque SdfFuncs in the reference): oracle-sampled voxels imported, meshed on the GPU
    fn = S.union(S.translate(S.with_color(S.sphere(f32(0.4)), (1.0, 0.2, 0.3)), (-1, 0, 0)),
                 S.translate(S.with_color(S.sphere(f32(0.2)), (0.1, 1.0, 0.3)), (1, 0, 0)))
    vals, cols = oracle.sample(oracle.numpy_sdf(fn), np.float32([-3] * 3), np.float32([3] * 3), 32, 32, 32)
    m = sk.Voxels(vals, cols, (-3,) * 3, (3,) * 3).ToMesh()
    assert len(m.Vertices) == 104 and m.Colors[0][0] > 0.5


@pytest.mark.parametrize("n,seed", [(24, 0), (64, 0), (33, 7)])
def test_white_noise_all_lewiner_cases(sk, oracle, n, seed):
    """Coverage input of SURVEY.md 8d: white noise reaches every ambiguous Lewiner branch (cases 3,4,6,7,10,12,13,
    face/interior tests, centre vertices) -- parity there is pinned only by the oracle restatement."""
    rng = np.random.default_rng(seed)
    vals = rng.uniform(-1, 1, (n, n, n)).astype(np.float32)
    cols = rng.uniform(0, 1, (n, n, n, 3)).astype(np.float32)
    mesh, om, gm = mesh_pair(sk, oracle, vals, cols, (-1, -1, -1), (1, 1, 1))
    assert all(om.case_hist[c] > 0 for c in range(1, 15)), om.case_hist
    assert_mesh_equal(mesh, om, "white noise %d" % n)


@pytest.mark.parametrize("dims", [(40, 23, 17), (130, 5, 4), (3, 3, 3), (2, 2, 2), (1, 4, 4), (4, 4, 1)])
def test_white_noise_ragged_grids(sk, oracle, dims):
    rng = np.random.default_rng(11)
    vals = rng.uniform(-1, 1, dims).astype(np.float32)
    cols = rng.uniform(0, 1, dims + (3,)).astype(np.float32)
    mesh, om, gm = mesh_pair(sk, oracle, vals, cols, (-1, -2, -3), (1, 2, 3))
    assert_mesh_equal(mesh, om, "ragged %s" % (dims,))


@pytest.mark.parametrize("step,iso", [(2, 0.0), (3, 0.0), (1, 0.25), (2, -0.1)])
def test_step_and_isovalue(sk, oracle, step, iso):
    """Public parameters of MarchingCubes.CreateMesh (MarchingCubes.cs:39) the reference's tests never vary."""
    rng = np.random.default_rng(2)
    vals = rng.uniform(-1, 1, (36, 31, 29)).astype(np.float32)
    cols = rng.uniform(0, 1, (36, 31, 29, 3)).astype(np.float32)
    mesh, om, gm = mesh_pair(sk, oracle, vals, cols, (-1, -1, -1), (1, 1, 1), iso=iso, step=step)
    assert len(om.vertices) > 0
    assert_mesh_equal(mesh, om, "step %d iso %g" % (step, iso))


def test_cube_index_census_matches(sk, oracle):
    """Cube indices / per-cell triangle counts: the GPU's totals must equal the oracle's per-cell debug arrays."""
    expr, mn, mx = scenes_list(sk)["readme"]
    vox = expr.ToSdf().ToVoxels(mn, mx, 64, 64, 64)
    gm = sk.MarchingCubes.CreateGpuMesh(vox)
    om = oracle.marching_cubes(vox.Values, vox.Colors, np.float32(mn), np.float32(mx), debug=True)
    active = int(((om.cell_index != 0) & (om.cell_index != 255)).sum())
    assert gm.stats()["active_cells"] == active == om.active_cells == 15218
    assert gm.counts() == (len(om.vertices), int(om.cell_ntris.sum())) == (15168, 30236)


# ---------------------------------------------------------------------------------------------- ray marcher

@pytest.mark.parametrize("name,w,h", [("readme", 192, 108), ("perf", 101, 57), ("csg50", 64, 48), ("sphere", 50, 30)])
def test_render_matches_oracle(sk, oracle, name, w, h):
    from sdfkit_b200 import numerics, scenes
    expr, _, _ = scenes_list(sk)[name]
    sdf = expr.ToSdf()
    img = sdf.ToImage(w, h, *scenes.CAMERA)
    view = numerics.create_look_at(*scenes.CAMERA)
    ref = oracle.render(sdf.lowered, w, h, view=view, bands=4)
    assert img.Array.shape == (h, w, 3)
    assert_bits_equal(img.Array, ref, name + " ToImage")
    assert np.isfinite(img.Array).all() and img.Array.max() <= 1.1 + 1e-6


def test_render_depth_goldens_and_parity(sk, oracle):
    # Tests/RayMarcherTests.cs:10-75 with SdfExpr equivalents of the opaque Sdfs
    E = sk.SdfExprs
    w, h = 50, 30
    sphere = sk.RayMarcher(w, h, E.Sphere(1.0).ToSdf()).RenderDepth()
    assert (sphere.Width, sphere.Height) == (w, h)
    assert abs(sphere[w // 2, h // 2] - 4.0) < 1e-2 and sphere[0, 0] > 9.0
    box = sk.RayMarcher(w, h, E.Box(1.0).ToSdf()).RenderDepth()
    assert abs(box[w // 2, h // 2] - 4.0) < 1e-2 and box[0, 0] > 9.0
    r = f32(0.25)
    cyl_sdf = E.Cylinder(r, r * 2).RepeatX(4 * r).ToSdf()
    cyl = sk.RayMarcher(w, h, cyl_sdf).RenderDepth()
    assert abs(cyl[w // 2, h // 2 - 2] - (5 - r)) < 1e-1 and cyl[0, 0] > 9.0
    plane = sk.RayMarcher(w, h, E.Solid(lambda p: p.Z).ToSdf()).RenderDepth()       # Sdfs.PlaneXY()
    assert abs(plane[w // 2, h // 2] - 5.0) < 1e-2 and plane[0, 0] < 9.0
    assert_bits_equal(cyl.Array, oracle.render_depth(cyl_sdf.lowered, w, h), "cylinder depth")


def test_render_row_bands_equal_full_image(sk):
    from sdfkit_b200 import scenes
    expr, _, _ = scenes.readme_scene()
    rm = sk.RayMarcher(160, 90, expr.ToSdf())
    from sdfkit_b200 import numerics
    rm.ViewTransform = numerics.create_look_at(*scenes.CAMERA)
    full = rm.Render().Array
    parts = [rm.Render(r0, r1).Array for r0, r1 in [(0, 23), (23, 46), (46, 69), (69, 90)]]
    assert_bits_equal(np.concatenate(parts), full, "row bands")


# ---------------------------------------------------------------------------------------------- z-slab sharding

@pytest.mark.parametrize("nslabs,step", [(2, 1), (3, 1), (8, 1), (2, 2)])
def test_slab_sharded_mesh_equals_single_gpu(sk, oracle, nslabs, step):
    """SURVEY.md 8e: an N-rank z-slab job (emulated sequentially on one GPU: slab sampling with halo, ghost-layer
    classification, offsets from the count exchange) must reproduce the single-GPU mesh exactly."""
    from sdfkit_b200 import dist, scenes
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    n = 72
    whole = sdf.ToMesh(mn, mx, n, n, n, step=step)
    sharded = dist.to_mesh_by_slabs(sdf, mn, mx, n, n, n, nslabs, step=step)
    assert len(whole.Vertices) > 0
    assert np.array_equal(sharded.Triangles, whole.Triangles)
    assert_bits_equal(sharded.Vertices, whole.Vertices, "slab vertices")
    assert_bits_equal(sharded.Colors, whole.Colors, "slab colours")
    assert_bits_equal(sharded.Normals, whole.Normals, "slab normals")
    assert_bits_equal(sharded.Min, whole.Min, "slab aabb")
    assert_bits_equal(sharded.Max, whole.Max, "slab aabb")


def test_layer_ranges_on_white_noise(sk, oracle):
    """Ghost-layer logic on the hardest input: mesh cell-layer ranges of a white-noise grid separately (all ambiguous
    cases, centre vertices on slab boundaries) and compare the concatenation with the oracle's whole mesh."""
    import ctypes as C
    from sdfkit_b200 import _native as N, dist, numerics
    rng = np.random.default_rng(21)
    n = 30
    vals = rng.uniform(-1, 1, (n, n, n)).astype(np.float32)
    cols = rng.uniform(0, 1, (n, n, n, 3)).astype(np.float32)
    vox = sk.Voxels(vals, cols, (-1, -1, -1), (1, 1, 1))
    om = oracle.marching_cubes(vals, cols, np.float32([-1] * 3), np.float32([1] * 3))
    M, Nn = numerics.mesh_transforms(vox.Min, vox.Max, n, n, n)
    M, Nn = N.f32c(M), N.f32c(Nn)
    ranges = [(0, 7), (7, 8), (8, 20), (20, 29)]
    meshes, counts = [], []
    for kb, ke in ranges:
        h, nv, nt = C.c_void_p(), C.c_int64(), C.c_int64()
        N.check(N.lib().sdfk_mesh_classify(vox.ctx.handle, vox.handle, 0.0, 1, kb, ke, C.byref(h), C.byref(nv), C.byref(nt)))
        meshes.append(sk.GpuMesh(h))
        counts.append((nv.value, nt.value))
    excl, tot = dist.exclusive_offsets(counts)
    assert tuple(tot) == (len(om.vertices), len(om.triangles))
    parts = []
    for m, (vb, tb) in zip(meshes, excl):
        N.check(N.lib().sdfk_mesh_emit(m.handle, int(vb), int(tb), N.fptr(M), N.fptr(Nn)))
        parts.append(m.download())
    merged = dist.merge_meshes(parts)
    assert_mesh_equal(merged, om, "white noise layer ranges")


def test_interleaved_slabs_equal_single_gpu(sk):
    """Round-robin multi-slab sharding (dist.ShardedMesher, what bench.py runs on N > 2 GPUs), emulated in one process:
    3 ranks x 2 slabs each must reproduce the single-GPU mesh exactly."""
    from sdfkit_b200 import dist, scenes
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    n, world, spr = 80, 3, 2
    whole = sdf.ToMesh(mn, mx, n, n, n)
    jobs = [dist.ShardedMesher(sdf, mn, mx, n, n, n, r, world, spr) for r in range(world)]
    counts = np.stack([j.sample_classify() for j in jobs])          # what the all-gather delivers to every rank
    parts = {}
    for j in jobs:
        offs, tot = j.offsets(counts)
        j.emit(offs)
        assert tuple(tot) == (len(whole.Vertices), len(whole.Triangles) // 3)
        for g, s in zip(j.slab_ids, j.slabs):
            parts[g] = s.mesh.download()
    merged = dist.merge_meshes([parts[g] for g in sorted(parts)])
    assert np.array_equal(merged.Triangles, whole.Triangles)
    assert_bits_equal(merged.Vertices, whole.Vertices, "interleaved slab vertices")
    assert_bits_equal(merged.Normals, whole.Normals, "interleaved slab normals")
    assert_bits_equal(merged.Colors, whole.Colors, "interleaved slab colours")
    for j in jobs:
        j.close()


def test_cost_balanced_slabs_equal_single_gpu(sk):
    """The cost-balanced partition (dist.plan_layers) only moves the cuts: the merged mesh must not change, and the
    slabs that hold the surface must come out thinner than the empty ones."""
    from sdfkit_b200 import dist, scenes
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    n, world = 96, 4
    whole = sdf.ToMesh(mn, mx, n, n, n)
    jobs = [dist.ShardedMesher(sdf, mn, mx, n, n, n, r, world, 1, balanced=True) for r in range(world)]
    layers = jobs[0].layers
    assert all(j.layers == layers for j in jobs) and layers[0][0] == 0 and layers[-1][1] == n - 1
    thick = [b - a for a, b in layers]
    assert min(thick[1:3]) < max(thick[0], thick[3])          # the spheres sit in the middle of z
    counts = np.stack([j.sample_classify() for j in jobs])
    parts = []
    for j in jobs:
        offs, _ = j.offsets(counts)
        j.emit(offs)
        parts.append(j.slabs[0].mesh.download())
    merged = dist.merge_meshes(parts)
    assert np.array_equal(merged.Triangles, whole.Triangles)
    assert_bits_equal(merged.Vertices, whole.Vertices, "balanced slab vertices")
    assert_bits_equal(merged.Normals, whole.Normals, "balanced slab normals")
    for j in jobs:
        j.close()


@pytest.mark.parametrize("name,dims,step", [("readme", (64, 64, 64), 1), ("perf", (50, 37, 29), 1), ("csg50", (96, 96, 48), 1),
                                            ("readme", (72, 72, 72), 2),
                                            ("readme", (256, 40, 70), 1), ("csg50", (512, 24, 33), 1), ("perf", (256, 9, 5), 2)])   # rows of whole tile pairs: the 8-voxels-per-lane sampler
def test_fused_to_mesh_equals_voxels_to_mesh(sk, oracle, name, dims, step):
    """Sdf.ToMesh samples distances only and evaluates vertex colours from the SDF (SURVEY.md 8f row 1): the mesh must be
    identical to the one made from fully materialised Voxels -- and to the oracle's."""
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    fused = sdf.ToMesh(mn, mx, nx, ny, nz, step=step)
    full = sdf.ToVoxels(mn, mx, nx, ny, nz).ToMesh(step=step)
    assert len(fused.Vertices) > 0
    assert np.array_equal(fused.Triangles, full.Triangles)
    assert_bits_equal(fused.Vertices, full.Vertices, "fused vertices")
    assert_bits_equal(fused.Normals, full.Normals, "fused normals")
    assert_bits_equal(fused.Colors, full.Colors, "fused colours")
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), nx, ny, nz, threads=4)
    om = oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx), step=step)
    assert_mesh_equal(fused, om, "fused %s" % name)


@pytest.mark.parametrize("dims,clip", [((256, 33, 70), True), ((512, 5, 40), False), ((256, 3, 3), True)])
def test_distance_only_sampler_8_per_lane_values_and_sign_blocks(sk, oracle, dims, clip):
    """sdfk_k_sample_dist8 (rows of whole tile pairs): distances equal the oracle's, and meshing from its sign blocks equals
    meshing from the distances."""
    from sdfkit_b200 import _native as N, scenes
    expr, mn, mx = scenes.readme_scene()
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    v = sk.Voxels._sample(sdf, mn, mx, nx, ny, nz, clip=clip, colors=False)
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), nx, ny, nz, clip_to_bounds=clip, threads=4)
    assert_bits_equal(v.Values, ov, "distances %s" % (dims,))
    a = v.ToMesh()
    sdf.ctx.set_option(N.OPT_SIGN_PLANES, 0)
    try:
        v2 = sk.Voxels._sample(sdf, mn, mx, nx, ny, nz, clip=clip, colors=False)
        b = v2.ToMesh()
    finally:
        sdf.ctx.set_option(N.OPT_SIGN_PLANES, 1)
    assert np.array_equal(a.Triangles, b.Triangles) and np.array_equal(bits(a.Vertices), bits(b.Vertices))
    assert np.array_equal(bits(a.Colors), bits(b.Colors)) and np.array_equal(bits(a.Normals), bits(b.Normals))


def test_distance_only_voxels_refuse_colors(sk):
    from sdfkit_b200 import scenes
    expr, mn, mx = scenes.readme_scene()
    v = sk.Voxels._sample(expr.ToSdf(), mn, mx, 16, 16, 16, clip=True, colors=False)
    assert v.Values.shape == (16, 16, 16)
    with pytest.raises(sk.SdfkError, match="hold no colours"):
        v.Colors


# ---------------------------------------------------------------------------------------------- sign planes (K2')

@pytest.mark.parametrize("name,dims,clip", [("readme", (64, 64, 64), True), ("perf", (50, 37, 29), True), ("readme", (260, 9, 7), True),
                                            ("csg50", (129, 40, 33), False), ("readme", (257, 6, 5), True), ("sphere", (2, 2, 2), False),
                                            ("readme", (128, 128, 20), True)])
def test_sign_plane_classify_equals_distance_classify(sk, oracle, name, dims, clip):
    """Marching cubes at iso 0 / step 1 finds the active cells from the sign planes the sampling kernel wrote (K2'); with the
    option off it reads the distances (K2).  Both must give the oracle's mesh, for ragged rows (nx % 128 in {0, 1, 2, 4, ...})
    and partial last tiles too."""
    from sdfkit_b200 import _native as N
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    ctx = sdf.ctx
    meshes = {}
    try:
        for opt in (1, 0):
            ctx.set_option(N.OPT_SIGN_PLANES, opt)
            vox = sdf.ToVoxels(mn, mx, nx, ny, nz, clipToBounds=clip)
            gm = sk.MarchingCubes.CreateGpuMesh(vox)
            assert gm.stats()["from_signs"] == bool(opt)
            meshes[opt] = gm.download()
            gm.destroy()
            fused = sdf.ToMesh(mn, mx, nx, ny, nz, clipToBounds=clip)
            assert np.array_equal(fused.Triangles, meshes[opt].Triangles)
            assert_bits_equal(fused.Vertices, meshes[opt].Vertices, "fused vertices (sign planes %d)" % opt)
    finally:
        ctx.set_option(N.OPT_SIGN_PLANES, 1)
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), nx, ny, nz, clip_to_bounds=clip, threads=4)
    om = oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx))
    for opt in (1, 0):
        assert_mesh_equal(meshes[opt], om, "%s %s sign planes %d" % (name, dims, opt))


def test_sign_planes_follow_the_stored_values(sk, oracle):
    """The sign planes describe the values actually stored: a later ClipToBounds invalidates them (K2 takes over), another
    iso value or step ignores them -- the mesh is the oracle's in every case."""
    from sdfkit_b200 import scenes
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    n = 48
    vox = sk.Voxels.SampleSdf(sdf, mn, mx, n, n, n)          # unclipped
    vox.ClipToBounds()
    gm = sk.MarchingCubes.CreateGpuMesh(vox)
    assert gm.stats()["from_signs"] is False
    m = gm.download()
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), n, n, n, clip_to_bounds=True, threads=4)
    assert_mesh_equal(m, oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx)), "clip after sampling")
    vox2 = sdf.ToVoxels(mn, mx, n, n, n)
    for iso, step in ((0.125, 1), (0.0, 2)):
        gm = sk.MarchingCubes.CreateGpuMesh(vox2, iso, step)
        assert gm.stats()["from_signs"] is False
        assert_mesh_equal(gm.download(), oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx), iso=iso, step=step), "iso %g step %d" % (iso, step))
    gm = sk.MarchingCubes.CreateGpuMesh(vox2)
    assert gm.stats()["from_signs"] is True


# ---------------------------------------------------------------------------------------------- pipelined Sdf.ToMesh

@pytest.mark.parametrize("name,dims,slabs,step,iso", [
    ("readme", (64, 64, 64), 1, 1, 0.0), ("readme", (64, 64, 64), 2, 1, 0.0), ("readme", (64, 64, 64), 5, 1, 0.0),
    ("readme", (64, 64, 64), 63, 1, 0.0), ("perf", (50, 37, 29), 3, 1, 0.0), ("csg50", (96, 96, 48), 4, 1, 0.0),
    ("readme", (72, 72, 72), 3, 2, 0.0), ("readme", (64, 64, 64), 4, 1, 0.125), ("sphere", (2, 2, 2), 0, 1, 0.0),
    ("sphere", (1, 1, 1), 0, 1, 0.0), ("readme", (260, 40, 300), 0, 1, 0.0)])
def test_pipelined_to_mesh_host(sk, oracle, name, dims, slabs, step, iso):
    """Sdf.ToMesh = sdfk_sdf_to_mesh_host: z-slabs software-pipelined on the device, mesh parts streamed to page-locked host
    memory.  Any slab count must give the oracle's mesh, bit for bit and in the reference's order."""
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    seen = []
    mesh = sdf.ToMesh(mn, mx, nx, ny, nz, isoValue=iso, step=step, slabs=slabs, progress=seen.append)
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), nx, ny, nz, threads=4)
    oseen = []
    om = oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx), iso=iso, step=step, progress=oseen.append)
    assert_mesh_equal(mesh, om, "pipelined %s %s slabs=%d" % (name, dims, slabs))
    assert np.array_equal(np.float32(seen), np.float32(oseen), equal_nan=True)   # IProgress<float> reports (MarchingCubes.cs:81); 0/0 on a 2^3 grid


def test_pipelined_to_mesh_buffers_are_recycled_safely(sk):
    """The page-locked arrays belong to the mesh: a second ToMesh must not overwrite the first one's data while it is alive."""
    from sdfkit_b200 import scenes
    e1, mn, mx = scenes.readme_scene()
    e2, mn2, mx2 = scenes.sphere()
    s1, s2 = e1.ToSdf(), e2.ToSdf()
    a = s1.ToMesh(mn, mx, 64, 64, 64)
    va, ta = a.Vertices.copy(), a.Triangles.copy()
    b = s2.ToMesh(mn2, mx2, 64, 64, 64)
    assert np.array_equal(a.Vertices, va) and np.array_equal(a.Triangles, ta)
    assert len(b.Vertices) == 4872 and len(b.Triangles) == 3 * 9740          # BASELINE config 1 counts
    del a
    c = s1.ToMesh(mn, mx, 64, 64, 64)                                        # reuses a's buffers
    assert np.array_equal(c.Vertices, va) and np.array_equal(c.Triangles, ta)
    assert len(b.Vertices) == 4872


@pytest.mark.parametrize("nslabs,chunks,colors", [(1, 0, True), (1, 5, False), (3, 4, False), (4, 16, True)])
def test_chunked_emit_to_host_equals_single_gpu(sk, oracle, nslabs, chunks, colors):
    """sdfk_mesh_emit_host (every rank's share of the mesh emitted in sub-ranges and streamed to its own page-locked host
    memory, global indices from the count all-gather): the concatenated shares are the single-GPU mesh, bit for bit."""
    from sdfkit_b200 import dist, scenes
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    n = 96
    whole = sdf.ToVoxels(mn, mx, n, n, n).ToMesh()
    jobs = [dist.ShardedMesher(sdf, mn, mx, n, n, n, r, nslabs, 1, colors=colors) for r in range(nslabs)]
    counts = np.stack([j.sample_classify() for j in jobs])
    parts = []
    for j in jobs:
        offs, tot = j.offsets(counts)
        parts += j.emit_host(offs, chunks)
    assert int(tot[0]) == len(whole.Vertices)
    merged = dist.merge_meshes(parts)
    assert np.array_equal(merged.Triangles, whole.Triangles)
    assert_bits_equal(merged.Vertices, whole.Vertices, "emit_host vertices")
    assert_bits_equal(merged.Normals, whole.Normals, "emit_host normals")
    assert_bits_equal(merged.Colors, whole.Colors, "emit_host colours")
    assert_bits_equal(merged.Min, whole.Min, "emit_host aabb min")
    assert_bits_equal(merged.Max, whole.Max, "emit_host aabb max")
    for j in jobs:
        j.close()


# ---------------------------------------------------------------------------------------------- packed (f32x2) evaluator

@pytest.mark.parametrize("name,dims", [("sphere", (33, 20, 17)), ("readme", (64, 64, 64)), ("perf", (50, 37, 29)), ("csg50", (96, 96, 48))])
def test_default_device_forms_equal_plain_scalar_body(sk, oracle, monkeypatch, name, dims):
    """The shared-guard device forms (default) and the plain scalar body (SDFK_PLAIN_BODY=1: what a host that only sends the
    scalar body gets) give identical voxels, meshes and images -- and both equal the oracle (other tests)."""
    from sdfkit_b200 import numerics, scenes
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    res = []
    for plain in ("0", "1"):
        monkeypatch.setenv("SDFK_PLAIN_BODY", plain)
        sdf = expr.ToSdf()
        vox = sdf.ToVoxels(mn, mx, nx, ny, nz)
        mesh = sdf.ToMesh(mn, mx, nx, ny, nz)
        img = sdf.ToImage(97, 55, *scenes.CAMERA)
        pts = np.random.default_rng(11).uniform(-4, 4, (5001, 3)).astype(np.float32)
        pts[:7] = [[0, 0, 0], [1.125, 0, 0], [-0.0, 0.0, -0.0], [1e-30, 0, 0], [3e38, 0, 0], [np.inf, 0, 0], [np.nan, 1, 1]]
        res.append((vox.Values.copy(), vox.Colors.copy(), mesh.Vertices.copy(), mesh.Colors.copy(), mesh.Normals.copy(), np.asarray(mesh.Triangles).copy(),
                    img.Array.copy(), sdf(pts)))
    for a, b in zip(*res):
        if a.dtype == np.float32:
            assert_bits_equal(a, b, name)
        else:
            assert np.array_equal(a, b)
    ref = oracle.eval_sdf(sdf.lowered, pts[:5])
    assert_bits_equal(res[0][7][:5], ref, name + " special points vs oracle")


def test_color_table_rewrite_is_bit_identical(sk, oracle, monkeypatch):
    """Opt-in colour-table form of a union of constant-coloured primitives (exprs._color_table_rewrite): same voxels and image."""
    import importlib
    from sdfkit_b200 import exprs, scenes
    expr, mn, mx = scenes.csg50()
    monkeypatch.setattr(exprs, "_CTAB", True)
    sdf = expr.ToSdf()
    assert "sdfk_ctab" in sdf.lowered.decls
    vox = sdf.ToVoxels(mn, mx, 96, 96, 48)
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), 96, 96, 48, clip_to_bounds=True, threads=4)
    assert_bits_equal(vox.Values, ov, "distances")
    assert_bits_equal(vox.Colors, oc, "colours")
    img = sdf.ToImage(64, 48, *scenes.CAMERA)
    from sdfkit_b200 import numerics
    assert_bits_equal(img.Array, oracle.render(sdf.lowered, 64, 48, view=numerics.create_look_at(*scenes.CAMERA), bands=2), "image")


def test_packed_sqrt_is_exhaustively_exact(sk):
    """sk2_sqrt (csrc/sdfk_prelude.h) against sqrt.rn.f32 for ALL 2^32 arguments (and scrambled partners in the other half)."""
    from sdfkit_b200 import _native as N
    assert N.Context.default().selftest_sqrt() == 0


@pytest.mark.parametrize("divisor", [1.125, 6.0, 3.0, 0.1, 7.0, 2.5, 1e-3, 1023.0, 0.33333334, 1.9999999, 1.0000001, -5.0])
def test_constant_division_is_exhaustively_exact(sk, divisor):
    """sk2_divc for this constant against div.rn.f32 for ALL 2^32 dividends; the lowering only uses it after this check."""
    import ctypes as C
    from sdfkit_b200 import _native as N
    ctx = N.Context.default()
    bad = C.c_int64(-1)
    N.check(N.lib().sdfk_constdiv_verify(ctx.handle, C.c_float(divisor), C.byref(bad)))
    assert bad.value == 0, "%d of 2^32 dividends differ for divisor %r" % (bad.value, divisor)
    assert ctx.constdiv_ok(divisor) is True
    assert ctx.constdiv_ok(0.0) is False and ctx.constdiv_ok(float("inf")) is False and ctx.constdiv_ok(1e-20) is False


def test_packed_body_uses_verified_fast_division(sk, monkeypatch):
    from sdfkit_b200 import scenes
    monkeypatch.setenv("SDFK_PACKED", "1")
    sdf = scenes.readme_scene()[0].ToSdf()
    assert "sk2_divc(" in sdf.lowered.body2 and len(sdf.lowered.fast_div) == 2      # / 1.125 and / 6
    assert "sk2_sqrt(" in sdf.lowered.body2 and "sk2_add_s(" in sdf.lowered.body2
    assert "sk2_" not in sdf.lowered.body                                            # the scalar body (what the oracle compiles) is untouched


@pytest.mark.parametrize("name,dims", [("sphere", (33, 20, 17)), ("readme", (64, 64, 64)), ("perf", (50, 37, 29)), ("csg50", (96, 96, 48))])
def test_packed_evaluator_is_bit_identical(sk, oracle, monkeypatch, name, dims):
    """SDFK_PACKED=1 (two points per instruction on the f32x2 pipe; off by default because it measured slower): voxels, mesh,
    delegate and image are still the oracle's, bit for bit."""
    from sdfkit_b200 import numerics, scenes
    monkeypatch.setenv("SDFK_PACKED", "1")
    expr, mn, mx = scenes_list(sk)[name]
    nx, ny, nz = dims
    sdf = expr.ToSdf()
    assert sdf.lowered.body2 and "sk2_" in sdf.lowered.body2
    vox = sdf.ToVoxels(mn, mx, nx, ny, nz)
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), nx, ny, nz, threads=4)
    assert_bits_equal(vox.Values, ov, name + " packed distances")
    assert_bits_equal(vox.Colors, oc, name + " packed colours")
    assert_mesh_equal(sdf.ToMesh(mn, mx, nx, ny, nz), oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx)), name + " packed ToMesh")
    pts = np.random.default_rng(5).uniform(-4, 4, (4099, 3)).astype(np.float32)
    assert_bits_equal(sdf(pts), oracle.eval_sdf(sdf.lowered, pts), name + " packed delegate")
    img = sdf.ToImage(97, 41, *scenes.CAMERA)
    ref = oracle.render(sdf.lowered, 97, 41, view=numerics.create_look_at(*scenes.CAMERA), bands=2)
    assert_bits_equal(img.Array, ref, name + " packed image")


def test_nan_and_inf_distances_classify_like_the_reference(sk, oracle):
    """An SDF that produces NaN (sqrt of a negative number) and +-inf (division by zero): `value > iso` is false for NaN in the
    reference (Cell.cs:221-228), so NaN corners count as inside.  Sign blocks (K2'), the distance classifier (K2) and the oracle
    must agree on the active cells and the index buffer (positions next to a NaN are NaN themselves: compared as bits)."""
    from sdfkit_b200 import _native as N
    expr = sk.SdfExprs.Solid(lambda p: sk.MathF.Sqrt(p.X + 0.31) + (p.Y * p.Y + p.Z * p.Z - 0.36) / (p.Z * p.Z))
    sdf = expr.ToSdf()
    mn, mx, n = (-1, -1, -1), (1, 1, 1), 33                      # 33: z = 0 is sampled exactly -> a division by zero plane
    ov, oc = oracle.to_voxels(sdf.lowered, np.float32(mn), np.float32(mx), n, n, n, threads=4)
    assert np.isnan(ov).any() and np.isinf(ov).any()
    om = oracle.marching_cubes(ov, oc, np.float32(mn), np.float32(mx))
    ctx = sdf.ctx
    try:
        for opt in (1, 0):
            ctx.set_option(N.OPT_SIGN_PLANES, opt)
            vox = sdf.ToVoxels(mn, mx, n, n, n)
            assert_bits_equal(vox.Values, ov, "NaN/inf distances")
            m = vox.ToMesh()
            assert np.array_equal(m.Triangles.reshape(-1, 3), om.triangles), "sign planes %d" % opt
            assert_bits_equal(m.Vertices, om.vertices, "vertices (sign planes %d)" % opt)
            assert_bits_equal(m.Normals, om.normals, "normals (sign planes %d)" % opt)
            f = sdf.ToMesh(mn, mx, n, n, n, slabs=3)
            assert np.array_equal(f.Triangles, m.Triangles)
            assert_bits_equal(f.Vertices, m.Vertices, "pipelined vertices (sign planes %d)" % opt)
    finally:
        ctx.set_option(N.OPT_SIGN_PLANES, 1)


def test_delegate_edge_cases(sk, oracle):
    from sdfkit_b200 import scenes
    sdf = scenes.perf_scene()[0].ToSdf()
    assert sdf(np.zeros((0, 3), dtype=np.float32)).shape == (0, 4)                      # empty batch
    one = np.float32([[0.25, -0.5, 1.0]])
    assert_bits_equal(sdf(one), oracle.eval_sdf(sdf.lowered, one), "single point")       # odd count: the pair kernel's tail
    odd = np.random.default_rng(1).uniform(-3, 3, (2049, 3)).astype(np.float32)          # one more than the reference's batch size
    assert_bits_equal(sdf(odd), oracle.eval_sdf(sdf.lowered, odd), "2049 points")
    with pytest.raises(ValueError):
        sdf(odd, np.zeros((5, 4), dtype=np.float32))


def test_render_tga_on_device_equals_save_tga(sk, tmp_path):
    """sdfk_render_bgr8: the TGA payload packed on the device is byte-identical to Render().SaveTga() (VectorData.cs:570-619)."""
    from sdfkit_b200 import numerics, scenes
    for name in ("readme", "perf"):
        sdf = scenes_list(sk)[name][0].ToSdf()
        rm = sk.RayMarcher(203, 77, sdf)
        rm.ViewTransform = numerics.create_look_at(*scenes.CAMERA)
        a, b = tmp_path / (name + "_host.tga"), tmp_path / (name + "_dev.tga")
        rm.Render().SaveTga(str(a))
        rm.RenderTga(str(b))
        assert a.read_bytes() == b.read_bytes()
        assert len(b.read_bytes()) == 18 + 203 * 77 * 3


def test_host_mesh_transform_equals_the_fused_device_transform(sk):
    """Mesh.Transform (Mesh.cs:47-64) applied on the host to an index-space mesh gives, bit for bit, the mesh whose transform was
    fused into the emit kernel (MarchingCubes.cs:85-90)."""
    from sdfkit_b200 import numerics, scenes
    expr, mn, mx = scenes.perf_scene()
    vox = expr.ToSdf().ToVoxels(mn, mx, 50, 37, 29)
    world = vox.ToMesh()
    gm = sk.MarchingCubes.CreateGpuMesh(vox, transform=False)
    index_space = gm.download()
    M, _ = numerics.mesh_transforms(vox.Min, vox.Max, vox.NX, vox.NY, vox.NZ)
    index_space.Transform(M)
    assert_bits_equal(index_space.Vertices, world.Vertices, "host-transformed vertices")
    assert_bits_equal(index_space.Normals, world.Normals, "host-transformed normals")
    assert_bits_equal(index_space.Min, world.Min, "aabb min")
    assert_bits_equal(index_space.Max, world.Max, "aabb max")
    f = expr.ToSdfFunc()                                            # SdfExprEx.ToSdfFunc: one point at a time
    assert f((0.1, 0.2, 0.3)).shape == (4,)


def test_store_bandwidth_probe(sk):
    """sdfk_ctx_store_bandwidth (bench.py's `write_only_peak`): a plausible HBM rate, and loud on bad arguments."""
    from sdfkit_b200 import _native as N
    ctx = sk.Context(0)
    g = ctx.store_bandwidth(1 << 30, 2)
    assert 1.0 < g < 20000.0                    # (GB/s; orders of magnitude slower under compute-sanitizer)
    with pytest.raises(N.SdfkError):
        ctx.store_bandwidth(1024, 1)            # less than one 16 KiB chunk
    ctx.close()


def test_bench_dump_outputs_is_the_mesh_of_the_timed_step(sk, tmp_path):
    """`bench.py --dump-outputs DIR` writes the mesh of the last timed step.  On a grid small enough to keep every row, that
    is the mesh Sdf.ToMesh makes of the same grid, bit for bit; the JSON line reports the --steps asked for."""
    import json
    import os
    import subprocess
    import sys
    from sdfkit_b200 import scenes
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = 96
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "0", "--grid", str(n), "--no-cpu", "--no-configs",
           "--no-strong", "--no-e2e", "--no-fused", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    expr, mn, mx = scenes.readme_scene()
    m = expr.ToSdf().ToMesh(mn, mx, n, n, n)
    d = {k: np.load(tmp_path / (k + ".npy")) for k in ("counts", "vertex_rows", "triangle_rows", "vertices", "colors", "normals", "triangles")}
    nv, nt = len(m.Vertices), len(m.Triangles) // 3
    assert d["counts"].tolist() == [nv, nt] == [line["vertices"], line["triangles"]]
    assert np.array_equal(d["vertex_rows"], np.arange(nv)) and np.array_equal(d["triangle_rows"], np.arange(nt))
    for k in ("vertices", "colors", "normals"):
        assert d[k].dtype == np.float32
        assert_bits_equal(d[k], getattr(m, k.capitalize()), k)
    assert d["triangles"].dtype == np.float64 and np.array_equal(d["triangles"], np.asarray(m.Triangles).reshape(-1, 3))
