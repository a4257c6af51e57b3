#!/usr/bin/env python3
"""bench.py -- the SdfKit hot path on B200: SdfExpr.ToSdf() -> Voxels sampling -> MarchingCubes meshing.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--grid N] [--scene readme|csg50|sphere]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one grid of the README RepeatXY scene (BASELINE.json): sample every
voxel (distance + colour, clip to bounds) into HBM, then mesh it (classify -> scan -> compact -> emit).  The SDF
is analytic, so the step has no input arrays: "inputs resident in HBM" is the compiled SDF module.
  N = 1: 1024^3 (the size BASELINE.json's metric is quoted on; 17.2 GB of voxels, fits one B200).
  N > 1: weak scaling -- an n^3 grid with n^3 ~= N * 1024^3 (2048^3 at N = 8, BASELINE config 4), z-slab sharded:
         every rank samples its slices + halo, classifies, the ranks all-gather their (vertices, triangles)
         counts over NCCL, and each emits its part of the mesh at the resulting global offsets.
`value` = voxels of the whole job / step time (device events, max over ranks).  `e2e` = the same metric through
the public API Sdf.ToMesh (host result: the mesh is copied back to host memory every step).
Outside the timed regions the line also carries
  parity_check (N > 1)  the N-rank job's output proven on the hardware it ran on: rank-ordered shares == the single-GPU
                        mesh (arrays and sha256 vs tests/golden/mesh_digests.json), slab boundaries == the CPU oracle;
  strong_1024           the SAME 1024^3 job on 1/2/4/.. GPUs through the multi-GPU context of the C ABI
                        (sdfk_ctx_create_multi: one process, N devices, one host mesh), device step and e2e;
  configs (N = 1)       BASELINE configs 3 (CSG-50 1024^3, FP32-bound) and 5 (ToImage 1920x1080, Perf/Program.cs protocol)
                        with their own FP32 rooflines and CPU baselines, and the Voxels.Values/Colors export rate.
--impl reference times the CPU restatement of the reference (the oracle) on a bounded sample of the workload.
--dump-outputs DIR writes the mesh of the last timed step as DIR/<name>.npy, so that two builds can be compared output for
output (the inputs are the same in every run: an analytic SDF on a fixed grid).
bench.py writes nothing into the tree it runs from, which may be read-only: the oracle compiles into a temporary directory.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True          # no __pycache__ in the tree for modules build() did not import
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "voxel_samples_per_s"
UNIT = "voxels/s"
WEAK_GRID = {1: 1024, 2: 1280, 4: 1624, 8: 2048}       # n^3 ~= N * 1024^3 (1280 = 10 full 128-voxel chunks per row)
DIGESTS = os.path.join(ROOT, "tests", "golden", "mesh_digests.json")


def workload_name(scene, n, world):
    return "README RepeatXY scene (%s): SdfExpr -> %d^3 Voxels (clip) + MarchingCubes, z-slab sharded over %d GPU(s)" % (scene, n, world)


def scene_by_name(name):
    from sdfkit_b200 import scenes
    return {"readme": scenes.readme_scene, "csg50": scenes.csg50, "sphere": scenes.sphere, "perf": scenes.perf_scene}[name]()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def fp32_peak():
    """Non-FMA FP32 lane-op rate (FMUL + FADD, what parity mode can issue): measured by tools/fp32_peak.py on this pool's
    B200 and committed with its clocks as profiles/fp32_peak.json; else the nominal 148 x 128 x 1.965 GHz."""
    try:
        with open(os.path.join(ROOT, "profiles", "fp32_peak.json")) as f:
            return float(json.load(f)["fp32_nofma_lane_ops_per_s"]), "measured (profiles/fp32_peak.json, tools/fp32_peak.py)"
    except Exception:
        return 148 * 128 * 1.965e9, "nominal 148 SMs x 128 lanes x 1.965 GHz"


def mesh_sha(m):
    import numpy as np
    return {k: hashlib.sha256(np.ascontiguousarray(getattr(m, a)).tobytes()).hexdigest()
            for k, a in (("vertices", "Vertices"), ("colors", "Colors"), ("normals", "Normals"), ("triangles", "Triangles"))}


DUMP_ROWS = 1 << 19        # rows kept of each mesh array: ~40 MB of .npy files in all


def dump_outputs(job, dev, out_dir):
    """The mesh the last timed step left on the device, i.e. what a caller of the step receives, as .npy files: vertices,
    colors, normals (float32 [rows, 3]) and triangles (float64 [rows, 3]; the int32 vertex ids are exact in float64).
    A mesh with more than DUMP_ROWS vertices (triangles) is represented by the same seeded sample of rows in every run;
    counts.npy holds the full (vertices, triangles) counts, vertex_rows.npy / triangle_rows.npy the rows kept."""
    import numpy as np
    import torch
    from sdfkit_b200 import dist as skd
    parts = [skd.mesh_device_tensors(s.mesh, dev) for s in job.slabs if s.mesh is not None]
    v, c, nrm, t = (torch.cat([p[a] for p in parts]) for a in range(4))

    def rows(n, seed):
        return np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(seed).choice(n, DUMP_ROWS, replace=False))
    vr, tr = rows(len(v), 1), rows(len(t), 2)
    vi, ti = torch.as_tensor(vr, device=dev), torch.as_tensor(tr, device=dev)
    out = {"counts": np.float64([len(v), len(t)]), "vertex_rows": vr.astype(np.float64), "triangle_rows": tr.astype(np.float64),
           "vertices": v[vi], "colors": c[vi], "normals": nrm[vi], "triangles": t[ti].double()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy() if torch.is_tensor(a) else a)


def golden_digest(scene, n):
    try:
        return json.load(open(DIGESTS))[scene][str(n)]
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed regions: through NVML in this process (nvidia_ml_py; a query
    costs microseconds), falling back to spawning nvidia-smi -- whose start-up holds a driver lock for milliseconds, which
    showed as 8 - 35 ms outliers in the wall-clock-timed e2e steps (round 1 and the first round-2 runs)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    mhz = float(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
                    try:
                        mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                    except Exception:
                        mask = int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                    self.samples.append([str(mhz), str(self.max_mhz)] + ["Active" if mask & b else "Not Active" for _, b in self.BITS])
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.05 if self.nvml is not None else 0.5)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# the CPU restatement of the reference (oracle): cpu_baseline leg and the reference arm
# ------------------------------------------------------------------------------------------------
def cpu_baseline(scene_name, n_sample, steps, warmup):
    """The CPU restatement of the reference path (oracle) on an n_sample^3 grid of the same scene and bounds:
    sampling on all host cores in 2048-sample batches (Voxels.cs:88), clip, single-threaded marching cubes
    (MarchingCubes.cs:39-92).  Returns (voxels/s, tris/s, detail)."""
    import numpy as np
    import oracle
    expr, mn, mx = scene_by_name(scene_name)
    cores = os.cpu_count() or 1
    sdf = oracle.compile_sdf(expr.Lower())
    mn, mx = np.float32(mn), np.float32(mx)
    times = []
    ntris = 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        v, c = oracle.sample(sdf, mn, mx, n_sample, n_sample, n_sample, threads=cores)
        t1 = time.perf_counter()
        oracle.clip(v, mn, mx)
        m = oracle.marching_cubes(v, c, mn, mx)
        t2 = time.perf_counter()
        ntris = len(m.triangles)
        if it >= warmup:
            times.append((t1 - t0, t2 - t1))
    ts = statistics.median([a for a, _ in times])
    tm = statistics.median([b for _, b in times])
    nvox = n_sample ** 3
    return nvox / (ts + tm), ntris / tm, {
        "sample_voxels_per_s": nvox / ts, "mesh_tris_per_s": ntris / tm, "mesh_cells_per_s": (n_sample - 1) ** 3 / tm,
        "sample_s": ts, "mesh_s": tm, "cores": cores, "grid": [n_sample] * 3, "triangles": ntris, "steps_timed": len(times), "warmup_done": warmup}


def cpu_baseline_expr(expr, mn, mx, n):
    """cpu_baseline for an arbitrary SdfExpr (one pass, no warm-up): the CPU leg of tools/run_configs.py's table."""
    import numpy as np
    import oracle
    cores = os.cpu_count() or 1
    sdf = oracle.compile_sdf(expr.Lower())
    mn, mx = np.float32(mn), np.float32(mx)
    t0 = time.perf_counter()
    v, c = oracle.sample(sdf, mn, mx, n, n, n, threads=cores)
    t1 = time.perf_counter()
    oracle.clip(v, mn, mx)
    m = oracle.marching_cubes(v, c, mn, mx)
    t2 = time.perf_counter()
    return {"cpu_grid": n, "cpu_cores": cores, "cpu_samples_per_s": n ** 3 / (t1 - t0), "cpu_tris_per_s": len(m.triangles) / (t2 - t1),
            "cpu_cells_per_s": (n - 1) ** 3 / (t2 - t1), "cpu_step_voxels_per_s": n ** 3 / (t2 - t0), "cpu_triangles": len(m.triangles)}


def cpu_baseline_render(expr, w, h):
    """The CPU restatement of RayMarcher.Render (row bands on all cores, RayMarcher.cs:50-61) on a w x h image."""
    import oracle
    from sdfkit_b200 import numerics, scenes
    cores = os.cpu_count() or 1
    sdf = oracle.compile_sdf(expr.Lower())
    view = numerics.create_look_at(*scenes.CAMERA)
    t0 = time.perf_counter()
    oracle.render(sdf, w, h, view=view, bands=cores)
    t = time.perf_counter() - t0
    return {"cpu_image": [w, h], "cpu_cores": cores, "cpu_render_ms": t * 1e3, "cpu_pixels_per_s": w * h / t}


CPU_SAMPLE_TEXT = ("the reference's CPU path restated in C++ (oracle/, g++ -O2 -ffp-contract=off; the .NET reference cannot run here): "
                   "sampling on %d threads in 2048-sample batches, marching cubes single-threaded like the reference; same scene and bounds "
                   "at %d^3 = 1/%d of the %d^3 workload's voxels -- a rate on a bounded sample, not the workload itself")


def run_reference(args):
    """The reference arm: the CPU restatement on the box's host cores.  It cannot finish the 1024^3 workload in minutes
    (17 GB of voxels, ~80 s per step), so every step is a bounded SAMPLE of it (default 512^3, the minimum SURVEY.md 8d
    allows); `config` names the grid that was really measured and `sample_of` / `same_config` say what it stands for."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_s = args.cpu_n
    warm = max(0, min(args.warmup, 1))          # one warm-up at most: a 512^3 step is ~10 s of CPU work
    val, tris, d = cpu_baseline(args.scene, n_s, max(1, args.steps), warm)
    n = args.n or WEAK_GRID.get(args.gpus, 1024)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": max(1, args.steps),
        "warmup": warm, "warmup_requested": args.warmup,
        "ms_per_step": 1e3 * (d["sample_s"] + d["mesh_s"]), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "README RepeatXY scene (%s): SdfExpr -> %d^3 Voxels (clip) + MarchingCubes on %d host cores (CPU restatement)" % (
                       args.scene, n_s, d["cores"]),
                   "grid": [n_s, n_s, n_s], "same_config": n_s == n,
                   "sample_of": {"workload": workload_name(args.scene, n, args.gpus), "grid": [n, n, n],
                                 "voxel_fraction": (n_s / n) ** 3,
                                 "note": "voxels/s and tris/s are rates; the CPU path's rate falls slightly with grid size (cache misses), "
                                         "so a rate measured on the smaller sample flatters the CPU"}},
        "tris_per_s": tris,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": d["cores"], "kind": "port",
                         "sample": CPU_SAMPLE_TEXT % (d["cores"], n_s, max(1, round((n / n_s) ** 3)), n), "detail": d},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# sub-records of the N = 1 line: BASELINE configs 3 and 5, voxel export
# ------------------------------------------------------------------------------------------------
def config3_record(sk, skd, ctx, reps, with_cpu):
    """BASELINE config 3: the 50-node CSG tree at 1024^3, sample + mesh, FP32-bound evaluation."""
    from sdfkit_b200 import scenes
    expr, mn, mx = scenes.csg50()
    n = 1024
    sdf = sk.GpuSdf(expr, ctx=ctx)
    slab = skd.SlabMesher(sdf, mn, mx, n, n, n, 0, skd.cells_along(n, 1), clip=True)
    ts, tt, st, nv, nt = [], [], None, 0, 0
    for it in range(2 + reps):
        ctx.mark(10)
        slab.sample()
        ctx.mark(11)
        nv, nt = slab.classify()
        slab.emit(0, 0)
        ctx.mark(12)
        if it >= 2:
            ts.append(ctx.elapsed(10, 11))
            tt.append(ctx.elapsed(10, 12))
            st = slab.mesh.stats()
    slab.close()
    fused = []
    for it in range(1 + reps):
        t0 = time.perf_counter()
        m = sdf.ToMesh(mn, mx, n, n, n)
        if it >= 1:
            fused.append((time.perf_counter() - t0) * 1e3)
    del m
    peak, src = fp32_peak()
    flops = sdf.lowered.flops
    k1 = statistics.mean(ts)
    ach = flops * float(n) ** 3 / (k1 * 1e-3)
    rec = {"workload": "config 3: CSG-50 (%d builder nodes, %d IEEE f32 ops/sample) -> 1024^3 Voxels (clip) + MarchingCubes, 1 GPU" % (sdf.lowered.node_count, flops),
           "grid": [n, n, n], "ms_per_step": statistics.mean(tt), "value": n ** 3 / (statistics.mean(tt) * 1e-3), "unit": UNIT,
           "sample_ms": k1, "samples_per_s": n ** 3 / (k1 * 1e-3), "mesh_ms": statistics.mean(tt) - k1,
           "stages_ms": {k: st[k] for k in ("classify_ms", "scan_ms", "compact_ms", "emit_ms")},
           "vertices": nv, "triangles": nt, "tris_per_s": nt / (statistics.mean(tt) * 1e-3),
           "roofline": {"kernel": "sdfk_k_sample (CSG-50)", "bound": "fp32", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s (IEEE f32 ops, no FMA)",
                        "frac": ach / peak, "peak_source": src, "flops_per_sample": flops, "launch_ms": k1,
                        "hbm_frac": 16.0 * n ** 3 / (k1 * 1e-3) / 1e9 / peaks()[0],
                        "evidence": "profiles/r02_ncu_k1_csg50.txt (FP32 pipe counters, issue-active, registers)"},
           "e2e": {"ms_per_step": statistics.mean(fused), "ms_per_step_median": statistics.median(fused), "value": n ** 3 / (statistics.mean(fused) * 1e-3), "unit": UNIT,
                   "note": "Sdf.ToMesh through the host API, mesh in host memory every step"}}
    if with_cpu:
        c = cpu_baseline_expr(expr, mn, mx, 256)
        rec["cpu_baseline"] = {"value": c["cpu_step_voxels_per_s"], "unit": UNIT, "cores": c["cpu_cores"], "kind": "port",
                               "sample": "same tree and bounds at 256^3 (1/64 of the voxels), one pass", "detail": c}
    sdf.Dispose()
    return rec


def config5_record(sk, ctx, with_cpu):
    """BASELINE config 5: ToImage 1920x1080 of the README scene; protocol of Perf/Program.cs:43-65 (3 loops through the
    public API, the first discarded, wall clock, host image), plus the kernel alone with its FP32 roofline."""
    import ctypes as C
    import torch
    from sdfkit_b200 import _native as N, numerics, scenes
    out = {}
    peak, src = fp32_peak()
    w, h = 1920, 1080
    for key, expr in (("readme", scenes.readme_scene()[0]), ("perf_program", scenes.perf_scene()[0])):
        sdf = sk.GpuSdf(expr, ctx=ctx)
        loops = []
        for i in range(3):
            t0 = time.perf_counter()
            img = sdf.ToImage(w, h, *scenes.CAMERA, depthIterations=40)
            loops.append((time.perf_counter() - t0) * 1e3)
        rm = sk.RayMarcher(w, h, sdf)
        rm.ViewTransform = numerics.create_look_at(*scenes.CAMERA)
        cam, ivp = rm.camera()
        buf = torch.empty((h, w, 3), dtype=torch.float32, device="cuda:%d" % ctx.device)
        ks = []
        for it in range(8):
            ctx.mark(10)
            N.check(N.lib().sdfk_render_device(ctx.handle, sdf.handle, w, h, N.fptr(cam), N.fptr(ivp), 1.0, 100.0, 40, 0, h, C.c_void_p(buf.data_ptr())))
            ctx.mark(11)
            if it >= 3:
                ks.append(ctx.elapsed(10, 11))
        flops = sdf.lowered.flops
        ops = (46 * flops + 70) * w * h
        k = statistics.mean(ks)
        e2e_ms = statistics.mean(loops[1:])
        rec = {"workload": "config 5: ToImage 1920x1080, camera (-2,2,4) -> 0, 40 iterations (%s scene)" % key,
               "protocol": "Perf/Program.cs:43-65: 3 x sdf.ToImage through the public API, first loop discarded, wall clock, float image in host memory",
               "loops_ms": loops, "ms_per_image": e2e_ms, "pixels_per_s": w * h / (e2e_ms * 1e-3), "d2h_bytes_per_image": w * h * 12,
               "kernel_ms": k, "kernel_pixels_per_s": w * h / (k * 1e-3), "sdf_evals_per_s": 46 * w * h / (k * 1e-3),
               "roofline": {"kernel": "sdfk_k_render", "bound": "fp32", "achieved": ops / (k * 1e-3) / 1e12, "peak": peak / 1e12,
                            "unit": "TFLOP/s (IEEE f32 ops, no FMA)", "frac": ops / (k * 1e-3) / peak, "peak_source": src,
                            "ops_per_pixel": 46 * flops + 70, "launch_ms": k},
               "checksum": float(img.Array.sum())}
        if with_cpu:
            c = cpu_baseline_render(expr, 480, 270)
            rec["cpu_baseline"] = {"value": c["cpu_pixels_per_s"], "unit": "pixels/s", "cores": c["cpu_cores"], "kind": "port",
                                   "sample": "same camera and scene at 480x270 (1/16 of the pixels), row bands on all cores", "detail": c}
        out[key] = rec
        sdf.Dispose()
    return out


def export_record(sk, ctx, sdf, mn, mx):
    """Voxels.Values / Voxels.Colors (Voxels.cs:8-9) in the C# layout, in page-locked host memory: chunked transpose +
    overlapped copies (sdfk_voxels_export), against the link's plain copy rate measured here."""
    import torch
    dev = "cuda:%d" % ctx.device
    a = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
    hbuf = torch.empty(1 << 28, dtype=torch.uint8, pin_memory=True)
    best = 1e9
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hbuf.copy_(a, non_blocking=True)
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    link = (1 << 28) / best / 1e9
    del a, hbuf
    rec = {"pcie_d2h_gbs_plain_copy": link, "grids": {}}
    for n in (512, 1024):
        try:
            vox = sdf.ToVoxels(mn, mx, n, n, n)
            ctx.synchronize()
            ts = []
            for it in range(3):
                vox._values = vox._colors = None
                t0 = time.perf_counter()
                v, c = vox.Values, vox.Colors
                ts.append(time.perf_counter() - t0)
            gb = 16.0 * n ** 3 / 1e9
            rec["grids"][str(n)] = {"bytes": 16 * n ** 3, "first_call_s": ts[0], "ms": min(ts[1:]) * 1e3, "gbs": gb / min(ts[1:]),
                                    "frac_of_link": gb / min(ts[1:]) / link,
                                    "note": "first call includes pinning the destination (cudaHostAlloc); later calls reuse it"}
            del v, c
            vox.Dispose()
        except Exception as ex:                      # a box without ~35 GB of pinnable host memory skips 1024^3
            rec["grids"][str(n)] = {"skipped": repr(ex)[:200]}
    return rec


# ------------------------------------------------------------------------------------------------
# strong scaling through the multi-GPU context of the C ABI (one process, N devices)
# ------------------------------------------------------------------------------------------------
def pcie_aggregate(ndevs):
    """Device -> page-locked host copy rate with 1, 2, 4, .. devices copying AT THE SAME TIME (256 MB each, best of 3): what the
    host side of the box can absorb -- the ceiling of any e2e number that lands a result in host memory."""
    import torch
    out = {}
    nb = 1 << 28
    for nd in ndevs:
        src = [torch.empty(nb, dtype=torch.uint8, device="cuda:%d" % d) for d in range(nd)]
        dst = [torch.empty(nb, dtype=torch.uint8, pin_memory=True) for _ in range(nd)]
        best = 1e9
        for _ in range(4):
            for d in range(nd):
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            for d in range(nd):
                with torch.cuda.device(d):
                    dst[d].copy_(src[d], non_blocking=True)
            for d in range(nd):
                torch.cuda.synchronize(d)
            best = min(best, time.perf_counter() - t0)
        out[str(nd)] = nd * nb / best / 1e9
        del src, dst
    return out


def strong_record(sk, expr, mn, mx, n, ndevs, steps, single_mesh_sha, scene, config4=True):
    """The same n^3 job on 1, 2, 4, .. devices behind sdfk_ctx_create_multi: (a) device-resident step = sharded Voxels
    (16 B/voxel) + MarchingCubes, (b) e2e = Sdf.ToMesh landing ONE host mesh.  Wall clock from call to completion on all
    devices (+ the slowest device's own event span); every result is compared with the single-GPU digest."""
    out = {"grid": [n, n, n], "scene": scene, "by_devices": {}, "pcie_d2h_aggregate_gbs": pcie_aggregate(ndevs),
           "note": "strong scaling: total work fixed; one process drives all devices through the C ABI (sdfk_ctx_create_multi), slabs cut by "
                   "the cost-balanced planner, counts exchanged in host memory, every device copies its share of the mesh to its offset of "
                   "one host result over its own PCIe link"}
    gold = golden_digest(scene, n)
    render_sha = [None]
    for nd in ndevs:
        ctx = sk.Context(devices=list(range(nd)))
        try:
            sdf = sk.GpuSdf(expr, ctx=ctx)
            vox = sdf.ToVoxels(mn, mx, n, n, n)
            wall, dev_ms = [], []
            for it in range(3 + steps):
                ctx.synchronize()
                ctx.timer_start()
                t0 = time.perf_counter()
                vox.Resample(sdf, clip=True)
                gm = sk.MarchingCubes.CreateGpuMesh(vox)
                t1 = time.perf_counter()
                d = ctx.timer_stop()
                if it >= 3:
                    wall.append((t1 - t0) * 1e3)
                    dev_ms.append(d)
                nv, nt = gm.counts()
                if it < 2 + steps:
                    gm.destroy()
            m = gm.download()
            sha_res = mesh_sha(m)
            gm.destroy()
            del m
            vox.Dispose()
            e2e = []
            for it in range(5 + steps):
                t0 = time.perf_counter()
                mesh = sdf.ToMesh(mn, mx, n, n, n)
                if it >= 5:
                    e2e.append((time.perf_counter() - t0) * 1e3)
            sha_e2e = mesh_sha(mesh)
            d2h = mesh.Vertices.nbytes * 3 + mesh.Triangles.nbytes
            del mesh
            rec = {"device_step_wall_ms": statistics.mean(wall), "device_step_wall_ms_median": statistics.median(wall),
                   "device_step_slowest_device_ms": statistics.mean(dev_ms),
                   "voxels_per_s": n ** 3 / (statistics.mean(wall) * 1e-3), "tris_per_s": nt / (statistics.mean(wall) * 1e-3),
                   "e2e_ms": statistics.mean(e2e), "e2e_ms_median": statistics.median(e2e), "e2e_voxels_per_s": n ** 3 / (statistics.mean(e2e) * 1e-3),
                   "d2h_bytes_per_step": d2h, "vertices": nv, "triangles": nt,
                   "equal_to_single_gpu": {"device_resident": sha_res == single_mesh_sha, "e2e": sha_e2e == single_mesh_sha},
                   "equal_to_golden_digest": None if gold is None else (sha_e2e == gold["sha256"])}
            # BASELINE config 5 on nd devices: the image in row bands (RayMarcher.cs:50-61), one per device, one host image
            from sdfkit_b200 import scenes as _sc
            imgs = []
            for it in range(6):
                t0 = time.perf_counter()
                img = sdf.ToImage(1920, 1080, *_sc.CAMERA, depthIterations=40)
                imgs.append((time.perf_counter() - t0) * 1e3)
            isha = hashlib.sha256(img.Array.tobytes()).hexdigest()
            if render_sha[0] is None:
                render_sha[0] = isha
            rec["toimage_1080p_ms"] = statistics.median(imgs[2:])
            rec["toimage_equal_to_single_gpu"] = isha == render_sha[0]
            del img
            # BASELINE config 4: the same scene at 2048^3 (137 GB of voxels if materialised) through Sdf.ToMesh on nd >= 2 devices
            if nd >= 2 and config4:
                try:
                    g4 = golden_digest(scene, 2048)
                    t4 = []
                    for it in range(4):
                        t0 = time.perf_counter()
                        m4 = sdf.ToMesh(mn, mx, 2048, 2048, 2048)
                        t4.append((time.perf_counter() - t0) * 1e3)
                        if it < 3:
                            del m4
                    rec["config4_2048"] = {"e2e_ms": statistics.median(t4[1:]), "e2e_voxels_per_s": 2048 ** 3 / (statistics.median(t4[1:]) * 1e-3),
                                           "vertices": int(len(m4.Vertices)), "triangles": int(len(m4.Triangles) // 3),
                                           "d2h_bytes_per_step": m4.Vertices.nbytes * 3 + m4.Triangles.nbytes,
                                           "equal_to_golden_digest": None if g4 is None else (mesh_sha(m4) == g4["sha256"])}
                    del m4
                except Exception as ex:
                    rec["config4_2048"] = {"error": repr(ex)[:300]}
            out["by_devices"][str(nd)] = rec
            sdf.Dispose()
        finally:
            ctx.close()
    one = out["by_devices"].get("1")
    if one:
        for nd, rec in out["by_devices"].items():
            rec["speedup_device_step"] = one["device_step_wall_ms"] / rec["device_step_wall_ms"]
            rec["speedup_e2e"] = one["e2e_ms"] / rec["e2e_ms"]
    return out


def run_ours(args):
    import numpy as np
    # stdout carries exactly one JSON line: library chatter (e.g. NCCL's version banner) is sent to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the SdfKit GPU path has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the mesh of a one-process run: use it with --gpus 1")
    torch.cuda.set_device(local)
    import torch.distributed as dist
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")     # host-side barriers while rank 0 alone drives all GPUs (strong_1024)
    import sdfkit_b200 as sk
    from sdfkit_b200 import dist as skd

    n = args.n or WEAK_GRID.get(world, int(round(1024 * world ** (1 / 3) / 8)) * 8)
    expr, mn, mx = scene_by_name(args.scene)
    ctx = sk.Context(local)
    t0 = time.perf_counter()
    sdf = sk.GpuSdf(expr, ctx=ctx)
    jit_s = time.perf_counter() - t0
    spr = args.slabs_per_rank or 1
    job = skd.ShardedMesher(sdf, mn, mx, n, n, n, rank, world, spr, clip=True, balanced=(world > 1 and not args.uniform_slabs))
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        counts = job.sample_classify()
        allc = skd.all_gather_int64(counts, device=dev) if world > 1 else counts[None]
        offs, tot = job.offsets(allc)
        job.emit(offs)
        return tot

    warm = max(args.warmup, 3)
    for _ in range(warm):
        tot = step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = ctx.launch_count()
    sample_ms, stage = [], {"classify_ms": [], "scan_ms": [], "compact_ms": [], "emit_ms": []}
    host = {"sample_classify": 0.0, "allgather": 0.0, "emit": 0.0}
    barrier()
    ctx.mark(0)
    w0 = time.perf_counter()
    for _ in range(args.steps):
        h0 = time.perf_counter()
        counts = np.zeros((spr, 2), dtype=np.int64)
        k1 = 0.0
        for k, s_ in enumerate(job.slabs):
            if s_.ke > s_.kb:
                ctx.mark(2)
                s_.sample()
                ctx.mark(3)
                counts[k] = s_.classify()                     # synchronises: the event pair is complete
                k1 += ctx.elapsed(2, 3)
        h1 = time.perf_counter()
        allc = skd.all_gather_int64(counts, device=dev) if world > 1 else counts[None]
        offs, tot = job.offsets(allc)
        h2 = time.perf_counter()
        job.emit(offs)
        h3 = time.perf_counter()
        host["sample_classify"] += (h1 - h0) * 1e3
        host["allgather"] += (h2 - h1) * 1e3
        host["emit"] += (h3 - h2) * 1e3
        sample_ms.append(k1)
        st = job.stats()
        for k in stage:
            stage[k].append(st[k])
    ctx.mark(1)
    barrier()
    wall = time.perf_counter() - w0
    dev_ms = ctx.elapsed(0, 1)
    launches = ctx.launch_count() - l0
    t = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = t.tolist()
    ms_per_step = dev_ms / args.steps
    nvox_total = n ** 3
    value = nvox_total / (ms_per_step * 1e-3)
    nverts_total, ntris_total = int(tot[0]), int(tot[1])
    last_allc, last_offs = allc, offs

    # dram__bytes_read + dram__bytes_write of one K1 launch from this round's committed ncu capture (same workload only)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_k1_traffic.json")))
        if world == 1 and n == 1024 and args.scene == "readme":
            traffic = float(tj["traffic_bytes"])
    except Exception:
        pass
    # ---- roofline of the dominant kernel (K1 sdfk_k_sample): 16 algorithmic bytes written per voxel, 0 read
    hbm, peak_src = peaks()
    # K1 only writes.  MEASURED_PEAKS.json's hbm_gbs is a COPY (read + write) rate; a pure store stream goes faster on this part
    # (torch fill_ / cudaMemset: ~7.5 TB/s), so the fraction of the copy peak can exceed 1.  Measured here, outside the timed
    # region, as context for `frac`: the library's store-only probe kernel (sdfk_ctx_store_bandwidth: one CTA per 16 KiB in
    # memory order, 4 GiB, CUDA events, best of 5).
    fill_gbs = None
    if rank == 0:
        try:
            fill_gbs = ctx.store_bandwidth(4 << 30, 5)
        except Exception:
            fill_gbs = None
    slab_vox = sum(n * n * (s_.z1 - s_.z0) for s_ in job.slabs if s_.ke > s_.kb)   # voxels this rank's K1 launches write per step (incl. halo slices)
    k1_ms = statistics.mean(sample_ms)
    achieved = 16.0 * slab_vox / (k1_ms * 1e-3) / 1e9
    mesh_ms = {k: statistics.mean(v) for k, v in stage.items()}
    cells = (n - 1) * (n - 1) * (n - 1)
    # per-rank view of the step (device stage times + host-side wall per phase), gathered to rank 0
    mine = [k1_ms] + [mesh_ms[k] for k in ("classify_ms", "scan_ms", "compact_ms", "emit_ms")] + [host[k] / args.steps for k in ("sample_classify", "allgather", "emit")]
    per_rank = torch.tensor(mine, dtype=torch.float64, device=dev)
    if world > 1:
        allr = [torch.empty_like(per_rank) for _ in range(world)]
        dist.all_gather(allr, per_rank)
        per_rank = torch.stack(allr)
    else:
        per_rank = per_rank[None]
    per_rank = per_rank.cpu().numpy()
    names = ["sample_ms", "classify_ms", "scan_ms", "compact_ms", "emit_ms", "host_sample_classify_ms", "host_allgather_ms", "host_emit_ms"]
    rank_stages = {nm: [round(float(x), 4) for x in per_rank[:, i]] for i, nm in enumerate(names)}
    mesh_total_ms = float(per_rank[:, 1:5].sum(axis=1).max())
    # meshing roofline (SURVEY.md 8d): bytes = 4 N (distance read once) + 12 U (colour of the corner voxels of active cells, U <= 8 active)
    # + 36 nverts + 12 ntris; and the bytes the sign-block formulation really needs: N/8 (one bit per voxel) instead of 4 N
    active = nverts_total                                   # ~1 created vertex per active cell in these scenes (stats carry the exact count per rank)
    mesh_bytes_8d = 4.0 * nvox_total + 12.0 * 8 * active + 36.0 * nverts_total + 12.0 * ntris_total
    mesh_bytes_signs = nvox_total / 8.0 + (4.0 + 12.0) * 8 * active + 36.0 * nverts_total + 12.0 * ntris_total
    mesh_s = max(mesh_total_ms * 1e-3, 1e-9)
    roofline_mesh = {"kernels": "K2' mc_classify_signs + K3 mc_scan x2 + K4a mc_compact + K4b mc_emit_tris/mc_emit_verts (slowest rank, summed)",
                     "bound": "hbm", "ms": mesh_total_ms, "tris_per_s": ntris_total / mesh_s, "cells_per_s": cells / mesh_s,
                     "algorithmic_bytes_8d": mesh_bytes_8d, "achieved_8d": mesh_bytes_8d / mesh_s / 1e9, "frac_8d": mesh_bytes_8d / mesh_s / 1e9 / hbm / world,
                     "algorithmic_bytes_sign_blocks": mesh_bytes_signs, "achieved_sign_blocks": mesh_bytes_signs / mesh_s / 1e9,
                     "frac_sign_blocks": mesh_bytes_signs / mesh_s / 1e9 / hbm / world, "peak": hbm, "unit": "GB/s",
                     "note": "8d: SURVEY.md 8(d)'s byte count (4 B/voxel distance re-read + colours of active corners + mesh out); sign_blocks: what the "
                             "shipped formulation must move (1 bit/voxel written by K1 + corner values and colours of active cells + mesh out) -- "
                             "the stages after classify are latency-bound gathers over ~1 % of the cells, far from the HBM line by construction"}

    # ---- the Sdf.ToMesh variant of the step: distance-only voxels (4 B/voxel), colours evaluated at the created vertices
    fused = None
    if not args.no_fused:
        fjob = skd.ShardedMesher(sdf, mn, mx, n, n, n, rank, world, spr, clip=True,
                                 balanced=(world > 1 and not args.uniform_slabs), colors=False)

        def fstep():
            counts = fjob.sample_classify()
            allc = skd.all_gather_int64(counts, device=dev) if world > 1 else counts[None]
            offs, tot_ = fjob.offsets(allc)
            fjob.emit(offs)
        for _ in range(3):
            fstep()
        barrier()
        ctx.mark(4)
        for _ in range(args.steps):
            fstep()
        ctx.mark(5)
        barrier()
        tf = torch.tensor([ctx.elapsed(4, 5) / args.steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tf, op=dist.ReduceOp.MAX)
        fused = {"ms_per_step": tf.item(), "value": nvox_total / (tf.item() * 1e-3), "unit": UNIT,
                 "note": "same step with distance-only voxels (what Sdf.ToMesh runs): 4 B/voxel written, vertex colours from the SDF"}
        fjob.close()

    # ---- e2e through the public API: Sdf.ToMesh(min, max, n, n, n) -> Mesh in host memory, every step
    e2e = None
    single_sha = None
    if not args.no_e2e:
        barrier()
        e_steps = max(3, min(args.steps, 10))
        e_times = []
        d2h = 0
        if world == 1:
            for _ in range(max(args.warmup, 5)):                 # warm: device + pinned host pools reach steady state
                mesh = sdf.ToMesh(mn, mx, n, n, n)               # (two result sets are alive while `mesh = sdf.ToMesh()` runs)
            torch.cuda.synchronize()
            e0 = time.perf_counter()
            for _ in range(e_steps):
                t_ = time.perf_counter()
                mesh = sdf.ToMesh(mn, mx, n, n, n)                # returns when the whole mesh is in host memory
                e_times.append(time.perf_counter() - t_)
            torch.cuda.synchronize()
            e_s = (time.perf_counter() - e0) / e_steps
            d2h = mesh.Vertices.nbytes * 3 + mesh.Triangles.nbytes + 24
            single_sha = mesh_sha(mesh)
            del mesh
        else:
            # N ranks: every rank delivers ITS share of the mesh (global indices from the count all-gather) into its own
            # page-locked host memory over its own PCIe link (sdfk_mesh_emit_host: emit in sub-ranges, copies overlapped);
            # the job's mesh is the concatenation of the shares in rank order
            # (slabs balanced for this path: an active cell also costs its ~60 bytes over PCIe, dist.ACTIVE_CELL_COST_E2E)
            ejob = skd.ShardedMesher(sdf, mn, mx, n, n, n, rank, world, spr, clip=True,
                                     balanced=(world > 1 and not args.uniform_slabs), colors=False,
                                     active_cell_cost=skd.ACTIVE_CELL_COST_E2E)

            def e2e_step():
                counts = ejob.sample_classify()
                allc = skd.all_gather_int64(counts, device=dev)
                offs, _ = ejob.offsets(allc)
                parts = ejob.emit_host(offs)
                return sum(m.Vertices.nbytes * 3 + m.Triangles.nbytes + 24 for m in parts)
            for _ in range(max(args.warmup, 5)):
                e2e_step()
            barrier()
            e0 = time.perf_counter()
            for _ in range(e_steps):
                t_ = time.perf_counter()
                d2h = e2e_step()
                e_times.append(time.perf_counter() - t_)
            barrier()
            e_s = (time.perf_counter() - e0) / e_steps
            ejob.close()
            tb = torch.tensor([float(d2h)], dtype=torch.float64, device=dev)
            dist.all_reduce(tb)
            d2h = int(tb.item())
        te = torch.tensor([e_s, statistics.median(e_times), max(e_times)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e_s, e_med, e_max = te.tolist()
        e2e = {"value": nvox_total / e_s, "unit": UNIT, "ms_per_step": e_s * 1e3, "steps": e_steps,
               "ms_per_step_median": e_med * 1e3, "ms_per_step_max": e_max * 1e3, "value_at_median": nvox_total / e_med,
               "ms_per_step_all_rank0": [round(x * 1e3, 3) for x in e_times],
               "h2d_bytes_per_step": 256, "d2h_bytes_per_step": int(d2h),
               "note": ("Sdf.ToMesh through the host API (sdfk_sdf_to_mesh_host: z-slabs pipelined, mesh parts streamed to page-locked "
                        "host memory while the next slabs are computed)" if world == 1 else
                        "per rank: distance-only sampling + classify, NCCL all-gather of the counts, chunked emit with every part "
                        "streamed to the rank's own page-locked host memory (sdfk_mesh_emit_host); d2h bytes summed over ranks") +
                       "; the SDF is analytic so the only host->device bytes are kernel parameters; the whole mesh (vertices, "
                       "colours, normals, triangles) lands in host memory every step; value = mean over the steps (median and max beside it, "
                       "max over ranks)"}

    clocks = sampler.stop() if sampler else None          # sampled over all timed regions above (main loop, fused, e2e)

    # ---- parity of the N-rank job, on the hardware and at the size it was timed (outside the timed regions)
    parity = None
    if world > 1 and not args.no_parity:
        parity = parity_check(sk, skd, dist, torch, ctx, sdf, job, last_allc, last_offs, expr, mn, mx, n, rank, world, dev, args.scene)
    if args.dump_outputs:
        dump_outputs(job, dev, args.dump_outputs)
    job.close()

    # ---- rank 0 alone: strong scaling through the multi-GPU C ABI, BASELINE configs 3 / 5, export, CPU baseline
    strong = cfgs = cpu = None
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    if rank == 0:
        ndev_max = min(torch.cuda.device_count(), max(world, 1))
        if not args.no_strong:
            if single_sha is None:
                m1 = sdf.ToMesh(mn, mx, 1024, 1024, 1024)
                single_sha = mesh_sha(m1)
                del m1
            elif n != 1024:
                single_sha = None
            try:
                strong = strong_record(sk, expr, mn, mx, 1024, [d for d in (1, 2, 4, 8) if d <= ndev_max], max(3, min(args.steps, 10)),
                                       single_sha, args.scene)
            except Exception as ex:
                strong = {"error": repr(ex)[:400]}
        if world == 1 and not args.no_configs:
            cfgs = {}
            try:
                cfgs["config3_csg50_1024"] = config3_record(sk, skd, ctx, 5, not args.no_cpu)
                cfgs["config5_toimage_1080p"] = config5_record(sk, ctx, not args.no_cpu)
                cfgs["voxels_export"] = export_record(sk, ctx, sdf, mn, mx)
            except Exception as ex:
                cfgs["error"] = repr(ex)[:400]
        if world == 1 and not args.no_cpu:
            val, tris, d = cpu_baseline(args.scene, args.cpu_n, 2, 0)
            cpu = {"value": val, "unit": UNIT, "cores": d["cores"], "kind": "port",
                   "sample": CPU_SAMPLE_TEXT % (d["cores"], args.cpu_n, max(1, round((n / args.cpu_n) ** 3)), n),
                   "tris_per_s": tris, "detail": d}
    if world > 1:
        dist.barrier(group=host_group)                      # the other ranks wait on the host, their GPUs idle

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(args.scene, n, world),
                       "grid": [n, n, n], "slabs_per_rank": spr, "slab_layers": [list(l) for l in job.layers], "sdf_nodes": sdf.lowered.node_count, "sdf_flops_per_sample": sdf.lowered.flops,
                       "l2": "working set %.1f GB per GPU >> 126 MB L2, no flush needed" % (16.0 * slab_vox / 1e9),
                       "parity_mode": "IEEE f32/f64, no FMA contraction (bit-exact vs the CPU oracle)"},
            "tris_per_s": ntris_total / (ms_per_step * 1e-3), "triangles": ntris_total, "vertices": nverts_total,
            "stages_ms": dict(sample_ms=k1_ms, **mesh_ms),
            "per_rank_ms": rank_stages,
            "roofline": {"kernel": "sdfk_k_sample", "bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s",
                         "frac": achieved / hbm, "traffic": traffic, "peak_source": peak_src,
                         "traffic_source": "profiles/r02_k1_traffic.json (ncu --set full of this kernel revision)" if traffic else None,
                         "algorithmic_bytes_per_launch": 16.0 * slab_vox, "launch_ms": k1_ms,
                         "write_only_peak": fill_gbs, "frac_of_write_only_peak": (achieved / fill_gbs) if fill_gbs else None,
                         "write_only_peak_source": "sdfk_ctx_store_bandwidth: 4 GiB from a store-only kernel in memory order, measured in this run (`peak` is the copy rate)"},
            "roofline_mesh": roofline_mesh,
            "wall_ms_per_step": wall_ms / args.steps, "jit_compile_s": jit_s, "gpu_launches": int(launches),
            "clocks": clocks, "e2e": e2e, "fused_to_mesh": fused, "parity_check": parity, "strong_1024": strong, "configs": cfgs,
            "cpu_baseline": cpu,
        }
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier(group=host_group)
        dist.destroy_process_group()


def parity_check(sk, skd, dist, torch, ctx, sdf, job, allc, offs, expr, mn, mx, n, rank, world, dev, scene):
    """What the timed N-rank job produced, checked where it ran: (a) the rank-ordered concatenation of the shares, gathered to
    rank 0 over NVLink (NCCL point-to-point, timed), equals the mesh one GPU makes of the same grid -- array for array, and
    its sha256 equals tests/golden/mesh_digests.json when that grid has an entry; (b) 4-slice slabs at both boundaries of
    every rank's z-slab equal the CPU oracle's SDF at the same positions (+ ClipToBounds); (c) the totals equal the
    all-gathered sums.  MarchingCubes.cs:54-92 numbers vertices layer-major, so shares concatenate in rank order."""
    import ctypes as C
    import numpy as np
    from sdfkit_b200 import _native as N, numerics
    out = {"grid": [n, n, n], "ranks": world}
    # (c) totals
    counts = np.asarray(allc, dtype=np.int64).reshape(world, -1, 2)
    mine_v = sum(s.mesh.counts()[0] for s in job.slabs if s.mesh is not None)
    mine_t = sum(s.mesh.counts()[1] for s in job.slabs if s.mesh is not None)
    tt = torch.tensor([mine_v, mine_t], dtype=torch.int64, device=dev)
    dist.all_reduce(tt)
    out["totals_vs_allgather"] = {"vertices": int(tt[0]), "triangles": int(tt[1]),
                                  "equal": bool(int(tt[0]) == int(counts[..., 0].sum()) and int(tt[1]) == int(counts[..., 1].sum()))}
    # (a) gather the shares to rank 0 over NVLink, slab by slab in global order (slab g belongs to rank g % world)
    spr = job.spr
    per_slab = counts.transpose(1, 0, 2).reshape(world * spr, 2)
    # (NCCL sets its point-to-point channels up on first use: one small untimed exchange first)
    skd.gather_rows(torch.zeros((4, 3), dtype=torch.float32, device=dev), [4] * world, dst=0)
    skd.gather_rows(torch.zeros((4, 3), dtype=torch.int32, device=dev), [4] * world, dst=0)
    gathered = [[], [], [], []]
    torch.cuda.synchronize()
    dist.barrier()
    g0 = time.perf_counter()
    nbytes = 0
    for s_idx in range(spr):
        slab = job.slabs[s_idx]
        if slab.mesh is not None:
            tens = skd.mesh_device_tensors(slab.mesh, dev)
        else:
            tens = [torch.empty((0, 3), dtype=torch.float32, device=dev)] * 3 + [torch.empty((0, 3), dtype=torch.int32, device=dev)]
        rows_v = [int(per_slab[s_idx * world + r][0]) for r in range(world)]
        rows_t = [int(per_slab[s_idx * world + r][1]) for r in range(world)]
        for a in range(4):
            res = skd.gather_rows(tens[a], rows_v if a < 3 else rows_t, dst=0)
            if rank == 0:
                gathered[a].append(res)
                nbytes += res.numel() * 4
    torch.cuda.synchronize()
    dist.barrier()
    g_ms = (time.perf_counter() - g0) * 1e3
    out["mesh_gather"] = {"ms": g_ms, "bytes": nbytes, "gbs": nbytes / (g_ms * 1e-3) / 1e9 if rank == 0 and g_ms > 0 else None,
                          "how": "dist.gather_rows: NCCL send/recv of every rank's device-resident share into rank 0's HBM at the all-gathered offsets"}
    if rank == 0:
        class M:
            pass
        m = M()
        arrs = [torch.cat(g).cpu().numpy() if g else np.zeros((0, 3)) for g in gathered]
        m.Vertices, m.Colors, m.Normals = arrs[0], arrs[1], arrs[2]
        m.Triangles = arrs[3].reshape(-1)
        sha_n = mesh_sha(m)
        one = sdf.ToMesh(mn, mx, n, n, n)                       # the whole grid on this rank's GPU alone (pipelined z-slabs)
        sha_1 = mesh_sha(one)
        eq = (len(one.Vertices) == len(m.Vertices) and len(one.Triangles) == len(m.Triangles) and
              all(np.array_equal(np.ascontiguousarray(getattr(one, k)).view(np.uint32), np.ascontiguousarray(getattr(m, k)).view(np.uint32))
                  for k in ("Vertices", "Colors", "Normals")) and np.array_equal(one.Triangles, m.Triangles))
        gold = golden_digest(scene, n)
        out["mesh_vs_single_gpu"] = {"equal": bool(eq), "sha256": sha_n, "sha256_single_gpu": sha_1,
                                     "golden_digest": None if gold is None else {"file": "tests/golden/mesh_digests.json", "equal": sha_n == gold["sha256"]}}
        del one, m, arrs
    gathered = None
    # (b) 4 slices at each boundary of this rank's slab(s) against the oracle (as tests/test_gpu_fullsize.py does at 1024^3)
    import oracle
    f = np.float32
    vmin, vmax = numerics.vec3(mn), numerics.vec3(mx)
    ok_b, checked = True, 0
    stride = max(1, n // 256)                                    # every stride-th x and y: 256 x 256 x 4 positions per boundary
    for slab in job.slabs:
        if slab.ke <= slab.kb:
            continue
        for z0 in sorted({slab.z0, max(slab.z0, slab.z1 - 4)}):
            nzl = min(4, slab.z1 - z0)
            h = C.c_void_p()
            N.check(N.lib().sdfk_voxels_sample_slab(sdf.ctx.handle, sdf.handle, N.fptr(vmin), N.fptr(vmax), n, n, n, 1, z0, z0 + nzl, C.byref(h)))
            vals = np.empty((n, n, nzl), dtype=np.float32)
            cols = np.empty((n, n, nzl, 3), dtype=np.float32)
            N.check(N.lib().sdfk_voxels_export(h, N.fptr(vals), N.fptr(cols)))
            N.lib().sdfk_voxels_destroy(h)
            d = ((vmax - vmin) / f(n)).astype(f)
            m0 = (vmin + f(0.5) * d).astype(f)
            ix, iy, iz = np.meshgrid(np.arange(0, n, stride), np.arange(0, n, stride), np.arange(z0, z0 + nzl), indexing="ij")
            pts = np.stack([m0[0] + ix.astype(f) * d[0], m0[1] + iy.astype(f) * d[1], m0[2] + iz.astype(f) * d[2]], axis=-1).astype(f)
            ref = oracle.eval_sdf(sdf.lowered, pts.reshape(-1, 3)).reshape(ix.shape + (4,))
            wall = (ix == 0) | (ix == n - 1) | (iy == 0) | (iy == n - 1) | (iz == 0) | (iz == n - 1)
            expect = np.where(wall, (vmax[0] - vmin[0]) / f(n), ref[..., 3]).astype(f)
            got_v = vals[::stride, ::stride, :]
            got_c = cols[::stride, ::stride, :, :]
            ok_b = ok_b and np.array_equal(got_v.view(np.uint32), expect.view(np.uint32)) and \
                np.array_equal(np.ascontiguousarray(got_c).view(np.uint32), np.ascontiguousarray(ref[..., :3]).view(np.uint32))
            checked += int(ix.size)
    tb = torch.tensor([1 if ok_b else 0, checked], dtype=torch.int64, device=dev)
    dist.all_reduce(tb, op=dist.ReduceOp.SUM)
    out["slab_boundaries_vs_oracle"] = {"equal": bool(int(tb[0]) == world), "voxels_checked": int(tb[1]),
                                        "how": "every rank re-samples 4 slices at both ends of its z-slab (sdfk_voxels_sample_slab + export) and compares "
                                               "distances (after ClipToBounds) and colours bit for bit with the CPU oracle on a %d-strided lattice" % stride}
    if rank == 0:
        out["ok"] = bool(out["totals_vs_allgather"]["equal"] and out["mesh_vs_single_gpu"]["equal"] and out["slab_boundaries_vs_oracle"]["equal"]
                         and (out["mesh_vs_single_gpu"]["golden_digest"] is None or out["mesh_vs_single_gpu"]["golden_digest"]["equal"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", dest="n", type=int, default=0, help="grid size override (default: 1024 per GPU-equivalent)")
    ap.add_argument("--scene", default="readme")
    ap.add_argument("--cpu-n", type=int, default=512, help="grid size of the bounded CPU sample (512^3: ~10 s of CPU work per step)")
    ap.add_argument("--slabs-per-rank", type=int, default=0, help="z-slabs dealt round-robin to every rank (default 1)")
    ap.add_argument("--uniform-slabs", action="store_true", help="equal-thickness z-slabs instead of the cost-balanced plan")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fused", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the N-rank parity block")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block (multi-GPU context of the C ABI)")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE config 3 / 5 / export sub-records (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the mesh of the last one as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computed")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
