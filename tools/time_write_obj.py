#!/usr/bin/env python3
"""Mesh.WriteObj on the device (sdfk_obj_write) for the README scene at 1024^3 through Sdf.ToMesh.

Prints the card and its power limit, the mesh's lines and text bytes, the device time of the length (+ scan) and format
kernels (torch.profiler's CUDA activity records over repeated calls after warm-up), the call's wall time into a sink that does
nothing, one that copies into a preallocated buffer and a file in the output directory, the ceiling (one cudaMemcpyAsync of as
many bytes device -> page-locked host), and the host writer's rate on the 256^3 mesh -- applied to 1024^3 it is an
extrapolation, not a measurement.  Also checks that the device's 256^3 file equals the host writer's, byte for byte.

    python tools/time_write_obj.py [outdir]        (where the timed files are written; default: a temporary directory)
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from sdfkit_b200 import _native as N  # noqa: E402
from sdfkit_b200 import scenes  # noqa: E402
from sdfkit_b200.voxels import Mesh  # noqa: E402

OWN_OUT = len(sys.argv) < 2
OUT = tempfile.mkdtemp(prefix="time_write_obj_") if OWN_OUT else sys.argv[1]
os.makedirs(OUT, exist_ok=True)
REPS = 10


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() or "unknown (nvidia-smi: %s)" % r.stderr.strip()


def obj_write(mesh, sink):
    v = N.f32c(mesh.Vertices).reshape(-1)
    n = N.f32c(mesh.Normals).reshape(-1)
    t = np.ascontiguousarray(mesh.Triangles, dtype=np.int32).reshape(-1)
    written = C.c_int64()
    N.check(N.lib().sdfk_obj_write(mesh.ctx.handle, N.fptr(v), len(v) // 3, N.fptr(n), len(n) // 3,
                                   t.ctypes.data_as(C.POINTER(C.c_int32)), len(t), sink, None, C.byref(written)))
    return written.value


def timed(fn, reps=REPS):
    fn()
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return np.median(ts) * 1e3, min(ts) * 1e3


def main():
    print("card: %s" % card(), flush=True)
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    mesh = sdf.ToMesh(mn, mx, 1024, 1024, 1024)
    nv, nt = len(mesh.Vertices), len(mesh.Triangles) // 3
    lines = nv + len(mesh.Normals) + nt

    null = N.WRITE_FN(lambda p, n, u: 0)
    nbytes = obj_write(mesh, null)
    print("README 1024^3: %d vertices, %d normals, %d triangles -> %d lines, %d bytes of OBJ text (%.1f B/line)"
          % (nv, len(mesh.Normals), nt, lines, nbytes, nbytes / lines), flush=True)

    ms_null = timed(lambda: obj_write(mesh, null))
    buf = np.empty(nbytes, dtype=np.uint8)
    pos = [0]

    def copy_sink(p, n, u):
        C.memmove(buf.ctypes.data + pos[0], p, n)
        pos[0] += n
        return 0
    copy_cb = N.WRITE_FN(copy_sink)

    def run_copy():
        pos[0] = 0
        obj_write(mesh, copy_cb)
    ms_copy = timed(run_copy)
    path = os.path.join(OUT, "readme1024.obj")

    def run_file():
        mesh.WriteObj(path)
    ms_file = timed(run_file, reps=3)
    assert os.path.getsize(path) == nbytes
    os.remove(path)

    # the ceiling: the same number of bytes, device -> page-locked host, one copy
    dsrc = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    hdst = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cp = []
    for i in range(REPS + 2):
        e0.record()
        hdst.copy_(dsrc, non_blocking=True)
        e1.record()
        e1.synchronize()
        if i >= 2:
            cp.append(e0.elapsed_time(e1))
    ms_ceiling = float(np.median(cp))
    del dsrc, hdst

    # device time of the kernels (a separate, profiled run)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(REPS):
            obj_write(mesh, null)
        torch.cuda.synchronize()
    kern = {}
    for a in prof.key_averages():
        for key, tag in (("length", "obj_line_bytes"), ("scan", "obj_scan"), ("format", "obj_format")):
            if tag in a.key:
                kern[key] = kern.get(key, 0.0) + a.device_time_total / 1e3 / REPS
    if kern:
        print("device time per call: length pass %.3f ms, scan %.3f ms, format pass %.3f ms (all chunks)"
              % (kern.get("length", 0.0), kern.get("scan", 0.0), kern.get("format", 0.0)))
    else:
        print("device time per call: not measured (the profiler recorded no obj_* kernels)")

    gb = nbytes / 1e9
    print("sdfk_obj_write wall (median / best of %d): do-nothing sink %.2f / %.2f ms (%.1f GB/s), copying sink %.2f / %.2f ms, "
          "file %.2f / %.2f ms (best of 3)" % (REPS, *ms_null, gb / ms_null[0] * 1e3, *ms_copy, *ms_file))
    print("ceiling: one %d-byte cudaMemcpyAsync device -> page-locked host %.2f ms (%.1f GB/s); do-nothing sink / ceiling = %.2fx"
          % (nbytes, ms_ceiling, gb / ms_ceiling * 1e3, ms_null[0] / ms_ceiling), flush=True)

    # the host writer on the 256^3 mesh, and the device's bytes for the same mesh
    m256 = sdf.ToMesh(mn, mx, 256, 256, 256)
    hp, dp = os.path.join(OUT, "readme256_host.obj"), os.path.join(OUT, "readme256_device.obj")
    t0 = time.perf_counter()
    Mesh(m256.Vertices, m256.Colors, m256.Normals, m256.Triangles, m256.Min, m256.Max).WriteObj(hp)
    th = time.perf_counter() - t0
    hb = os.path.getsize(hp)
    m256.WriteObj(dp)
    same = open(hp, "rb").read() == open(dp, "rb").read()
    os.remove(hp)
    os.remove(dp)
    print("host writer, README 256^3: %d bytes in %.2f s = %.2f MB/s; device file identical: %s"
          % (hb, th, hb / th / 1e6, same))
    print("host writer at 1024^3 (EXTRAPOLATED from the 256^3 rate, not measured): %.0f s for %d bytes"
          % (nbytes / (hb / th), nbytes))
    assert same
    if OWN_OUT:
        os.rmdir(OUT)


if __name__ == "__main__":
    main()
