#!/usr/bin/env python3
"""MarchingCubes.CreateMesh on resident voxels of the README scene, 1024^3 (one meshing job) and 2048^3 (sub-slabs), on
ONE device.

Prints the card and its power limit, then per size: the sub-slab count, the device time of the device-resident mesh
(sdfk_mesh_create between two CUDA events on the context's stream; the call ends in a synchronise, so the host wall time
of the call is printed too), and the wall time of Voxels.ToMesh, which adds the download of the mesh into page-locked host
memory.  Median and minimum over REPS calls after two warm-up calls.  The voxels are sampled once per size and kept.
A size whose voxels do not fit the free device memory is reported as skipped.

    python tools/time_large_voxel_mesh.py [sizes...]        (default: 1024 2048)
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from sdfkit_b200 import scenes  # noqa: E402
from sdfkit_b200.voxels import MarchingCubes  # noqa: E402

REPS = 10


def sub_slab_layers(n):
    """Cell layers per sub-slab of an n^3 grid at step 1 (mesh_max_layers in sdfk_api.cu); n - 1 when one job holds the grid."""
    per_layer = (n - 1) ** 2
    if (n - 1) * per_layer <= 0xFFFFFFF0:
        return n - 1
    return max(8, min(0xF0000000 // per_layer - 2, (3 << 30) // (n * n)))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() or "unknown (nvidia-smi: %s)" % r.stderr.strip()


def stats(ts):
    return "median %.2f ms, min %.2f ms" % (float(np.median(ts)), float(np.min(ts)))


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [1024, 2048]
    print("card: %s" % card())
    expr, mn, mx = scenes.readme_scene()
    sdf = expr.ToSdf()
    ctx = sdf.ctx
    for n in sizes:
        free, _ = torch.cuda.mem_get_info(0)
        if free < n ** 3 * 16 + (12 << 30):
            print("%d^3: skipped, %.1f GB free on the device" % (n, free / 1e9))
            continue
        vox = sdf.ToVoxels(mn, mx, n, n, n)
        ncz, layers = n - 1, sub_slab_layers(n)
        print("%d^3: %d cell layers, sub-slabs of %d layers -> %d meshing job(s)" % (n, ncz, layers, -(-ncz // layers)))
        dev, wall, full = [], [], []
        for rep in range(REPS + 2):
            ctx.timer_start()
            t0 = time.perf_counter()
            gm = MarchingCubes.CreateGpuMesh(vox)
            t1 = time.perf_counter()
            ms = ctx.timer_stop()
            nv, nt = gm.counts()
            gm.destroy()
            t2 = time.perf_counter()
            mesh = vox.ToMesh()
            t3 = time.perf_counter()
            del mesh
            if rep >= 2:
                dev.append(ms)
                wall.append((t1 - t0) * 1e3)
                full.append((t3 - t2) * 1e3)
        print("  %d vertices, %d triangles" % (nv, nt))
        print("  sdfk_mesh_create, device (CUDA events): %s" % stats(dev))
        print("  sdfk_mesh_create, host wall:            %s" % stats(wall))
        print("  Voxels.ToMesh incl. download, wall:     %s" % stats(full))
        vox.Dispose()
        del vox
        torch.cuda.synchronize()


if __name__ == "__main__":
    main()
