"""Time sr_get_points on the cfg4 workload and the host loop it replaces.

cfg4 (bench.py --workload cfg4): 8 refractive, distorted 1920x1080 views.  All views are run through sr_run_view and
sr_cross_check, then, per view:
  - call_ms:   one sr_get_points fetch (count, compaction, copies into pageable numpy buffers; it ends in a
               synchronise), median over warm calls timed with the host clock;
  - kernel_ms / copy_ms: device time of the points_* kernels and of the device-to-host copies of one call,
               from torch.profiler (CUDA activities) over the same number of calls, in a separate pass.
The host side is MultiViewStereo::pointCloud() without setKeepPointCloud (Camera::unproject per pixel on one thread),
timed by tests/cpp/point_cloud_test.cpp on the same views in the same run; the driver also checks that the class's
GPU cloud equals that host loop's.

    python tools/point_cloud_timing.py [--calls 10] [--out point_cloud_timing.json]

Prints the GPU name and power limit and the host CPU beside the numbers, as one JSON object.
"""
import argparse
import json
import os
import platform
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
from stereoreconstruction_b200 import capi, scenes  # noqa: E402

CROSS_CHECK = 5.0  # bench.py's multi-view cross-check threshold


def gpu_name_and_power():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown (nvidia-smi failed)"


def cpu_name():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor() or "unknown"


def device_split(ctx, view, calls):
    """(kernel ms, copy ms) of one sr_get_points call: device times summed over `calls` profiled calls."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            ctx.points(view)
        torch.cuda.synchronize()
    kern = copy = 0.0
    for ev in prof.events():
        name = ev.name
        dt = getattr(ev, "device_time", None)
        if dt is None:
            dt = ev.cuda_time
        if "points_" in name and "kernel" in name:
            kern += dt
        elif "Memcpy DtoH" in name:
            copy += dt
    return kern / 1e3 / calls, copy / 1e3 / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    wl = bench.workload("cfg4")
    w, h, V, P = wl["w"], wl["h"], wl["V"], wl["params"]
    ctx = capi.Context(0)
    ctx.set_views(wl["cams"], [np.zeros((h, w, 4), np.uint8)] * V, None)
    ctx.set_params(P)
    imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), wl["surf"], wl["seed"], wl["cell"])
    ctx.set_views(wl["cams"], imgs, None)
    ctx.set_params(P)
    nbrs = bench.neighbours_for(wl)
    for v in range(V):
        ctx.run_view(v, nbrs[v])
    ctx.cross_check(False, CROSS_CHECK)
    ctx.synchronize()

    views = []
    for v in range(V):
        for _ in range(2):  # warm-up
            ctx.points(v)
        ts = []
        for _ in range(args.calls):
            t0 = time.perf_counter()
            xyz, _, _ = ctx.points(v)
            ts.append((time.perf_counter() - t0) * 1e3)
        views.append(dict(view=v, points=int(len(xyz)), call_ms=statistics.median(ts)))
    for v in range(V):
        views[v]["kernel_ms"], views[v]["copy_ms"] = device_split(ctx, v, args.calls)
    ctx.close()

    # the host loop, timed by the C++ driver on the same views (label mode, as above)
    from test_gpu_point_cloud import write_scene
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "point_cloud_test")
        pkg = os.path.join(ROOT, "stereoreconstruction_b200")
        subprocess.run(["g++", "-std=c++17", "-O2", "-Wno-deprecated-declarations", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "point_cloud_test.cpp"), "-L", pkg, "-lsr_b200", "-lz",
                        "-Wl,-rpath," + pkg, "-o", exe], check=True)
        scene = os.path.join(tmp, "scene.bin")
        write_scene(scene, wl["cams"], imgs, None)
        r = subprocess.run([exe, scene, "-", str(P.min_depth), str(P.max_depth), str(P.num_levels), str(CROSS_CHECK), "0"],
                           capture_output=True, text=True, check=True)
        host_line = r.stdout.strip().splitlines()[-1]
    fields = dict(kv.split("=") for kv in host_line.split()[1:])

    res = dict(
        workload=wl["desc"], gpu=gpu_name_and_power(), host_cpu=cpu_name(), calls_per_view=args.calls,
        views=views,
        gpu_call_ms_total=sum(x["call_ms"] for x in views),
        gpu_kernel_ms_total=sum(x["kernel_ms"] for x in views),
        gpu_copy_ms_total=sum(x["copy_ms"] for x in views),
        host_loop_ms_total=float(fields["host_ms"]),
        host_loop_points=int(fields["host"]), class_gpu_points=int(fields["kept"]),
        class_gpu_vs_host_max_rel=float(fields["max_rel"]), class_gpu_vs_host_same_rgb=fields["same_rgb"] == "1",
    )
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
