"""Time sr_fuse_points on the cfg4 workload against the per-view sr_get_points fetches it replaces, and compare the
two clouds against the scene's known geometry.

cfg4 (bench.py --workload cfg4): 8 refractive, distorted 1920x1080 views.  All views are run through sr_run_view
(label mode) and sr_cross_check at bench.py's threshold 5, then on those maps:
  - count_ms / fetch_ms: one sr_fuse_points call with capacity 0 (count only) and one count-then-fetch
    (Context.fuse_points), CUDA events on the context stream, median of --calls warm calls;
  - kernel_ms / copy_ms: device time of the fuse_* and points_scan kernels and of the device-to-host copies of
    one fetch, from torch.profiler (CUDA activities) over --calls fetches in a separate pass;
  - points_fetch_ms: the 8 per-view sr_get_points fetches (Context.points) on the same maps, same timing;
  - points: fused against concatenated;
  - quality: of each cloud, the fraction of points with |z - f(x, y)| <= one label step and the median |z - f(x, y)|.

    python tools/fuse_timing.py [--calls 10] [--min-views 1] [--out fuse_timing.json]

Prints the GPU name and power limit, read in the same process, beside the numbers, as one JSON object.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from stereoreconstruction_b200 import capi, scenes  # noqa: E402

CROSS_CHECK = 5.0  # bench.py's multi-view cross-check threshold


def gpu_name_and_power():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--min-views", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import ctypes as C
    import torch
    from torch.profiler import ProfilerActivity, profile

    wl = bench.workload("cfg4")
    w, h, V, P = wl["w"], wl["h"], wl["V"], wl["params"]
    ctx = capi.Context(0)
    ctx.set_views(wl["cams"], [np.zeros((h, w, 4), np.uint8)] * V, None)
    ctx.set_params(P)
    imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), wl["surf"], wl["seed"], wl["cell"])
    ctx.set_views(wl["cams"], imgs, None)
    ctx.set_params(P)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    nbrs = bench.neighbours_for(wl)
    for v in range(V):
        ctx.run_view(v, nbrs[v])
    ctx.cross_check(False, CROSS_CHECK)
    ctx.synchronize()
    mv = args.min_views
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        ts = []
        for rep in range(args.calls + 2):  # two warm-up calls
            ctx.synchronize()
            ev0.record(stream)
            fn()
            ev1.record(stream)
            torch.cuda.synchronize()
            if rep >= 2:
                ts.append(ev0.elapsed_time(ev1))
        return statistics.median(ts)

    n = C.c_int64(0)
    count = lambda: ctx._ck(ctx._L.sr_fuse_points(ctx._h, CROSS_CHECK, mv, 0, None, None, None, C.byref(n)))
    res = dict(workload=wl["desc"], gpu=gpu_name_and_power(), max_dist=CROSS_CHECK, min_views=mv,
               calls=args.calls)
    res["count_ms"] = timed(count)
    res["fetch_ms"] = timed(lambda: ctx.fuse_points(CROSS_CHECK, mv))
    res["points_fetch_ms"] = timed(lambda: [ctx.points(v) for v in range(V)])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.calls):
            ctx.fuse_points(CROSS_CHECK, mv)
        torch.cuda.synchronize()
    kern = copy = 0.0
    for ev in prof.events():
        dt = getattr(ev, "device_time", None)
        dt = ev.cuda_time if dt is None else dt
        if ("fuse_" in ev.name or "points_scan" in ev.name) and "kernel" in ev.name:
            kern += dt
        elif "Memcpy DtoH" in ev.name:
            copy += dt
    res["kernel_ms"], res["copy_ms"] = kern / 1e3 / args.calls, copy / 1e3 / args.calls

    step = (P.max_depth - P.min_depth) / (P.num_levels - 1)
    surf = wl["surf"]

    def quality(xyz):
        e = np.abs(xyz[:, 2] - surf.z(xyz[:, 0], xyz[:, 1]))
        return dict(points=int(len(xyz)), within_step=round(float((e <= step).mean()), 4),
                    median_abs_z_err=round(float(np.median(e)), 4))
    res["label_step"] = step
    res["fused"] = quality(ctx.fuse_points(CROSS_CHECK, mv)[0])
    res["concatenated"] = quality(np.concatenate([ctx.points(v)[0] for v in range(V)]))
    ctx.close()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
