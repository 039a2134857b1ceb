"""Time sr_mrf_select on the cfg4 workload, the cost of keeping the peak lists it reads, and its effect on the depth
maps against the scene's known geometry.

cfg4 (bench.py --workload cfg4): 8 refractive, distorted 1920x1080 views, 256 depth levels.  Per mode (label, curve):
  - run_ms / run_keep_ms: all 8 sr_run_view(_curve) calls and a synchronise, without and with keep_cost_volume & 2
    (median of --reps timed passes after one warm-up, host clock);
  - mrf_ms: one sr_mrf_select per view with the defaults, CUDA events on the context stream around the call
    (which ends in the energy download); mrf0_ms the same with iterations = 0 (prep, labelling and energy only);
    per_iteration_ms = (mrf_ms - mrf0_ms) / iterations;
  - quality: per MRF setting and for the winner-take-all (WTA), over the in-mask pixels of all views, "cover" = the
    fraction with a depth (finite, not -1) and "within_step" = the fraction within one label step of the true depth
    (p - C) . n of the height field hit by the pixel's ray, before and after sr_cross_check (bench.py's threshold).

    python tools/mrf_timing.py [--reps 3] [--modes label,curve] [--out mrf_timing.json]

Prints the GPU name and power limit, read in the same process, beside the numbers, as one JSON object.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from stereoreconstruction_b200 import capi, scenes  # noqa: E402

CROSS_CHECK = 5.0  # bench.py's multi-view cross-check threshold
# MRF settings compared with the defaults: (smooth_weight, smooth_trunc)
SETTINGS = [None, (0.02, 8.0), (0.05, 8.0), (0.1, 8.0), (0.3, 4.0)]


def gpu_name_and_power():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown (nvidia-smi failed)"


def quality(ctx, depths, truth, step):
    """(cover, within_step) of the given maps, and after sr_cross_check on them."""
    def stats(ds):
        cov = ok = tot = 0
        for d, t in zip(ds, truth):
            have = np.isfinite(d) & (d != -1.0)
            cov += have.sum()
            ok += (have & (np.abs(d - t) <= step)).sum()
            tot += d.size
        return round(cov / tot, 4), round(ok / tot, 4)
    for v, d in enumerate(depths):
        ctx.set_depth(v, d)
    ctx.cross_check(False, CROSS_CHECK)
    after = [ctx.depth(v) for v in range(len(depths))]
    b, a = stats(depths), stats(after)
    return dict(cover=b[0], within_step=b[1], cover_cross_checked=a[0], within_step_cross_checked=a[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--modes", default="label,curve")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    wl = bench.workload("cfg4")
    w, h, V, P = wl["w"], wl["h"], wl["V"], wl["params"]
    ctx = capi.Context(0)
    ctx.set_views(wl["cams"], [np.zeros((h, w, 4), np.uint8)] * V, None)
    ctx.set_params(P)
    imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), wl["surf"], wl["seed"], wl["cell"])
    truth = []
    for v in range(V):
        p = wl["surf"].hit(ctx.unproject_grid(v))
        c = wl["cams"][v]
        truth.append((p - np.array(c.C[:])) @ np.array(c.prin_dir[:]))
    ctx.set_views(wl["cams"], imgs, None)
    nbrs = bench.neighbours_for(wl)
    step = (P.max_depth - P.min_depth) / (P.num_levels - 1)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    defaults = capi.mrf_params_default()

    res = dict(workload=wl["desc"], gpu=gpu_name_and_power(),
               mrf_defaults=dict((f, getattr(defaults, f)) for f, _ in defaults._fields_), modes={})
    for mode in args.modes.split(","):
        run = ctx.run_view_curve if mode == "curve" else ctx.run_view

        def run_all(keep):
            P.keep_cost_volume = keep
            ctx.set_params(P)
            ts = []
            for rep in range(args.reps + 1):
                ctx.synchronize()
                t0 = time.perf_counter()
                for v in range(V):
                    run(v, nbrs[v])
                ctx.synchronize()
                if rep:
                    ts.append((time.perf_counter() - t0) * 1e3)
            return statistics.median(ts)
        out = dict(run_ms=run_all(0), run_keep_ms=run_all(2))

        # every view once more with the lists kept: its WTA map and lists, then the MRF timings on those lists
        wta, lists, mrf_ms, mrf0_ms = [], [], [], []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def timed(v, p):
            ctx.flush()
            ev0.record(stream)
            ctx.mrf_select(v, p)
            ev1.record(stream)
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1)
        for v in range(V):
            run(v, nbrs[v])
            wta.append(ctx.depth(v))
            lists.append(ctx.peaks(v))
            timed(v, capi.mrf_params_default(iterations=0))  # warm-up
            mrf0_ms.append(statistics.median(timed(v, capi.mrf_params_default(iterations=0)) for _ in range(args.reps)))
            mrf_ms.append(statistics.median(timed(v, defaults) for _ in range(args.reps)))
        out.update(mrf_ms_per_view=statistics.median(mrf_ms), mrf0_ms_per_view=statistics.median(mrf0_ms),
                   per_iteration_ms=(statistics.median(mrf_ms) - statistics.median(mrf0_ms)) / defaults.iterations)
        q = dict(wta=quality(ctx, wta, truth, step))
        for s in SETTINGS:
            p = capi.mrf_params_default() if s is None else capi.mrf_params_default(smooth_weight=s[0], smooth_trunc=s[1])
            ds = []
            for v in range(V):
                ctx.set_peaks(v, lists[v])
                ctx.mrf_select(v, p)
                ds.append(ctx.depth(v))
            name = "mrf_defaults" if s is None else f"mrf_weight{s[0]}_trunc{s[1]}"
            q[name] = quality(ctx, ds, truth, step)
        out["quality"] = q
        res["modes"][mode] = out
        print(json.dumps({mode: out}), flush=True)
    ctx.close()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
