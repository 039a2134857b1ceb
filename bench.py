#!/usr/bin/env python
"""bench.py — cost-volume throughput (build + aggregate + WTA) in Mpix*disp/s.

One "step" = the full dense-matching job of the workload: every reference view of the synthetic
8-view refractive scene (BASELINE.json configs[3], "cfg4", the configuration north_star quotes
its target on) through sr_run_view: stage (1) refractive tap-volume build, stages (2)+(3)
support-weight aggregation with fused WTA.  Metric = sum over reference views of H*W*D / time.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload cfg4|cfg5|cfg3|small] [--partition views|rows] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); reference views are dealt to ranks (north_star:
"by reference view for multi-view runs") or, with --partition rows, every rank takes a row band of
every view; no collective on the data path; the total work is fixed, so scaling is "strong".
`--impl reference` times the reference's own MultiViewStereo (oracle/_ref, compiled from the
reference's sources where they lie) — or the CPU oracle port when that library is absent — on a
bounded row band with all host threads.

What the line carries beyond the contract keys (all measured in this run unless a source is named):
  roofline          HBM view of the dominant kernel (contract) + `issue`: the instruction-issue view
                    (warp-instructions per unit from the committed ncu capture x this run's units, over
                    the SM issue rate at this run's clock) with the FMA/FP64 pipe utilisations
  cpu_baseline      the oracle port in label mode on a band of a mid-arc view (doubles as the
                    full-size parity check), `reference_itself` (the reference's curve search on the
                    same band, with the GPU's curve mode checked against ITS depths)
  like_for_like     GPU label mode / port label mode, GPU curve mode / reference curve mode
  job               MultiViewStereo::runTask end to end: upload, all views, gather (N > 1), cross-check, download
  parity_vs_1gpu    (N > 1) the ranks' maps against rank 0's solo recomputation, bit for bit
  secondary         (N > 1) the other partition (row bands) timed and checked the same way
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from stereoreconstruction_b200 import scenes, sharding, types as T  # noqa: E402

METRIC = "cost-volume Mpix*disp/s (build+aggregate+WTA)"
UNIT = "Mpix*disp/s"
# --dump-outputs: 3 float64 maps x 8 views x 2^18 pixels = 48 MiB, under the 64 MB a dump may take
DUMP_PIXELS = 1 << 18


def dump_pixels(h, w):
    """The flat pixel indices --dump-outputs keeps of an h x w map: all of them, or a fixed seeded sample."""
    return np.sort(np.random.default_rng(0).choice(h * w, min(h * w, DUMP_PIXELS), replace=False))


def workload(name):
    """Returns dict(w,h,V,D,params,cams,max_nbrs,desc)."""
    if name == "cfg4":
        w, h, V, D = 1920, 1080, 8, 256
    elif name == "cfg5":
        w, h, V, D = 3840, 2160, 8, 512
    elif name == "small":
        w, h, V, D = 480, 270, 8, 64
    elif name == "cfg3":
        w, h, V, D = 1920, 1080, 2, 256
    else:
        raise SystemExit(f"unknown workload {name}")
    if name == "cfg3":
        cams, _ = scenes.rectified_pair(w, h, z0=100.0)
        P = T.default_params(False, 100.0, 500.0, D, radius=16, weight_kind=T.SR_WEIGHT_ADAPTIVE)
        desc = "cfg3: synthetic rectified 1920x1080 pair, 256 disparities, AdaptiveWeight 33x33, NCC, both directions"
        surf = scenes.HeightField(z0=167.0, amp=20.0, lx=25.0, ly=18.0)
        cell = 3.5 * 167.0 / cams[0].K[0]
        seed = 1234
    else:
        cams = scenes.arc_cameras(V, w, h)
        P = T.default_params(True, 350.0, 650.0, D)  # GeodesicWeight r=2, NCC, 3 neighbours (reference defaults)
        desc = (f"{name}: synthetic refractive {V}-view {w}x{h}, {D} depth hypotheses, tilted planar interface "
                f"(n=1.333), lens distortion, GeodesicWeight r=2, 3 nearest neighbour views, all reference views")
        surf = scenes.HeightField(z0=0.0, amp=25.0, lx=90.0, ly=70.0)
        cell = 3.5 * 500.0 / cams[0].K[0]
        seed = 4321 if name != "cfg5" else 8765
    return dict(name=name, w=w, h=h, V=V, D=D, params=P, cams=cams, desc=desc, surf=surf, cell=cell, seed=seed)


def neighbours_for(wl, ctx=None):
    if wl["name"] == "cfg3":
        return [[1], [0]]
    return scenes.nearest_neighbours(wl["cams"], 3)


def sample_view(wl):
    """The reference view the CPU samples run on: mid-arc, so that its neighbours lie on both sides."""
    return 0 if wl["name"] == "cfg3" else wl["V"] // 2


def host_threads():
    """All host threads for the OpenMP-parallel CPU arms.  torchrun exports OMP_NUM_THREADS=1 for N > 1:
    the count is set explicitly, in the environment (read by libgomp when it loads) and through libgomp."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ.pop("OMP_THREAD_LIMIT", None)
    try:
        ctypes.CDLL("libgomp.so.1", mode=ctypes.RTLD_GLOBAL).omp_set_num_threads(n)
    except OSError:
        pass
    return n


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([time.time()] + [c.strip() for c in line.split(",")])
        except Exception:
            pass

    def finish(self, t_begin=None, t_end=None):
        """Samples inside [t_begin, t_end] (the timed region); when the region is shorter than two
        sampling periods, all samples since the sampler started (warm-up steps + timed region, the
        same load) are used and `window` says so."""
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        rows, window = self.rows, "warmup+timed"
        if t_begin is not None:
            inside = [r for r in self.rows if t_begin <= r[0] <= t_end]
            if len(inside) >= 2:
                rows, window = inside, "timed"
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "window": window}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "window": window}


def cpu_sample(wl, imgs, rows, steps=1, warmup=0, target_s=12.0):
    """Times the CPU oracle (all host threads) on a row band of the mid-arc reference view of the workload.
    rows <= 0: a short probe sizes the band so that one timed pass takes about `target_s`."""
    from oracle import oracle_api as O
    host_threads()
    sc = O.Scene(wl["cams"], imgs)
    nb = neighbours_for(wl)
    P = T.SrParams.from_buffer_copy(wl["params"])
    v0 = sample_view(wl)

    last = {}

    def run(nrows):
        r0 = (wl["h"] - nrows) // 2
        P.row_begin, P.row_end = r0, r0 + nrows
        t0 = time.perf_counter()
        if wl["name"] == "cfg3":
            od, oi, ob, _ = sc.twoview_label(P, 0, 1)
        else:
            od, oi, ob, _, _ = sc.mvs_view(P, v0, nb[v0])
        dt = time.perf_counter() - t0
        last.update(depth=od[r0:r0 + nrows], index=oi[r0:r0 + nrows], best=ob[r0:r0 + nrows], r0=r0, rows=nrows, view=v0)
        return dt, r0

    if rows <= 0:
        probe = max(2, min(wl["h"], O.num_threads()))  # one row per thread
        tp, _ = run(probe)
        rows = int(max(probe, min(wl["h"], probe * target_s / max(tp, 1e-3))))
        rows -= rows % max(1, O.num_threads())  # whole rows per thread under the static schedule
        rows = max(rows, probe)
    times = []
    r0 = 0
    for i in range(warmup + steps):
        dt, r0 = run(rows)
        if i >= warmup:
            times.append(dt)
    units = rows * wl["w"] * wl["D"]
    t = sum(times) / len(times)
    cpu_sample.last = last  # the band's outputs: compared with the GPU's for the same rows (parity at full size)
    return units / t / 1e6, t, O.num_threads(), (f"{rows} rows x {wl['w']} px x {wl['D']} labels of reference view {v0} "
                                               f"(rows {r0}..{r0 + rows})")


def reference_sample(wl, imgs, rows, steps=1, warmup=0, target_s=12.0):
    """Times the REFERENCE'S OWN MultiViewStereo::computeInitialEstimate (stereo/multiviewstereo.cpp compiled
    where it lies, oracle/_ref/libref.so; its tbb::parallel_for over rows on all host threads) on a row
    band of the mid-arc reference view of the workload: the reference view's mask is reduced to the band (the
    class skips pixels outside its mask), the neighbours are the ones its runTask() rule selects.  This is the
    reference's live formulation — candidates are the pixels of the rasterised epipolar curve that the D
    depth labels span — so a unit of work is still one (pixel, depth label).  Returns None when the
    prebuilt library is not there (then the oracle port is timed instead)."""
    from oracle import oracle_api as O
    if wl["name"] == "cfg3" or O.ref_lib() is None:
        return None
    host_threads()
    P = wl["params"]
    nb = neighbours_for(wl)
    h = wl["h"]
    v0 = sample_view(wl)
    threads = [1]
    last = {}

    def timed(nrows, r0):
        # a fresh task object per pass: narrowing the view's mask to the band cannot be undone
        band = O.RefMVS(wl["cams"], imgs, None, P.min_depth, P.max_depth, P.num_levels, 5.0, image_scale=P.image_scale)
        threads[0] = band.num_threads()
        for v in range(wl["V"]):
            band.set_neighbours(v, nb[v])
        band.mask_rows(v0, r0, r0 + nrows)
        t0 = time.perf_counter()
        d, _ = band.initial_estimate(v0)
        dt = time.perf_counter() - t0
        band.close()
        last.update(depth=d[r0:r0 + nrows], r0=r0, rows=nrows, view=v0)
        return dt

    if rows <= 0:
        probe = max(2, min(h, host_threads()))  # about one row per thread
        tp = timed(probe, (h - probe) // 2)
        rows = int(max(probe, min(h, probe * target_s / max(tp, 1e-3))))
        rows -= rows % max(1, threads[0])
        rows = max(rows, probe)
    r0 = (h - rows) // 2
    times = []
    for i in range(warmup + steps):
        dt = timed(rows, r0)
        if i >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    units = rows * wl["w"] * wl["D"]
    reference_sample.last = last
    return units / t / 1e6, t, threads[0], (f"{rows} rows x {wl['w']} px x {wl['D']} depth levels of reference view {v0} "
                                         f"(rows {r0}..{r0 + rows}), MultiViewStereo::computeInitialEstimate of the reference itself")


def render_on_cpu(wl):
    """The workload's images rendered through the ORACLE's unproject (the reference arm has no GPU code on its
    path); the GPU arm renders the same scene through its own unproject (equal to 1e-11)."""
    from oracle import oracle_api as O
    w, h = wl["w"], wl["h"]
    cams = O.as_cam_array(wl["cams"])

    def rays(v):
        out = np.empty((h, w, 6), dtype=np.float64)
        O.lib().orc_unproject_grid(ctypes.byref(cams[v]), w, h, ctypes.c_double(wl["params"].image_scale),
                                   out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
        return out

    return scenes.render_views(wl["V"], rays, wl["surf"], wl["seed"], wl["cell"])


def same_maps(a, b):
    """Elementwise equality with NaN == NaN."""
    if a.dtype.kind == "f":
        return (a == b) | (np.isnan(a) & np.isnan(b))
    return a == b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip job / curve-mode / secondary / parity legs (profiling aid)")
    ap.add_argument("--views", type=int, default=0, help="only the first N reference views (profiling aid; 0 = all)")
    ap.add_argument("--partition", default="views", choices=["views", "rows"],
                    help="multi-GPU: deal reference views to ranks (default) or give every rank a row band of every view")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what their last step returned for each reference view (depth, "
                         "depth_index, best_cost) as DIR/<name>_view<v>.npy, float64, at a fixed seeded sample of "
                         f"{DUMP_PIXELS} pixels per view (the whole map when it is smaller)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or (world > 1 and args.partition == "rows")):
        raise SystemExit("--dump-outputs needs --impl ours and whole views per rank (--partition views)")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = workload(args.workload)
    w, h, V, D = wl["w"], wl["h"], wl["V"], wl["D"]
    cpu_rows = args.cpu_rows  # 0: sized by a probe to ~12 s of CPU work

    # ------------------------------------------------------------------ reference arm (the reference's own CPU code)
    if args.impl == "reference":
        if rank != 0:
            return
        cores = host_threads()
        imgs = render_on_cpu(wl)  # the same rendered scene as the GPU arm
        kind, note = "reference", ("the reference's own MultiViewStereo (stereo/multiviewstereo.cpp compiled where it lies, "
                                   "oracle/_ref; its tbb::parallel_for over rows on all host threads); each step = the bounded "
                                   "sample; same rendered images as the GPU arm, mid-arc reference view")
        got = reference_sample(wl, imgs, cpu_rows, steps=max(1, args.steps), warmup=min(args.warmup, 1))
        if got is None:
            kind, note = "port", "CPU oracle (restated reference, OpenMP over rows); each step = the bounded sample"
            got = cpu_sample(wl, imgs, cpu_rows, steps=max(1, args.steps), warmup=min(args.warmup, 1))
        val, t, cores_used, sample = got
        line = {
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["desc"], "note": note, "host_threads_available": cores},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores_used, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (CUDA)
    import torch
    import torch.distributed as dist
    from stereoreconstruction_b200 import capi

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = capi.Context(local_rank)
    stream = torch.cuda.Stream()  # an explicit stream: the library launches on it, the events time it
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    # synthetic, photo-consistent inputs rendered through the GPU's own unproject
    cams = wl["cams"]
    blank = [np.zeros((h, w, 4), np.uint8)] * V
    ctx.set_views(cams, blank, None)
    ctx.set_params(wl["params"])
    cache = os.environ.get("SR_BENCH_IMAGE_CACHE")  # A/B aid: several runs in one session render the scene once
    if cache and os.path.exists(cache):
        imgs = list(np.load(cache)["imgs"])
    else:
        imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), wl["surf"], wl["seed"], wl["cell"])
        if cache:
            np.savez(cache, imgs=np.stack(imgs))
    pinned = [torch.from_numpy(im).pin_memory() for im in imgs]
    imgs_p = [p.numpy() for p in pinned]
    ctx.set_views(cams, imgs_p, None)
    nbrs = neighbours_for(wl)
    ref_views = list(range(V if args.views <= 0 else min(V, args.views)))
    units_total = len(ref_views) * h * w * D
    full_params = T.SrParams.from_buffer_copy(wl["params"])

    def partition(kind):
        """(my views, my row band) under the views / rows partition."""
        if kind == "rows" and world > 1:
            return list(ref_views), sharding.row_bands(h, world)[rank]
        return [v for v in sharding.partition_views(V, world)[rank] if v in ref_views], (0, h)

    def set_rows(b0, b1):
        P = T.SrParams.from_buffer_copy(full_params)
        P.row_begin, P.row_end = (b0, b1) if (b0, b1) != (0, h) else (0, 0)
        ctx.set_params(P)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_steps(views, steps, warmup):
        """(ms per step on the device, max over ranks; wall-clock bounds of the timed region)."""
        for _ in range(warmup):
            for v in views:
                ctx.run_view(v, nbrs[v])
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_begin = time.time()
        ev0.record(stream)
        for _ in range(steps):
            for v in views:
                ctx.run_view(v, nbrs[v])
        ctx.flush()  # the views run on the library's internal lanes: order them before the event
        ev1.record(stream)
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1)) / steps, t_begin, time.time()

    def parity_vs_solo(kind, views, band):
        """The maps this run's ranks produced against rank 0's solo recomputation (full rows, no sharding):
        every rank contributes one of its views (views partition) or its band of view 0 (rows partition)."""
        if world == 1:
            return None
        b0, b1 = band
        pv = views[0] if views else -1
        mine_i = torch.from_numpy(ctx.depth_index(pv)).cuda() if pv >= 0 else torch.zeros((h, w), dtype=torch.int32, device="cuda")
        mine_d = torch.from_numpy(ctx.depth(pv)).cuda() if pv >= 0 else torch.zeros((h, w), dtype=torch.float64, device="cuda")
        meta = torch.tensor([pv, b0, b1], device="cuda", dtype=torch.int64)
        metas = [torch.zeros_like(meta) for _ in range(world)]
        gi = [torch.zeros_like(mine_i) for _ in range(world)]
        gd = [torch.zeros_like(mine_d) for _ in range(world)]
        dist.all_gather(metas, meta)
        dist.all_gather(gi, mine_i)
        dist.all_gather(gd, mine_d)
        out = None
        if rank == 0:
            set_rows(0, h)
            solo, checked, bad_i, bad_d, npx = {}, [], 0, 0, 0
            for r in range(world):
                v, r0, r1 = (int(x) for x in metas[r].tolist())
                if v < 0 or r1 <= r0:
                    continue
                if v not in solo:
                    ctx.run_view(v, nbrs[v])
                    solo[v] = (ctx.depth_index(v).copy(), ctx.depth(v).copy())
                si, sd = solo[v]
                bad_i += int((gi[r].cpu().numpy()[r0:r1] != si[r0:r1]).sum())
                bad_d += int((~same_maps(gd[r].cpu().numpy()[r0:r1], sd[r0:r1])).sum())
                npx += (r1 - r0) * w
                checked.append({"rank": r, "view": v, "rows": [r0, r1]})
            out = {"partition": kind, "checked": checked, "pixels": npx, "index_mismatches": bad_i,
                   "depth_mismatches": bad_d, "identical": bad_i == 0 and bad_d == 0}
        barrier()
        return out

    # ------------------------------------------------------------------ headline: K timed steps
    my_views, my_band = partition(args.partition)
    set_rows(*my_band)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        for v in my_views:
            ctx.run_view(v, nbrs[v])
    barrier()
    launches0 = ctx.launch_count()
    ms_per_step, t_begin, t_end = timed_steps(my_views, args.steps, 0)
    clocks = sampler.finish(t_begin, t_end)
    launches = ctx.launch_count() - launches0
    if args.dump_outputs:  # before the legs below recompute (or cross-check) any view
        os.makedirs(args.dump_outputs, exist_ok=True)
        pick = dump_pixels(h, w)
        for v in my_views:
            for name, a in (("depth", ctx.depth(v)), ("depth_index", ctx.depth_index(v)), ("best_cost", ctx.best_cost(v))):
                np.save(os.path.join(args.dump_outputs, f"{name}_view{v}.npy"), a.reshape(-1)[pick].astype(np.float64))
    # per-stage device times: one more step with the library's per-stage events on (which serialises the
    # views on the context stream: a kernel's duration is then its own, not stretched by the overlap)
    ctx.set_profiling(True)
    for v in my_views:
        ctx.run_view(v, nbrs[v])
    stages = ctx.stage_ms()
    if os.environ.get("SR_MATCH_STATS"):
        print("match stats:", ctx.match_stats(), file=sys.stderr)
        print("build stats:", ctx.build_stats(), file=sys.stderr)
    ctx.set_profiling(False)
    value = units_total / (ms_per_step * 1e-3) / 1e6
    parity_n = None if args.no_extras else parity_vs_solo(args.partition, my_views, my_band)
    set_rows(*my_band)

    # ------------------------------------------------------------------ end to end through the C ABI with host buffers
    # H2D of the images this rank needs + run + D2H of what MultiViewStereo::fetch pulls per view it computed
    # (f64 depth map + int32 index map), all inside the timed region, pinned host memory on both sides.
    idx_host = [torch.empty((h, w), dtype=torch.int32).pin_memory().numpy() for _ in my_views]
    dep_host = [torch.empty((h, w), dtype=torch.float64).pin_memory().numpy() for _ in my_views]
    needed = set(my_views) | {n for v in my_views for n in nbrs[v]}
    imgs_e2e = [imgs_p[v] if v in needed else None for v in range(V)]  # the others stay camera-only

    def e2e_step():
        ctx.set_views(cams, imgs_e2e, None)
        set_rows(*my_band)
        for v in my_views:
            ctx.run_view(v, nbrs[v])
        for k, v in enumerate(my_views):
            ctx.depth(v, out=dep_host[k])
            ctx.depth_index(v, out=idx_host[k])

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 2))
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e_val = units_total / e2e_s / 1e6
    rows_frac = (my_band[1] - my_band[0]) / h
    d2h_bytes = int(len(my_views) * h * w * 12)

    # ------------------------------------------------------------------ the whole job (MultiViewStereo::runTask)
    job = None
    if not args.no_extras and wl["name"] != "cfg3" and len(ref_views) == V:
        if world > 1:  # the library's own gather: NCCL broadcasts from the owners (sr_comm_allgather_*)
            uid = [capi.Context.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            ctx.comm_init(uid[0], rank, world)
        owner = sharding.view_owner(V, world)
        bands = sharding.row_bands(h, world)

        def job_step():
            ctx.set_views(cams, imgs_e2e, None)
            set_rows(*my_band)
            for v in my_views:
                ctx.run_view(v, nbrs[v])
            ctx.synchronize()  # (only to attribute the gather and the cross-check their own times)
            g0 = time.perf_counter()
            if world > 1:
                if args.partition == "rows":
                    for v in range(V):
                        ctx.allgather_rows(v, [b[0] for b in bands], [b[1] for b in bands])
                else:
                    ctx.allgather_views(owner)
                ctx.synchronize()
            g1 = time.perf_counter()
            ctx.cross_check(False, 5.0)
            ctx.synchronize()
            g2 = time.perf_counter()
            for k, v in enumerate(my_views):
                ctx.depth(v, out=dep_host[k])
            return g1 - g0, g2 - g1

        job_step()
        barrier()
        t0 = time.perf_counter()
        ga, cc = job_step()
        barrier()
        job_s = max_over_ranks(time.perf_counter() - t0)
        job = {"value": units_total / job_s / 1e6, "unit": UNIT, "seconds_per_step": job_s,
               "allgather_ms": max_over_ranks(ga) * 1e3, "cross_check_ms": max_over_ranks(cc) * 1e3,
               "what": "upload + all reference views + depth-map gather (N > 1: sr_comm_allgather_*, NCCL) + cross-check "
                       "(threshold 5) + download of the cross-checked f64 depth maps: MultiViewStereo::runTask"}
        ctx.set_views(cams, imgs_p, None)  # every image again for the legs below

    # ------------------------------------------------------------------ the other partition (N > 1)
    secondary = None
    if world > 1 and not args.no_extras and wl["name"] != "cfg3":
        other = "rows" if args.partition == "views" else "views"
        ctx.set_views(cams, imgs_p, None)
        o_views, o_band = partition(other)
        set_rows(*o_band)
        o_ms, _, _ = timed_steps(o_views, max(1, min(args.steps, 2)), 1)
        secondary = {"partition": other, "value": units_total / (o_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": o_ms,
                     "parity_vs_1gpu": parity_vs_solo(other, o_views, o_band)}
        set_rows(*my_band)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ------------------------------------------------------------------ rooflines of the dominant kernel
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    n_nbr = len(nbrs[my_views[0]])
    n_match = max(1, stages["match_launches"])
    match_ms = stages["match_ms"] / n_match / rows_frac  # per full view
    build_ms = stages["build_ms"] / n_match / rows_frac
    # SURVEY §8d: 8 B per pixel*disparity (volume written once by build, read once by
    # aggregate+WTA) + H*W*(4*(1+N_nbr)+4) per reference view; the match launch owns the read half
    # and the per-pixel terms.
    alg_bytes_match = h * w * D * 4 + h * w * (4 * (1 + n_nbr) + 4)
    alg_bytes_view = h * w * D * 8 + h * w * (4 * (1 + n_nbr) + 4)
    achieved = alg_bytes_match / (match_ms * 1e-3) / 1e9
    pipe_gbs = alg_bytes_view / ((match_ms + build_ms) * 1e-3) / 1e9
    kname = "match_mvs_screen2_kernel" if wl["name"] != "cfg3" else "match_kernel"
    counters = {}
    try:  # per-launch counters of the committed ncu capture of this workload (tools/make_profiles.py)
        with open(os.path.join(ROOT, "profiles", "r2_counters.json")) as f:
            counters = json.load(f).get(wl["name"], {})
    except (OSError, ValueError):
        pass
    kc = counters.get(kname, {})
    traffic = kc.get("dram_bytes")
    issue = None
    sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
    if kc.get("inst_executed") and kc.get("units"):
        n_sm = 148
        per_unit = kc["inst_executed"] / kc["units"]           # warp-instructions per (pixel, label) of one launch
        inst_view = per_unit * h * w * D                       # ... of one full view of THIS workload
        slots_per_s = 4 * n_sm * sm_mhz * 1e6                  # one warp-instruction per scheduler per clock
        min_ms = inst_view / slots_per_s * 1e3
        issue = {"bound": "issue", "warp_instr_per_unit": per_unit, "warp_instr_per_unit_per_neighbour": per_unit / n_nbr,
                 "issue_slots_per_s": slots_per_s, "sm_mhz": sm_mhz, "min_ms_per_view": min_ms,
                 "measured_ms_per_view": match_ms - kc.get("other_ms_in_stage", 0.0), "frac": min_ms / max(match_ms, 1e-9),
                 "pipe_fma_pct": kc.get("pipe_fma_pct"), "pipe_fp64_pct": kc.get("pipe_fp64_pct"),
                 "pipe_lsu_pct": kc.get("pipe_lsu_pct"), "issue_active_pct": kc.get("issue_active_pct"),
                 "source": "profiles/r2_counters.json (ncu --set full of this kernel on this workload) x this run's clock and time",
                 "note": "FMA pipe accepts one warp-instruction per 2 clocks per scheduler (FFMA2 = full FP32 rate): "
                         "its share of the label loop bounds the kernel before issue does (DESIGN.md section 5)"}
        bk = counters.get("build_refr_kernel")
        if bk and bk.get("inst_executed") and bk.get("units"):
            b_min = bk["inst_executed"] / bk["units"] * h * w * D * n_nbr / slots_per_s * 1e3
            issue["build"] = {"warp_instr_per_unit_per_neighbour": bk["inst_executed"] / bk["units"], "min_ms_per_view": b_min,
                              "measured_ms_per_view": build_ms, "frac": b_min / max(build_ms, 1e-9),
                              "pipe_fp64_pct": bk.get("pipe_fp64_pct"), "issue_active_pct": bk.get("issue_active_pct")}
    roofline = {
        "bound": "hbm", "kernel": kname + " (support-weight aggregation of the photo-consistency cost + fused WTA)",
        "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs, "traffic": traffic,
        "traffic_source": "profiles/r2_counters.json (dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full)" if traffic else None,
        "peak_source": peak_src, "match_ms_per_view": match_ms, "build_ms_per_view": build_ms,
        "pipeline_achieved_gbs": pipe_gbs, "pipeline_frac": pipe_gbs / peak_gbs,
        "issue": issue,
    }

    # ------------------------------------------------------------------ CPU legs (rank 0, N = 1 only)
    cpu = None
    like = None
    if not args.no_cpu and world == 1:
        v0 = sample_view(wl)
        val, t, cores, sample = cpu_sample(wl, imgs, cpu_rows)
        cpu = {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "seconds": t}
        like = {"label_mode_gpu_e2e_over_port": e2e_val / val, "label_mode_gpu_over_port": value / val}
        # The oracle's outputs for that band are the checker of the GPU's at the benchmark's full size.
        o = cpu_sample.last
        if v0 in my_views and o:
            ra, rb = o["r0"], o["r0"] + o["rows"]
            ctx.run_view(v0, nbrs[v0])
            gi, gd, gb = ctx.depth_index(v0)[ra:rb], ctx.depth(v0)[ra:rb], ctx.best_cost(v0)[ra:rb]
            mism = gi != o["index"]
            lab = ~mism & (o["index"] >= 0)
            with np.errstate(invalid="ignore"):
                rel = np.abs(gb[lab] - o["best"][lab]) / np.maximum(np.abs(o["best"][lab]), 1e-300)
            cpu["parity"] = {
                "pixels": int(mism.size), "index_mismatch_rate": float(mism.mean()),
                "depth_equal_where_index_equal": bool(same_maps(gd, o["depth"])[~mism].all()),
                "max_rel_cost_diff": float(rel.max()) if rel.size else None,
                "max_abs_cost_diff": float(np.abs(gb[lab] - o["best"][lab]).max()) if rel.size else None,  # (two-view costs can be ~0)
                "labelled_fraction": float(lab.mean()),
            }
        # ... and the reference's own MultiViewStereo (oracle/_ref, when the prebuilt library is there) on a band
        # of the same view: its live curve formulation, timed beside the port, and the checker of the GPU's curve
        # mode at full size (optional: never fails the line)
        try:
            got = reference_sample(wl, imgs, 0, target_s=8.0)
        except Exception as e:  # noqa: BLE001
            got = None
            cpu["reference_itself"] = {"unavailable": str(e)[:200]}
        if got:
            cpu["reference_itself"] = {"value": got[0], "unit": UNIT, "cores": got[2], "kind": "reference",
                                       "sample": got[3], "seconds": got[1]}
        if wl["name"] != "cfg3" and not args.no_extras:
            # GPU curve mode (the reference's live formulation) on the sample view: throughput and parity
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx.run_view_curve(v0, nbrs[v0])
            ctx.flush()
            ev0.record(stream)
            ctx.run_view_curve(v0, nbrs[v0])
            ev1.record(stream)
            torch.cuda.synchronize()
            curve_ms = ev0.elapsed_time(ev1)
            curve_val = h * w * D / (curve_ms * 1e-3) / 1e6
            like["gpu_curve_mode"] = {"value": curve_val, "unit": UNIT, "ms_per_view": curve_ms}
            if got:
                like["curve_mode_gpu_over_reference"] = curve_val / got[0]
                r = reference_sample.last
                ra, rb = r["r0"], r["r0"] + r["rows"]
                gd = ctx.depth(v0)[ra:rb]
                rd = r["depth"]
                with np.errstate(invalid="ignore", divide="ignore"):
                    close = same_maps(gd, rd) | (np.abs(gd - rd) <= 1e-9 * np.maximum(np.abs(rd), 1e-300))
                cpu["reference_itself"]["gpu_curve_mode_parity"] = {
                    "pixels": int(close.size), "depth_mismatch_rate_1e-9_rel": float((~close).mean()),
                    "finite_fraction": float(np.isfinite(rd).mean())}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "views_per_rank": len(my_views), "neighbours": n_nbr,
                   "l2": "inputs larger than L2 (tap volume %.1f GB per view streams through HBM)" % (n_nbr * h * w * D * 4 / 1e9),
                   "partition": ("row bands of every reference view" if (args.partition == "rows" and world > 1)
                                 else "reference views round-robin over ranks"),
                   "precision": ("every output (index, depth, winning cost) is decided in FP64; FP32 only screens labels "
                                 "that provably cannot win, and labels between exactly projected anchors are interpolated "
                                 "under a pixel-boundary guard (DESIGN.md section 3)")},
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(len(needed) * h * w * 4),
                "d2h_bytes_per_step": d2h_bytes, "seconds_per_step": e2e_s,
                "d2h": "f64 depth map + int32 index map of every view this rank computed (what MultiViewStereo::fetch pulls)"},
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "like_for_like": like,
        "job": job,
        "parity_vs_1gpu": parity_n,
        "secondary": secondary,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
