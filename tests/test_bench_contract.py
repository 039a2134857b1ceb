"""bench.py prints ONE JSON line with the benchmark's keys: `--impl reference` (the reference's own
MultiViewStereo from oracle/_ref when it is there, else the oracle port) on the CPU, and the CUDA arm's
`--dump-outputs` on the GPU.  (profiles/r1_bench_default.json is a committed copy of a CUDA arm line.)"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--workload", "small", "--steps", "1", "--warmup", "0", "--cpu-rows", "8"])
    assert d["impl"] == "reference" and d["unit"] == "Mpix*disp/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    from oracle import oracle_api as O
    if O.ref_lib() is not None:
        assert cb["kind"] == "reference" and "of the reference itself" in cb["sample"]


def test_dump_pixels_sample_large_maps():
    import bench
    assert (bench.dump_pixels(270, 480) == np.arange(270 * 480)).all()  # the small workload: whole maps
    p = bench.dump_pixels(1080, 1920)                                    # cfg4: a fixed sample
    assert p.size == bench.DUMP_PIXELS and (np.diff(p) > 0).all() and 0 <= p[0] and p[-1] < 1080 * 1920
    assert (p == bench.dump_pixels(1080, 1920)).all()
    assert 3 * 8 * p.size * 8 <= 64e6  # depth, index and cost of 8 views in float64


@pytest.mark.gpu
def test_dump_outputs_is_complete_and_reproducible(tmp_path):
    """--dump-outputs writes every reference view's maps (float64, under 64 MB); a second run with another
    --steps dumps the same values and times twice the launches; the values are the maps sr_run_view returns."""
    common = ["--gpus", "1", "--workload", "small", "--warmup", "1", "--no-cpu", "--no-extras"]
    a = _run(common + ["--steps", "1", "--dump-outputs", str(tmp_path / "a")])
    b = _run(common + ["--steps", "2", "--dump-outputs", str(tmp_path / "b")])
    assert a["steps"] == 1 and b["steps"] == 2 and b["gpu_launches"] == 2 * a["gpu_launches"] > 0
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(f"{m}_view{v}.npy" for m in ("depth", "depth_index", "best_cost") for v in range(8))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64e6
    for n in names:
        x, y = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert x.dtype == np.float64 and x.shape == (480 * 270,)
        assert ((x == y) | (np.isnan(x) & np.isnan(y))).all(), n
    assert (np.load(tmp_path / "a" / "depth_index_view3.npy") >= 0).any()  # not vacuous: labels were found
    # the same view through the C ABI directly, with the bench's inputs
    import bench
    from stereoreconstruction_b200 import capi, scenes
    wl = bench.workload("small")
    w, h, V = wl["w"], wl["h"], wl["V"]
    ctx = capi.Context(0)
    try:
        ctx.set_views(wl["cams"], [np.zeros((h, w, 4), np.uint8)] * V, None)
        ctx.set_params(wl["params"])
        imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), wl["surf"], wl["seed"], wl["cell"])
        ctx.set_views(wl["cams"], imgs, None)
        ctx.run_view(3, bench.neighbours_for(wl)[3])
        pick = bench.dump_pixels(h, w)
        for name, direct in (("depth", ctx.depth(3)), ("depth_index", ctx.depth_index(3)), ("best_cost", ctx.best_cost(3))):
            x, y = np.load(tmp_path / "a" / f"{name}_view3.npy"), direct.reshape(-1)[pick].astype(np.float64)
            assert ((x == y) | (np.isnan(x) & np.isnan(y))).all(), name
    finally:
        ctx.close()
