"""The two empirical bounds of the screened MVS path under load they were not tuned on, with the kernels'
own self-check counters read (SR_MATCH_STATS=1):

  * the FP32 screen's error bars (sr_screen2.cuh: eps = e0 + e1 * kappa per label) — every verified label
    must lie inside its bar (`outside_error_bar == 0`), and the reserved slot 7 of the counters reads 0
    (`prescreen_false_drops == 0`, sr_b200.h);
  * the anchor interpolation of the refractive build (sr_build_refr.cuh) — with the switch on every
    interpolated label is also projected exactly, `tap_mismatches == 0`.

Inputs: adversarial images made in image space (not photo-consistent, so NCC matches only by accident and
the tie-breaks are exercised): near-constant windows with single outliers, 0/255 checkerboards and step
edges (support weights from 1 down to below the 1e-10 cut-off inside one window), +-1 gray level noise
(ill-conditioned windows: the FP64-only paths), ramps, and random scenes / the bunny fixture.  Results are
compared with the oracle as everywhere else; the reference rule being protected is the candidate selection
of stereo/multiviewstereo.cpp:589-602,654-660.

Also here: the two internal lanes, which must not change a single output bit (SR_LANES=1 vs the default),
and a context that is re-used with larger and smaller images (peak lists kept, label mode on the lanes, curve
mode)."""
import numpy as np
import pytest

from oracle import oracle_api as O
from stereoreconstruction_b200 import capi, scenes, types as T
from scene_util import refractive_arc_scene

pytestmark = pytest.mark.gpu


def _stats_ctx(monkeypatch, **env):
    monkeypatch.setenv("SR_MATCH_STATS", "1")
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    return capi.Context(0)


def _check_counters(c, need_interpolated=True):
    ms, bs = c.match_stats(), c.build_stats()
    assert ms["outside_error_bar"] == 0, ms
    assert ms["prescreen_false_drops"] == 0, ms
    assert ms["max_screen_err"] < 5e-3, ms
    assert bs["tap_mismatches"] == 0, bs
    if need_interpolated:
        assert bs["interpolated"] > 0, bs
    return ms, bs


def _compare_with_oracle(c, cams, imgs, ms, P, ref, nbrs):
    c.set_views(cams, imgs, ms)
    c.set_params(P)
    c.run_view(ref, nbrs)
    gi, gd, gb = c.depth_index(ref), c.depth(ref), c.best_cost(ref)
    od, oi, ob, _, _ = O.Scene(cams, imgs, ms).mvs_view(P, ref, nbrs)
    mism = gi != oi
    assert mism.mean() <= 1e-4, f"index mismatch rate {mism.mean()}"
    assert ((gd == od) | (np.isnan(gd) & np.isnan(od)))[~mism].all()
    lab = ~mism & (oi >= 0)
    if lab.any():
        assert np.abs(gb[lab] - ob[lab]).max() <= 1e-12
    return gi


def adversarial_images(kind, V, w, h, seed):
    rng = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    imgs = []
    for v in range(V):
        if kind == "outliers":      # near-constant windows with one outlier
            g = np.full((h, w), 120 + v, np.int32)
            g[rng.rand(h, w) < 0.04] = rng.choice([0, 255])
            rgb = np.dstack([g, g, g])
        elif kind == "checker":     # 0 / 255 extremes, period 3: many exact ties between labels
            g = (((xx + v) // 3 + yy // 3) % 2) * 255
            rgb = np.dstack([g, g, g])
        elif kind == "steps":       # strong colour edges: geodesic / adaptive weights span 1 .. < 1e-10 in a window
            g = ((xx + 2 * v) // 7 % 2) * 255
            rgb = np.dstack([g, 255 - g, (yy // 5 % 2) * 255])
        elif kind == "lowcontrast":  # +-1 gray level: ill-conditioned windows, the FP64-only paths
            g = 128 + rng.randint(-1, 2, size=(h, w))
            rgb = np.dstack([g, g, g])
        elif kind == "ramp":        # smooth ramps with a little noise: ncc close to 1 for many labels
            g = np.clip((xx * 255) // w + rng.randint(-2, 3, size=(h, w)), 0, 255)
            rgb = np.dstack([g, (yy * 255) // h, g])
        else:
            raise ValueError(kind)
        im = np.empty((h, w, 4), np.uint8)
        im[..., :3] = np.clip(rgb, 0, 255)
        im[..., 3] = 255
        imgs.append(im)
    return imgs


@pytest.mark.parametrize("kind", ["outliers", "checker", "steps", "lowcontrast", "ramp"])
@pytest.mark.parametrize("weight_kind", [T.SR_WEIGHT_GEODESIC, T.SR_WEIGHT_ADAPTIVE])
def test_adversarial_windows(monkeypatch, kind, weight_kind):
    V, w, h = 4, 72, 44
    cams = scenes.arc_cameras(V, w, h, arc_deg=22.0)
    imgs = adversarial_images(kind, V, w, h, seed=11)
    P = T.default_params(True, 430.0, 570.0, 40, weight_kind=weight_kind)
    c = _stats_ctx(monkeypatch)
    try:
        _compare_with_oracle(c, cams, imgs, None, P, 1, [0, 2, 3])
        _check_counters(c)
    finally:
        c.close()


@pytest.mark.parametrize("seed", [3, 17, 29])
def test_random_scenes_inside_their_bars(monkeypatch, seed):
    """The photo-consistent random scenes of test_gpu_random, this time with the counters read."""
    from test_gpu_random import random_case
    cams, imgs, masks, (lo, hi, D), kw, rng = random_case(100 + seed)
    V = len(cams)
    ref = int(rng.randint(V))
    nbrs = [v for v in range(V) if v != ref][:3]
    P = T.default_params(True, lo, hi, D, radius=min(2, kw["radius"]), weight_kind=kw["weight_kind"])
    c = _stats_ctx(monkeypatch)
    try:
        _compare_with_oracle(c, cams, imgs, masks, P, ref, nbrs)
        refr = any(cams[j].is_refractive for j in nbrs)
        _check_counters(c, need_interpolated=refr and P.num_levels > 8)
    finally:
        c.close()


def test_bunny_inside_its_bars(monkeypatch):
    """The reference's own example data (1/4 size, injected interface): real masks, flat regions."""
    from bunny_util import load
    cams, imgs, ms, scale = load(refractive=True)
    P = T.default_params(True, 30.0, 55.0, 100)
    P.image_scale = scale
    c = _stats_ctx(monkeypatch)
    try:
        c.set_views(cams, imgs, ms)
        c.set_params(P)
        nb = c.select_neighbours(3)
        _compare_with_oracle(c, cams, imgs, ms, P, 2, nb[2])
        st, _ = _check_counters(c)
        assert st["screened"] > 0 and st["verified"] > 0
    finally:
        c.close()


def _views_out(c, cams, imgs, ms, P, order, mode="run_view"):
    c.set_views(cams, imgs, ms)
    c.set_params(P)
    nb = c.select_neighbours(3)
    for v in order:
        getattr(c, mode)(v, nb[v])
    return [(c.depth_index(v).copy(), c.depth(v).copy(), c.best_cost(v).copy()) for v in range(len(cams))]


def _run_views(monkeypatch, env, cams, imgs, ms, P, order, mode="run_view"):
    monkeypatch.delenv("SR_LANES", raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    c = capi.Context(0)
    out = _views_out(c, cams, imgs, ms, P, order, mode)
    c.close()
    return out


def _same(a, b):
    return (a[0] == b[0]).all() and ((a[1] == b[1]) | (np.isnan(a[1]) & np.isnan(b[1]))).all() and \
        ((a[2] == b[2]) | (np.isnan(a[2]) & np.isnan(b[2]))).all()


def test_lanes_are_bit_invisible(monkeypatch):
    cams, imgs, ms, _ = refractive_arc_scene(V=5, w=112, h=72, masks=True)
    P = T.default_params(True, 420.0, 580.0, 48)
    order = [0, 1, 2, 3, 4, 2, 2, 0]  # (the same view twice in a row lands on different lanes)
    base = _run_views(monkeypatch, {"SR_LANES": 1}, cams, imgs, ms, P, order)
    for env in ({}, {"SR_LANES": 2}):
        got = _run_views(monkeypatch, env, cams, imgs, ms, P, order)
        for v in range(len(cams)):
            assert _same(base[v], got[v]), (env, v)


def test_context_reused_with_larger_images_and_peaks(monkeypatch):
    """The context's grow-only buffers follow the image size.  First the peak-list buffer (ADVICE r1: it used to
    keep its first allocation) against the oracle; then label mode on the default lanes and curve mode, each
    through small -> large -> small images and label counts in one context, bit for bit against a fresh
    context of each size."""
    c = capi.Context(0)
    try:
        for (w, h) in [(48, 32), (96, 64)]:
            cams, imgs, ms, _ = refractive_arc_scene(V=3, w=w, h=h, masks=False)
            P = T.default_params(True, 420.0, 580.0, 16)
            P.keep_cost_volume = 2
            c.set_views(cams, imgs, ms)
            c.set_params(P)
            c.run_view(1, [0, 2])
            out = c.peaks(1)
            od, oi, ob, _, pk = O.Scene(cams, imgs, ms).mvs_view(P, 1, [0, 2], want_peaks=True)
            gi = c.depth_index(1)
            assert (gi != oi).mean() <= 1e-4
            same = gi == oi
            assert (out[..., 1][same] == pk[..., 1][same]).mean() > 1 - 1e-3  # depths of the kept pairs
            assert np.abs(out[..., 0][same] - pk[..., 0][same]).max() <= 1e-9
    finally:
        c.close()
    monkeypatch.delenv("SR_LANES", raising=False)
    for mode in ("run_view", "run_view_curve"):
        c = capi.Context(0)
        try:
            for (w, h, D) in [(48, 32, 16), (96, 64, 24), (48, 32, 16)]:
                cams, imgs, ms, _ = refractive_arc_scene(V=4, w=w, h=h, masks=True)
                P = T.default_params(True, 420.0, 580.0, D)
                order = [1, 2, 0, 1]  # (label mode: both lanes run views of every size)
                got = _views_out(c, cams, imgs, ms, P, order, mode)
                want = _run_views(monkeypatch, {}, cams, imgs, ms, P, order, mode)
                assert (got[1][0] >= 0).mean() > 0.1
                for v in range(len(cams)):
                    assert _same(got[v], want[v]), (mode, w, h, v)
        finally:
            c.close()
