"""Every compiled variant of the MVS match path against the oracle, at the sizes where its addressing differs.

Which kernel runs depends on the image width, the radius and SR_MATCH_STATS (launch_match_screen in
sr_match_dispatch.cuh, screen_pitch in sr_kernels.cuh):

  * r <= 2: match_mvs_screen2_kernel<R, false, PITCH> with the FP32 row pitch a compile-time constant
    (1024, 2048, 4096; 0 = run-time pitch for w > 4096, which equals w at w = 16384), and
    <R, true, 0> with statistics;
  * r = 3, 5, 16: the lane-group match_mvs_screen_kernel<R, G, STATS>;
  * SR_MATCH_SCREEN=0: the all-FP64 match_kernel<R, G, NCC_MVS>.

The wide scenes (h = 48, widths at and one past each pitch) compute only rows 19..27: a band whose first row
and row count are not multiples of the 4-row screen tile, and whose last 32-pixel tile holds one pixel when
w % 32 == 1.  Each case runs three arms, (a) the default context, (b) SR_MATCH_STATS=1 and (c)
SR_MATCH_SCREEN=0; each must match the oracle, and (a) and (b) must agree bit for bit.  Curve mode runs the
same dispatch; at w = 4097 the epipolar curves are longer than the initial curve volume (2D + 64 planes), so
the volume is refilled.  A two-view case at w = 16384 has taps far left of and beyond x = 4096.

test_cases_exercise_what_they_claim (no GPU) checks on the oracle alone that the fixtures reach these
paths: projections inside the neighbours' interior rows, a mostly labelled band, curves longer than the
initial volume at w = 4097 and shorter at w = 1025, two-view taps left of 0 and right of 4096."""
import functools

import numpy as np
import pytest

from oracle import oracle_api as O
from stereoreconstruction_b200 import capi, types as T
from scene_util import refractive_arc_scene, cost_close

H = 48
BAND = (19, 28)              # row_begin, row_end: 9 rows from row 19
REF, NBRS = 1, [0, 2]        # adjacent views on the arc: every projection of the band stays in rows 9..35
DEPTHS = (420.0, 580.0)
LABEL_D, CURVE_D = 24, 16
WIDE = [1024, 1025, 2048, 2049, 4096, 4097, 16384]
RADII = [1, 2, 3, 5]
CURVE_WIDTHS = [1025, 4097]  # curves of ~70 and ~230 pixels against an initial volume of 2 * 16 + 64 = 96
KNOBS = ("SR_MATCH_STATS", "SR_MATCH_SCREEN", "SR_TAP_BUDGET_MB")


@functools.lru_cache(maxsize=None)
def wide_scene(w):
    f = 1600.0 * w / 1920.0  # arc_cameras' focal length: the texture cell spans ~3.5 pixels at every width
    cams, imgs, _, _ = refractive_arc_scene(V=4, w=w, h=H, arc_deg=25.0, cell=3.5 * 500.0 / f)
    return cams, imgs, O.Scene(cams, imgs)


def band_params(multi_view, D, radius):
    P = T.default_params(multi_view, *DEPTHS, D, radius=radius)
    P.row_begin, P.row_end = BAND
    return P


@functools.lru_cache(maxsize=None)
def oracle_label(w, radius):
    od, oi, ob, _, _ = wide_scene(w)[2].mvs_view(band_params(True, LABEL_D, radius), REF, NBRS)
    return oi, od, ob


def band_endpoints(w, nbr):
    """Projections into view nbr of the band pixels' points at min_depth and at max_depth (pointFromDepth:
    the ray meets the plane normal to the reference's principal direction at that depth)."""
    cams, _, sc = wide_scene(w)
    rays = sc.unproject_grid(REF)[BAND[0]:BAND[1]].reshape(-1, 6)
    s, d = rays[:, :3], rays[:, 3:]
    prin, C = np.array(cams[REF].prin_dir[:]), np.array(cams[REF].C[:])
    nrm = prin / np.linalg.norm(prin)
    out = []
    for depth in DEPTHS:
        t = (nrm @ (C + depth * prin) - s @ nrm) / (d @ nrm)
        xy, ok = sc.project_points(nbr, s + t[:, None] * d)
        assert ok.all()
        out.append(xy)
    return out


def test_cases_exercise_what_they_claim():
    r_max = max(RADII)
    for w in WIDE:
        for nbr in NBRS:
            ends = band_endpoints(w, nbr)
            ys = np.concatenate([e[:, 1] for e in ends])
            assert r_max <= ys.min() and ys.max() < H - r_max, (w, nbr, ys.min(), ys.max())
            extent = (np.abs(ends[0] - ends[1]).sum(axis=1)).max()
            if w == 4097:   # the curve volume must be refilled
                assert extent > 2 * CURVE_D + 64, (w, nbr, extent)
            if w == 1025:   # the curve volume holds every curve
                assert extent + 1 < 2 * CURVE_D + 64, (w, nbr, extent)
        for r in RADII:
            oi = oracle_label(w, r)[0]
            assert (oi[BAND[0]:BAND[1]] >= 0).mean() > 0.5, (w, r)
            assert (oi[:BAND[0]] == -2).all() and (oi[BAND[1]:] == -2).all()
    # two-view: taps left of the image and beyond x = 4096 (the two-view build keeps out-of-image taps)
    xs = np.concatenate([e[:, 0] for e in band_endpoints(16384, 0)])
    assert xs.min() < -500 and xs.max() > 4096


# ---- GPU ----------------------------------------------------------------------------------------------

def _run(monkeypatch, env, cams, imgs, masks, P, nbrs=NBRS, mode="run_view"):
    """One view in a fresh context created under env; (index, depth, best) and, with statistics, the counters."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = capi.Context(0)
    try:
        c.set_views(cams, imgs, masks)
        c.set_params(P)
        getattr(c, mode)(REF, nbrs)
        out = (c.depth_index(REF), c.depth(REF), c.best_cost(REF))
        stats = (c.match_stats(), c.build_stats()) if env.get("SR_MATCH_STATS") == "1" else None
    finally:
        c.close()
    for k in env:
        monkeypatch.delenv(k)
    return out, stats


def _same(a, b):
    return all(((x == y) | (np.isnan(x) & np.isnan(y))).all() for x, y in zip(a, b))


def _rows(P, h):
    r0 = max(P.row_begin, 0)
    return r0, (P.row_end if 0 < P.row_end < h else h)


def _check_label(g, o, P, cost_bar=1e-12):
    """index mismatch rate <= 1e-4, depths equal where the indices are, winning cost within cost_bar (MVS) or
    cost_close (two-view, cost_bar=None); nothing written outside the row band.  Returns the mismatch rate."""
    gi, gd, gb = g
    oi, od, ob = o
    r0, r1 = _rows(P, gi.shape[0])
    assert (gi[:r0] == -1).all() and (gi[r1:] == -1).all(), "index written outside the row band"
    gi, gd, gb, oi, od, ob = (m[r0:r1] for m in (gi, gd, gb, oi, od, ob))
    mism = gi != oi
    assert mism.mean() <= 1e-4, f"index mismatch rate {mism.mean()}"
    assert ((gd == od) | (np.isnan(gd) & np.isnan(od)))[~mism].all()
    lab = ~mism & (oi >= 0)
    assert lab.mean() > 0.5
    if cost_bar is None:
        assert not cost_close(gb[lab], ob[lab]).any()
    else:
        assert np.abs(gb[lab] - ob[lab]).max() <= cost_bar
    return float(mism.mean())


def _check_counters(ms, bs):
    assert ms["outside_error_bar"] == 0, ms
    assert ms["prescreen_false_drops"] == 0, ms
    assert ms["max_screen_err"] < 5e-3, ms
    assert ms["screened"] > 0, ms  # the FP32 screen judged interior windows (not everything sent to slow_cost)
    assert bs["tap_mismatches"] == 0, bs


def _report(case, rate, ms):
    print(f"{case}: mismatch rate {rate:.1e}, screened {ms['screened']}, verified {ms['verified']}, "
          f"forced {ms['forced']}, max_screen_err {ms['max_screen_err']:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("radius", RADII)
@pytest.mark.parametrize("w", WIDE)
def test_wide_band_label_mode(monkeypatch, w, radius):
    cams, imgs, _ = wide_scene(w)
    P = band_params(True, LABEL_D, radius)
    o = oracle_label(w, radius)
    a, _ = _run(monkeypatch, {}, cams, imgs, None, P)                          # PITCH variants, lanes on
    b, (ms, bs) = _run(monkeypatch, {"SR_MATCH_STATS": "1"}, cams, imgs, None, P)  # PITCH = 0, statistics
    c, _ = _run(monkeypatch, {"SR_MATCH_SCREEN": "0"}, cams, imgs, None, P)     # all-FP64 match_kernel
    rates = [_check_label(arm, o, P) for arm in (a, b, c)]
    assert _same(a, b), "default and statistics builds of the screen differ"
    _check_counters(ms, bs)
    assert bs["interpolated"] > 0, bs
    _report(f"label w={w} r={radius}", max(rates), ms)


@pytest.mark.gpu
def test_mvs_radius_16(monkeypatch):
    """match_mvs_screen_kernel<16, 32, *>: one 32-lane group per pixel, 33 x 33 windows on a masked scene."""
    cams, imgs, masks, _ = refractive_arc_scene(V=4, w=64, h=40, masks=True)
    P = T.default_params(True, *DEPTHS, LABEL_D, radius=16)
    od, oi, ob, _, _ = O.Scene(cams, imgs, masks).mvs_view(P, REF, [0, 2, 3])
    a, _ = _run(monkeypatch, {}, cams, imgs, masks, P, nbrs=[0, 2, 3])
    b, (ms, bs) = _run(monkeypatch, {"SR_MATCH_STATS": "1"}, cams, imgs, masks, P, nbrs=[0, 2, 3])
    gi, gd, gb = a
    mism = gi != oi
    assert mism.mean() <= 1e-4, f"index mismatch rate {mism.mean()}"
    assert ((gd == od) | (np.isnan(gd) & np.isnan(od)))[~mism].all()
    lab = ~mism & (oi >= 0)
    assert lab.mean() > 0.5
    assert np.abs(gb[lab] - ob[lab]).max() <= 1e-12
    assert _same(a, b)
    _check_counters(ms, bs)
    _report("label 64x40 r=16", float(mism.mean()), ms)


def _depth_equal(g, o):
    with np.errstate(invalid="ignore"):
        return (g == o) | (np.isnan(g) & np.isnan(o)) | (np.abs(g - o) <= 1e-9 * np.abs(o))


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [2, 3])
@pytest.mark.parametrize("w", CURVE_WIDTHS)
def test_wide_band_curve_mode(monkeypatch, w, radius):
    """Curve mode: screen variants at w = 1025 (pitch 2048) and 4097 (run-time pitch), the refilled curve
    volume at 4097, and row bands of the tap budget (one row; several rows that the refill shrinks)."""
    cams, imgs, sc = wide_scene(w)
    P = band_params(True, CURVE_D, radius)
    od, _, ob, _, _ = sc.mvs_view(P, REF, NBRS, curve_mode=True)
    a, _ = _run(monkeypatch, {}, cams, imgs, None, P, mode="run_view_curve")
    b, (ms, _) = _run(monkeypatch, {"SR_MATCH_STATS": "1"}, cams, imgs, None, P, mode="run_view_curve")
    gi, gd, gb = a
    r0, r1 = BAND
    assert (gi[:r0] == -1).all() and (gi[r1:] == -1).all(), "index written outside the row band"
    gi, gd, gb, odb, obb = gi[r0:r1], gd[r0:r1], gb[r0:r1], od[r0:r1], ob[r0:r1]
    ok = _depth_equal(gd, odb)
    assert ok.mean() >= 1 - 1e-4, f"depth mismatch rate {1 - ok.mean()}"
    have = ok & (odb > 0) & np.isfinite(odb)
    assert have.mean() > 0.5
    assert np.abs(gb[have] - obb[have]).max() <= 1e-12
    assert (gi[have] >= 0).all()
    if w == 4097:  # a winner past the initial volume: the refilled volume was searched
        assert gi.max() >= 2 * CURVE_D + 64, gi.max()
    assert _same(a, b), "default and statistics builds of the screen differ"
    assert ms["outside_error_bar"] == 0 and ms["screened"] > 0, ms
    # row bands: one row each, and (16 MB) bands of several rows that the first refill shrinks
    for budget in ("1", "16"):
        banded, _ = _run(monkeypatch, {"SR_TAP_BUDGET_MB": budget}, cams, imgs, None, P, mode="run_view_curve")
        assert _same(banded, a), f"SR_TAP_BUDGET_MB={budget} changed the result"
    _report(f"curve w={w} r={radius}", float(1 - ok.mean()), ms)


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [2, 5])
def test_twoview_label_16384(monkeypatch, radius):
    """Two-view label mode at the widest image: taps from x ~ -950 to past 16384 in 16-bit fields, and windows
    entirely outside the image."""
    cams, imgs, sc = wide_scene(16384)
    P = band_params(False, LABEL_D, radius)
    od, oi, ob, _ = sc.twoview_label(P, REF, 0)
    g, _ = _run(monkeypatch, {}, cams, imgs, None, P, nbrs=[0])
    rate = _check_label(g, (oi, od, ob), P, cost_bar=None)
    print(f"two-view w=16384 r={radius}: mismatch rate {rate:.1e}")
