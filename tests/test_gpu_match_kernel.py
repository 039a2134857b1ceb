"""The all-FP64 match kernel, match_kernel<R, G, COST> (sr_kernels.cuh), against the oracle at every compiled
radius, on ill-conditioned windows, with the winning cost held to the reference's selection margin.

The kernel serves two-view label mode (NCC and SAD), two-view curve mode, and MVS whenever the FP32 screen is
off: a kept cost volume (keep_cost_volume & 1), kept peak lists (& 2) or SR_MATCH_SCREEN=0.  Lanes per pixel
(LanesFor in sr_match_dispatch.cuh): G = 1, 1, 2, 4, 4, 32 at r = 1, 2, 3, 4, 5, 16.

Its fast path sums the neighbour side in one pass (s3 = S2 - 2 meanR S1 + nact meanR^2); the reference sums
it in two.  On a nearly flat window under geodesic weights (every weight exp(0) = 1) the one-pass form loses
digits; the reference's rules compare costs with no margin beyond 1e-10 (two-view: cost + 1e-10 < minCost,
and the 0.95 ratio test) or by exact equality (MVS ties), so each arm holds the winning cost to 1e-10
(two-view) or 1e-12 (MVS NCC) wherever the index agrees with the oracle.

Scenes: 4 views of scenes.arc_cameras(4, 72, 44, arc_deg=22.0).  Image kinds: the five adversarial kinds of
test_gpu_screen_hardening; "dots" (flat gray, about 4 % of the pixels one level brighter: the ill-conditioned
case); "holes" (textured, with masks whose holes leave r = 1 windows of exactly 4 and 5 active taps, SAD's
`<= 4` degenerate rule); "textured" (refractive_arc_scene with masks, a control).  At r = 16 only a row band
is computed, with fewer labels.

  A  two-view label mode, NCC and SAD, kept FP32 volume;
  B  unscreened MVS: SR_MATCH_SCREEN=0, keep_cost_volume = 1, keep_cost_volume = 2 (peak lists), on the kinds
     without engineered ties (MVS_KINDS); on "dots" and "lowcontrast" the peak-list NCCs, entry by entry;
  C  two-view curve mode at r = 3 and 16;
  D  support weights in list mode, window centres at corners, edges and masked pixels.

test_fixtures_reach_the_ill_conditioned_regime (no GPU) checks on the oracle that the fixtures reach what the
arms claim."""
import functools

import numpy as np
import pytest

from oracle import oracle_api as O
from stereoreconstruction_b200 import capi, scenes, types as T
from scene_util import refractive_arc_scene, cost_close
from test_gpu_screen_hardening import adversarial_images

V, W, H = 4, 72, 44
REF, NBR, NBRS = 1, 2, [0, 2, 3]
DEPTHS = (430.0, 570.0)
LABELS, LABELS16 = 24, 8
BAND16 = (16, 22)            # r = 16: rows computed
RADII = [1, 2, 3, 4, 5, 16]
WEIGHTS = [T.SR_WEIGHT_GEODESIC, T.SR_WEIGHT_ADAPTIVE]
KINDS = ["outliers", "checker", "steps", "lowcontrast", "ramp", "dots", "holes", "textured"]
# Unscreened MVS keeps the reference's winner only where no two labels tie: its NCC is not the reference's to
# the last bit, and MultiViewStereo breaks ties by exact equality.  The kinds built to tie are left out of arm B
# (DESIGN.md section 1, "Known deviations").
MVS_KINDS = ["ramp", "holes", "textured"]
# The kinds whose MVS winners tie: arm B compares their peak-list NCCs label by label instead.
MVS_TIE_KINDS = ["dots", "lowcontrast"]
# Two-view NCC where the reference window is exactly flat (every w*gl equal, as on the 0/255 plateaus of "steps"
# under geodesic weights) on lane groups (G = 2, 4): the reference's s2 is exactly 0 and the lanes' is rounding
# noise, so the 0.95 ratio test decides on noise (DESIGN.md section 1).  Of the fixtures only "steps" has such
# windows at these radii.
TWOVIEW_FLAT_LANES = {("steps", 3, T.SR_WEIGHT_GEODESIC, T.SR_COST_NCC_TWOVIEW),
                      ("steps", 4, T.SR_WEIGHT_GEODESIC, T.SR_COST_NCC_TWOVIEW)}
CURVE_KINDS = ["dots", "lowcontrast", "holes", "textured"]
COSTS = [T.SR_COST_NCC_TWOVIEW, T.SR_COST_SAD_TWOVIEW]
GPU = pytest.mark.gpu


def dots_images(seed=5):
    """Flat gray (a different level per view) with about 4 % of the pixels raised by one level in R, G and B."""
    rng = np.random.RandomState(seed)
    imgs = []
    for v in range(V):
        g = np.full((H, W), 118 + 3 * v, np.int32)
        g[rng.rand(H, W) < 0.04] += 1
        im = np.empty((H, W, 4), np.uint8)
        im[..., :3] = g[..., None]
        im[..., 3] = 255
        imgs.append(im)
    return imgs


def hole_masks(seed=9):
    """Half of the pixels of one half of each view masked out: the reference view's holes are in its left half
    (its windows there have 1..9 active taps and project into the neighbours' hole-free half, the fast path);
    the other views' holes are in their right half (the exact tap filter, slow_cost)."""
    rng = np.random.RandomState(seed)
    ms = []
    for v in range(V):
        m = np.full((H, W), 255, np.uint8)
        cols = slice(2, W // 2) if v == REF else slice(W // 2, W - 2)
        m[4:H - 4, cols][rng.rand(H - 8, m[:, cols].shape[1]) < 0.5] = 0
        ms.append(m)
    return ms


@functools.lru_cache(maxsize=None)
def fixture(kind):
    """(cams, imgs, masks, oracle scene) of one image kind."""
    if kind in ("holes", "textured"):
        cams, imgs, ms, _ = refractive_arc_scene(V=V, w=W, h=H, arc_deg=22.0, masks=kind == "textured")
        if kind == "holes":
            ms = hole_masks()
    else:
        cams = scenes.arc_cameras(V, W, H, arc_deg=22.0)
        imgs = dots_images() if kind == "dots" else adversarial_images(kind, V, W, H, seed=11)
        ms = None
    return cams, imgs, ms, O.Scene(cams, imgs, ms)


def params(multi_view, radius, weight, **kw):
    P = T.default_params(multi_view, *DEPTHS, LABELS16 if radius == 16 else LABELS, radius=radius,
                         weight_kind=weight, **kw)
    if radius == 16:
        P.row_begin, P.row_end = BAND16
    return P


def rows(radius):
    return slice(*BAND16) if radius == 16 else slice(0, H)


@functools.lru_cache(maxsize=None)
def oracle_twoview(kind, radius, weight, cost):
    P = params(False, radius, weight, cost_kind=cost, keep_cost_volume=1)
    od, oi, ob, ov = fixture(kind)[3].twoview_label(P, REF, NBR, want_volume=True)
    return oi, od, ob, np.transpose(ov, (2, 0, 1))  # volume [D][rows][w]


@functools.lru_cache(maxsize=None)
def oracle_curve(kind, radius, weight, cost):
    P = params(False, radius, weight, cost_kind=cost)
    return fixture(kind)[3].twoview_curve(P, REF, NBR)


@functools.lru_cache(maxsize=None)
def oracle_mvs(kind, radius, weight):
    P = params(True, radius, weight)
    od, oi, ob, _, pk = fixture(kind)[3].mvs_view(P, REF, NBRS, want_peaks=True)
    return oi, od, ob, pk


def labelled(idx, best, radius):
    """Pixels of the computed rows the oracle labels with a cost below the 120 / 1000 sentinels."""
    r = rows(radius)
    return (idx[r] >= 0) & (best[r] < 120.0)


def one_pass_twoview_ncc(gl, gr, wt):
    """The fast path's one-pass two-view NCC (match_kernel's fast_one) in float64 NumPy, one window per row of
    gl, gr, wt ((N, WN) arrays, every tap valid)."""
    act = wt > 1e-10
    wt = np.where(act, wt, 0.0)
    c1 = np.where(act, gl, 0.0)
    totW, SL, nact = wt.sum(1), (wt * c1).sum(1), act.sum(1)
    meanL, inv = SL / totW, 1.0 / totW
    dl = np.where(act, wt * c1 - meanL[:, None], 0.0)
    s2, SD = (dl * dl).sum(1), dl.sum(1)
    p = wt * gr
    S1, S2, S3 = p.sum(1), (p * p).sum(1), (wt * dl * gr).sum(1)
    meanR = S1 * inv
    s1 = S3 - meanR * SD
    s3 = S2 - 2.0 * meanR * S1 + nact * meanR * meanR
    with np.errstate(invalid="ignore", divide="ignore"):
        v = 255.0 * (1.0 - np.abs(s1) / np.sqrt(s2 * s3))
    return np.where(v < 120.0, v, 120.0)


def gray(im):
    rgb = im[..., :3].astype(np.float64)
    return (0.11 * rgb[..., 0] + 0.59 * rgb[..., 1]) + 0.3 * rgb[..., 2]  # RGBA::toGray


def test_fixtures_reach_the_ill_conditioned_regime():
    # every arm A and C case has costs to compare: not every label at the 120 / 1000 sentinels
    for kind in KINDS:
        for radius in RADII:
            for weight in WEIGHTS:
                for cost in COSTS:
                    oi, _, ob, _ = oracle_twoview(kind, radius, weight, cost)
                    assert labelled(oi, ob, radius).mean() > 0.2, (kind, radius, weight, cost)
    for kind in CURVE_KINDS:
        for radius in (3, 16):
            for weight in WEIGHTS:
                for cost in COSTS:
                    od, ob, _ = oracle_curve(kind, radius, weight, cost)
                    r = rows(radius)
                    assert (np.isfinite(od[r]) & (ob[r] < 120.0)).mean() > 0.2, (kind, radius, weight, cost)
    # the one-pass sums differ from the reference's two passes by more than the selection margin on "dots"
    cams, imgs, _, sc = fixture("dots")
    gL, gR = gray(imgs[REF]), gray(imgs[NBR])
    rng = np.random.RandomState(1)
    for radius in (2, 5):
        n = 400
        x1, x2 = rng.randint(radius, W - radius - 1, (2, n))
        y1, y2 = rng.randint(radius, H - radius - 1, (2, n))
        P = params(False, radius, T.SR_WEIGHT_GEODESIC)
        want = np.array([sc.cost(P, REF, NBR, *a) for a in zip(x1, y1, x2, y2)])
        wt = sc.weights(REF, T.SR_WEIGHT_GEODESIC, radius, x1, y1).reshape(n, -1)
        k = np.arange(-radius, radius + 1)
        win = lambda g, x, y: g[y[:, None, None] + k[None, :, None], x[:, None, None] + k[None, None, :]].reshape(n, -1)
        got = one_pass_twoview_ncc(win(gL, x1, y1), win(gR, x2, y2), wt)
        diff = np.abs(got - want)
        assert (diff > 1e-10).sum() > 0, (radius, diff.max())
        assert (wt == 1.0).all(axis=1).any()  # geodesic-flat windows: every weight exp(0) = 1
    # r = 1 windows (reference side, two-view validity: white and x + 1 < w, y + 1 < h) of 4 and 5 active taps
    ms = fixture("holes")[2][REF]
    valid = np.zeros((H + 2, W + 2), np.int32)
    valid[1:H, 1:W] = ms[:H - 1, :W - 1] == 255
    count = sum(valid[1 + dy:H + 1 + dy, 1 + dx:W + 1 + dx] for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    centre = valid[1:H + 1, 1:W + 1] == 1
    assert (centre & (count == 4)).sum() > 20 and (centre & (count == 5)).sum() > 20


# ---- GPU ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _load(c, kind):
    cams, imgs, ms, _ = fixture(kind)
    c.set_views(cams, imgs, ms)


def _same(a, b):
    return (a == b) | (np.isnan(a) & np.isnan(b))


def _check_winner(g, o, radius, cost_bar):
    """Index mismatch rate <= 1e-4 (sentinels compared too), depths equal where the indices are, winning cost
    within cost_bar where the indices agree and the cost is finite.  Returns (mismatch rate, worst cost diff)."""
    r = rows(radius)
    gi, gd, gb = (m[r] for m in g)
    oi, od, ob = (m[r] for m in o)
    mism = gi != oi
    assert mism.mean() <= 1e-4, f"index mismatch rate {mism.mean()}"
    assert _same(gd, od)[~mism].all(), "depth differs where the index agrees"
    fin = ~mism & np.isfinite(ob)
    assert _same(gb, ob)[~mism & ~np.isfinite(ob)].all()
    diff = float(np.abs(gb[fin] - ob[fin]).max()) if fin.any() else 0.0
    assert diff <= cost_bar, f"winning cost differs by {diff:.3g}"
    return float(mism.mean()), diff


@GPU
@pytest.mark.parametrize("weight", WEIGHTS)
@pytest.mark.parametrize("radius", RADII)
@pytest.mark.parametrize("kind", KINDS)
def test_twoview_label(ctx, kind, radius, weight):
    """Arm A: two-view label mode, NCC and SAD, the 0.95 ratio test, the FP32 volume kept."""
    _load(ctx, kind)
    for cost in [c for c in COSTS if (kind, radius, weight, c) not in TWOVIEW_FLAT_LANES]:
        P = params(False, radius, weight, cost_kind=cost, keep_cost_volume=1)
        ctx.set_params(P)
        ctx.run_view(REF, [NBR])
        g = (ctx.depth_index(REF), ctx.depth(REF), ctx.best_cost(REF))
        gv = ctx.cost_volume(1)[0]
        oi, od, ob, ov = oracle_twoview(kind, radius, weight, cost)
        rate, diff = _check_winner(g, (oi, od, ob), radius, 1e-10)
        assert not cost_close(gv, ov).any(), f"cost volume mismatches: {cost_close(gv, ov).sum()}"
        print(f"A {kind} r={radius} w={weight} cost={cost}: mismatch {rate:.1e}, winning cost diff {diff:.2e}")


def _mvs_outputs(c):
    return c.depth_index(REF), c.depth(REF), c.best_cost(REF)


@GPU
@pytest.mark.parametrize("weight", WEIGHTS)
@pytest.mark.parametrize("radius", RADII)
@pytest.mark.parametrize("kind", MVS_KINDS)
def test_mvs_unscreened(ctx, monkeypatch, kind, radius, weight):
    """Arm B: match_kernel<R, G, NCC_MVS> through SR_MATCH_SCREEN=0, a kept cost volume and kept peak lists."""
    oi, od, ob, pk = oracle_mvs(kind, radius, weight)
    cams, imgs, ms, _ = fixture(kind)
    monkeypatch.setenv("SR_MATCH_SCREEN", "0")
    c = capi.Context(0)
    try:
        c.set_views(cams, imgs, ms)
        c.set_params(params(True, radius, weight))
        c.run_view(REF, NBRS)
        arms = {"screen=0": _mvs_outputs(c)}
    finally:
        c.close()
    monkeypatch.delenv("SR_MATCH_SCREEN")
    _load(ctx, kind)
    for keep in (1, 2):
        ctx.set_params(params(True, radius, weight, keep_cost_volume=keep))
        ctx.run_view(REF, NBRS)
        arms[f"keep={keep}"] = _mvs_outputs(ctx)
    gp = ctx.peaks(REF)
    for name, g in arms.items():
        rate, diff = _check_winner(g, (oi, od, ob), radius, 1e-12)
        print(f"B {kind} r={radius} w={weight} {name}: mismatch {rate:.1e}, winning ncc diff {diff:.2e}")
    r = rows(radius)
    same = (arms["keep=2"][0] == oi)[r]
    if ms is not None:
        same &= ms[REF][r] == 255
    gz, oz = gp[r][same][..., 1], pk[r][same][..., 1]
    assert (gz == oz).all(), "peak depths differ"
    pdiff = float(np.abs(gp[r][same][..., 0] - pk[r][same][..., 0]).max())
    assert pdiff <= 1e-12, f"peak ncc differs by {pdiff:.3g}"
    assert (pk[r][same][..., -1, 0] > 0).any()  # some lists hold entries


@GPU
@pytest.mark.parametrize("weight", WEIGHTS)
@pytest.mark.parametrize("radius", RADII)
@pytest.mark.parametrize("kind", MVS_TIE_KINDS)
def test_mvs_peak_nccs_on_ill_conditioned_windows(ctx, kind, radius, weight):
    """Arm B on the ill-conditioned kinds, whose winners tie (exact-equality tie-breaks are the screen's job): every
    kept (ncc, depth) pair whose depth equals the oracle's pair at the same list position holds its NCC to 1e-12."""
    _, _, _, pk = oracle_mvs(kind, radius, weight)
    _load(ctx, kind)
    ctx.set_params(params(True, radius, weight, keep_cost_volume=2))
    ctx.run_view(REF, NBRS)
    r = rows(radius)
    gp, op = ctx.peaks(REF)[r], pk[r]
    same = (gp[..., 1] == op[..., 1]) & (op[..., 0] > 0)
    assert same.sum() > 100, same.sum()
    diff = float(np.abs(gp[..., 0][same] - op[..., 0][same]).max())
    assert diff <= 1e-12, f"peak ncc differs by {diff:.3g}"
    print(f"B peaks {kind} r={radius} w={weight}: {same.sum()} pairs, ncc diff {diff:.2e}")


@GPU
@pytest.mark.parametrize("weight", WEIGHTS)
@pytest.mark.parametrize("radius", [3, 16])
@pytest.mark.parametrize("kind", CURVE_KINDS)
def test_twoview_curve(ctx, kind, radius, weight):
    """Arm C: two-view curve mode (bestTap and curve_depth on lane groups of 2 and 32), to the bars of
    test_gpu_curve.test_twoview_curve_matches_oracle."""
    _load(ctx, kind)
    r = rows(radius)
    for cost in COSTS:
        ctx.set_params(params(False, radius, weight, cost_kind=cost))
        ctx.run_view_curve(REF, [NBR])
        gd, gb = ctx.depth(REF)[r], ctx.best_cost(REF)[r]
        od, ob, cnt = (m[r] for m in oracle_curve(kind, radius, weight, cost))
        with np.errstate(invalid="ignore"):
            ok = _same(gd, od) | (np.abs(gd - od) <= 1e-9 * np.abs(od))
        assert ok.mean() >= 1 - 1e-4, f"depth mismatch rate {1 - ok.mean()}"
        fin = ok & np.isfinite(od)
        assert fin.mean() > 0.05 and cnt.max() > 4  # (the short baseline gives curves of <= 7 candidates)
        assert not cost_close(gb[fin], ob[fin]).any()
        print(f"C {kind} r={radius} w={weight} cost={cost}: depth mismatch {1 - ok.mean():.1e}")


@GPU
@pytest.mark.parametrize("weight", WEIGHTS)
@pytest.mark.parametrize("radius", RADII)
def test_support_weights(ctx, radius, weight):
    """Arm D: sr_compute_weights (list mode) against the oracle.  Adaptive: weights_adaptive_kernel at every
    radius.  Geodesic: weights_geodesic_kernel<true, 1> at r = 1, <true, 2> at r = 2, and from r = 3 up
    <false, 0> (the grid in W, the radius a run-time value)."""
    rng = np.random.RandomState(radius)
    ex = [0, W - 1, 0, W - 1] + [0] * 3 + [W - 1] * 3 + list(rng.randint(1, W - 1, 6))
    ey = [0, 0, H - 1, H - 1] + list(rng.randint(1, H - 1, 6)) + [0] * 3 + [H - 1] * 3
    for kind in ("steps", "holes"):
        _, _, ms, sc = fixture(kind)
        cx, cy = list(ex), list(ey)
        if ms is not None:  # masked window centres
            my, mx = np.nonzero(ms[REF] == 0)
            pick = rng.choice(mx.size, 12, replace=False)
            cx += list(mx[pick])
            cy += list(my[pick])
        cx += list(rng.randint(0, W, 40))
        cy += list(rng.randint(0, H, 40))
        cx, cy = np.array(cx, np.int32), np.array(cy, np.int32)
        _load(ctx, kind)
        g = ctx.weights(REF, weight, radius, cx, cy)
        o = sc.weights(REF, weight, radius, cx, cy)
        assert np.allclose(g, o, rtol=1e-13, atol=1e-300), (kind, np.abs(g - o).max())
        assert (o < 1e-10).any() and (o == 1.0).any()  # weights below the cut-off and exp(0) both occur
