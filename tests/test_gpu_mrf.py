"""sr_mrf_select (the MRF stage on the peak lists) against the NumPy restatement of tests/mrf_util.py bit for bit,
against exact dynamic programming on chains, against the winner-take-all of real runs in its limit, on synthetic
outliers at 1920x1080, in the pipeline (cross-check, depth image, point cloud) and in MultiViewStereo::setMrf."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from stereoreconstruction_b200 import capi, scenes, types as T
from stereoreconstruction_b200.types import SrMrfParams
import mrf_util as M
from scene_util import refractive_arc_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "stereoreconstruction_b200")
SR_ERR_INVALID, SR_ERR_STATE, SR_ERR_CANCELLED = 1, 3, 4  # include/sr_b200.h
P = T.default_params(True, 420.0, 580.0, 64)


def mrf(**kw):
    return capi.mrf_params_default(**kw)


def holes_mask(h, w, rng):
    m = np.where(rng.rand(h, w) < 0.85, 255, 0).astype(np.uint8)
    if h > 4 and w > 4:
        m[h // 3:h // 2, w // 3:w // 2] = 0
    return m


def context(h, w, mask, params=P):
    ctx = capi.Context(0)
    ctx.set_views(scenes.arc_cameras(2, w, h), [np.zeros((h, w, 4), np.uint8)] * 2, [mask, None])
    ctx.set_params(params)
    return ctx


def run_both(ctx, lists, mask, mp, params=P):
    """GPU maps and energy after sr_set_peaks + sr_mrf_select on view 0, and the oracle's."""
    d0, b0, i0 = ctx.depth(0), ctx.best_cost(0), ctx.depth_index(0)
    ctx.set_peaks(0, lists)
    e = ctx.mrf_select(0, mp)
    got = (ctx.depth(0), ctx.best_cost(0), ctx.depth_index(0), e)
    want = M.mrf_select(lists, mask, params, mp, d0, b0, i0)
    return got, want


def assert_same(got, want):
    d, b, i, e = got
    _, wd, wb, wi, we = want
    assert np.array_equal(d, wd, equal_nan=True)
    assert np.array_equal(b, wb, equal_nan=True)
    assert (i == wi).all()
    assert e == pytest.approx(we, rel=1e-12, abs=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (33, 17), (160, 256)])
@pytest.mark.parametrize("iterations", [0, 1, 9])
def test_equals_oracle(shape, iterations):
    h, w = shape
    rng = np.random.RandomState(h * 1000 + w + iterations)
    mask = holes_mask(h, w, rng) if h * w > 1 else np.full((1, 1), 255, np.uint8)
    lists = M.random_lists(h, w, rng, P)
    ctx = context(h, w, mask)
    for mp in (mrf(iterations=iterations), mrf(iterations=iterations, smooth_weight=0.4, smooth_trunc=3.0,
                                                unknown_cost=0.7, unknown_pair=0.9)):
        assert_same(*run_both(ctx, lists, mask, mp))
    ctx.close()


@pytest.mark.gpu
def test_equals_oracle_many_iterations_and_odd_params():
    h, w = 47, 61
    rng = np.random.RandomState(11)
    mask = holes_mask(h, w, rng)
    Q = T.default_params(True, 10.0, 100.0, 100, ncc_threshold=0.5)
    lists = M.random_lists(h, w, rng, Q)
    ctx = context(h, w, mask, Q)
    for mp in (mrf(iterations=40), mrf(iterations=5, smooth_weight=0.0, smooth_trunc=0.0, unknown_pair=0.0),
               mrf(iterations=3, unknown_cost=1e30, smooth_weight=-0.0, unknown_pair=1e30)):
        assert_same(*run_both(ctx, lists, mask, mp, Q))
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 41), (41, 1)])
def test_chain_equals_viterbi(shape):
    h, w = shape
    rng = np.random.RandomState(h + 2 * w)
    lists = M.random_lists(h, w, rng, P, adversarial=False)
    mask = np.full(shape, 255, np.uint8)
    ctx = context(h, w, mask)
    mp = mrf(iterations=max(h, w) + 1, smooth_weight=0.3, smooth_trunc=6.0, unknown_pair=0.5, unknown_cost=0.8)
    ctx.set_peaks(0, lists)
    e = ctx.mrf_select(0, mp)
    unary, zs = M.prepare(lists, P)
    best, vlab = M.viterbi_chain(unary.reshape(M.K, -1), zs.reshape(M.K, -1), mp)
    idx = ctx.depth_index(0).reshape(-1)
    lab = np.where(idx < 0, M.U, idx)
    assert (lab == vlab).all() or abs(e - best) <= 1e-6 * abs(best), (e, best)
    ctx.close()


@pytest.fixture(scope="module")
def full_scene():
    w, h, V = 1920, 1080, 3
    cams = scenes.arc_cameras(V, w, h)
    ctx = capi.Context(0)
    ctx.set_views(cams, [np.zeros((h, w, 4), np.uint8)] * V, None)
    surf = scenes.HeightField(z0=0.0, amp=25.0, lx=90.0, ly=70.0)
    imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), surf, seed=4321, cell=3.5 * 500.0 / cams[0].K[0])
    ctx.close()
    return cams, imgs


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [False, True])
def test_wta_limit_on_a_real_run(full_scene, curve):
    """Huge unknown_cost with no smoothness (or no iterations): the run's own depth and best maps, slot 8 where
    the WTA found a candidate and SR_INDEX_NONE elsewhere."""
    cams, imgs = full_scene
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, None)
    ctx.set_params(T.default_params(True, 350.0, 650.0, 64, keep_cost_volume=2))
    (ctx.run_view_curve if curve else ctx.run_view)(0, [1, 2])
    d, b, i = ctx.depth(0), ctx.best_cost(0), ctx.depth_index(0)
    found = i >= 0
    assert found.mean() > 0.5
    parallel = found & ~np.isfinite(d)  # a curve-mode winner whose z is not finite is no hypothesis
    assert parallel.sum() == 0
    cmp = ~parallel
    for mp in (mrf(unknown_cost=1e30, smooth_weight=0.0, unknown_pair=0.0), mrf(unknown_cost=1e30, iterations=0)):
        ctx.mrf_select(0, mp)
        assert d[cmp].tobytes() == ctx.depth(0)[cmp].tobytes()
        assert b[cmp].tobytes() == ctx.best_cost(0)[cmp].tobytes()
        assert (ctx.depth_index(0)[cmp] == np.where(found, 8, T.SR_INDEX_NONE)[cmp]).all()
    ctx.close()


def outlier_lists(h, w, rng):
    """A smooth surface at a random slot with ncc 0.97; on 20 % of the pixels a decoy at a random depth with ncc
    0.99 in another slot; the rest padding.  Returns the lists, the true depth and the decoy mask."""
    yy, xx = np.mgrid[0:h, 0:w]
    truth = 500.0 + 60.0 * np.sin(xx / 300.0) * np.cos(yy / 200.0)
    lists = np.zeros((h, w, 9, 2))
    lists[..., 1] = -1.0
    ts = rng.randint(0, 9, size=(h, w))
    ds = (ts + rng.randint(1, 9, size=(h, w))) % 9
    decoy = rng.rand(h, w) < 0.2
    np.put_along_axis(lists[..., 0], ts[..., None], 0.97, -1)
    np.put_along_axis(lists[..., 1], ts[..., None], truth[..., None], -1)
    dz = rng.uniform(P.min_depth, P.max_depth, size=(h, w))
    cur0 = np.take_along_axis(lists[..., 0], ds[..., None], -1)[..., 0]
    cur1 = np.take_along_axis(lists[..., 1], ds[..., None], -1)[..., 0]
    np.put_along_axis(lists[..., 0], ds[..., None], np.where(decoy, 0.99, cur0)[..., None], -1)
    np.put_along_axis(lists[..., 1], ds[..., None], np.where(decoy, dz, cur1)[..., None], -1)
    return lists, truth, decoy


@pytest.mark.gpu
def test_outliers_removed_at_full_size():
    h, w = 1080, 1920
    rng = np.random.RandomState(2024)
    lists, truth, decoy = outlier_lists(h, w, rng)
    mask = np.full((h, w), 255, np.uint8)
    ctx = context(h, w, mask)
    ctx.set_peaks(0, lists)
    e_wta = ctx.mrf_select(0, mrf(iterations=0))  # the argmin of the unary term: the decoys
    d = ctx.depth(0)
    assert (d[decoy] != truth[decoy]).mean() > 0.999
    e = ctx.mrf_select(0)
    d = ctx.depth(0)
    step = (P.max_depth - P.min_depth) / (P.num_levels - 1)
    restored = np.abs(d[decoy] - truth[decoy]) <= step
    assert restored.mean() >= 0.99, restored.mean()
    assert (d[~decoy] == truth[~decoy]).mean() >= 0.99
    assert e < e_wta
    ctx.close()


@pytest.mark.gpu
def test_pipeline_and_state():
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=96, h=64, masks=True)
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    Q = T.default_params(True, 420.0, 580.0, 32, keep_cost_volume=2)
    ctx.set_params(Q)
    nbrs = ctx.select_neighbours(3)
    V = len(cams)
    for v in range(V):
        ctx.run_view_curve(v, nbrs[v])
    peaks = ctx.peaks(V - 1)
    e1 = ctx.mrf_select(V - 1)
    maps1 = [x.copy() for x in (ctx.depth(V - 1), ctx.best_cost(V - 1), ctx.depth_index(V - 1))]
    e2 = ctx.mrf_select(V - 1)
    maps2 = (ctx.depth(V - 1), ctx.best_cost(V - 1), ctx.depth_index(V - 1))
    assert e1 == e2 and all(a.tobytes() == b.tobytes() for a, b in zip(maps1, maps2))
    assert ctx.peaks(V - 1).tobytes() == peaks.tobytes()
    # cross-check, depth image and point cloud after the MRF == after sr_set_depth with the MRF's depth map
    before = [ctx.depth(v) for v in range(V)]
    ctx.cross_check(False, 12.0)
    after = [ctx.depth(v) for v in range(V)]
    img, pts = ctx.depth_image(V - 1), ctx.points(V - 1)
    for v in range(V):
        ctx.set_depth(v, before[v])
    ctx.cross_check(False, 12.0)
    for v in range(V):
        assert np.array_equal(after[v], ctx.depth(v), equal_nan=True)
    assert (img == ctx.depth_image(V - 1)).all()
    for x, y in zip(pts, ctx.points(V - 1)):
        assert x.tobytes() == y.tobytes()
    # cancel between iterations leaves the maps as they were
    ctx.set_peaks(V - 1, peaks)
    ctx.set_depth(V - 1, before[V - 1])
    d0 = ctx.depth(V - 1)
    L = capi.lib()
    L.sr_request_cancel(ctx._h)
    p = mrf(iterations=4)
    assert L.sr_mrf_select(ctx._h, V - 1, C.byref(p), None) == SR_ERR_CANCELLED
    L.sr_clear_cancel(ctx._h)
    assert ctx.depth(V - 1).tobytes() == d0.tobytes()
    # errors
    rc = lambda view, q: L.sr_mrf_select(ctx._h, view, C.byref(q), None)
    assert rc(0, mrf()) == SR_ERR_STATE  # lists of view V - 1 only
    for bad in (dict(iterations=-1), dict(unknown_cost=-1.0), dict(unknown_cost=float("nan")),
                dict(smooth_weight=float("inf")), dict(smooth_trunc=-0.5), dict(unknown_pair=2e30),
                dict(smooth_weight=1e20, smooth_trunc=1e20)):
        assert rc(V - 1, mrf(**bad)) == SR_ERR_INVALID, bad
    for bad in (dict(ncc_threshold=1.0), dict(ncc_threshold=float("nan")), dict(max_depth=420.0),
                dict(row_begin=8), dict(row_end=32)):
        ctx.set_params(T.default_params(True, **dict(dict(min_depth=420.0, max_depth=580.0, num_levels=32), **bad)))
        assert rc(V - 1, mrf()) == SR_ERR_INVALID, bad
    ctx.set_params(Q)
    assert rc(V - 1, mrf()) == 0
    assert L.sr_mrf_select(ctx._h, V, C.byref(mrf()), None) == SR_ERR_INVALID
    ctx.set_params(T.default_params(True, 420.0, 580.0, 32))  # a run without keep_cost_volume & 2 drops the lists
    ctx.run_view(0, nbrs[0])
    assert rc(V - 1, mrf()) == SR_ERR_STATE
    ctx.close()
    fresh = capi.Context(0)
    assert capi.lib().sr_mrf_select(fresh._h, 0, C.byref(mrf()), None) == SR_ERR_STATE
    fresh.close()


def test_mrf_params_layout():
    assert C.sizeof(SrMrfParams) == 40
    assert SrMrfParams.unknown_cost.offset == 8 and SrMrfParams.unknown_pair.offset == 32
    src = open(os.path.join(ROOT, "include", "sr_b200.h")).read()
    body = src[src.index("typedef struct sr_mrf_params"):src.index("} sr_mrf_params;")]
    assert [f for f, _ in SrMrfParams._fields_] == ["iterations", "unknown_cost", "smooth_weight", "smooth_trunc",
                                                     "unknown_pair"]
    for f, _ in SrMrfParams._fields_:
        assert f + ";" in body


def test_defaults_are_in_range():
    p = mrf()
    assert p.iterations > 0 and p.unknown_cost > 0 and p.smooth_weight > 0 and p.smooth_trunc > 0
    assert p.unknown_pair > 0


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    """tests/cpp/mrf_class_test.cpp built against the library."""
    out = str(tmp_path_factory.mktemp("mrf") / "mrf_class_test")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-Wno-deprecated-declarations", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "mrf_class_test.cpp"), "-L", PKG, "-lsr_b200", "-lz",
           "-Wl,-rpath," + PKG, "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return out


def test_driver_builds(driver):
    assert os.path.exists(driver)


@pytest.mark.gpu
@pytest.mark.parametrize("use_mrf", [True, False])
def test_class_equals_the_abi_sequence(driver, tmp_path, use_mrf):
    from test_gpu_point_cloud import write_scene
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=96, h=64, masks=True)
    scene = str(tmp_path / "scene.bin")
    write_scene(scene, cams, imgs, ms)
    cross = 12.0
    r = subprocess.run([driver, scene, str(tmp_path), "420", "580", "32", str(cross), "1", str(int(use_mrf))],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    V, h, w = len(cams), 64, 96
    got = np.fromfile(str(tmp_path / "depth.bin"), np.float64).reshape(V, h, w)
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    ctx.set_params(T.default_params(True, 420.0, 580.0, 32, keep_cost_volume=2 if use_mrf else 0))
    nbrs = ctx.select_neighbours(3)
    for v in range(V):
        ctx.run_view_curve(v, nbrs[v])
        if use_mrf:
            ctx.mrf_select(v)
    ctx.cross_check(False, cross)
    for v in range(V):
        assert np.array_equal(got[v], ctx.depth(v), equal_nan=True), v
    ctx.close()
