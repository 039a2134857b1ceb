"""Edge cases of the label-mode path on the GPU against the oracle: degenerate label counts, images
smaller than the window, fully masked views, descending depth ranges, scaled images, air (n = 1)
cameras through the screened MVS path, many / single neighbours."""
import numpy as np
import pytest

from oracle import oracle_api as O
from stereoreconstruction_b200 import capi, scenes, types as T
from scene_util import refractive_arc_scene, cost_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _compare_mvs(ctx, cams, imgs, ms, P, ref, nbrs, min_labelled=0.0):
    ctx.set_views(cams, imgs, ms)
    ctx.set_params(P)
    ctx.run_view(ref, nbrs)
    gi, gd, gb = ctx.depth_index(ref), ctx.depth(ref), ctx.best_cost(ref)
    sc = O.Scene(cams, imgs, ms)
    od, oi, ob, _, _ = sc.mvs_view(P, ref, nbrs)
    mism = gi != oi
    assert mism.mean() <= 1e-4, f"index mismatch rate {mism.mean()}"
    same = ~mism
    assert ((gd == od) | (np.isnan(gd) & np.isnan(od)))[same].all()
    lab = same & (oi >= 0)
    assert lab.mean() >= min_labelled
    if lab.any():
        assert np.abs(gb[lab] - ob[lab]).max() <= 1e-12
    return gi


def _compare_two(ctx, cams, imgs, ms, P, a, b):
    ctx.set_views(cams, imgs, ms)
    ctx.set_params(P)
    ctx.run_view(a, [b])
    gi, gd, gb = ctx.depth_index(a), ctx.depth(a), ctx.best_cost(a)
    sc = O.Scene(cams, imgs, ms)
    od, oi, ob, _ = sc.twoview_label(P, a, b, root_mode=1)
    mism = gi != oi
    assert mism.mean() <= 1e-4, f"index mismatch rate {mism.mean()}"
    same = ~mism
    assert ((gd == od) | (np.isnan(gd) & np.isnan(od)))[same].all()
    lab = same & (oi >= 0)
    if lab.any():
        assert not cost_close(gb[lab], ob[lab]).any()
    return gi


@pytest.mark.parametrize("D", [2, 3, 5, 9])
def test_few_labels(ctx, D):
    """Label counts below / around the anchor stride of the refractive build."""
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=64, h=40, masks=True)
    _compare_mvs(ctx, cams, imgs, ms, T.default_params(True, 470.0, 530.0, D), 1, [0, 2, 3])
    _compare_two(ctx, cams, imgs, ms, T.default_params(False, 470.0, 530.0, D, radius=2), 1, 2)


def test_image_smaller_than_window(ctx):
    """Every window touches a border: the exact tap filter decides everything."""
    cams, imgs, ms, _ = refractive_arc_scene(V=3, w=9, h=7, masks=False, cell=3.0)
    _compare_mvs(ctx, cams, imgs, None, T.default_params(True, 420.0, 580.0, 12, radius=5), 1, [0, 2])
    _compare_two(ctx, cams, imgs, None, T.default_params(False, 420.0, 580.0, 12, radius=5), 0, 1)


def test_fully_masked_reference_and_neighbour(ctx):
    cams, imgs, ms, _ = refractive_arc_scene(V=3, w=48, h=32, masks=True)
    P = T.default_params(True, 420.0, 580.0, 16)
    ms0 = [m.copy() for m in ms]
    ms0[1][:] = 0  # the reference view is masked out entirely: every pixel stays +INF / MASKED
    gi = _compare_mvs(ctx, cams, imgs, ms0, P, 1, [0, 2])
    assert (gi == T.SR_INDEX_MASKED).all() and np.isinf(ctx.depth(1)).all()
    ms1 = [m.copy() for m in ms]
    ms1[0][:] = 0  # a neighbour is masked out entirely: it contributes no candidate
    _compare_mvs(ctx, cams, imgs, ms1, P, 1, [0, 2])
    gi = _compare_mvs(ctx, cams, imgs, ms1, P, 1, [0])
    assert (gi[ms[1] == 255] == T.SR_INDEX_NONE).all()  # no candidate at all -> depth -1
    assert (ctx.depth(1)[ms[1] == 255] == -1.0).all()


def test_descending_depth_range(ctx):
    """maxDepth < minDepth: labels run far -> near, the MVS tie-break 'deeper wins' flips direction."""
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=64, h=40, masks=True)
    _compare_mvs(ctx, cams, imgs, ms, T.default_params(True, 580.0, 420.0, 48), 2, [0, 1, 3], min_labelled=0.05)
    _compare_two(ctx, cams, imgs, ms, T.default_params(False, 580.0, 420.0, 24, radius=2), 2, 1)


def test_air_cameras_through_screened_path(ctx):
    """n = 1 (no interface), with and without lens distortion: bit-exact projection path + screen."""
    for distortion in (True, False):
        cams, imgs, ms, _ = refractive_arc_scene(V=4, w=80, h=48, masks=True, interface=False, distortion=distortion)
        assert not cams[0].is_refractive
        _compare_mvs(ctx, cams, imgs, ms, T.default_params(True, 420.0, 580.0, 40), 1, [0, 2, 3], min_labelled=0.05)


def test_mixed_refractive_and_air_neighbours(ctx):
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=80, h=48, masks=True)
    air, _, _, _ = refractive_arc_scene(V=4, w=80, h=48, masks=True, interface=False)
    mixed = [cams[0], cams[1], air[2], cams[3]]
    _compare_mvs(ctx, mixed, imgs, ms, T.default_params(True, 420.0, 580.0, 32), 1, [0, 2, 3])


def test_image_scale_half(ctx):
    """Cameras calibrated at full resolution, images (already scaled) at half: pixel centres are
    divided by the scale before unproject, projections multiplied by it (multiviewstereo.cpp:572,774)."""
    w, h = 64, 40
    cams = scenes.arc_cameras(4, 2 * w, 2 * h, arc_deg=25.0)
    P = T.default_params(True, 420.0, 580.0, 24, image_scale=0.5)
    dummy = [np.zeros((h, w, 4), np.uint8)] * 4
    sc0 = O.Scene(cams, dummy)
    surf = scenes.HeightField(z0=0.0, amp=15.0, lx=60.0, ly=45.0)
    imgs = scenes.render_views(4, lambda v: sc0.unproject_grid(v, scale=0.5), surf, seed=77, cell=28.0)
    _compare_mvs(ctx, cams, imgs, None, P, 1, [0, 2, 3], min_labelled=0.05)
    P2 = T.default_params(False, 420.0, 580.0, 24, radius=3, image_scale=0.5)
    _compare_two(ctx, cams, imgs, None, P2, 1, 2)


def test_single_and_seven_neighbours(ctx):
    cams, imgs, ms, _ = refractive_arc_scene(V=8, w=64, h=40, masks=False, arc_deg=40.0)
    P = T.default_params(True, 420.0, 580.0, 24)
    _compare_mvs(ctx, cams, imgs, None, P, 3, [4])
    _compare_mvs(ctx, cams, imgs, None, P, 3, [0, 1, 2, 4, 5, 6, 7], min_labelled=0.05)


def test_bad_arguments_fail_loudly(ctx):
    cams, imgs, ms, _ = refractive_arc_scene(V=3, w=32, h=24, masks=False)
    ctx.set_views(cams, imgs, None)
    with pytest.raises(capi.SrError):
        ctx.set_params(T.default_params(True, 420.0, 580.0, 1))  # fewer than two labels
    with pytest.raises(capi.SrError):
        ctx.set_params(T.default_params(True, 420.0, 580.0, 8, radius=9))  # unsupported radius
    for run in (ctx.run_view, ctx.run_view_curve):  # label and curve mode share their argument checks
        ctx.set_params(T.default_params(True, 420.0, 580.0, 8))
        with pytest.raises(capi.SrError):
            run(0, [0])  # a view cannot be its own neighbour
        with pytest.raises(capi.SrError):
            run(5, [0])
        ctx.set_params(T.default_params(True, 420.0, 580.0, 8, row_begin=10, row_end=10))
        with pytest.raises(capi.SrError):
            run(0, [1, 2])  # empty row range
        ctx.set_params(T.default_params(False, 420.0, 580.0, 8))
        with pytest.raises(capi.SrError):
            run(0, [1, 2])  # two-view selection takes exactly one neighbour


def test_camera_only_views(ctx):
    """rgba8[i] == NULL: a view this context only needs the camera of (another rank computes it)."""
    cams, imgs, ms, _ = refractive_arc_scene(V=5, w=64, h=40, masks=False)
    P = T.default_params(True, 420.0, 580.0, 16)
    ctx.set_views(cams, imgs, None)
    ctx.set_params(P)
    ctx.run_view(1, [0, 2])
    want = ctx.depth_index(1).copy()
    ctx.set_views(cams, [imgs[0], imgs[1], imgs[2], None, None], None)
    ctx.set_params(P)
    ctx.run_view(1, [0, 2])
    assert (ctx.depth_index(1) == want).all()
    with pytest.raises(capi.SrError):
        ctx.run_view(1, [0, 3])
    with pytest.raises(capi.SrError):
        ctx.run_view(4, [0, 2])
