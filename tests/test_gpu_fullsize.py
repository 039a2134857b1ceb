"""BASELINE.json's full sizes (cfg4: 1920x1080, 256 labels, refractive, 3 neighbours) on the GPU,
through size-independent properties — the oracle needs ~15 minutes per view at this size:
  * the screened MVS path picks the same label at every pixel as the all-FP64 kernel;
  * the build's interpolation self-check finds no differing tap, the screen no value outside its bar;
  * two row bands computed separately equal the whole view (row sharding is bit-invisible);
  * the depth map reconstructs the rendered surface (the images are photo-consistent renders of a
    known height field through the refractive cameras)."""
import numpy as np
import pytest

from stereoreconstruction_b200 import capi, scenes, types as T

pytestmark = pytest.mark.gpu

W, H, V, D = 1920, 1080, 8, 256


@pytest.fixture(scope="module")
def cfg4():
    cams = scenes.arc_cameras(V, W, H)
    P = T.default_params(True, 350.0, 650.0, D)
    surf = scenes.HeightField(z0=0.0, amp=25.0, lx=90.0, ly=70.0)
    c = capi.Context(0)
    c.set_views(cams, [np.zeros((H, W, 4), np.uint8)] * V, None)
    c.set_params(P)
    rays = {v: c.unproject_grid(v) for v in (2, 3, 4, 5)}
    imgs = scenes.render_views(V, lambda v: rays[v] if v in rays else rays[3], surf, 4321, 3.5 * 500.0 / cams[0].K[0])
    c.close()
    return cams, imgs, P, surf, rays[3]


def _run(monkeypatch, cams, imgs, P, env, row_bands=None):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = capi.Context(0)
    c.set_views(cams, imgs, None)
    if row_bands is None:
        c.set_params(P)
        c.run_view(3, [2, 4, 5])
    else:
        for (r0, r1) in row_bands:
            Q = T.SrParams.from_buffer_copy(P)
            Q.row_begin, Q.row_end = r0, r1
            c.set_params(Q)
            c.run_view(3, [2, 4, 5])
    out = (c.depth_index(3).copy(), c.depth(3).copy(), c.best_cost(3).copy())
    stats = (c.match_stats(), c.build_stats()) if env.get("SR_MATCH_STATS") == "1" else None
    c.close()
    for k in env:
        monkeypatch.delenv(k)
    return out, stats


def test_cfg4_full_size_properties(cfg4, monkeypatch):
    cams, imgs, P, surf, rays3 = cfg4
    (i1, d1, b1), stats = _run(monkeypatch, cams, imgs, P, {"SR_MATCH_STATS": "1"})
    ms, bs = stats
    assert bs["interpolated"] > 1e9 and bs["tap_mismatches"] == 0
    # every verified label inside its own error bar (one-pass screen: the bar follows the label's cancellation,
    # e0 + e1 * kappa, typically 1e-5 .. 1e-4), and the reserved slot 7 (prescreen_false_drops) reads 0
    assert ms["outside_error_bar"] == 0 and ms["max_screen_err"] < 1e-4 and ms["prescreen_false_drops"] == 0
    # screened path == all-FP64 kernel, same taps
    (i0, d0, b0), _ = _run(monkeypatch, cams, imgs, P, {"SR_MATCH_SCREEN": "0"})
    assert (i0 == i1).all(), f"{(i0 != i1).sum()} of {i0.size} pixels differ"
    lab = i0 >= 0
    assert lab.mean() > 0.5
    assert np.abs(b0[lab] - b1[lab]).max() <= 1e-9
    # anchors-only build (every label projected exactly is the stride-1 limit): the generic
    # build_kernel projects every label with its own FP32/FP64 Newton — same taps, same result
    (i2, _, _), _ = _run(monkeypatch, cams, imgs, P, {"SR_BUILD_REFR": "0"})
    assert (i2 != i1).mean() <= 1e-6
    # row bands
    (i3, d3, _), _ = _run(monkeypatch, cams, imgs, P, {}, row_bands=[(0, 500), (500, H)])
    assert (i3 == i1).all() and ((d3 == d1) | (np.isnan(d3) & np.isnan(d1))).all()
    # the reconstruction: depth of the rendered surface along the principal axis of view 3
    hit = surf.hit(rays3)
    prin = np.array(cams[3].prin_dir)
    true_depth = (hit - np.array(cams[3].C)) @ prin
    step = (P.max_depth - P.min_depth) / (D - 1)
    err = np.abs(d1[lab] - true_depth[lab])
    assert np.median(err) < 2 * step, np.median(err)
