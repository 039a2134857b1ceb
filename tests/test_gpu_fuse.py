"""sr_fuse_points (one de-duplicated point cloud of all views' depth maps) against the NumPy restatement of its
model in tests/fuse_util.py, and MultiViewStereo::setFusePointCloud against Context.fuse_points.

The CPU tests check the restatement itself: that the fixtures reach every rule, that none of their decisions is a
near-tie (so the exact comparisons on the GPU are well posed), the two identities with sr_get_points' cloud, and
that fusion does what it is for on a scene with known geometry.  The GPU tests compare the library with the
restatement run on the library's own unproject and projection, so only the fusion logic is under test."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree

import fuse_util as F
from oracle import oracle_api as O
from stereoreconstruction_b200 import capi, scenes, types as T
from scene_util import refractive_arc_scene
from test_gpu_point_cloud import MIN_DEPTHS, reference_points, sentinel_depths, write_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "stereoreconstruction_b200")
SR_ERR_INVALID, SR_ERR_STATE = 1, 3  # include/sr_b200.h
CROSS = 12.0                          # cross-check threshold of the arc scene (label step 5.16)
MAX_DISTS = (1.0, CROSS, 1000.0)      # nothing but near-duplicates / the cross-check's / every projection with a point


@pytest.fixture(scope="module")
def small_scene():
    return refractive_arc_scene(V=4, w=96, h=64, masks=True)


def oracle_maps(scene, levels=32, curve=False):
    cams, imgs, ms, _ = scene
    P = T.default_params(True, 420.0, 580.0, levels)
    sc = O.Scene(cams, imgs, ms)
    nb = sc.select_neighbours(3)
    return P, sc, [sc.mvs_view(P, v, nb[v], curve_mode=curve)[0] for v in range(len(cams))]


def oracle_fuse(sc, cams, imgs, depths, min_depth, max_dist, min_views, scale=1.0):
    rays = [sc.unproject_grid(v, scale) for v in range(len(cams))]
    return F.fuse(cams, rays, lambda u, X: sc.project_points(u, X), depths, imgs, min_depth, scale, max_dist, min_views)


def lib_fuse(ctx, cams, imgs, min_depth, max_dist, min_views):
    """The restatement on the library's geometry and its current maps (ctx.params.image_scale)."""
    rays = [ctx.unproject_grid(v) for v in range(ctx.V)]
    depths = [ctx.depth(v) for v in range(ctx.V)]
    return F.fuse(cams, rays, lambda u, X: ctx.project_points(u, X), depths, imgs, min_depth,
                  ctx.params.image_scale, max_dist, min_views)


def lib_view_points(ctx):
    """Every view's points as sr_get_points computes them, in the layout of fuse_util.view_points."""
    out = []
    for v in range(ctx.V):
        xyz, _, pix = ctx.points(v)
        pts = np.full((ctx.h * ctx.w, 3), np.nan)
        pts[pix] = xyz
        has = np.zeros(ctx.h * ctx.w, bool)
        has[pix] = True
        out.append((pts, has))
    return out


def concat_points(cams, rays, depths, imgs, min_depth):
    """sr_get_points over the views, concatenated, as the restatement returns clouds."""
    xyz, rgb, src = [], [], []
    for v in range(len(cams)):
        p, idx, _ = reference_points(cams[v], rays[v], depths[v], min_depth)
        xyz.append(p)
        rgb.append(imgs[v][..., :3].reshape(-1, 3)[idx])
        src.append(np.stack([np.full(len(idx), v), idx], 1).astype(np.int32))
    return np.concatenate(xyz), np.concatenate(rgb), np.concatenate(src)


# ---- CPU: the restatement and its fixtures ------------------------------------------------------------------------

def test_restatement_reaches_every_rule(small_scene):
    """Measured: on the masked 4-view arc scene (96x64, 24576 pixels) after the oracle's label-mode run, at
    max_dist 12 with min_views 1 and 2, kept pixels have support 0 to 3 (support 0 with min_views 0), 1590 and
    5840 pixels fail min_views, 9167 and 6780 are not emitted because a lower view keeps them, 46 and 250 are emitted
    although a confirming lower view's pixel is not kept, and matches are rejected off-image (81), for a pixel
    without a point (7779) and by distance (8985).  The sentinel maps add every reason a pixel has no point."""
    cams, imgs, ms, _ = small_scene
    P, sc, depths = oracle_maps(small_scene)
    seen = dict(kept_support=set(), dropped=0, blocked=0, lower_unkept=0, off_image=0, no_point=0, distance=0)

    def note(r):
        for v in range(len(cams)):
            seen["kept_support"] |= set(np.unique(r["support"][v][r["kept"][v]]).tolist())
            seen["dropped"] += int(((r["support"][v] >= 0) & ~r["kept"][v]).sum())
            seen["blocked"] += int(r["blocked"][v].sum())
            seen["lower_unkept"] += int(r["lower_unkept"][v].sum())
        for k in ("off_image", "no_point", "distance"):
            seen[k] += r["reject"][k]
    for mv in (0, 1, 2):
        note(oracle_fuse(sc, cams, imgs, depths, P.min_depth, CROSS, mv))
    h, w = imgs[0].shape[:2]
    for min_depth in MIN_DEPTHS:
        sent = [sentinel_depths(h, w, min_depth, seed=v)[0] for v in range(len(cams))]
        r = oracle_fuse(O.Scene(cams, imgs), cams, imgs, sent, min_depth, 1000.0, 1)
        note(r)
        assert r["reject"]["no_point"] > 0
    assert seen["kept_support"] == {0, 1, 2, 3}, seen
    for k in ("dropped", "blocked", "lower_unkept", "off_image", "no_point", "distance"):
        assert seen[k] > 0, (k, seen)


def test_restatement_has_no_near_ties(small_scene):
    """No agreement distance within 1e-9 * max(1, max_dist) of max_dist and no projected coordinate within 1e-9
    of an integer, on the fixtures the GPU tests compare exactly (label and curve mode, every max_dist)."""
    cams, imgs, ms, _ = small_scene
    for curve in (False, True):
        P, sc, depths = oracle_maps(small_scene, curve=curve)
        for md in MAX_DISTS:
            assert oracle_fuse(sc, cams, imgs, depths, P.min_depth, md, 1)["ties"] == (0, 0), (curve, md)


def test_restatement_identities(small_scene):
    """max_dist 0 with min_views 0, and a single view with min_views 0, give sr_get_points' clouds concatenated,
    bit for bit; a single view with min_views >= 1 gives nothing."""
    cams, imgs, ms, _ = small_scene
    P, sc, depths = oracle_maps(small_scene)
    rays = [sc.unproject_grid(v) for v in range(len(cams))]
    xyz, rgb, src = concat_points(cams, rays, depths, imgs, P.min_depth)
    r = oracle_fuse(sc, cams, imgs, depths, P.min_depth, 0.0, 0)
    assert r["xyz"].tobytes() == xyz.tobytes() and (r["rgb"] == rgb).all() and (r["source"] == src).all()
    one = O.Scene(cams[:1], imgs[:1])
    r = oracle_fuse(one, cams[:1], imgs[:1], depths[:1], P.min_depth, CROSS, 0)
    x1, g1, s1 = concat_points(cams[:1], rays[:1], depths[:1], imgs[:1], P.min_depth)
    assert r["xyz"].tobytes() == x1.tobytes() and (r["rgb"] == g1).all() and (r["source"] == s1).all()
    assert len(oracle_fuse(one, cams[:1], imgs[:1], depths[:1], P.min_depth, CROSS, 1)["xyz"]) == 0


def test_fusion_quality_small_scale():
    """On the oracle's label-mode maps of a 4-view 192x128 masked arc scene (32 levels, step 5.16), cross-checked
    at 12, then fused at max_dist 12, min_views 1.  Measured: 18277 fused points against 59516 concatenated; median
    |z - f(x, y)| 3.81 against 4.10; coverage of view 0's in-mask true surface points within one label step 0.876
    against 0.954 (ratio 0.918: one point per surface sample sits near fewer of view 0's true points than four
    overlapping clouds do)."""
    w, h = 192, 128
    f = scenes.arc_cameras(4, w, h)[0].K[0]
    scene = refractive_arc_scene(V=4, w=w, h=h, cell=3.5 * 500.0 / f, masks=True)
    cams, imgs, ms, surf = scene
    P, sc, depths = oracle_maps(scene)
    step = (P.max_depth - P.min_depth) / (P.num_levels - 1)
    rays = [sc.unproject_grid(v) for v in range(len(cams))]
    cc = sc.crosscheck_mvs(P, depths, CROSS)
    cat = concat_points(cams, rays, cc, imgs, P.min_depth)[0]
    fused = oracle_fuse(sc, cams, imgs, cc, P.min_depth, CROSS, 1)["xyz"]
    truth = surf.hit(rays[0])[ms[0] == 255]

    def quality(c):
        e = np.abs(c[:, 2] - surf.z(c[:, 0], c[:, 1]))
        return float(np.median(e)), float((cKDTree(c).query(truth)[0] <= step).mean())
    (med_f, cov_f), (med_c, cov_c) = quality(fused), quality(cat)
    assert len(fused) < 0.4 * len(cat), (len(fused), len(cat))
    assert med_f < 0.98 * med_c, (med_f, med_c)
    assert cov_f >= 0.88 * cov_c, (cov_f, cov_c)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def run_scene(scene, curve, cross):
    cams, imgs, ms, _ = scene
    P = T.default_params(True, 420.0, 580.0, 32)
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    ctx.set_params(P)
    nb = ctx.select_neighbours(3)
    for v in range(len(cams)):
        (ctx.run_view_curve if curve else ctx.run_view)(v, nb[v])
    if cross:
        ctx.cross_check(False, CROSS)
    return ctx, P


@pytest.mark.gpu
@pytest.mark.parametrize("cross", [False, True], ids=["raw", "cross_checked"])
@pytest.mark.parametrize("curve", [False, True], ids=["label", "curve"])
def test_g1_parity(small_scene, curve, cross):
    cams, imgs, ms, _ = small_scene
    ctx, P = run_scene(small_scene, curve, cross)
    pts = lib_view_points(ctx)
    deps = [ctx.depth(v) for v in range(ctx.V)]
    total = 0
    for md in MAX_DISTS:
        for mv in (0, 1, 2, 3):
            want = lib_fuse(ctx, cams, imgs, P.min_depth, md, mv)
            assert want["ties"] == (0, 0), (md, mv)
            got = ctx.fuse_points(md, mv)
            total += F.assert_same_cloud(got, want, f"max_dist={md} min_views={mv}")
            # on the library's own points every sum and mean is the same IEEE operation in the same order
            exact = F.fuse(cams, None, lambda u, X: ctx.project_points(u, X), deps, imgs, P.min_depth, 1.0, md, mv,
                           points=pts)
            assert_bits(got, (exact["xyz"], exact["rgb"], exact["source"]))
    assert total > 0
    ctx.close()


@pytest.mark.gpu
def test_g2_sentinels_and_image_scale(small_scene):
    cams, imgs, ms, _ = small_scene
    h, w = imgs[0].shape[:2]
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    for scale in (1.0, 0.5):
        for min_depth in MIN_DEPTHS:
            ctx.set_params(T.default_params(True, min_depth, 1000.0, 32, image_scale=scale))
            for v in range(len(cams)):
                ctx.set_depth(v, sentinel_depths(h, w, min_depth, seed=v)[0])
            for md, mv in ((1000.0, 0), (1000.0, 1), (100.0, 1)):
                want = lib_fuse(ctx, cams, imgs, min_depth, md, mv)
                assert want["ties"] == (0, 0)
                F.assert_same_cloud(ctx.fuse_points(md, mv), want, f"scale={scale} min_depth={min_depth}")
    ctx.close()


def assert_bits(a, b):
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()


def concat_lib_points(ctx):
    pts = [ctx.points(v) for v in range(ctx.V)]
    return (np.concatenate([p[0] for p in pts]), np.concatenate([p[1] for p in pts]),
            np.concatenate([np.stack([np.full(len(p[2]), v, np.int32), p[2]], 1) for v, p in enumerate(pts)]))


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [False, True], ids=["label", "curve"])
def test_g3_identities(small_scene, curve):
    cams, imgs, ms, _ = small_scene
    ctx, P = run_scene(small_scene, curve, True)
    assert_bits(ctx.fuse_points(0.0, 0), concat_lib_points(ctx))
    depth0 = ctx.depth(0)
    ctx.close()
    one = capi.Context(0)
    one.set_views(cams[:1], imgs[:1], ms[:1])
    one.set_params(P)
    one.set_depth(0, depth0)
    assert_bits(one.fuse_points(CROSS, 0), concat_lib_points(one))
    assert len(one.fuse_points(CROSS, 0)[0]) > 0 and len(one.fuse_points(CROSS, 1)[0]) == 0
    one.close()


def height_field_views(V, w, h, seed):
    """V views of a height field with depths near the truth (+-2 units of noise) and 20 % NaN holes."""
    cams = scenes.arc_cameras(V, w, h, f=1600.0, distortion=None)
    imgs = scenes.noise_images(V, w, h, seed=seed)
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, None)
    ctx.set_params(T.default_params(True, 350.0, 650.0, 64))
    surf = scenes.HeightField(z0=0.0, amp=25.0, lx=90.0, ly=70.0)
    rng = np.random.RandomState(seed)
    for v in range(V):
        c = cams[v]
        d = (surf.hit(ctx.unproject_grid(v)) - np.array(c.C[:])) @ np.array(c.prin_dir[:])
        d = d + rng.uniform(-2.0, 2.0, size=d.shape)
        d[rng.rand(h, w) < 0.2] = np.nan
        ctx.set_depth(v, d)
    return ctx, cams, imgs


@pytest.mark.gpu
@pytest.mark.parametrize("V,w,h", [(2, 1, 64), (3, 4097, 3), (2, 16384, 2), (8, 1920, 1080)])
def test_g4_sizes(V, w, h):
    """Against the restatement run on the library's own points (sr_get_points), bit for bit: at the edges of the
    16384-wide view the NumPy plane intersection differs from the library's in the 12th digit (7e-12), which
    sr_get_points' own tests hold to 1e-9."""
    ctx, cams, imgs = height_field_views(V, w, h, seed=w + h)
    pts = lib_view_points(ctx)
    deps = [ctx.depth(v) for v in range(V)]
    for md, mv in ((3.0, 1), (10.0, 0)):
        want = F.fuse(cams, None, lambda u, X: ctx.project_points(u, X), deps, imgs, 350.0, 1.0, md, mv, points=pts)
        assert want["ties"] == (0, 0) and len(want["xyz"]) > 0
        assert_bits(ctx.fuse_points(md, mv), (want["xyz"], want["rgb"], want["source"]))
    ctx.close()


@pytest.mark.gpu
def test_g4_strict_agreement(small_scene):
    """Two views with the same camera, image and map: every pixel's point is also the other view's point at
    distance exactly 0, so max_dist 0 confirms nothing (the strict <) and any positive max_dist confirms every
    pixel whose projection comes back to it, whose fused point (X + X) / 2 is X."""
    cams, imgs, ms, _ = small_scene
    ctx, P = run_scene(small_scene, False, True)
    depth = ctx.depth(0)
    ctx.close()
    two = capi.Context(0)
    two.set_views([cams[0], cams[0]], [imgs[0], imgs[0]], [ms[0], ms[0]])
    two.set_params(P)
    two.set_depth(0, depth)
    two.set_depth(1, depth)
    xyz, rgb, pix = two.points(0)
    assert len(xyz) > 1000
    assert len(two.fuse_points(0.0, 1)[0]) == 0
    fx, frgb, fsrc = two.fuse_points(1e-9, 1)
    assert (fsrc[:, 0] == 0).all() and len(fsrc) >= 0.99 * len(pix)
    sel = np.searchsorted(pix, fsrc[:, 1])
    assert (pix[sel] == fsrc[:, 1]).all()
    assert fx.tobytes() == np.ascontiguousarray(xyz[sel]).tobytes() and (frgb == rgb[sel]).all()
    two.close()


def raw_fuse(ctx, max_dist, min_views, capacity, xyz=None, rgb=None, src=None, count=True):
    n = C.c_int64(-5)
    p = lambda a: None if a is None else a.ctypes.data
    rc = ctx._L.sr_fuse_points(ctx._h, float(max_dist), int(min_views), int(capacity), p(xyz), p(rgb), p(src),
                               C.byref(n) if count else None)
    return rc, n.value


@pytest.mark.gpu
def test_g5_errors_and_state(small_scene):
    cams, imgs, ms, _ = small_scene
    ctx = capi.Context(0)
    assert raw_fuse(ctx, CROSS, 1, 0)[0] == SR_ERR_STATE  # no views
    ctx.set_views(cams, imgs, ms)
    assert raw_fuse(ctx, CROSS, 1, 0)[0] == SR_ERR_STATE  # no params
    ctx.close()
    ctx, P = run_scene(small_scene, False, True)
    buf = np.zeros((16, 3)), np.zeros((16, 3), np.uint8)
    assert raw_fuse(ctx, CROSS, 1, 0, count=False)[0] == SR_ERR_INVALID
    assert raw_fuse(ctx, CROSS, 1, 16, None, buf[1])[0] == SR_ERR_INVALID
    assert raw_fuse(ctx, CROSS, 1, 16, buf[0], None)[0] == SR_ERR_INVALID
    assert raw_fuse(ctx, CROSS, 1, -1)[0] == SR_ERR_INVALID
    for md in (-1.0, np.nan, np.inf):
        assert raw_fuse(ctx, md, 1, 0)[0] == SR_ERR_INVALID
    assert raw_fuse(ctx, CROSS, -1, 0)[0] == SR_ERR_INVALID
    assert raw_fuse(ctx, CROSS, len(cams), 0) == (0, 0)  # min_views > V - 1
    depths = [ctx.depth(v).tobytes() for v in range(len(cams))]
    index = [ctx.depth_index(v).tobytes() for v in range(len(cams))]
    rc, n = raw_fuse(ctx, CROSS, 1, 0)
    assert rc == 0 and n > 1
    xyz, rgb, src = np.full((n, 3), 7.25), np.full((n, 3), 0xAB, np.uint8), np.full((n, 2), -7, np.int32)
    assert raw_fuse(ctx, CROSS, 1, n - 1, xyz, rgb, src) == (SR_ERR_INVALID, n)
    assert (xyz == 7.25).all() and (rgb == 0xAB).all() and (src == -7).all()
    assert raw_fuse(ctx, CROSS, 1, n, xyz, rgb, src) == (0, n)
    assert raw_fuse(ctx, CROSS, 1, n, xyz, rgb, None) == (0, n)  # the source is optional
    a, b = ctx.fuse_points(CROSS, 1), ctx.fuse_points(CROSS, 1)
    assert_bits(a, b)
    assert_bits((xyz, rgb, src), a)
    assert [ctx.depth(v).tobytes() for v in range(len(cams))] == depths
    assert [ctx.depth_index(v).tobytes() for v in range(len(cams))] == index
    # a context reused from larger images gives what a fresh one gives
    big, _, _ = height_field_views(4, 320, 200, seed=3)
    big.fuse_points(10.0, 1)
    big.set_views(cams, imgs, ms)
    big.set_params(P)
    for v in range(len(cams)):
        big.set_depth(v, np.frombuffer(depths[v]).reshape(imgs[0].shape[:2]))
    assert_bits(big.fuse_points(CROSS, 1), a)
    big.close()
    ctx.close()
    # a view this context has only the camera of
    ctx = capi.Context(0)
    ctx.set_views(cams, [imgs[0], None, imgs[2], imgs[3]], None)
    ctx.set_params(P)
    assert raw_fuse(ctx, CROSS, 1, 0)[0] == SR_ERR_STATE
    ctx.close()


@pytest.mark.gpu
def test_g6_ordered_after_the_runs():
    """Straight after sr_run_view on the lanes, without a synchronise, fusion waits for every view."""
    w, h, V = 1920, 1080, 3
    cams = scenes.arc_cameras(V, w, h)
    ctx = capi.Context(0)
    ctx.set_views(cams, [np.zeros((h, w, 4), np.uint8)] * V, None)
    surf = scenes.HeightField(z0=0.0, amp=25.0, lx=90.0, ly=70.0)
    imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), surf, seed=4321, cell=3.5 * 500.0 / cams[0].K[0])
    ctx.set_views(cams, imgs, None)
    ctx.set_params(T.default_params(True, 350.0, 650.0, 64))
    ctx.run_view(0, [1, 2])
    ctx.run_view(1, [0, 2])
    ctx.run_view(2, [0, 1])
    now = ctx.fuse_points(5.0, 1)
    ctx.synchronize()
    later = ctx.fuse_points(5.0, 1)
    assert len(later[0]) > 0
    assert_bits(now, later)
    ctx.close()


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    """tests/cpp/fuse_test.cpp built against the library."""
    out = str(tmp_path_factory.mktemp("fuse") / "fuse_test")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-Wno-deprecated-declarations", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "fuse_test.cpp"), "-L", PKG, "-lsr_b200", "-lz",
           "-Wl,-rpath," + PKG, "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return out


def test_fuse_driver_builds(driver):
    assert os.path.exists(driver)


@pytest.mark.gpu
def test_g7_class(small_scene, driver, tmp_path):
    cams, imgs, ms, _ = small_scene
    h, w = imgs[0].shape[:2]
    scene = str(tmp_path / "scene.bin")
    write_scene(scene, cams, imgs, ms)
    r = subprocess.run([driver, scene, str(tmp_path), "420", "580", "32", str(CROSS), "0"], capture_output=True,
                       text=True, timeout=1800)
    assert r.returncode == 0, r.stdout + r.stderr
    m = re.search(r"fuse off_fused=(\d+) off_points=(\d+) fused1=(\d+) fused2=(\d+)", r.stdout)
    assert m, r.stdout
    assert int(m[1]) == 0
    V, n = len(cams), h * w
    load = lambda name, dt: np.fromfile(str(tmp_path / name), dt)
    d_off = load("depth_off.bin", np.float64).reshape(V, h, w)
    for k in (1, 2):
        assert load(f"depth_{k}.bin", np.float64).tobytes() == d_off.tobytes()
    # with the flag off, pointCloud() is the host loop's cloud of the unchanged maps
    sc = O.Scene(cams, imgs)
    rays = [sc.unproject_grid(v) for v in range(V)]
    want_xyz, want_rgb, _ = concat_points(cams, rays, list(d_off), imgs, 420.0)
    off_xyz = load("off_xyz.bin", np.float64).reshape(-1, 3)
    assert off_xyz.shape == want_xyz.shape and int(m[2]) == len(want_xyz)
    assert (np.abs(off_xyz - want_xyz) <= 1e-9 * np.maximum(1.0, np.abs(want_xyz))).all()
    assert (load("off_rgb.bin", np.uint8).reshape(-1, 3) == want_rgb).all()
    # the class's fused cloud is Context.fuse_points(threshold, k) on the same maps
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    ctx.set_params(T.default_params(True, 420.0, 580.0, 32))
    for v in range(V):
        ctx.set_depth(v, d_off[v])
    for k in (1, 2):
        xyz, rgb, _ = ctx.fuse_points(CROSS, k)
        assert len(xyz) == int(m[2 + k]) > 0
        assert load(f"fused{k}_xyz.bin", np.float64).tobytes() == xyz.tobytes()
        assert load(f"fused{k}_rgb.bin", np.uint8).tobytes() == rgb.tobytes()
    ctx.close()
