"""sr_get_points (the coloured point cloud of a depth map, MultiViewStereo's PLY export on the GPU) against a
NumPy reference over the oracle's Camera::unproject, and MultiViewStereo::setKeepPointCloud against the class's
own host loop.

The reference applies pointFromDepth (stereo/multiviewstereo.cpp:740-750) and the filter of
MultiViewStereo::pointCloud: plane normal prin_dir through C + n d, intersection rejected when |n.dir| < 1e-10
or t < 1e-10 (util/ray.cpp:78-88), pixels skipped when d is not finite or d + 1e-5 < min_depth."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import oracle_api as O
from stereoreconstruction_b200 import capi, scenes, types as T
from scene_util import refractive_arc_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "stereoreconstruction_b200")
# min_depth of the sentinel fixtures: 10 lies closer than the interface (plane_d 25), where the plane through
# C + n d is behind the refracted ray's source; 400 lies beyond it, where a depth within the 1e-5 slack keeps its point
MIN_DEPTHS = (10.0, 400.0)
SR_ERR_INVALID, SR_ERR_STATE = 1, 3  # include/sr_b200.h


def reference_points(cam, rays, depth, min_depth):
    """(xyz (n,3), pixel (n,), per-rule exclusion counts) of one view; rays = the oracle's (h,w,6) unproject grid."""
    src, d = rays[..., :3].reshape(-1, 3), rays[..., 3:].reshape(-1, 3)
    dep = depth.reshape(-1)
    n = np.array(cam.prin_dir[:])
    nrm = n / np.linalg.norm(n)
    finite = np.isfinite(dep)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        below = finite & (dep + 1e-5 < min_depth)
        x0 = np.array(cam.C[:])[None, :] + dep[:, None] * n[None, :]
        dist = x0 @ nrm
        nd = d @ nrm
        t = ((dist[:, None] * nrm[None, :] - src) @ nrm) / nd
        miss = finite & ~below & ((np.abs(nd) < 1e-10) | (t < 1e-10))
        keep = finite & ~below & ~miss
        p = src + t[:, None] * d
    idx = np.flatnonzero(keep).astype(np.int32)
    return p[idx], idx, dict(nonfinite=int((~finite).sum()), below=int(below.sum()), miss=int(miss.sum()),
                             kept=int(keep.sum()))


def assert_matches(got, cam, rays, depth, img, min_depth):
    xyz, rgb, pix = got
    want_xyz, want_pix, _ = reference_points(cam, rays, depth, min_depth)
    assert pix.shape == want_pix.shape and (pix == want_pix).all()
    err = np.abs(xyz - want_xyz) / np.maximum(1.0, np.abs(want_xyz))
    assert err.size == 0 or err.max() <= 1e-9, err.max()
    assert (rgb == img[..., :3].reshape(-1, 3)[pix]).all()
    return len(pix)


def sentinel_depths(h, w, min_depth, seed=7):
    """A depth map holding every case the filter and the intersection distinguish: NaN, +INF and -1, depths just
    below min_depth (excluded) and within its 1e-5 slack (kept unless the plane is behind the ray's source), 12
    (with min_depth 10: a plane behind the refracted ray's source on the interface, excluded), and ordinary
    depths.  Returns the map and the flat pixel indices of each case."""
    rng = np.random.RandomState(seed)
    d = rng.uniform(420.0, 580.0, size=(h, w))
    flat = d.reshape(-1)
    cases = dict(nan=np.nan, inf=np.inf, minus1=-1.0, below=min_depth - 2e-5, slack=min_depth - 0.5e-5, near=12.0)
    pick = rng.permutation(flat.size)[:len(cases) * 40]
    where = {}
    for k, (name, v) in enumerate(cases.items()):
        where[name] = pick[k * 40:(k + 1) * 40]
        flat[where[name]] = v
    return d, where


@pytest.fixture(scope="module")
def small_scene():
    return refractive_arc_scene(V=4, w=96, h=64, masks=True)


def test_reference_exercises_every_rule(small_scene):
    """CPU: on the sentinel fixture the reference excludes pixels by each rule and still keeps most of them, so the
    GPU comparisons below cover every branch of the filter and the intersection."""
    cams, imgs, ms, _ = small_scene
    h, w = imgs[0].shape[:2]
    sc = O.Scene(cams, imgs)
    near, far = MIN_DEPTHS
    depth, where = sentinel_depths(h, w, near)
    _, pix, c = reference_points(cams[0], sc.unproject_grid(0), depth, near)
    assert c["nonfinite"] == 80 and c["below"] == 80 and c["miss"] >= 40
    assert not np.isin(where["near"], pix).any() and c["kept"] > 0.2 * h * w
    # beyond the interface the two depths around min_depth fall on either side of the 1e-5 slack
    depth, where = sentinel_depths(h, w, far)
    _, pix, c = reference_points(cams[0], sc.unproject_grid(0), depth, far)
    assert np.isin(where["slack"], pix).all() and not np.isin(where["below"], pix).any()
    assert c["kept"] > 0.2 * h * w


def raw_points(ctx, view, capacity, xyz=None, rgb=None, pix=None):
    n = C.c_int64(-5)
    p = lambda a: None if a is None else a.ctypes.data
    rc = ctx._L.sr_get_points(ctx._h, int(view), int(capacity), p(xyz), p(rgb), p(pix), C.byref(n))
    return rc, n.value


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [False, True], ids=["label", "curve"])
def test_scene_after_cross_check(small_scene, curve):
    cams, imgs, ms, _ = small_scene
    P = T.default_params(True, 420.0, 580.0, 32)
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    ctx.set_params(P)
    nb = ctx.select_neighbours(3)
    for v in range(len(cams)):
        (ctx.run_view_curve if curve else ctx.run_view)(v, nb[v])
    ctx.cross_check(False, 12.0)
    sc = O.Scene(cams, imgs, ms)
    total = 0
    for v in range(len(cams)):
        total += assert_matches(ctx.points(v), cams[v], sc.unproject_grid(v), ctx.depth(v), imgs[v], P.min_depth)
    assert total > 0
    ctx.close()


@pytest.mark.gpu
def test_sentinels_and_image_scale(small_scene):
    cams, imgs, ms, _ = small_scene
    h, w = imgs[0].shape[:2]
    sc = O.Scene(cams, imgs)
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    for scale in (1.0, 0.5):
        for min_depth in MIN_DEPTHS:
            ctx.set_params(T.default_params(True, min_depth, 1000.0, 32, image_scale=scale))
            for v in range(len(cams)):
                depth, _ = sentinel_depths(h, w, min_depth, seed=v)
                ctx.set_depth(v, depth)
                got = ctx.points(v)
                assert assert_matches(got, cams[v], sc.unproject_grid(v, scale), depth, imgs[v], min_depth) > 0.2 * h * w
    # an all-NaN map has no points, with and without output buffers
    ctx.set_depth(1, np.full((h, w), np.nan))
    assert raw_points(ctx, 1, 0) == (0, 0)
    xyz, rgb, pix = ctx.points(1)
    assert xyz.shape == (0, 3) and rgb.shape == (0, 3) and pix.shape == (0,)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 64), (4097, 3), (16384, 2), (1920, 1080)])
def test_sizes(w, h):
    """Rows narrower than a block, one partial block past a multiple of 256, the widest rows, and a full-size view."""
    cams = scenes.arc_cameras(2, w, h, f=1600.0, distortion=None)
    imgs = scenes.noise_images(2, w, h, seed=w + h)
    rng = np.random.RandomState(w)
    depth = rng.uniform(420.0, 580.0, size=(h, w))
    depth[rng.rand(h, w) < 0.3] = np.nan
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, None)
    ctx.set_params(T.default_params(True, 420.0, 580.0, 32))
    ctx.set_depth(1, depth)
    a = ctx.points(1)
    assert assert_matches(a, cams[1], O.Scene(cams, imgs).unproject_grid(1), depth, imgs[1], 420.0) > 0
    b = ctx.points(1)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    ctx.close()


@pytest.mark.gpu
def test_buffers_and_state(small_scene):
    cams, imgs, ms, _ = small_scene
    h, w = imgs[0].shape[:2]
    ctx = capi.Context(0)
    ctx.set_views(cams, imgs, ms)
    assert raw_points(ctx, 0, 0)[0] == SR_ERR_STATE  # before sr_set_params
    ctx.set_params(T.default_params(True, MIN_DEPTHS[0], 1000.0, 32))
    ctx.set_depth(0, sentinel_depths(h, w, MIN_DEPTHS[0])[0])
    rc, n = raw_points(ctx, 0, 0)
    assert rc == 0 and n > 1
    xyz = np.full((n, 3), 7.25)
    rgb = np.full((n, 3), 0xAB, np.uint8)
    pix = np.full(n, -7, np.int32)
    assert raw_points(ctx, 0, n - 1, xyz, rgb, pix) == (SR_ERR_INVALID, n)  # the count is reported
    assert (xyz == 7.25).all() and (rgb == 0xAB).all() and (pix == -7).all()
    assert raw_points(ctx, 0, n, xyz, rgb, pix) == (0, n)
    assert (pix >= 0).all()
    assert raw_points(ctx, len(cams), 0)[0] == SR_ERR_INVALID and raw_points(ctx, -1, 0)[0] == SR_ERR_INVALID
    ctx.close()
    # a view this context has only the camera of
    ctx = capi.Context(0)
    ctx.set_views(cams, [imgs[0], None, imgs[2], imgs[3]], None)
    ctx.set_params(T.default_params(True, MIN_DEPTHS[0], 1000.0, 32))
    assert raw_points(ctx, 1, 0)[0] == SR_ERR_STATE
    assert raw_points(ctx, 0, 0)[0] == 0
    ctx.close()


@pytest.mark.gpu
def test_ordered_after_the_view_it_reads():
    """Right after sr_run_view, without a synchronise, the depth image and the point cloud of that view wait for it
    (the view runs on a lane of its own): each equals what the same call returns after sr_synchronize."""
    w, h, V = 1920, 1080, 3
    cams = scenes.arc_cameras(V, w, h)
    ctx = capi.Context(0)
    ctx.set_views(cams, [np.zeros((h, w, 4), np.uint8)] * V, None)
    surf = scenes.HeightField(z0=0.0, amp=25.0, lx=90.0, ly=70.0)
    imgs = scenes.render_views(V, lambda v: ctx.unproject_grid(v), surf, seed=4321, cell=3.5 * 500.0 / cams[0].K[0])
    ctx.set_views(cams, imgs, None)
    P = T.default_params(True, 350.0, 650.0, 64)
    ctx.set_params(P)
    ctx.run_view(0, [1, 2])
    img_now = ctx.depth_image(0)
    ctx.run_view(1, [0, 2])
    pts_now = ctx.points(1)
    ctx.synchronize()
    assert (img_now == ctx.depth_image(0)).all()
    pts = ctx.points(1)
    assert len(pts[2]) > 0
    for x, y in zip(pts_now, pts):
        assert x.tobytes() == y.tobytes()
    ctx.close()


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    """tests/cpp/point_cloud_test.cpp built against the library (as __graft_entry__.build() builds its harness)."""
    out = str(tmp_path_factory.mktemp("point_cloud") / "point_cloud_test")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-Wno-deprecated-declarations", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "point_cloud_test.cpp"), "-L", PKG, "-lsr_b200", "-lz",
           "-Wl,-rpath," + PKG, "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return out


def write_scene(path, cams, imgs, masks):
    """The driver's input: int32 V, w, h; the camera PODs; RGBA8 images with the mask in alpha."""
    h, w = imgs[0].shape[:2]
    with open(path, "wb") as f:
        f.write(np.array([len(cams), w, h], np.int32).tobytes())
        for c in cams:
            f.write(bytes(c))
        for v, im in enumerate(imgs):
            x = np.ascontiguousarray(im, np.uint8).copy()
            if masks is not None:
                x[..., 3] = np.where(masks[v] == 255, 255, 0)
            f.write(x.tobytes())


def run_driver(exe, scene, outdir, mind, maxd, levels, cross, curve):
    r = subprocess.run([exe, scene, outdir, str(mind), str(maxd), str(levels), str(cross), str(int(curve))],
                       capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout + r.stderr
    m = re.search(r"points kept=(\d+) host=(\d+) same_rgb=(\d) max_rel=(\S+) host_ms=(\S+)", r.stdout)
    assert m, r.stdout
    return dict(kept=int(m[1]), host=int(m[2]), same_rgb=m[3] == "1", max_rel=float(m[4]), host_ms=float(m[5]))


def test_driver_builds(driver):
    assert os.path.exists(driver)


@pytest.mark.gpu
def test_class_keeps_the_host_loops_cloud(small_scene, driver, tmp_path):
    cams, imgs, ms, _ = small_scene
    scene = str(tmp_path / "scene.bin")
    write_scene(scene, cams, imgs, ms)
    res = run_driver(driver, scene, str(tmp_path), 420.0, 580.0, 32, 12.0, True)
    assert res["kept"] == res["host"] > 0 and res["same_rgb"] and res["max_rel"] <= 1e-9, res
    kx = np.fromfile(str(tmp_path / "kept_xyz.bin"), np.float64).reshape(-1, 3)
    hx = np.fromfile(str(tmp_path / "host_xyz.bin"), np.float64).reshape(-1, 3)
    assert kx.shape == hx.shape == (res["kept"], 3)
    assert (np.abs(kx - hx) <= 1e-9 * np.maximum(1.0, np.abs(hx))).all()
    assert (np.fromfile(str(tmp_path / "kept_rgb.bin"), np.uint8) == np.fromfile(str(tmp_path / "host_rgb.bin"), np.uint8)).all()
