"""Pins oracle/oracle.cpp against the REFERENCE'S OWN leaf sources and classes (util/lineiter.cpp, util/ray.cpp,
util/vectorimage.cpp, stereo/adaptiveweight.cpp, stereo/geodesicweight.cpp, project/camera.cpp,
stereo/multiviewstereo.cpp, stereo/twoviewstereo.cpp), compiled from the reference's source tree into
oracle/_ref/libref.so (`make -C oracle REF=<reference source tree>`, see oracle/Makefile).
Bit-exact for the leaves and the classes; to rounding (1e-12) for the camera model, whose matrix algebra goes
through a stand-in for Eigen on the reference side.

Where oracle/_ref is not built, every test compares with a stored copy in tests/golden/ref_pins/
(tests/golden/make_ref_pins.py; SOURCE.json there says which code wrote it).  The copy in the repository was
written without the reference: it is the ORACLE's output on these inputs, which these tests found equal to the
reference's (bit for bit; to rounding for the camera model) when oracle/_ref was last built.  Against it the
tests are regression pins of the oracle, not an independent check against the reference; with oracle/_ref
built they are that check again."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle_api as O

REF = O.ref_lib()
PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pins")
MVS_COMBOS = [(i, d, a) for a in (False, True) for (i, d) in ((True, True), (False, True), (False, False))]
TWO_COMBOS = [(True, True), (False, False)]


def stored(name):
    return np.load(os.path.join(PINS, name + ".npz"))


def mvs_name(interface, distortion, adaptive):
    return f"mvs_i{int(interface)}_d{int(distortion)}_a{int(adaptive)}"


def two_name(interface, distortion):
    return f"two_i{int(interface)}_d{int(distortion)}"


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


# ---- inputs (shared with tests/golden/make_ref_pins.py) ----------------------------------------------
def line_cases():
    rng = np.random.RandomState(11)
    cases = [(0, 0, 10, 3), (10, 3, 0, 0), (5, 5, 5, 5), (0, 0, 0, 9), (7, 2, 7, -6), (-5, -5, 70, 60),
             (-20, 10, 90, 12), (30, -40, 31, 90), (63, 47, 0, 0), (64, 48, -1, -1), (100, 100, 200, 150)]
    for _ in range(400):
        cases.append(tuple(int(v) for v in rng.randint(-40, 110, 4)))
    return cases, 64, 48


def ray_cases():
    rng = np.random.RandomState(5)
    out = []
    for _ in range(500):
        s1, d1, s2, d2, pn = (rng.normal(size=3) for _ in range(5))
        out.append((s1, d1, s2, d2, pn, float(rng.normal() * 3), float(rng.uniform(0.6, 1.7))))
    return out


def leaf_image():
    rng = np.random.RandomState(2)
    h, w = 37, 53
    img = rng.randint(0, 256, size=(h, w, 4)).astype(np.uint8)
    img[..., 3] = 255
    img[5:9, 7:12] = 255  # a WHITE patch
    return img


def sample_points(w, h):
    rng = np.random.RandomState(9)
    return [(float(rng.uniform(-2, w + 1)), float(rng.uniform(-2, h + 1))) for _ in range(2000)]


def grid_points(w, h):
    return [(x, y) for x in range(-2, w + 2) for y in range(-2, h + 2)]


def weight_centres(w, h):
    rng = np.random.RandomState(4)
    cx = np.concatenate([rng.randint(0, w, 30), [0, w - 1, 0, w - 1]]).astype(np.int32)
    cy = np.concatenate([rng.randint(0, h, 30), [0, 0, h - 1, h - 1]]).astype(np.int32)
    return cx, cy


WEIGHT_CASES = [(kind, radius) for kind in (0, 1) for radius in (1, 2, 5, 9)]


def cameras():
    """Cameras covering every branch: refractive + distorted (cfg4's), refractive only, distorted
    only, plain pinhole."""
    from stereoreconstruction_b200 import scenes
    out = []
    for interface, dist in ((True, (-0.1, 0.05, 0.001, 0.001, 0.0)), (True, (0.0,) * 5),
                            (False, (-0.1, 0.05, 0.001, 0.001, 0.0)), (False, (0.0,) * 5)):
        out += scenes.arc_cameras(4, 640, 480, arc_deg=40.0, interface=interface, distortion=dist)[1:3]
    return out


def unproject_pixels():
    rng = np.random.RandomState(3)
    xy = np.concatenate([rng.uniform(-20, 660, (400, 1)), rng.uniform(-20, 500, (400, 1))], axis=1)
    return np.ascontiguousarray(np.concatenate([xy, [[319.5, 239.5], [0.5, 0.5], [639.5, 479.5]]]))


def project_points():
    """Per camera: 600 points in front and in view (along the oracle's pixel rays), 200 anywhere."""
    rng = np.random.RandomState(4)
    out = []
    for c in cameras():
        sc = O.Scene([c], [np.zeros((480, 640, 4), np.uint8)])
        rays = sc.unproject_grid(0).reshape(-1, 6)
        rays = rays[rng.randint(0, rays.shape[0], 600)]
        pts = rays[:, :3] + rng.uniform(200, 900, (600, 1)) * rays[:, 3:]
        out.append(np.ascontiguousarray(np.concatenate([pts, rng.uniform(-400, 400, (200, 3)) + [0, 0, 100]])))
    return out


def projection_matrices():
    """P of the first two cameras, scaled by 3.7 (the reference normalises P by its third row)."""
    out = []
    for c in cameras()[:2]:
        K, R = np.array(c.K[:]).reshape(3, 3), np.array(c.R[:]).reshape(3, 3)
        out.append(np.ascontiguousarray(K @ np.hstack([R, np.array(c.t[:])[:, None]]) * 3.7))
    return out


def mvs_scene(interface, distortion):
    from scene_util import refractive_arc_scene
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=96, h=64, masks=True, interface=interface, distortion=distortion)
    return cams, imgs, ms


def mvs_curve_pixels():
    rng = np.random.RandomState(8)
    return [(int(rng.randint(4, 92)), int(rng.randint(4, 60))) for _ in range(40)]


def two_cost_windows():
    rng = np.random.RandomState(1)
    out = []
    for _ in range(150):
        x1, y1 = int(rng.randint(0, 96)), int(rng.randint(0, 64))
        x2, y2 = int(rng.randint(-3, 99)), int(rng.randint(-3, 67))
        out.append((x1, y1, x2, y2))
    return out


def label_pixels(mask, n, seed):
    rng = np.random.RandomState(seed)
    ys, xs = np.nonzero(mask == 255)
    pick = rng.choice(len(ys), n, replace=False)
    return list(zip(ys[pick], xs[pick]))


def _pod(c):
    return O.as_cam_array([c])


# ---- the reference itself (oracle/_ref) -----------------------------------------------------------
def ref_lines():
    cases, w, h = line_cases()
    counts, pts, ok, out = [], [], [], []
    for (x0, y0, x1, y1) in cases:
        for clip in (0, 1):
            buf = np.empty((4096, 2), np.int32)
            n = REF.ref_line(x0, y0, x1, y1, clip, w, h, _ip(buf), 4096)
            counts.append(n)
            pts.append(buf[:min(n, 4096)].copy())
        a = np.array([x0, y0, x1, y1], dtype=np.int32)
        ok.append(REF.ref_clip_line(_ip(a), w, h))
        out.append(a)
    return dict(counts=np.array(counts), points=np.concatenate(pts), clip_ok=np.array(ok), clip_out=np.array(out))


def ref_rays():
    d = {k: [] for k in ("intersect_ok", "intersect", "refract_ok", "refract", "closest")}
    for (s1, d1, s2, d2, pn, pd, n) in ray_cases():
        b, b6, c6 = np.full(3, np.nan), np.empty(6), np.empty(6)
        d["intersect_ok"].append(REF.ref_intersect(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), _dp(b)))
        d["intersect"].append(b)
        d["refract_ok"].append(REF.ref_refract(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), C.c_double(n), _dp(b6)))
        d["refract"].append(b6)
        REF.ref_closest_points(_dp(s1), _dp(d1), _dp(s2), _dp(d2), _dp(c6))
        d["closest"].append(c6)
    return {k: np.array(v) for k, v in d.items()}


def _ref_image(image):
    h, w = image.shape[:2]
    REF.ref_image_create.restype = C.c_void_p
    return C.c_void_p(REF.ref_image_create(image.ctypes.data_as(C.c_void_p), w, h))


def ref_samples():
    image = leaf_image()
    h, w = image.shape[:2]
    r = _ref_image(image)
    out = {}
    for key, pts in (("sample", sample_points(w, h)), ("grid", grid_points(w, h))):
        vals = np.empty((len(pts), 4))
        for i, (x, y) in enumerate(pts):
            REF.ref_sample(r, C.c_double(x), C.c_double(y), _dp(vals[i]))
        out[key] = vals
    cx, cy = weight_centres(w, h)
    for kind, radius in WEIGHT_CASES:
        wts = np.empty((cx.size, 2 * radius + 1, 2 * radius + 1))
        REF.ref_weights(r, kind, radius, cx.size, _ip(cx), _ip(cy), _dp(wts))
        out[f"weights_k{kind}_r{radius}"] = wts
    REF.ref_image_destroy(r)
    return out


def ref_cameras():
    derived, rays, xy, ok, from_p = [], [], [], [], []
    pix = unproject_pixels()
    for c, pts in zip(cameras(), project_points()):
        got = O.OrcCamera()
        REF.ref_camera_derived(_pod(c), C.byref(got))
        derived.append(bytes(got))
        r = np.empty((len(pix), 6))
        REF.ref_camera_unproject(_pod(c), len(pix), _dp(pix), _dp(r))
        rays.append(r)
        p, k = np.empty((len(pts), 2)), np.empty(len(pts), np.int32)
        REF.ref_camera_project(_pod(c), len(pts), _dp(pts), _dp(p), _ip(k))
        xy.append(p)
        ok.append(k)
    for P in projection_matrices():
        got = O.OrcCamera()
        REF.ref_camera_from_P(_dp(P), C.byref(got))
        from_p.append(bytes(got))
    return dict(derived=np.frombuffer(b"".join(derived), np.uint8), unproject=np.array(rays), project_xy=np.array(xy),
                project_ok=np.array(ok), from_P=np.frombuffer(b"".join(from_p), np.uint8))


def ref_mvs(interface, distortion, adaptive):
    import golden_cases as G
    cams, imgs, ms = mvs_scene(interface, distortion)
    mind, maxd, D, cross = G.REF_MVS_CASES["arc"]
    ref = O.RefMVS(cams, imgs, ms, mind, maxd, D, cross, adaptive=adaptive)
    after, nb = ref.run()
    before, peak_pix, peaks = [], [], []
    for v in range(len(cams)):
        d, pk = ref.initial_estimate(v)
        before.append(d)
        pix = np.flatnonzero(ms[v] == 255)
        peak_pix.append(pix)
        peaks.append(pk.reshape(-1, 9, 2)[pix])
    counts, pts, costs = [], [], []
    for (x, y) in mvs_curve_pixels():
        curve = ref.curve(1, 2, x, y)
        counts.append(len(curve))
        pts.append(curve)
        for (px, py) in curve[:: max(1, len(curve) // 5)]:
            costs.append(ref.cost_ncc(1, 2, x, y, px, py))
    ref.close()
    # maps as (views, pixels): the layout of the stored copy, which keeps a sample of the pixels
    return dict(neighbours=np.array([r + [-1] * (3 - len(r)) for r in nb], np.int32),
                before=np.array(before).reshape(len(cams), -1), after=np.asarray(after).reshape(len(cams), -1),
                peak_pix=peak_pix, peaks=peaks, curve_counts=np.array(counts),
                curve_points=np.concatenate(pts), costs=np.array(costs))


def ref_two(interface, distortion):
    import golden_cases as G
    cams, imgs, ms = mvs_scene(interface, distortion)
    a, b, mind, maxd, D = G.REF_TWO_CASES["arc"]
    ref = O.RefTwoView(cams[a], cams[b], imgs[a], imgs[b], ms[a], ms[b], mind, maxd, D)
    before = np.array(ref.search()).reshape(2, -1)  # (views, pixels), as in ref_mvs
    after = np.array(ref.run()).reshape(2, -1)
    costs = np.array([[ref.cost(sad, 0, *win) for sad in (0, 1)] for win in two_cost_windows()])
    ref.close()
    return dict(before=before, after=after, costs=costs)


def ref_label_mvs():
    """The depth-label sweep composed from the reference's compiled pieces (see the test)."""
    import golden_cases as G
    from stereoreconstruction_b200 import types as T
    cams, imgs, ms = G.arc_scene()
    mind, maxd, D, cross = G.REF_MVS_CASES["arc"]
    P = T.default_params(True, mind, maxd, D)
    sc = O.Scene(cams, imgs, ms)
    ref_view = 1
    nb = [int(v) for v in sc.select_neighbours(3)[ref_view]]
    ref = O.RefMVS(cams, imgs, ms, mind, maxd, D, cross)
    depths = _label_depths(P, D)
    cam = cams[ref_view]
    n, Cc = _prin_dir(cam), np.array(cam.C[:])
    h, w = ms[0].shape
    label, depth, cost = [], [], []
    for y, x in label_pixels(ms[ref_view], 120, 12):
        ray = np.empty(6)
        REF.ref_camera_unproject(_pod(cam), 1, _dp(np.array([x + 0.5, y + 0.5])), _dp(ray))
        best = None  # (cost, depth, label)
        for j in nb:
            pts, ok = np.empty((D, 3)), np.zeros(D, bool)
            for d in range(D):
                x0 = Cc + n * depths[d]
                out3 = np.empty(3)
                ok[d] = REF.ref_intersect(_dp(ray[:3].copy()), _dp(ray[3:].copy()), _dp(n.copy()), C.c_double(n.dot(x0)), _dp(out3)) != 0
                pts[d] = out3
            xy, pok = np.empty((D, 2)), np.empty(D, np.int32)
            REF.ref_camera_project(_pod(cams[j]), D, _dp(np.ascontiguousarray(pts)), _dp(xy), _ip(pok))
            for d in range(D):
                if not ok[d] or not pok[d]:
                    continue
                tx, ty = int(xy[d, 0]), int(xy[d, 1])  # truncation, multiviewstereo.cpp:773-775
                if not (0 <= tx < w and 0 <= ty < h) or ms[j][ty, tx] != 255:
                    continue
                c = ref.cost_ncc(ref_view, j, int(x), int(y), tx, ty)
                if c > 0.95 and (best is None or (c, depths[d]) > best[:2]):
                    best = (c, depths[d], d)
        label.append(-1 if best is None else best[2])
        depth.append(-1.0 if best is None else best[1])
        cost.append(np.nan if best is None else best[0])
    ref.close()
    return dict(label=np.array(label), depth=np.array(depth), cost=np.array(cost))


def ref_label_two():
    """The two-view label sweep composed from the reference's compiled pieces (see the test)."""
    import golden_cases as G
    from stereoreconstruction_b200 import types as T
    cams, imgs, ms = G.arc_scene()
    a, b, mind, maxd, D = G.REF_TWO_CASES["arc"]
    P = T.default_params(False, mind, maxd, D)
    ref = O.RefTwoView(cams[a], cams[b], imgs[a], imgs[b], ms[a], ms[b], mind, maxd, D)
    depths = _label_depths(P, D)
    cam = cams[a]
    n, Cc = _prin_dir(cam), np.array(cam.C[:])
    label, depth, cost = [], [], []
    for y, x in label_pixels(ms[a], 60, 13):
        ray = np.empty(6)
        REF.ref_camera_unproject(_pod(cam), 1, _dp(np.array([x + 0.5, y + 0.5])), _dp(ray))
        pts, ok = np.empty((D, 3)), np.zeros(D, bool)
        for d in range(D):
            out3 = np.empty(3)
            ok[d] = REF.ref_intersect(_dp(ray[:3].copy()), _dp(ray[3:].copy()), _dp(n.copy()),
                                      C.c_double(n.dot(Cc + n * depths[d])), _dp(out3)) != 0
            pts[d] = out3
        xy, pok = np.empty((D, 2)), np.empty(D, np.int32)
        REF.ref_camera_project(_pod(cams[b]), D, _dp(np.ascontiguousarray(pts)), _dp(xy), _ip(pok))
        min_cost, second, dep, index = np.inf, np.inf, np.nan, -1
        for d in range(D):
            if not ok[d] or not pok[d]:
                continue
            c = ref.cost(0, 0, int(x), int(y), int(xy[d, 0] - 0.5), int(xy[d, 1] - 0.5))
            if c + 1e-10 < min_cost:
                second, min_cost, dep, index = min_cost, c, depths[d], d
        if index >= 0 and min_cost > 0.95 * second:
            dep, index = np.inf, -3
        label.append(index)
        depth.append(dep)
        cost.append(min_cost)
    ref.close()
    return dict(label=np.array(label), depth=np.array(depth), cost=np.array(cost))


def _label_depths(P, D):
    L = O.lib()
    L.orc_depth_from_label.restype = C.c_double
    pp = O.as_params(P)
    return np.array([L.orc_depth_from_label(C.byref(pp), d) for d in range(D)])


def _prin_dir(cam):
    n = np.array(cam.prin_dir[:])
    return n / np.sqrt(n.dot(n))


def reference(name, live, *args):
    """The values the test compares with: the reference's, computed by oracle/_ref when it is built; else the
    stored copy (see the module docstring for what wrote it)."""
    return live(*args) if REF is not None else stored(name)


def kept(want, key, n):
    """Indices (along the first axis, or flat pixels of a map) of the entries of `key` that `want` holds: all n
    of them from oracle/_ref, a fixed seeded sample in the stored copy (its `<key>_idx`)."""
    return np.asarray(want[key + "_idx"]) if key + "_idx" in want else np.arange(n)


# ---- the tests ----------------------------------------------------------------------------------
def test_line_iterator_and_clip_match_reference():
    L = O.lib()
    want = reference("lines", ref_lines)
    cases, w, h = line_cases()
    off, k = 0, 0
    for j, i in enumerate(kept(want, "clip_ok", len(cases))):
        x0, y0, x1, y1 = cases[i]
        for clip in (0, 1):
            buf = np.empty((4096, 2), dtype=np.int32)
            n = L.orc_line(x0, y0, x1, y1, clip, w, h, _ip(buf), 4096)
            assert n == want["counts"][k], (x0, y0, x1, y1, clip)
            m = min(n, 4096)
            assert (buf[:m] == want["points"][off:off + m]).all(), (x0, y0, x1, y1, clip)
            off += m
            k += 1
        a = np.array([x0, y0, x1, y1], dtype=np.int32)
        ok = L.orc_clip_line(_ip(a), w, h)
        assert ok == want["clip_ok"][j]
        if ok:
            assert (a == want["clip_out"][j]).all()
    assert off == len(want["points"]) and k == len(want["counts"])


def test_ray_ops_match_reference():
    L = O.lib()
    want = reference("rays", ref_rays)
    cases = ray_cases()
    for i, j in enumerate(kept(want, "closest", len(cases))):
        s1, d1, s2, d2, pn, pd, n = cases[j]
        a = np.full(3, np.nan)
        ra = L.orc_intersect(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), _dp(a))
        assert ra == want["intersect_ok"][i]
        if ra:
            assert (a == want["intersect"][i]).all()
        a6 = np.empty(6)
        ra = L.orc_refract(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), C.c_double(n), _dp(a6))
        assert ra == want["refract_ok"][i] and (a6 == want["refract"][i]).all()
        L.orc_closest_points(_dp(s1), _dp(d1), _dp(s2), _dp(d2), _dp(a6))
        assert (a6 == want["closest"][i]).all()


@pytest.fixture(scope="module")
def samples():
    return reference("samples", ref_samples)


def _identity_scene(image):
    from stereoreconstruction_b200 import types as T
    return O.Scene([T.make_camera(np.eye(3), np.eye(3), np.zeros(3))], [image])


def test_pixel_sample_gray_match_reference(samples):
    image = leaf_image()
    h, w = image.shape[:2]
    sc = _identity_scene(image)
    L = O.lib()
    a = np.empty(4)
    pts = sample_points(w, h)
    for j, i in enumerate(kept(samples, "sample", len(pts))):
        x, y = pts[i]
        L.orc_sample(sc.ptr, 0, C.c_double(x), C.c_double(y), _dp(a))
        assert _same(a, samples["sample"][j]), (x, y)
    pts = grid_points(w, h)
    for j, i in enumerate(kept(samples, "grid", len(pts))):
        x, y = pts[i]
        # sampleInt(x,y) == sample((double)x,(double)y) of the reference
        L.orc_sample_int(sc.ptr, 0, x, y, _dp(a))
        assert _same(a, samples["grid"][j]), (x, y)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("radius", [1, 2, 5, 9])
def test_weights_match_reference(samples, kind, radius):
    image = leaf_image()
    h, w = image.shape[:2]
    cx, cy = weight_centres(w, h)
    mine = _identity_scene(image).weights(0, kind, radius, cx, cy)
    key = f"weights_k{kind}_r{radius}"
    assert (mine[kept(samples, key, cx.size)] == samples[key]).all()


# ---- project/camera.cpp: the reference's own Camera class ------------------------------------------
@pytest.fixture(scope="module")
def camera_ref():
    return reference("cameras", ref_cameras)


def _cams_from_bytes(buf):
    n = C.sizeof(O.OrcCamera)
    return [O.OrcCamera.from_buffer_copy(bytes(buf[i * n:(i + 1) * n])) for i in range(len(buf) // n)]


def test_camera_derived_state_matches_reference(camera_ref):
    """Camera::set / setLensDistortion / setRefractiveIndex / setPlane (camera.cpp:205-222,302-342):
    Kinv, Rinv, C, the principal ray and the two flags, as the host code derives them."""
    for c, got in zip(cameras(), _cams_from_bytes(camera_ref["derived"]), strict=True):
        for f in ("K", "R", "t", "dist", "plane_n"):
            assert np.allclose(np.array(getattr(got, f)[:]), np.array(getattr(c, f)[:]), rtol=0, atol=1e-15), f
        for f in ("Kinv", "Rinv", "C", "prin_dir"):
            assert np.allclose(np.array(getattr(got, f)[:]), np.array(getattr(c, f)[:]), rtol=1e-13, atol=1e-13), f
        assert got.plane_d == c.plane_d and got.n == c.n
        assert got.is_refractive == c.is_refractive and got.is_distorted == c.is_distorted


def test_camera_unproject_matches_reference(camera_ref):
    """Camera::unproject (camera.cpp:423-459): distortion removal (5 fixed-point rounds), K^-1, refract
    at the interface, local -> global."""
    xy = unproject_pixels()
    xy = xy[kept(camera_ref, "unproject", len(xy))]
    L = O.lib()
    cams = cameras()
    assert len(camera_ref["unproject"]) == len(cams)
    for c, ref in zip(cams, camera_ref["unproject"]):
        got = np.empty((len(xy), 6))
        for i, (x, y) in enumerate(xy):
            L.orc_unproject(_pod(c), C.c_double(x), C.c_double(y), _dp(got[i]))
        assert np.isfinite(ref).all()
        assert np.abs(got - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("root_mode", [0, 1])
def test_camera_project_matches_reference(camera_ref, root_mode):
    """Camera::project + projectRefraction (camera.cpp:95-138,380-419) — the quartic's coefficients, the
    root acceptance test, the point on the interface, K, distortion with the reference's y-from-distorted-x
    — against the oracle in both root modes (0: the same quartic + acceptance order; 1: the monotone
    1-D solve the GPU uses).  The GSL call inside the reference is answered by the restated solver."""
    cams = cameras()
    assert len(camera_ref["project_xy"]) == len(cams)
    for c, pts, ref_xy, ref_ok in zip(cams, project_points(), camera_ref["project_xy"], camera_ref["project_ok"]):
        pts = pts[kept(camera_ref, "project_xy", len(pts))]
        sc = O.Scene([c], [np.zeros((480, 640, 4), np.uint8)])
        xy, ok = sc.project_points(0, pts, root_mode=root_mode)
        assert (ok != 0).mean() > 0.5
        same = (ok != 0) == (ref_ok != 0)
        assert same.mean() >= 0.995, same.mean()  # acceptance at the +-1e-3 band edges may differ by rounding
        both = (ok != 0) & (ref_ok != 0)
        err = np.abs(xy[both] - ref_xy[both]).max(axis=1)
        assert np.quantile(err, 0.995) <= 1e-8, np.quantile(err, 0.995)
        # a different accepted root is only possible inside the |y| < 1e-3 acceptance band (DESIGN.md section 2)
        assert (err > 1e-6).mean() <= 0.005


def test_camera_from_projection_matrix_matches_reference(camera_ref):
    """Camera::setP -> updateOthers (camera.cpp:251-288): RQ factorisation as the host code does it."""
    from stereoreconstruction_b200 import types as T
    got_all = _cams_from_bytes(camera_ref["from_P"])
    assert len(got_all) == 2
    for c, P, got in zip(cameras()[:2], projection_matrices(), got_all):
        mine = T.camera_from_P(P)
        for f in ("K", "R", "t", "C", "prin_dir"):
            a, b = np.array(getattr(got, f)[:]), np.array(getattr(mine, f)[:])
            assert np.allclose(a, b, rtol=1e-9, atol=1e-9), (f, a, b)
        # (the reference divides P by the SQUARED norm of its third row, :252: a scaled P gives a scaled K)
        assert np.allclose(np.array(got.K[:]) / got.K[8], np.array(c.K[:]), rtol=1e-9, atol=1e-7)


# ---- stereo/multiviewstereo.cpp: the reference's own MultiViewStereo, end to end ---------------------
@pytest.mark.parametrize("adaptive", [False, True])
@pytest.mark.parametrize("interface,distortion", [(True, True), (False, True), (False, False)])
def test_mvs_end_to_end_matches_reference(interface, distortion, adaptive):
    """initialize() -> runTask() of the reference's own class (neighbour rule, rasterised epipolar curves,
    weighted NCC, K = 9 peak lists, selection, cross-check; multiviewstereo.cpp:193-247,325-475,524-810) on a
    masked 4-view scene — refractive + distorted, air + distorted, air + pinhole: the oracle reproduces
    every output BIT FOR BIT.  (The stored copy keeps the maps and peak lists at a sample of the pixels.)"""
    import golden_cases as G
    from stereoreconstruction_b200 import types as T
    want = reference(mvs_name(interface, distortion, adaptive), ref_mvs, interface, distortion, adaptive)
    cams, imgs, ms = mvs_scene(interface, distortion)
    mind, maxd, D, cross = G.REF_MVS_CASES["arc"]
    sc = O.Scene(cams, imgs, ms)
    P = T.default_params(True, mind, maxd, D, weight_kind=T.SR_WEIGHT_ADAPTIVE if adaptive else T.SR_WEIGHT_GEODESIC)
    nb = [[int(v) for v in r if v >= 0] for r in want["neighbours"]]
    assert nb == [[int(v) for v in r] for r in sc.select_neighbours(3)]
    before = []
    for v in range(len(cams)):
        od, _, _, _, op = sc.mvs_view(P, v, nb[v], curve_mode=True, root_mode=0, want_peaks=True)
        before.append(od)
        pix = kept(want, "before", od.size)
        assert _same(od.reshape(-1)[pix], want["before"][v])
        pix = np.asarray(want["peak_pix"][v])
        assert pix.size > 0 and (ms[v].reshape(-1)[pix] == 255).all()
        assert (op.reshape(-1, 9, 2)[pix] == want["peaks"][v]).all()
        assert (np.isfinite(od) & (od > 0)).mean() > 0.3
    after = sc.crosscheck_mvs(P, before, cross)
    for v in range(len(cams)):
        assert _same(after[v].reshape(-1)[kept(want, "after", after[v].size)], want["after"][v])
        assert 0.2 < (np.isfinite(after[v]) & (after[v] > 0)).mean() < (np.isfinite(before[v]) & (before[v] > 0)).mean()
    # the file-local cost function and the public curve of single pixels
    off, k = 0, 0
    for i, (x, y) in enumerate(mvs_curve_pixels()):
        n = int(want["curve_counts"][i])
        curve = want["curve_points"][off:off + n]
        off += n
        mine = sc.epipolar_curve(P, 1, 2, x, y, True, 0)
        assert curve.shape == mine.shape and (curve == mine).all()
        for (px, py) in curve[:: max(1, len(curve) // 5)]:
            assert want["costs"][k] == sc.cost(P, 1, 2, x, y, int(px), int(py))
            k += 1
    assert off == len(want["curve_points"]) and k == len(want["costs"])


# ---- stereo/twoviewstereo.cpp: the reference's own TwoViewStereo, end to end ----------------------------
@pytest.mark.parametrize("interface,distortion", [(True, True), (False, False)])
def test_twoview_end_to_end_matches_reference(interface, distortion):
    """constructor -> computeCostVolumes -> crossCheck of the reference's own class (live rasterised-curve
    search with the second-best test in both directions, cross-check; twoviewstereo.cpp:89-124,233-500,
    596-672) and its two cost functions (cost_ncc :909-977, cost_sad :864-905, windows over borders and
    masked pixels included): the oracle reproduces every output BIT FOR BIT.  (The reference's unqualified
    abs(sum1) is the floating overload of its author's toolchain: ref_shim/precompiled_shim.hpp.)"""
    import golden_cases as G
    from stereoreconstruction_b200 import types as T
    want = reference(two_name(interface, distortion), ref_two, interface, distortion)
    cams, imgs, ms = mvs_scene(interface, distortion)
    a, b, mind, maxd, D = G.REF_TWO_CASES["arc"]
    sc = O.Scene(cams, imgs, ms)
    P = T.default_params(False, mind, maxd, D)
    ol, _, cl = sc.twoview_curve(P, a, b, root_mode=0)
    orr, _, _ = sc.twoview_curve(P, b, a, root_mode=0)
    pix = kept(want, "before", ol.size)
    assert _same(want["before"][0], ol.reshape(-1)[pix]) and _same(want["before"][1], orr.reshape(-1)[pix])
    assert np.isfinite(ol).mean() > 0.3 and np.isinf(ol).any() and cl.max() > 5
    wl, wr = sc.crosscheck_two(P, a, b, ol, orr, 1.0, root_mode=0)
    pix = kept(want, "after", wl.size)
    assert _same(want["after"][0], wl.reshape(-1)[pix]) and _same(want["after"][1], wr.reshape(-1)[pix])
    for i, (x1, y1, x2, y2) in enumerate(two_cost_windows()):
        for sad, kind in ((0, T.SR_COST_NCC_TWOVIEW), (1, T.SR_COST_SAD_TWOVIEW)):
            P2 = T.default_params(False, mind, maxd, D, cost_kind=kind)
            r_, o_ = want["costs"][i][sad], sc.cost(P2, a, b, x1, y1, x2, y2)
            assert r_ == o_ or (np.isnan(r_) and np.isnan(o_)), (sad, x1, y1, x2, y2, r_, o_)


def test_label_mode_is_the_reference_pieces_composed():
    """The depth-label sweep (north_star's cost volume + WTA) is compiled out of the reference
    (twoviewstereo.cpp:283,308-329), so it cannot be run there.  Here it is COMPOSED from the reference's own
    compiled pieces — Camera::unproject, intersect (pointFromDepth), Camera::project, the MultiViewStereo
    cost_ncc — with only the loop and the selection rule (multiviewstereo.cpp:589-602,654-660) written in
    this test (ref_label_mvs), for 120 random pixels: index, depth and winning cost equal the oracle's label mode."""
    import golden_cases as G
    from stereoreconstruction_b200 import types as T
    want = reference("label_mvs", ref_label_mvs)
    cams, imgs, ms = G.arc_scene()
    mind, maxd, D, cross = G.REF_MVS_CASES["arc"]
    P = T.default_params(True, mind, maxd, D)
    sc = O.Scene(cams, imgs, ms)
    ref_view = 1
    nb = [int(v) for v in sc.select_neighbours(3)[ref_view]]
    od, oi, ob, _, _ = sc.mvs_view(P, ref_view, nb, root_mode=0)
    pixels = label_pixels(ms[ref_view], 120, 12)
    assert len(want["label"]) == len(pixels) == 120
    labelled = 0
    for (y, x), lab, dep, cost in zip(pixels, want["label"], want["depth"], want["cost"]):
        if lab < 0:
            assert oi[y, x] == -1 and od[y, x] == -1
        else:
            labelled += 1
            assert oi[y, x] == lab and od[y, x] == dep and ob[y, x] == cost, (x, y, lab, oi[y, x], ob[y, x])
    assert labelled > 30


def test_twoview_label_mode_is_the_reference_pieces_composed():
    """The same for the two-view label sweep (twoviewstereo.cpp:308-329 — the compiled-out branch — with the
    live path's second-best test :304-305): Camera::unproject, intersect, Camera::project and
    TwoViewStereo::cost_ncc are the reference's own compiled code; the loop, the tap rule
    (x*scale - 0.5, truncated by the callee's int parameters) and the selection are written in ref_label_two."""
    import golden_cases as G
    from stereoreconstruction_b200 import types as T
    want = reference("label_two", ref_label_two)
    cams, imgs, ms = G.arc_scene()
    a, b, mind, maxd, D = G.REF_TWO_CASES["arc"]
    P = T.default_params(False, mind, maxd, D)
    sc = O.Scene(cams, imgs, ms)
    od, oi, ob, _ = sc.twoview_label(P, a, b, root_mode=0)
    pixels = label_pixels(ms[a], 60, 13)
    assert len(want["label"]) == len(pixels) == 60
    finite = 0
    for (y, x), index, depth, min_cost in zip(pixels, want["label"], want["depth"], want["cost"]):
        assert oi[y, x] == index, (x, y, index, oi[y, x])
        assert (od[y, x] == depth) or (np.isnan(depth) and np.isnan(od[y, x]))
        if index != -1:
            assert ob[y, x] == min_cost
        finite += np.isfinite(depth)
    assert finite > 10
