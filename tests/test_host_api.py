"""The C++ class API (include/stereo, include/project, include/util) end to end on the GPU.

tests/cpp/host_api_test.cpp is compiled by __graft_entry__.build() against the C-ABI library and
drives Project / ImageSet / Camera / MultiViewStereo / TwoViewStereo / GeodesicWeight /
AdaptiveWeight the way the reference GUI does (gui/widgets/stereowidget.cpp:974-1002).  This test
writes a project XML + RGBA PNGs (alpha = mask), runs the harness, and checks its raw outputs
against the C ABI called directly with the harness's own camera PODs, and against the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from stereoreconstruction_b200 import capi, types as T
from scene_util import refractive_arc_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "stereoreconstruction_b200", "host_api_test")


def write_project(tmp, cams, imgs, masks):
    from PIL import Image
    os.makedirs(os.path.join(tmp, "images"), exist_ok=True)
    xml = ["<project>", " <cameras>"]
    for i, c in enumerate(cams):
        K = np.array(c.K).reshape(3, 3)
        R = np.array(c.R).reshape(3, 3)
        t = np.array(c.t)
        P = K @ np.hstack([R, t[:, None]])
        attrs = " ".join(f'm{r + 1}{k + 1}="{P[r, k]:.17g}"' for r in range(3) for k in range(4))
        xml.append(f'  <camera id="cam{i}" name="view {i}">')
        xml.append(f"   <projectionMatrix {attrs}/>")
        d = list(c.dist)
        xml.append(f'   <lensDistortion k1="{d[0]:.17g}" k2="{d[1]:.17g}" p1="{d[2]:.17g}" p2="{d[3]:.17g}" k3="{d[4]:.17g}"/>')
        if c.is_refractive:
            kn = K @ np.array(c.plane_n)
            xml.append(f'   <refractiveInterface px="{kn[0] / kn[2]:.17g}" py="{kn[1] / kn[2]:.17g}" '
                       f'dist="{c.plane_d:.17g}" refractiveRatio="{c.n:.17g}"/>')
        xml.append("  </camera>")
    xml += [" </cameras>", " <imageSets>", '  <imageSet root="images" id="set0" name="synthetic arc">']
    for i, (im, m) in enumerate(zip(imgs, masks)):
        rgba = im.copy()
        rgba[..., 3] = m
        Image.fromarray(rgba, "RGBA").save(os.path.join(tmp, "images", f"v{i}.png"))
        xml.append(f'   <image for="cam{i}" default="yes" file="v{i}.png"/>')
    xml += ["  </imageSet>", " </imageSets>", "</project>"]
    path = os.path.join(tmp, "project.xml")
    with open(path, "w") as f:
        f.write("\n".join(xml))
    return path


def test_harness_is_built():
    assert os.path.exists(HARNESS), "run __graft_entry__.build()"


@pytest.mark.gpu
def test_cpp_class_api_end_to_end(tmp_path):
    cams, imgs, ms, _ = refractive_arc_scene(V=4, w=96, h=64, masks=True)
    h, w = imgs[0].shape[:2]
    proj = write_project(str(tmp_path), cams, imgs, ms)
    out = str(tmp_path)
    mind, maxd, levels, cross = 420.0, 580.0, 32, 12.0
    r = subprocess.run([HARNESS, proj, "set0", out, str(mind), str(maxd), str(levels), str(cross)],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stderr

    # the camera PODs the C++ Camera class derived from the XML (setP -> RQ decomposition)
    raw = np.fromfile(os.path.join(out, "cams.bin"), dtype=np.uint8)
    V = len(cams)
    assert raw.size == V * C.sizeof(T.SrCamera)
    pods = [T.SrCamera.from_buffer_copy(raw[i * C.sizeof(T.SrCamera):(i + 1) * C.sizeof(T.SrCamera)].tobytes()) for i in range(V)]
    for a, b in zip(pods, cams):  # the decomposition recovers the cameras the XML was written from
        assert np.allclose(np.array(a.K), np.array(b.K), rtol=1e-9, atol=1e-7)
        assert np.allclose(np.array(a.R), np.array(b.R), atol=1e-10)
        assert np.allclose(np.array(a.C), np.array(b.C), atol=1e-7)
        assert np.allclose(np.array(a.plane_n), np.array(b.plane_n), atol=1e-10)
        assert a.is_refractive == b.is_refractive and a.is_distorted == b.is_distorted

    # MultiViewStereo == the C ABI driven directly with the same PODs (bit for bit), == oracle
    masks = [np.where(m == 255, 255, 0).astype(np.uint8) for m in ms]
    rgba = []
    for im, m in zip(imgs, ms):
        x = im.copy()
        x[..., 3] = m
        rgba.append(x)
    ctx = capi.Context(0)
    ctx.set_views(pods, rgba, masks)
    P = T.default_params(True, mind, maxd, levels)
    ctx.set_params(P)
    nb = ctx.select_neighbours(3)
    for v in range(V):
        ctx.run_view(v, nb[v])
    ctx.cross_check(False, cross)
    from oracle import oracle_api as O
    sc = O.Scene(pods, rgba, masks)
    before = []
    for v in range(V):
        od, _, _, _, _ = sc.mvs_view(P, v, nb[v])
        before.append(od)
    want = sc.crosscheck_mvs(P, before, cross)
    for v in range(V):
        gd = np.fromfile(os.path.join(out, f"mvs_v{v}_depth.bin"), dtype=np.float64).reshape(h, w)
        gi = np.fromfile(os.path.join(out, f"mvs_v{v}_index.bin"), dtype=np.int32).reshape(h, w)
        gn = np.fromfile(os.path.join(out, f"mvs_v{v}_nbrs.bin"), dtype=np.int32)
        assert list(gn) == nb[v]
        d = ctx.depth(v)
        assert ((gd == d) | (np.isnan(gd) & np.isnan(d))).all()
        assert (gi == ctx.depth_index(v)).all()
        assert ((gd == want[v]) | (np.isnan(gd) & np.isnan(want[v]))).mean() > 1 - 1e-4
        img = np.fromfile(os.path.join(out, f"mvs_v{v}_image.bin"), dtype=np.uint8).reshape(h, w, 4)
        fin = np.isfinite(gd) & (masks[v] == 255) & ~(gd + 1e-5 < mind)
        t = np.clip((gd[fin] - mind) / (maxd - mind), 0, 1)
        assert (img[..., 0][fin] == (255 * t).astype(np.int64)).all()  # colorFromDepth, multiviewstereo.cpp:257-278
        assert (img[..., 0][~fin] == 255).all()
        assert np.isfinite(gd).sum() > 0

    # MultiViewStereo in curve mode (the reference's live search) == sr_run_view_curve directly
    ctx.set_views(pods, rgba, masks)
    ctx.set_params(P)
    for v in range(V):
        ctx.run_view_curve(v, nb[v])
    ctx.cross_check(False, cross)
    for v in range(V):
        gd = np.fromfile(os.path.join(out, f"mvs_curve_v{v}_depth.bin"), dtype=np.float64).reshape(h, w)
        d = ctx.depth(v)
        assert ((gd == d) | (np.isnan(gd) & np.isnan(d))).all()
    # ... and its peak lists (setKeepPeaks) == sr_get_peaks directly
    P.keep_cost_volume = 2
    ctx.set_params(P)
    ctx.run_view_curve(0, nb[0])
    gp = np.fromfile(os.path.join(out, "mvs_curve_v0_peaks.bin"), dtype=np.float64).reshape(h, w, 9, 2)
    assert (gp == ctx.peaks(0)).all() and (gp[..., -1, 0] > 0.95).any()
    P.keep_cost_volume = 0

    # TwoViewStereo (no masks, radius 2, cross-check 30) == the C ABI directly
    two = [pods[0], pods[1]]
    plain = [rgba[0], rgba[1]]  # QImage(file) keeps the alpha byte; the mask argument was null
    ctx.set_views(two, plain, None)
    P2 = T.default_params(False, mind, maxd, levels, radius=2)
    ctx.set_params(P2)
    ctx.run_view(0, [1])
    ctx.run_view(1, [0])
    ctx.cross_check(True, 30.0)
    for name, v in (("left", 0), ("right", 1)):
        gd = np.fromfile(os.path.join(out, f"two_{name}_depth.bin"), dtype=np.float64).reshape(h, w)
        d = ctx.depth(v)
        assert ((gd == d) | (np.isnan(gd) & np.isnan(d))).all()
    li = np.fromfile(os.path.join(out, "two_left_image.bin"), dtype=np.uint8).reshape(h, w, 4)
    gd = np.fromfile(os.path.join(out, "two_left_depth.bin"), dtype=np.float64).reshape(h, w)
    assert (li[..., :3][~np.isfinite(gd)] == 0).all() and np.isfinite(gd).sum() > 0
    # the public epipolar-curve preview against the oracle's curve (two-view flavour, no mask)
    sc2 = O.Scene(two, plain, None)
    curve = np.fromfile(os.path.join(out, "two_curve.bin"), dtype=np.int32).reshape(-1, 2)
    want_curve = sc2.epipolar_curve(P2, 0, 1, w // 2, h // 2, mvs=False)
    assert curve.shape == want_curve.shape and (curve == want_curve).all()

    # weight functors == sr_compute_weights == oracle
    wv = np.fromfile(os.path.join(out, "weights.bin"), dtype=np.float64).reshape(2, 5, 5)
    cx, cy = np.array([w // 3], np.int32), np.array([h // 2], np.int32)
    sc1 = O.Scene([pods[0]], [rgba[0]], None)
    assert np.allclose(wv[0], sc1.weights(0, T.SR_WEIGHT_GEODESIC, 2, cx, cy)[0], rtol=1e-13, atol=1e-300)
    assert np.allclose(wv[1], sc1.weights(0, T.SR_WEIGHT_ADAPTIVE, 2, cx, cy)[0], rtol=1e-13, atol=1e-300)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fix_index", [True, False])
def test_refraction_calibration_matches_oracle(tmp_path, fix_index):
    """RefractionCalibration::calibrate (stereo/refractioncalibration.cpp:289-404; util/lm.cpp): the C++
    class — LM loop on the host, every residual from sr_calibration_residuals_batch — against the
    oracle's literal point-by-point restatement of the same loops on the same correspondences."""
    from oracle import oracle_api as O
    from calib_util import calibration_problem
    cams, pairs, pix, truth, start = calibration_problem(O.Scene)
    V, n = len(cams), len(pairs)
    h, w = 480, 640
    blank = [np.zeros((h, w, 4), np.uint8)] * V
    xml = write_project(str(tmp_path), cams, blank, [np.full((h, w), 255, np.uint8)] * V)
    fixed = np.zeros(truth.size, np.uint8)
    fixed[0] = fix_index  # the GUI always fixes the refractive index (stereowidget.cpp:577-578)

    def run(flags, model):
        prob = os.path.join(str(tmp_path), f"problem{flags}.bin")
        with open(prob, "wb") as f:
            f.write(np.array([n, flags], np.int32).tobytes())
            f.write(np.ascontiguousarray(pairs, np.int32).tobytes())
            f.write(np.ascontiguousarray(pix, np.float64).tobytes())
            f.write(np.ascontiguousarray(model, np.float64).tobytes())
            f.write(fixed.tobytes())
        r = subprocess.run([HARNESS, "--calibrate", xml, prob, str(tmp_path)], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        out = np.fromfile(os.path.join(str(tmp_path), "calib.bin"), dtype=np.float64)
        return out[:truth.size], out[truth.size:]

    # the cameras the harness loads from the XML carry the true interface: the model is what decides
    gm, (it, c0, c1, total, avg, err0, ok, _restored) = run(0, start)
    om, oit, oc0, oc1 = O.calibration_lm(cams, pairs, pix, start, fixed)
    assert ok == 1.0
    assert it == oit and it >= 5
    # (finite differences with steps down to 1e-4 amplify the ~1e-12 residual differences between the GPU and the
    # oracle, and the normal's pixel x is weakly determined: a 1e-13 relative change of the input pixels moves
    # the oracle's own answer by 1e-6)
    assert abs(c0 - oc0) <= 1e-9 * oc0 and abs(c1 - oc1) <= 1e-5 * oc1
    assert c1 < 1e-2 * c0                      # it calibrates: chi^2 drops by orders of magnitude ...
    assert np.allclose(gm, om, rtol=1e-5, atol=1e-3)
    assert abs(total - c1) <= 1e-12 * c1 and abs(avg - total / n) <= 1e-12 * avg
    res = O.calibration_residuals(_with_model(cams, om), pairs[:1], pix[:1])
    assert abs(err0 - abs(res[0])) <= 1e-4 * max(1.0, abs(res[0]))
    py_err = np.abs(gm - truth)[2::3]
    assert (py_err < 2.0).all()                # ... and the well-determined parameters are recovered

    # the reference's text as written: its gradient attribution leaves H singular, nothing is accepted
    gm2, (it2, c0b, c1b, *_rest) = run(1, start)
    om2, oit2, _, oc1b = O.calibration_lm(cams, pairs, pix, start, fixed, exact_attribution=False)
    assert (gm2 == start).all() and (om2 == start).all() and it2 == oit2 and c1b == c0b
    # ... and its solve test skips every successful solve
    gm3, (it3, *_r3) = run(2, start)
    om3, oit3, _, _ = O.calibration_lm(cams, pairs, pix, start, fixed, literal_check=True)
    assert (gm3 == start).all() and (om3 == start).all() and it3 == oit3 == 5


def _with_model(cams, model):
    """Cameras re-configured as RefractiveCalibrationFunction::update does (:238-251)."""
    import copy
    out = []
    for v, c in enumerate(cams):
        c = copy.copy(c)
        Kinv = np.array(c.Kinv[:]).reshape(3, 3)
        nrm = Kinv @ np.array([model[3 * v + 1], model[3 * v + 2], 1.0])
        nrm /= np.linalg.norm(nrm)
        for i in range(3):
            c.plane_n[i] = nrm[i]
        c.plane_d = model[3 * v + 3]
        c.n = model[0]
        out.append(c)
    return out


def bunny_cameras():
    """The 8 cameras of the reference's example/project.xml (tests/golden/bunny/cameras.json)."""
    import json
    from bunny_util import DIR
    meta = json.load(open(os.path.join(DIR, "cameras.json")))
    return [T.camera_from_P(c["P"], dist=c["dist"]) for c in meta["cameras"]]


def projection_matrices(cams):
    """What write_project puts into the XML for each camera."""
    out = []
    for c in cams:
        K, R, t = (np.array(getattr(c, f)[:]) for f in ("K", "R", "t"))
        out.append(K.reshape(3, 3) @ np.hstack([R.reshape(3, 3), t[:, None]]))
    return out


def test_host_camera_class_matches_reference_camera(tmp_path):
    """CPU: the C++ `Project` + `Camera` classes of include/ (XML -> Camera::setP -> updateOthers -> toPod) on
    the 8 cameras of the reference's example/project.xml (tests/golden/bunny/cameras.json), against the
    REFERENCE'S OWN Camera::setP (project/camera.cpp compiled where it lies, oracle/_ref): K, R, t, C, the
    principal ray and the inverses agree to rounding.  Where oracle/_ref is not built, the comparison is with
    tests/golden/ref_pins/host_cameras.npz, which holds this C++ Camera class's own output from when it agreed
    with the reference (tests/golden/make_ref_pins.py): a regression pin, not an independent check."""
    from oracle import oracle_api as O
    REF = O.ref_lib()
    cams = bunny_cameras()
    n = C.sizeof(T.SrCamera)
    if REF is not None:
        refs = []
        for P in projection_matrices(cams):
            ref = O.OrcCamera()
            REF.ref_camera_from_P(np.ascontiguousarray(P).ctypes.data_as(C.POINTER(C.c_double)), C.byref(ref))
            refs.append(ref)
    else:
        buf = np.load(os.path.join(ROOT, "tests", "golden", "ref_pins", "host_cameras.npz"))["cams"].tobytes()
        refs = [O.OrcCamera.from_buffer_copy(buf[i * n:(i + 1) * n]) for i in range(len(buf) // n)]
    assert len(refs) == len(cams)
    h, w = 8, 8
    blank = [np.zeros((h, w, 4), np.uint8)] * len(cams)
    xml = write_project(str(tmp_path), cams, blank, [np.full((h, w), 255, np.uint8)] * len(cams))
    r = subprocess.run([HARNESS, "--cameras", xml, str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = open(os.path.join(str(tmp_path), "cams.bin"), "rb").read()
    assert len(raw) == n * len(cams)
    for i, (c, ref) in enumerate(zip(cams, refs)):
        host = T.SrCamera.from_buffer_copy(raw[i * n:(i + 1) * n])
        for f in ("K", "Kinv", "R", "Rinv", "t", "C", "prin_dir"):
            a, b = np.array(getattr(host, f)[:]), np.array(getattr(ref, f)[:])
            assert np.allclose(a, b, rtol=1e-9, atol=1e-9), (i, f, np.abs(a - b).max())
        assert host.is_distorted == 1 and np.allclose(np.array(host.dist[:]), np.array(c.dist[:]), rtol=0, atol=1e-15)
