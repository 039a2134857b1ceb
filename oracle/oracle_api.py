"""ctypes binding of the CPU oracle (oracle/oracle.cpp).

TEST INFRASTRUCTURE.  Import only from tests/, __graft_entry__.smoke() and the cpu_baseline /
--impl reference legs of bench.py.  The product package never imports this module.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_REF = None


class OrcCamera(C.Structure):
    """Same layout as include/sr_b200.h::sr_camera (kept separate on purpose)."""
    _fields_ = [
        ("K", C.c_double * 9), ("Kinv", C.c_double * 9), ("R", C.c_double * 9),
        ("Rinv", C.c_double * 9), ("t", C.c_double * 3), ("C", C.c_double * 3),
        ("dist", C.c_double * 5), ("plane_n", C.c_double * 3), ("plane_d", C.c_double),
        ("n", C.c_double), ("prin_dir", C.c_double * 3),
        ("is_refractive", C.c_int32), ("is_distorted", C.c_int32),
    ]


class OrcParams(C.Structure):
    """Same layout as include/sr_b200.h::sr_params."""
    _fields_ = [
        ("min_depth", C.c_double), ("max_depth", C.c_double), ("num_levels", C.c_int32),
        ("image_scale", C.c_double), ("radius", C.c_int32), ("weight_kind", C.c_int32),
        ("cost_kind", C.c_int32), ("depth_kind", C.c_int32), ("select_kind", C.c_int32),
        ("second_best_factor", C.c_double), ("ncc_threshold", C.c_double),
        ("keep_cost_volume", C.c_int32), ("row_begin", C.c_int32), ("row_end", C.c_int32),
    ]


def _cpu_stamp():
    try:
        with open("/proc/cpuinfo") as f:
            txt = f.read()
        flags = [l for l in txt.splitlines() if l.startswith("flags")][:1]
        model = [l for l in txt.splitlines() if l.startswith("model name")][:1]
        return hashlib.sha1(("".join(model + flags)).encode()).hexdigest()
    except OSError:
        return "unknown"


def build(verbose=False):
    """Compile the oracle (and oracle/_ref when REF names the reference's source tree, see Makefile).  -march=native is used,
    so the library is rebuilt when the host CPU differs from the one it was built on."""
    os.makedirs(os.path.join(_HERE, "_build"), exist_ok=True)
    stamp = os.path.join(_HERE, "_build", "cpu.stamp")
    cur = _cpu_stamp()
    old = None
    if os.path.exists(stamp):
        with open(stamp) as f:
            old = f.read().strip()
    if old != cur:
        with open(stamp, "w") as f:
            f.write(cur)
    env = dict(os.environ)
    env.pop("CXX", None)
    r = subprocess.run(["make", "-C", _HERE, "all"], capture_output=True, text=True, env=env)
    if verbose or r.returncode != 0:
        print(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)


def lib():
    global _LIB
    if _LIB is None:
        build()
        L = C.CDLL(os.path.join(_HERE, "_build", "liboracle.so"))
        L.orc_scene_create.restype = C.c_void_p
        L.orc_cost.restype = C.c_double
        L.orc_depth_from_label.restype = C.c_double
        L.orc_snell_root.restype = C.c_double
        L.orc_snell_root.argtypes = [C.c_double] * 4
        _LIB = L
    return _LIB


def ref_lib():
    """The reference's own sources compiled from its source tree (oracle/_ref/libref.so), or
    None when neither the reference tree nor a prebuilt library is available."""
    global _REF
    if _REF is None:
        build()
        p = os.path.join(_HERE, "_ref", "libref.so")
        if not os.path.exists(p):
            return None
        _REF = C.CDLL(p)
    return _REF


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def as_cam_array(cams):
    arr = (OrcCamera * len(cams))()
    for i, c in enumerate(cams):
        C.memmove(C.byref(arr[i]), C.byref(c), C.sizeof(OrcCamera))
    return arr


def as_params(p):
    q = OrcParams()
    C.memmove(C.byref(q), C.byref(p), C.sizeof(OrcParams))
    return q


class Scene:
    """V views (camera POD + RGBA8 image + mask byte plane) held by the oracle."""

    def __init__(self, cams, images, masks=None):
        L = lib()
        self.V = len(cams)
        self.h, self.w = images[0].shape[:2]
        self._imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        self._masks = None
        img_ptrs = (C.c_void_p * self.V)(*[im.ctypes.data for im in self._imgs])
        mask_ptrs = None
        if masks is not None:
            self._masks = [np.ascontiguousarray(m, dtype=np.uint8) for m in masks]
            mask_ptrs = (C.c_void_p * self.V)(*[m.ctypes.data for m in self._masks])
        self._cams = as_cam_array(cams)
        self.ptr = C.c_void_p(L.orc_scene_create(self.V, self._cams, img_ptrs, mask_ptrs, self.w, self.h))

    def __del__(self):
        try:
            lib().orc_scene_destroy(self.ptr)
        except Exception:
            pass

    def cam(self, i):
        return self._cams[i]

    # -- leaves ------------------------------------------------------------------------
    def unproject_grid(self, view, scale=1.0):
        out = np.empty((self.h, self.w, 6), dtype=np.float64)
        lib().orc_unproject_grid(C.byref(self._cams[view]), self.w, self.h, C.c_double(scale), _dp(out))
        return out

    def project_points(self, view, xyz, root_mode=1):
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        n = xyz.shape[0]
        xy = np.empty((n, 2), dtype=np.float64)
        ok = np.empty(n, dtype=np.int32)
        lib().orc_project_points(C.byref(self._cams[view]), n, _dp(xyz), root_mode, _dp(xy), _ip(ok))
        return xy, ok

    def weights(self, view, kind, radius, cx, cy):
        cx = np.ascontiguousarray(cx, dtype=np.int32)
        cy = np.ascontiguousarray(cy, dtype=np.int32)
        wn = 2 * radius + 1
        out = np.empty((cx.size, wn, wn), dtype=np.float64)
        lib().orc_weights(self.ptr, view, kind, radius, cx.size, _ip(cx), _ip(cy), _dp(out))
        return out

    def cost(self, params, va, vb, x1, y1, x2, y2):
        p = as_params(params)
        return lib().orc_cost(self.ptr, C.byref(p), va, vb, int(x1), int(y1), int(x2), int(y2))

    def epipolar_curve(self, params, ref, nbr, x, y, mvs, root_mode=1, max_pts=1 << 16):
        p = as_params(params)
        out = np.empty((max_pts, 2), dtype=np.int32)
        n = lib().orc_epipolar_curve(self.ptr, C.byref(p), ref, nbr, x, y, int(mvs), root_mode, _ip(out), max_pts)
        return out[:min(n, max_pts)].copy()

    # -- the path ----------------------------------------------------------------------
    def twoview_label(self, params, a, b, root_mode=1, want_volume=False):
        p = as_params(params)
        h, w = self.h, self.w
        r0 = max(p.row_begin, 0)
        r1 = p.row_end if 0 < p.row_end < h else h
        depth = np.full((h, w), np.nan)
        index = np.full((h, w), -2, dtype=np.int32)
        best = np.full((h, w), np.nan)
        vol = np.empty((r1 - r0, w, p.num_levels)) if want_volume else None
        lib().orc_twoview_label(self.ptr, C.byref(p), a, b, root_mode, _dp(depth), _ip(index), _dp(best),
                                _dp(vol) if want_volume else None)
        return depth, index, best, vol

    def twoview_curve(self, params, a, b, root_mode=1):
        p = as_params(params)
        h, w = self.h, self.w
        depth = np.full((h, w), np.nan)
        best = np.full((h, w), np.nan)
        count = np.zeros((h, w), dtype=np.int32)
        lib().orc_twoview_curve(self.ptr, C.byref(p), a, b, root_mode, _dp(depth), _dp(best), _ip(count))
        return depth, best, count

    def mvs_view(self, params, ref, nbrs, curve_mode=False, root_mode=1, want_volume=False, want_peaks=False):
        p = as_params(params)
        h, w = self.h, self.w
        r0 = max(p.row_begin, 0)
        r1 = p.row_end if 0 < p.row_end < h else h
        nbrs = np.ascontiguousarray(nbrs, dtype=np.int32)
        depth = np.full((h, w), np.inf)
        index = np.full((h, w), -2, dtype=np.int32)
        best = np.full((h, w), np.nan)
        vol = np.empty((nbrs.size, r1 - r0, w, p.num_levels)) if want_volume else None
        peaks = np.zeros((h, w, 9, 2)) if want_peaks else None
        lib().orc_mvs_view(self.ptr, C.byref(p), ref, _ip(nbrs), nbrs.size, int(curve_mode), root_mode,
                           _dp(depth), _ip(index), _dp(best), _dp(vol) if want_volume else None,
                           _dp(peaks) if want_peaks else None)
        return depth, index, best, vol, peaks

    def select_neighbours(self, max_n=3):
        out = np.full((self.V, max_n), -1, dtype=np.int32)
        counts = np.zeros(self.V, dtype=np.int32)
        lib().orc_select_neighbours(self.ptr, max_n, _ip(out), _ip(counts))
        return [list(out[i, :counts[i]]) for i in range(self.V)]

    def crosscheck_two(self, params, l, r, depth_l, depth_r, thresh=1.0, root_mode=1):
        p = as_params(params)
        dl = np.array(depth_l, dtype=np.float64, order="C")
        dr = np.array(depth_r, dtype=np.float64, order="C")
        lib().orc_crosscheck_two(self.ptr, C.byref(p), l, r, _dp(dl), _dp(dr), C.c_double(thresh), root_mode)
        return dl, dr

    def crosscheck_mvs(self, params, depths, thresh, root_mode=1, snapshot=False):
        p = as_params(params)
        ds = [np.array(d, dtype=np.float64, order="C") for d in depths]
        ptrs = (C.c_void_p * self.V)(*[d.ctypes.data for d in ds])
        lib().orc_crosscheck_mvs(self.ptr, C.byref(p), ptrs, C.c_double(thresh), root_mode, int(snapshot))
        return ds


def calibration_residuals(cams, pairs, pixels):
    """RefractiveCalibrationFunction::diff (stereo/refractioncalibration.cpp:175-201) per correspondence."""
    pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    pixels = np.ascontiguousarray(pixels, dtype=np.float64).reshape(-1, 4)
    out = np.empty(pairs.shape[0], dtype=np.float64)
    lib().orc_calibration_residuals(as_cam_array(cams), pairs.shape[0], _ip(pairs), _dp(pixels), _dp(out))
    return out


def calibration_lm(cams, pairs, pixels, model, fixed, max_iterations=100, epsilon=1.0, literal_check=False,
                   exact_attribution=True):
    """RefractionCalibration::calibrate (stereo/refractioncalibration.cpp:363-378): util/lm.cpp's loop around
    the residual above.  model = [n, (px, py, dist) x V].  Returns (model, iterations, chi2_before, chi2_after)."""
    pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    pixels = np.ascontiguousarray(pixels, dtype=np.float64).reshape(-1, 4)
    m = np.array(model, dtype=np.float64)
    fx = np.ascontiguousarray(fixed, dtype=np.uint8)
    assert m.size == 1 + 3 * len(cams) == fx.size
    chi = np.zeros(2)
    L = lib()
    L.orc_calibration_lm.restype = C.c_int
    it = L.orc_calibration_lm(as_cam_array(cams), len(cams), pairs.shape[0], _ip(pairs), _dp(pixels), _dp(m),
                              fx.ctypes.data_as(C.c_void_p), int(max_iterations), C.c_double(epsilon),
                              int(literal_check), int(exact_attribution), _dp(chi))
    return m, it, chi[0], chi[1]


class RefMVS:
    """The REFERENCE'S OWN MultiViewStereo (stereo/multiviewstereo.cpp compiled where it lies into
    oracle/_ref/libref.so, see ref_glue_mvs.cpp), driven as the GUI drives it: initialize() ->
    runTask().  images: RGBA8 (h,w,4); masks: uint8 (h,w), 255 = WHITE, written into the alpha byte
    the reference reads its mask from."""

    def __init__(self, cams, images, masks, min_depth, max_depth, num_levels, cross_check, image_scale=1.0, adaptive=False):
        """adaptive=True: the build of the same reference file whose `WeightFunc` typedef names AdaptiveWeight
        (ref_glue_mvs_ada.cpp) instead of GeodesicWeight."""
        self.R = ref_lib()
        if self.R is None:
            raise RuntimeError("oracle/_ref/libref.so is not available")
        self._p = "ref_mvsa_" if adaptive else "ref_mvs_"
        self.V = len(cams)
        self.h, self.w = images[0].shape[:2]
        self._rgba = []
        for im, m in zip(images, masks if masks is not None else [None] * self.V):
            a = np.ascontiguousarray(im, dtype=np.uint8).copy()
            a[..., 3] = 255 if m is None else m
            self._rgba.append(a)
        ptrs = (C.c_void_p * self.V)(*[a.ctypes.data for a in self._rgba])
        self._f('create').restype = C.c_void_p
        self._h = C.c_void_p(self._f('create')(self.V, as_cam_array(cams), ptrs, self.w, self.h, C.c_double(min_depth),
                                                   C.c_double(max_depth), int(num_levels), C.c_double(cross_check),
                                                   C.c_double(image_scale)))
        assert self._f('num_views')(self._h) == self.V

    def _f(self, name):
        return getattr(self.R, self._p + name)

    def close(self):
        if self._h:
            self._f('destroy')(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self):
        """runTask(): (depths after the cross-check (V,h,w), neighbour lists)."""
        after = np.empty((self.V, self.h, self.w))
        nb = np.empty((self.V, 3), np.int32)
        self._f('run')(self._h, _dp(after), _ip(nb))
        return after, [[int(v) for v in row if v >= 0] for row in nb]

    def initial_estimate(self, view):
        """computeInitialEstimate(view) (call run() first: it selects the neighbours): depths before
        the cross-check (h,w) and the K = 9 peak pairs (h,w,9,2)."""
        d = np.empty((self.h, self.w))
        pk = np.empty((self.h, self.w, 9, 2))
        self._f('initial_estimate')(self._h, int(view), _dp(d), _dp(pk))
        return d, pk

    def set_neighbours(self, view, nbrs):
        nb = np.ascontiguousarray(nbrs, dtype=np.int32)
        self._f('set_neighbours')(self._h, int(view), _ip(nb), int(nb.size))

    def mask_rows(self, view, row_begin, row_end):
        """Reduce the view's mask to rows [row_begin, row_end): the class skips pixels outside its mask."""
        self._f('mask_rows')(self._h, int(view), int(row_begin), int(row_end))

    def num_threads(self):
        return self._f('num_threads')()

    def cost_ncc(self, a, b, x1, y1, x2, y2):
        self._f('cost_ncc').restype = C.c_double
        return self._f('cost_ncc')(self._h, a, b, int(x1), int(y1), int(x2), int(y2))

    def curve(self, a, b, x, y, max_pts=1 << 14):
        out = np.empty((max_pts, 2), np.int32)
        n = self._f('curve')(self._h, a, b, int(x), int(y), _ip(out), max_pts)
        return out[:min(n, max_pts)].copy()


class RefTwoView:
    """The REFERENCE'S OWN TwoViewStereo (stereo/twoviewstereo.cpp compiled where it lies, ref_glue_two.cpp):
    constructor -> computeCostVolumes / computeDepthMaps.  masks: uint8 (h,w) with 255 = WHITE, or None
    (the null QImage the reference treats as all-WHITE)."""

    def __init__(self, cam_l, cam_r, img_l, img_r, mask_l, mask_r, min_depth, max_depth, num_levels, image_scale=1.0):
        self.R = ref_lib()
        if self.R is None:
            raise RuntimeError("oracle/_ref/libref.so is not available")
        self.h, self.w = img_l.shape[:2]
        self._keep = [np.ascontiguousarray(img_l, np.uint8), np.ascontiguousarray(img_r, np.uint8),
                      None if mask_l is None else np.ascontiguousarray(mask_l, np.uint8),
                      None if mask_r is None else np.ascontiguousarray(mask_r, np.uint8)]
        vp = [C.c_void_p(a.ctypes.data) if a is not None else None for a in self._keep]
        self.R.ref_two_create.restype = C.c_void_p
        self._h = C.c_void_p(self.R.ref_two_create(as_cam_array([cam_l]), as_cam_array([cam_r]), vp[0], vp[1], vp[2], vp[3],
                                                   self.w, self.h, C.c_double(min_depth), C.c_double(max_depth),
                                                   int(num_levels), C.c_double(image_scale)))

    def close(self):
        if self._h:
            self.R.ref_two_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _two(self, fn):
        l, r = np.empty((self.h, self.w)), np.empty((self.h, self.w))
        fn(self._h, _dp(l), _dp(r))
        return l, r

    def search(self):
        """computeCostVolumes: (left, right) depths before the cross-check."""
        return self._two(self.R.ref_two_search)

    def run(self):
        """computeDepthMaps: search + cross-check."""
        return self._two(self.R.ref_two_run)

    def cost(self, sad, direction, x1, y1, x2, y2):
        self.R.ref_two_cost.restype = C.c_double
        return self.R.ref_two_cost(self._h, int(sad), int(direction), int(x1), int(y1), int(x2), int(y2))


def stats_reset():
    lib().orc_stats_reset()


def stats():
    out = (C.c_longlong * 5)()
    md = C.c_double()
    lib().orc_stats_get(out, C.byref(md))
    return {"project_calls": out[0], "quartic_fail": out[1], "root_mismatch": out[2],
            "no_root": out[3], "max_root_diff": md.value}


def num_threads():
    return lib().orc_num_threads()
