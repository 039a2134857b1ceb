"""ctypes binding of the C ABI (include/sr_b200.h) — used by the parity tests and bench.py.

The product is the CUDA library; this module only marshals numpy arrays across the ABI.  It
fails loudly when the library is missing or no CUDA device is present: there is no fallback.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from .types import SrCamera, SrParams

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SR_LIB") or os.path.join(_PKG, "libsr_b200.so")  # SR_LIB: A/B kernel variants
_LIB = None

NVCC_FLAGS = ["-std=c++17", "-O3", "-fmad=false", "-DSR_FEW_RADII", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "--shared", "-Xcompiler", "-fPIC"]
SOURCES = ["csrc/sr_capi.cu"]
HEADERS = ["csrc/" + f for f in sorted(os.listdir(os.path.join(_PKG, "csrc"))) if f.endswith(".cuh")] + ["../include/sr_b200.h"]

EXPORTS = [
    "sr_ctx_create", "sr_ctx_destroy", "sr_last_error", "sr_request_cancel", "sr_clear_cancel",
    "sr_set_stream", "sr_params_default", "sr_launch_count", "sr_set_profiling", "sr_get_stage_ms", "sr_get_match_stats", "sr_get_build_stats", "sr_set_views", "sr_set_params",
    "sr_run_view", "sr_run_view_curve", "sr_select_neighbours", "sr_cross_check", "sr_flush", "sr_synchronize",
    "sr_get_depth_index", "sr_get_depth", "sr_get_best_cost", "sr_get_cost_volume", "sr_get_peaks", "sr_set_depth",
    "sr_get_depth_image", "sr_get_points", "sr_unproject_grid", "sr_project_points", "sr_compute_weights", "sr_calibration_residuals",
    "sr_calibration_residuals_batch",
    "sr_comm_unique_id", "sr_comm_init", "sr_comm_allgather_views", "sr_comm_allgather_rows",
]


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(os.path.join(_PKG, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> stereoreconstruction_b200/libsr_b200.so
    (in-tree, so the built library travels with the repository snapshot)."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + ["-o", LIB_PATH] + [os.path.join(_PKG, s) for s in SOURCES] + ["-lcudart", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(" ".join(cmd))
        print(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.sr_last_error.restype = C.c_char_p
        L.sr_last_error.argtypes = [C.c_void_p]
        L.sr_launch_count.restype = C.c_int64
        L.sr_launch_count.argtypes = [C.c_void_p]
        L.sr_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.sr_ctx_destroy.argtypes = [C.c_void_p]
        L.sr_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.sr_get_cost_volume.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.sr_get_points.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.POINTER(C.c_int64)]
        _LIB = L
    return _LIB


class SrError(RuntimeError):
    pass


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """One sr_ctx (one CUDA device)."""

    def __init__(self, device=0):
        self._L = lib()
        self._h = C.c_void_p()
        rc = self._L.sr_ctx_create(int(device), C.byref(self._h))
        if rc != 0:
            raise SrError(f"sr_ctx_create failed ({rc}): {self._L.sr_last_error(None).decode()}")
        self.V = self.w = self.h = 0
        self.params = None
        self._keep = []

    def close(self):
        if self._h:
            self._L.sr_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise SrError(f"sr error {rc}: {self._L.sr_last_error(self._h).decode()}")

    def calibration_residuals(self, cams, pairs, pixels):
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        pixels = np.ascontiguousarray(pixels, dtype=np.float64).reshape(-1, 4)
        out = np.empty(pairs.shape[0], dtype=np.float64)
        arr = (SrCamera * len(cams))(*cams)
        self._ck(self._L.sr_calibration_residuals(self._h, len(cams), arr, pairs.shape[0], _p(pairs), _p(pixels), _p(out)))
        return out

    def calibration_residuals_batch(self, cam_sets, pairs, pixels):
        """cam_sets: M lists of the same number of cameras -> (M, n) residuals in one launch."""
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        pixels = np.ascontiguousarray(pixels, dtype=np.float64).reshape(-1, 4)
        M, V = len(cam_sets), len(cam_sets[0])
        out = np.empty((M, pairs.shape[0]), dtype=np.float64)
        arr = (SrCamera * (M * V))(*[c for cs in cam_sets for c in cs])
        self._ck(self._L.sr_calibration_residuals_batch(self._h, M, V, arr, pairs.shape[0], _p(pairs), _p(pixels), _p(out)))
        return out

    def peaks(self, view):
        out = np.empty((self.h, self.w, 9, 2), dtype=np.float64)
        self._ck(self._L.sr_get_peaks(self._h, int(view), _p(out)))
        return out

    def build_stats(self):
        out = np.zeros(4, np.uint64)
        self._ck(self._L.sr_get_build_stats(self._h, _p(out)))
        return dict(interpolated=int(out[0]), guard_fallbacks=int(out[1]), tap_mismatches=int(out[2]))

    def match_stats(self):
        """Counters of sr_get_match_stats.  prescreen_false_drops is slot 7, reserved and always 0 since the
        subset-bound sweep it counted was removed; the key stays so that callers reading it keep working."""
        out = np.zeros(8, np.uint64)
        self._ck(self._L.sr_get_match_stats(self._h, _p(out)))
        return dict(pixels=int(out[0]), screened=int(out[1]), forced=int(out[2]), verified=int(out[3]),
                    fp64_only_pixels=int(out[4]),
                    max_screen_err=float(np.array([out[5]], np.uint64).view(np.uint32)[0:1].view(np.float32)[0]),
                    outside_error_bar=int(out[6]), prescreen_false_drops=int(out[7]))

    # -- setup -------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(self._L.sr_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def set_views(self, cams, images, masks=None):
        V = len(cams)
        h, w = next(im for im in images if im is not None).shape[:2]
        imgs = [None if im is None else np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        for im in imgs:
            assert im is None or im.shape == (h, w, 4)
        arr = (SrCamera * V)(*cams)
        ip = (C.c_void_p * V)(*[None if im is None else im.ctypes.data for im in imgs])  # None: camera only
        mp = None
        ms = None
        if masks is not None:
            ms = [None if m is None else np.ascontiguousarray(m, dtype=np.uint8) for m in masks]
            mp = (C.c_void_p * V)(*[None if m is None else m.ctypes.data for m in ms])
        self._ck(self._L.sr_set_views(self._h, V, arr, ip, mp, w, h))
        self._keep = [imgs, ms]
        self.V, self.w, self.h = V, w, h

    def set_params(self, params):
        self.params = SrParams.from_buffer_copy(params)
        self._ck(self._L.sr_set_params(self._h, C.byref(self.params)))

    # -- the path ------------------------------------------------------------------------
    def run_view(self, ref, nbrs):
        nb = np.ascontiguousarray(nbrs, dtype=np.int32)
        self._ck(self._L.sr_run_view(self._h, int(ref), _p(nb), int(nb.size)))

    def run_view_curve(self, ref, nbrs):
        nb = np.ascontiguousarray(nbrs, dtype=np.int32)
        self._ck(self._L.sr_run_view_curve(self._h, int(ref), _p(nb), int(nb.size)))

    def select_neighbours(self, max_n=3):
        out = np.full((self.V, max_n), -1, dtype=np.int32)
        cnt = np.zeros(self.V, dtype=np.int32)
        self._ck(self._L.sr_select_neighbours(self._h, max_n, _p(out), _p(cnt)))
        return [[int(v) for v in out[i, :cnt[i]]] for i in range(self.V)]

    def cross_check(self, two_view, threshold):
        self._ck(self._L.sr_cross_check(self._h, int(two_view), C.c_double(threshold)))

    def flush(self):
        """Orders every view enqueued so far before the context stream (no host synchronisation)."""
        self._ck(self._L.sr_flush(self._h))

    def synchronize(self):
        self._ck(self._L.sr_synchronize(self._h))

    def launch_count(self):
        return int(self._L.sr_launch_count(self._h))

    def set_profiling(self, on):
        self._ck(self._L.sr_set_profiling(self._h, int(on)))

    def stage_ms(self):
        out = (C.c_double * 4)()
        self._ck(self._L.sr_get_stage_ms(self._h, out))
        return {"build_ms": out[0], "match_ms": out[1], "bands": int(out[2]), "match_launches": int(out[3])}

    # -- results -------------------------------------------------------------------------
    def depth_index(self, view, out=None):
        out = np.empty((self.h, self.w), dtype=np.int32) if out is None else out
        self._ck(self._L.sr_get_depth_index(self._h, view, _p(out)))
        return out

    def depth(self, view, out=None):
        out = np.empty((self.h, self.w), dtype=np.float64) if out is None else out
        self._ck(self._L.sr_get_depth(self._h, view, _p(out)))
        return out

    def best_cost(self, view):
        out = np.empty((self.h, self.w), dtype=np.float64)
        self._ck(self._L.sr_get_best_cost(self._h, view, _p(out)))
        return out

    def cost_volume(self, num_nbrs):
        p = self.params
        r0 = max(p.row_begin, 0)
        r1 = p.row_end if 0 < p.row_end < self.h else self.h
        out = np.empty((num_nbrs, p.num_levels, r1 - r0, self.w), dtype=np.float32)
        self._ck(self._L.sr_get_cost_volume(self._h, _p(out), out.size))
        return out

    def set_depth(self, view, depth):
        d = np.ascontiguousarray(depth, dtype=np.float64)
        self._ck(self._L.sr_set_depth(self._h, view, _p(d)))

    def depth_image(self, view, mvs=True):
        out = np.empty((self.h, self.w, 4), dtype=np.uint8)
        self._ck(self._L.sr_get_depth_image(self._h, view, int(mvs), _p(out)))
        return out

    def points(self, view):
        """The coloured point cloud of the view's depth map (sr_get_points): xyz (n, 3) float64, rgb (n, 3) uint8
        and the pixel index y * w + x (n,) int32 of every point, in row-major pixel order."""
        n = C.c_int64(0)
        self._ck(self._L.sr_get_points(self._h, int(view), 0, None, None, None, C.byref(n)))
        xyz = np.empty((n.value, 3), dtype=np.float64)
        rgb = np.empty((n.value, 3), dtype=np.uint8)
        pixel = np.empty(n.value, dtype=np.int32)
        if n.value:
            self._ck(self._L.sr_get_points(self._h, int(view), n.value, _p(xyz), _p(rgb), _p(pixel), C.byref(n)))
        return xyz, rgb, pixel

    # -- building blocks -------------------------------------------------------------------
    def unproject_grid(self, view):
        out = np.empty((self.h, self.w, 6), dtype=np.float64)
        self._ck(self._L.sr_unproject_grid(self._h, view, _p(out)))
        return out

    def project_points(self, view, xyz):
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        n = xyz.shape[0]
        xy = np.empty((n, 2), dtype=np.float64)
        ok = np.empty(n, dtype=np.int32)
        self._ck(self._L.sr_project_points(self._h, view, n, _p(xyz), _p(xy), _p(ok)))
        return xy, ok

    def weights(self, view, kind, radius, cx, cy):
        cx = np.ascontiguousarray(cx, dtype=np.int32)
        cy = np.ascontiguousarray(cy, dtype=np.int32)
        wn = 2 * radius + 1
        out = np.empty((cx.size, wn, wn), dtype=np.float64)
        self._ck(self._L.sr_compute_weights(self._h, view, kind, radius, cx.size, _p(cx), _p(cy), _p(out)))
        return out

    # -- multi-GPU ---------------------------------------------------------------------------
    @staticmethod
    def comm_unique_id():
        buf = (C.c_char * 128)()
        rc = lib().sr_comm_unique_id(buf)
        if rc != 0:
            raise SrError(f"sr_comm_unique_id failed: {lib().sr_last_error(None).decode()}")
        return bytes(buf)

    def comm_init(self, uid, rank, nranks):
        buf = (C.c_char * 128).from_buffer_copy(uid)
        self._ck(self._L.sr_comm_init(self._h, buf, rank, nranks))

    def allgather_views(self, owner):
        o = np.ascontiguousarray(owner, dtype=np.int32)
        self._ck(self._L.sr_comm_allgather_views(self._h, _p(o)))

    def allgather_rows(self, view, row_begin, row_end):
        b = np.ascontiguousarray(row_begin, dtype=np.int32)
        e = np.ascontiguousarray(row_end, dtype=np.int32)
        self._ck(self._L.sr_comm_allgather_rows(self._h, view, _p(b), _p(e)))
