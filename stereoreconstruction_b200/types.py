"""POD structs of the C ABI (include/sr_b200.h) as ctypes Structures, plus the host-side
camera derivations of the reference's Camera class (project/camera.cpp) in numpy.

These are *inputs* to the hot path (the reference's Project/ImageSet/Camera data model,
SURVEY.md §8b); nothing here computes matching costs.
"""
import ctypes as C

import numpy as np

SR_WEIGHT_ADAPTIVE, SR_WEIGHT_GEODESIC = 0, 1
SR_COST_NCC_TWOVIEW, SR_COST_NCC_MVS, SR_COST_SAD_TWOVIEW = 0, 1, 2
SR_DEPTH_LINEAR, SR_DEPTH_INV5 = 0, 1
SR_SELECT_TWOVIEW, SR_SELECT_MVS = 0, 1
SR_INDEX_NONE, SR_INDEX_MASKED, SR_INDEX_REJECTED = -1, -2, -3


class SrCamera(C.Structure):
    _fields_ = [
        ("K", C.c_double * 9), ("Kinv", C.c_double * 9), ("R", C.c_double * 9),
        ("Rinv", C.c_double * 9), ("t", C.c_double * 3), ("C", C.c_double * 3),
        ("dist", C.c_double * 5), ("plane_n", C.c_double * 3), ("plane_d", C.c_double),
        ("n", C.c_double), ("prin_dir", C.c_double * 3),
        ("is_refractive", C.c_int32), ("is_distorted", C.c_int32),
    ]


class SrParams(C.Structure):
    _fields_ = [
        ("min_depth", C.c_double), ("max_depth", C.c_double), ("num_levels", C.c_int32),
        ("image_scale", C.c_double), ("radius", C.c_int32), ("weight_kind", C.c_int32),
        ("cost_kind", C.c_int32), ("depth_kind", C.c_int32), ("select_kind", C.c_int32),
        ("second_best_factor", C.c_double), ("ncc_threshold", C.c_double),
        ("keep_cost_volume", C.c_int32), ("row_begin", C.c_int32), ("row_end", C.c_int32),
    ]


class SrMrfParams(C.Structure):
    _fields_ = [
        ("iterations", C.c_int32), ("unknown_cost", C.c_double), ("smooth_weight", C.c_double),
        ("smooth_trunc", C.c_double), ("unknown_pair", C.c_double),
    ]


def default_params(multi_view, min_depth=10.0, max_depth=100.0, num_levels=100, **kw):
    """File-scope constants of the reference: two-view r=5 (stereo/twoviewstereo.cpp:64-80),
    MVS r=2 (stereo/multiviewstereo.cpp:90-102); both typedef GeodesicWeight."""
    p = SrParams()
    p.min_depth, p.max_depth, p.num_levels = min_depth, max_depth, num_levels
    p.image_scale = 1.0
    p.weight_kind = SR_WEIGHT_GEODESIC
    p.second_best_factor = 0.95
    p.ncc_threshold = 0.95
    p.keep_cost_volume = 0
    p.row_begin, p.row_end = 0, 0
    if multi_view:
        p.radius, p.cost_kind, p.depth_kind, p.select_kind = 2, SR_COST_NCC_MVS, SR_DEPTH_LINEAR, SR_SELECT_MVS
    else:
        p.radius, p.cost_kind, p.depth_kind, p.select_kind = 5, SR_COST_NCC_TWOVIEW, SR_DEPTH_INV5, SR_SELECT_TWOVIEW
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def _orthonormalize(M):
    """Gram-Schmidt on columns + tiny->0, project/camera.cpp:143-165."""
    M = np.array(M, dtype=np.float64)
    for i in range(3):
        accum = np.zeros(3)
        for j in range(i):
            vi, vj = M[:, i].copy(), M[:, j].copy()
            accum += vj * (vi.dot(vj) / vj.dot(vj))
        M[:, i] -= accum
        M[:, i] /= np.linalg.norm(M[:, i])
    M[np.abs(M) < 1e-10] = 0.0
    return M


def _inv3(M):
    """Closed-form 3x3 inverse (cofactors), as Eigen's Matrix3d::inverse()."""
    M = np.asarray(M, dtype=np.float64)
    c = np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            r = [k for k in range(3) if k != i]
            s = [k for k in range(3) if k != j]
            c[i, j] = (-1) ** (i + j) * (M[r[0], s[0]] * M[r[1], s[1]] - M[r[0], s[1]] * M[r[1], s[0]])
    det = M[0, 0] * c[0, 0] + M[0, 1] * c[0, 1] + M[0, 2] * c[0, 2]
    return c.T / det


def make_camera(K, R, t, dist=None, plane_normal=None, plane_d=0.0, n=1.0):
    """Camera::set(K,R,t) + setLensDistortion + setRefractiveIndex + setPlane
    (project/camera.cpp:205-222, 292-342)."""
    cam = SrCamera()
    K = np.array(K, dtype=np.float64).reshape(3, 3)
    R = _orthonormalize(np.array(R, dtype=np.float64).reshape(3, 3))
    t = np.array(t, dtype=np.float64).reshape(3)
    Kinv = _inv3(K)
    Rinv = R.T.copy()
    Cc = Rinv @ (-t)
    # updatePrincipleRay, camera.cpp:292-298
    tcol = K[:, 2]
    d = Kinv @ (tcol / tcol[2])
    prin = Rinv @ (d / np.linalg.norm(d))
    prin = prin / np.linalg.norm(prin)  # Ray3d::setDirection normalises again (ray.hpp:41)
    cam.K[:] = K.ravel()
    cam.Kinv[:] = Kinv.ravel()
    cam.R[:] = R.ravel()
    cam.Rinv[:] = Rinv.ravel()
    cam.t[:] = t
    cam.C[:] = Cc
    dist = np.zeros(5) if dist is None else np.array(dist, dtype=np.float64)
    cam.dist[:] = dist
    cam.is_distorted = int(np.any(np.abs(dist) > 1e-10))  # camera.cpp:305-309
    if plane_normal is None:
        pn = np.array([0.0, 0.0, 1.0])
    else:
        pn = np.array(plane_normal, dtype=np.float64)
        pn = pn / np.linalg.norm(pn)  # Plane3d ctor, plane.hpp:33
    cam.plane_n[:] = pn
    cam.plane_d = float(plane_d)
    cam.n = float(n)
    cam.is_refractive = int(abs(n - 1.0) > 1e-10 and abs(plane_d) > 1e-10)  # camera.cpp:329,339
    cam.prin_dir[:] = prin
    return cam


def set_interface_px(cam, px, py, plane_d, n):
    """<refractiveInterface px py dist refractiveRatio>: normal = K^-1 (px,py,1)
    (project/project.cpp:173-181)."""
    Kinv = np.array(cam.Kinv[:]).reshape(3, 3)
    pn = Kinv @ np.array([px, py, 1.0])
    pn = pn / np.linalg.norm(pn)
    cam.plane_n[:] = pn
    cam.plane_d = float(plane_d)
    cam.n = float(n)
    cam.is_refractive = int(abs(n - 1.0) > 1e-10 and abs(plane_d) > 1e-10)
    return cam


def camera_from_P(P, dist=None):
    """Camera::setP -> updateOthers: RQ factorisation of the 3x4 projection matrix
    (project/camera.cpp:251-288)."""
    P = np.array(P, dtype=np.float64).reshape(3, 4)
    P = P / np.dot(P[2, :3], P[2, :3])  # squaredNorm, camera.cpp:252
    M = P[:, :3]
    J = np.array([[0, 0, 1.0], [0, 1.0, 0], [1.0, 0, 0]])
    Q, Rq = np.linalg.qr((J @ M).T)  # Householder, same sign convention as Eigen (beta=-sign*norm)
    R = J @ Q.T
    K = J @ Rq.T @ J
    for axis in (2, 1, 0):
        if K[axis, axis] < 0:
            K[axis, axis] = -K[axis, axis]
            R[axis, :] = -R[axis, :]
        if K[axis, 2] < 0:
            K[axis, 2] = -K[axis, 2]
    R = _orthonormalize(R)
    Kinv = _inv3(K)
    t = Kinv @ P[:, 3]
    return make_camera(K, R, t, dist=dist)
