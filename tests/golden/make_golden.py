#!/usr/bin/env python
"""Generates the committed golden fixtures of tests/golden/.

  REF=<reference source tree> python tests/golden/make_golden.py     (builds oracle/_ref from that tree first)

ref_leaves.npz    outputs of the REFERENCE'S OWN sources (util/lineiter.cpp, util/ray.cpp,
                  util/vectorimage.cpp, stereo/adaptiveweight.cpp, stereo/geodesicweight.cpp,
                  project/camera.cpp compiled where they lie into oracle/_ref/libref.so) on seeded inputs.  They pin the oracle
                  — and through it the CUDA path — on machines without the reference's sources.
ref_mvs.npz       END-TO-END outputs of the reference's own MultiViewStereo class (stereo/multiviewstereo.cpp
                  + project/camera.cpp + the leaves, compiled where they lie, driven initialize() ->
                  runTask() by oracle/ref_glue_mvs.cpp): neighbour lists, depths before and after the
                  cross-check, the K = 9 peak lists of one view — on the small refractive arc scene and
                  on the bunny fixture with and without the injected interface (BASELINE configs[1]).
ref_two.npz       the same for the reference's own TwoViewStereo class (stereo/twoviewstereo.cpp): both
                  directions of the live curve search before and after the cross-check, on the arc scene and
                  on the bunny pair 7310085 / 7310087 with and without the interface (BASELINE configs[0]).
oracle_scenes.npz outputs of the CPU oracle (oracle/oracle.cpp) on two small seeded scenes (a
                  masked refractive 4-view arc and a rectified pair): depth-index maps, depths,
                  winning costs, one cost volume, cross-check results.  The reference ships no
                  expected outputs (SURVEY §4), so these are regression + GPU-parity vectors.
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle_api as O  # noqa: E402
from stereoreconstruction_b200 import types as T  # noqa: E402
import golden_cases as G  # noqa: E402


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def ref_leaves():
    REF = O.ref_lib()
    if REF is None:
        raise SystemExit("oracle/_ref/libref.so is not built: run `make -C oracle REF=<reference source tree>`")
    out = {}
    # --- LineIterator / clipLine (util/lineiter.hpp:32-118, util/lineiter.cpp:44-88)
    cases, w, h = G.line_cases()
    pts, counts, clipped, clip_ok = [], [], [], []
    for (x0, y0, x1, y1) in cases:
        for clip in (0, 1):
            buf = np.empty((4096, 2), np.int32)
            n = REF.ref_line(x0, y0, x1, y1, clip, w, h, _ip(buf), 4096)
            counts.append(n)
            pts.append(buf[:n].copy())
        a = np.array([x0, y0, x1, y1], np.int32)
        clip_ok.append(REF.ref_clip_line(_ip(a), w, h))
        clipped.append(a)
    out["line_counts"] = np.array(counts, np.int32)
    out["line_points"] = np.concatenate(pts) if pts else np.zeros((0, 2), np.int32)
    out["clip_ok"] = np.array(clip_ok, np.int32)
    out["clip_out"] = np.array(clipped, np.int32)
    # --- intersect / refract / closestPoints (util/ray.cpp:53-106)
    rays = G.ray_cases()
    inter, inter_ok, refr, refr_ok, closest = [], [], [], [], []
    for (s1, d1, s2, d2, pn, pd, n) in rays:
        a = np.full(3, np.nan)
        inter_ok.append(REF.ref_intersect(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), _dp(a)))
        inter.append(a)
        b = np.empty(6)
        refr_ok.append(REF.ref_refract(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), C.c_double(n), _dp(b)))
        refr.append(b)
        c = np.empty(6)
        REF.ref_closest_points(_dp(s1), _dp(d1), _dp(s2), _dp(d2), _dp(c))
        closest.append(c)
    out["intersect"], out["intersect_ok"] = np.array(inter), np.array(inter_ok, np.int32)
    out["refract"], out["refract_ok"] = np.array(refr), np.array(refr_ok, np.int32)
    out["closest"] = np.array(closest)
    # --- VectorImage::sample / toGray, AdaptiveWeight, GeodesicWeight
    img = G.leaf_image()
    hh, ww = img.shape[:2]
    REF.ref_image_create.restype = C.c_void_p
    r = C.c_void_p(REF.ref_image_create(img.ctypes.data_as(C.c_void_p), ww, hh))
    xy = G.sample_points(ww, hh)
    samp = np.empty((len(xy), 4))
    for i, (x, y) in enumerate(xy):
        REF.ref_sample(r, C.c_double(x), C.c_double(y), _dp(samp[i]))
    out["sample"] = samp
    cx, cy = G.weight_centres(ww, hh)
    for kind in (0, 1):
        for radius in G.WEIGHT_RADII:
            wn = (2 * radius + 1) ** 2
            buf = np.empty((cx.size, wn))
            REF.ref_weights(r, kind, radius, cx.size, _ip(cx), _ip(cy), _dp(buf))
            out[f"weights_k{kind}_r{radius}"] = buf
    REF.ref_image_destroy(r)
    # --- Camera::unproject / Camera::project (project/camera.cpp:95-138,380-459)
    cams, pix, pts = G.camera_cases()
    for i, c in enumerate(cams):
        pod = O.as_cam_array([c])
        rays = np.empty((len(pix), 6))
        REF.ref_camera_unproject(pod, len(pix), _dp(pix), _dp(rays))
        xy = np.empty((len(pts[i]), 2))
        ok = np.empty(len(pts[i]), np.int32)
        REF.ref_camera_project(pod, len(pts[i]), _dp(pts[i]), _dp(xy), _ip(ok))
        out[f"cam{i}_rays"], out[f"cam{i}_xy"], out[f"cam{i}_ok"] = rays, xy, ok
    return out


def oracle_scenes():
    out = {}
    cams, imgs, ms = G.arc_scene()
    sc = O.Scene(cams, imgs, ms)
    nb = sc.select_neighbours(3)
    out["arc_neighbours"] = np.array([[int(v) for v in r] for r in nb], np.int32)
    for name, P in G.arc_mvs_params().items():
        depths = []
        for ref in range(len(cams)):
            od, oi, ob, _, _ = sc.mvs_view(P, ref, nb[ref])
            out[f"{name}_v{ref}_index"], out[f"{name}_v{ref}_depth"], out[f"{name}_v{ref}_best"] = oi, od, ob
            depths.append(od)
        if name == "arc_mvs_geo_r2":
            after = sc.crosscheck_mvs(P, depths, G.ARC_CROSS_THRESH)
            for v, d in enumerate(after):
                out[f"{name}_v{v}_crosschecked"] = d
    for name, (P, a, b) in G.arc_twoview_params().items():
        od, oi, ob, ov = sc.twoview_label(P, a, b, root_mode=1, want_volume=True)
        out[f"{name}_index"], out[f"{name}_depth"], out[f"{name}_best"] = oi, od, ob
        out[f"{name}_volume"] = np.transpose(ov, (2, 0, 1)).astype(np.float32)
    cams2, imgs2 = G.rectified_scene()
    sc2 = O.Scene(cams2, imgs2)
    P = G.rectified_params()
    for (a, b) in ((0, 1), (1, 0)):
        od, oi, ob, _ = sc2.twoview_label(P, a, b, root_mode=1)
        out[f"rect_{a}{b}_index"], out[f"rect_{a}{b}_depth"], out[f"rect_{a}{b}_best"] = oi, od, ob
    return out


def ref_mvs():
    """The reference's own MultiViewStereo (stereo/multiviewstereo.cpp through oracle/ref_glue_mvs.cpp),
    initialize() -> runTask(), on the small arc scene and on the bunny fixture (BASELINE configs[1])."""
    out = {}
    for name, (mind, maxd, D, cross) in G.REF_MVS_CASES.items():
        cams, imgs, ms, scale = G.ref_mvs_inputs(name)
        cams = G.settled_cameras(cams)
        ref = O.RefMVS(cams, imgs, ms, mind, maxd, D, cross, image_scale=scale, adaptive=G.ref_mvs_adaptive(name))
        after, nb = ref.run()
        out[f"{name}_cams"] = G.cams_to_bytes(cams)
        out[f"{name}_neighbours"] = np.array([r + [-1] * (3 - len(r)) for r in nb], np.int32)
        keep = G.ref_mvs_kept_views(name, len(cams))
        before = []
        for v in range(len(cams)):
            d, pk = ref.initial_estimate(v)
            before.append(d)
            if v == 1:
                r0, r1 = G.ref_mvs_peak_rows(name, d.shape[0])
                out[f"{name}_peaks_v1"] = pk[r0:r1]
        before = np.array(before)
        out[f"{name}_views"] = np.array(keep, np.int32)
        out[f"{name}_before"] = before[keep]
        if len(keep) == len(cams):
            # the cross-check only ever replaces a depth by NaN: the mask of those pixels IS the map after it
            nan_after = np.isnan(after)
            rebuilt = np.where(nan_after, np.nan, before)
            assert ((rebuilt == after) | (np.isnan(rebuilt) & np.isnan(after))).all()
            out[f"{name}_after_nan"] = np.packbits(nan_after)
        ref.close()
    return out


def ref_two():
    """The reference's own TwoViewStereo (stereo/twoviewstereo.cpp through oracle/ref_glue_two.cpp):
    both directions of the live curve search, before and after the cross-check."""
    out = {}
    for name, (a, b, mind, maxd, D) in G.REF_TWO_CASES.items():
        cams, imgs, ms, scale = G.ref_mvs_inputs(name)
        cams = G.settled_cameras([cams[a], cams[b]])
        ref = O.RefTwoView(cams[0], cams[1], imgs[a], imgs[b], ms[a], ms[b], mind, maxd, D, image_scale=scale)
        bl, br = ref.search()
        al, ar = ref.run()
        ref.close()
        out[f"{name}_cams"] = G.cams_to_bytes(cams)
        out[f"{name}_before"] = np.array([bl, br])
        out[f"{name}_after"] = np.array([al, ar])
    return out


if __name__ == "__main__":
    O.build()
    np.savez_compressed(os.path.join(HERE, "ref_two.npz"), **ref_two())
    np.savez_compressed(os.path.join(HERE, "ref_mvs.npz"), **ref_mvs())
    np.savez_compressed(os.path.join(HERE, "ref_leaves.npz"), **ref_leaves())
    np.savez_compressed(os.path.join(HERE, "oracle_scenes.npz"), **oracle_scenes())
    for f in ("ref_leaves.npz", "oracle_scenes.npz", "ref_mvs.npz", "ref_two.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
