#!/usr/bin/env python
"""Writes tests/golden/ref_pins/*.npz: what the reference returned for the inputs of tests/test_oracle_vs_ref.py
and tests/test_host_api.py::test_host_camera_class_matches_reference_camera, so that those comparisons run where
oracle/_ref (the reference's sources compiled where they lie, oracle/Makefile) is not built.

  python tests/golden/make_ref_pins.py

With oracle/_ref built, every value comes from the reference itself (the tests' own ref_* functions).  Without
it, the values come from the code those tests pinned to the reference on exactly these inputs: the oracle,
bit for bit for the leaves, curves, costs and end-to-end classes, and to the tests' tolerances for the camera
model; the C++ Camera class for the host camera test (DESIGN.md section 2).  Large outputs are kept at a fixed
seeded sample of their entries (shrink(); `<key>_idx` says which), so that the fixtures stay small.
"""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle_api as O  # noqa: E402
from stereoreconstruction_b200 import types as T  # noqa: E402
import golden_cases as G  # noqa: E402
import test_oracle_vs_ref as V  # noqa: E402

OUT = os.path.join(HERE, "ref_pins")


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def cams_bytes(cams):
    return np.frombuffer(b"".join(bytes(O.as_cam_array([c])[0]) for c in cams), np.uint8)


# ---- the same values from the code pinned to the reference ------------------------------------------
def lines():
    L = O.lib()
    cases, w, h = V.line_cases()
    counts, pts, ok, out = [], [], [], []
    for (x0, y0, x1, y1) in cases:
        for clip in (0, 1):
            buf = np.empty((4096, 2), np.int32)
            n = L.orc_line(x0, y0, x1, y1, clip, w, h, _ip(buf), 4096)
            counts.append(n)
            pts.append(buf[:min(n, 4096)].copy())
        a = np.array([x0, y0, x1, y1], np.int32)
        ok.append(L.orc_clip_line(_ip(a), w, h))
        out.append(a)
    return dict(counts=np.array(counts), points=np.concatenate(pts), clip_ok=np.array(ok), clip_out=np.array(out))


def rays():
    L = O.lib()
    d = {k: [] for k in ("intersect_ok", "intersect", "refract_ok", "refract", "closest")}
    for (s1, d1, s2, d2, pn, pd, n) in V.ray_cases():
        b, b6, c6 = np.full(3, np.nan), np.empty(6), np.empty(6)
        d["intersect_ok"].append(L.orc_intersect(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), _dp(b)))
        d["intersect"].append(b)
        d["refract_ok"].append(L.orc_refract(_dp(s1), _dp(d1), _dp(pn), C.c_double(pd), C.c_double(n), _dp(b6)))
        d["refract"].append(b6)
        L.orc_closest_points(_dp(s1), _dp(d1), _dp(s2), _dp(d2), _dp(c6))
        d["closest"].append(c6)
    return {k: np.array(v) for k, v in d.items()}


def samples():
    L = O.lib()
    image = V.leaf_image()
    h, w = image.shape[:2]
    sc = V._identity_scene(image)
    out = {}
    vals = np.empty((2000, 4))
    for i, (x, y) in enumerate(V.sample_points(w, h)):
        L.orc_sample(sc.ptr, 0, C.c_double(x), C.c_double(y), _dp(vals[i]))
    out["sample"] = vals
    grid = V.grid_points(w, h)
    vals = np.empty((len(grid), 4))
    for i, (x, y) in enumerate(grid):
        L.orc_sample_int(sc.ptr, 0, x, y, _dp(vals[i]))
    out["grid"] = vals
    cx, cy = V.weight_centres(w, h)
    for kind, radius in V.WEIGHT_CASES:
        out[f"weights_k{kind}_r{radius}"] = sc.weights(0, kind, radius, cx, cy)
    return out


def cameras():
    L = O.lib()
    cams = V.cameras()
    pix = V.unproject_pixels()
    unproject, xy, ok = [], [], []
    for c, pts in zip(cams, V.project_points()):
        r = np.empty((len(pix), 6))
        for i, (x, y) in enumerate(pix):
            L.orc_unproject(O.as_cam_array([c]), C.c_double(x), C.c_double(y), _dp(r[i]))
        unproject.append(r)
        p, k = O.Scene([c], [np.zeros((480, 640, 4), np.uint8)]).project_points(0, pts, root_mode=0)
        xy.append(p)
        ok.append(k)
    return dict(derived=cams_bytes(cams), unproject=np.array(unproject), project_xy=np.array(xy),
                project_ok=np.array(ok), from_P=cams_bytes([T.camera_from_P(P) for P in V.projection_matrices()]))


def mvs(interface, distortion, adaptive):
    cams, imgs, ms = V.mvs_scene(interface, distortion)
    mind, maxd, D, cross = G.REF_MVS_CASES["arc"]
    sc = O.Scene(cams, imgs, ms)
    P = T.default_params(True, mind, maxd, D, weight_kind=T.SR_WEIGHT_ADAPTIVE if adaptive else T.SR_WEIGHT_GEODESIC)
    nb = [[int(v) for v in r] for r in sc.select_neighbours(3)]
    before, peaks, pk_pix = [], [], []
    for v in range(len(cams)):
        od, _, _, _, op = sc.mvs_view(P, v, nb[v], curve_mode=True, root_mode=0, want_peaks=True)
        before.append(od)
        pk_pix.append(np.flatnonzero(ms[v] == 255))
        peaks.append(op.reshape(-1, 9, 2)[pk_pix[-1]])
    after = sc.crosscheck_mvs(P, before, cross)
    counts, pts, costs = [], [], []
    for (x, y) in V.mvs_curve_pixels():
        curve = sc.epipolar_curve(P, 1, 2, x, y, True, 0)
        counts.append(len(curve))
        pts.append(curve)
        for (px, py) in curve[:: max(1, len(curve) // 5)]:
            costs.append(sc.cost(P, 1, 2, x, y, int(px), int(py)))
    return dict(neighbours=np.array([r + [-1] * (3 - len(r)) for r in nb], np.int32),
                before=np.array(before).reshape(len(cams), -1), after=np.array(after).reshape(len(cams), -1), peak_pix=pk_pix, peaks=peaks, curve_counts=np.array(counts),
                curve_points=np.concatenate(pts), costs=np.array(costs))


def two(interface, distortion):
    cams, imgs, ms = V.mvs_scene(interface, distortion)
    a, b, mind, maxd, D = G.REF_TWO_CASES["arc"]
    sc = O.Scene(cams, imgs, ms)
    P = T.default_params(False, mind, maxd, D)
    bl = sc.twoview_curve(P, a, b, root_mode=0)[0]
    br = sc.twoview_curve(P, b, a, root_mode=0)[0]
    al, ar = sc.crosscheck_two(P, a, b, bl, br, 1.0, root_mode=0)
    costs = [[sc.cost(T.default_params(False, mind, maxd, D, cost_kind=k), a, b, *win)
              for k in (T.SR_COST_NCC_TWOVIEW, T.SR_COST_SAD_TWOVIEW)] for win in V.two_cost_windows()]
    return dict(before=np.array([bl, br]).reshape(2, -1), after=np.array([al, ar]).reshape(2, -1), costs=np.array(costs))


def label_mvs():
    cams, imgs, ms = G.arc_scene()
    mind, maxd, D, _ = G.REF_MVS_CASES["arc"]
    sc = O.Scene(cams, imgs, ms)
    nb = [int(v) for v in sc.select_neighbours(3)[1]]
    od, oi, ob, _, _ = sc.mvs_view(T.default_params(True, mind, maxd, D), 1, nb, root_mode=0)
    pix = V.label_pixels(ms[1], 120, 12)
    return dict(label=np.array([oi[p] for p in pix]), depth=np.array([od[p] for p in pix]),
                cost=np.array([ob[p] if oi[p] >= 0 else np.nan for p in pix]))


def label_two():
    cams, imgs, ms = G.arc_scene()
    a, b, mind, maxd, D = G.REF_TWO_CASES["arc"]
    od, oi, ob, _ = O.Scene(cams, imgs, ms).twoview_label(T.default_params(False, mind, maxd, D), a, b, root_mode=0)
    pix = V.label_pixels(ms[a], 60, 13)
    return dict(label=np.array([oi[p] for p in pix]), depth=np.array([od[p] for p in pix]),
                cost=np.array([ob[p] for p in pix]))


def host_cameras():
    """Camera::setP of the bunny fixture's cameras: the reference's when oracle/_ref is built, else the C++
    Camera class (include/project/camera.hpp, the harness's --cameras mode)."""
    import test_host_api as H
    cams = H.bunny_cameras()
    if V.REF is not None:
        out = []
        for P in H.projection_matrices(cams):
            ref = O.OrcCamera()
            V.REF.ref_camera_from_P(np.ascontiguousarray(P).ctypes.data_as(C.POINTER(C.c_double)), C.byref(ref))
            out.append(bytes(ref))
        return dict(cams=np.frombuffer(b"".join(out), np.uint8))
    with tempfile.TemporaryDirectory() as tmp:
        blank = [np.zeros((8, 8, 4), np.uint8)] * len(cams)
        xml = H.write_project(tmp, cams, blank, [np.full((8, 8), 255, np.uint8)] * len(cams))
        subprocess.run([H.HARNESS, "--cameras", xml, tmp], check=True, capture_output=True)
        return dict(cams=np.fromfile(os.path.join(tmp, "cams.bin"), np.uint8))


def _pick(rng, n, k, always=()):
    rest = np.setdiff1d(np.arange(n), always)
    return np.sort(np.concatenate([rng.choice(rest, min(k, rest.size), replace=False), always])).astype(np.int32)


def shrink(name, d, seed):
    """Fixed seeded samples of the large outputs; `<key>_idx` holds the kept indices (first axis, or flat pixels)."""
    rng = np.random.RandomState(seed)
    d = dict(d)

    def keep(key, idx, axis=0, also=()):
        for k in (key,) + also:
            d[k] = np.take(np.asarray(d[k]), idx, axis=axis)
        d[key + "_idx"] = idx

    if name == "lines":
        idx = _pick(rng, len(d["clip_ok"]), 100, always=np.arange(11))  # (+ the hand-written cases)
        starts = np.concatenate([[0], np.cumsum(np.minimum(d["counts"], 4096))])
        pairs = np.stack([2 * idx, 2 * idx + 1], axis=1).reshape(-1)
        d["points"] = np.concatenate([d["points"][starts[p]:starts[p + 1]] for p in pairs]).astype(np.int16)
        d["counts"] = d["counts"][pairs]
        keep("clip_ok", idx, also=("clip_out",))
    elif name == "rays":
        keep("closest", _pick(rng, len(d["closest"]), 150), also=("intersect_ok", "intersect", "refract_ok", "refract"))
    elif name == "samples":
        keep("sample", _pick(rng, len(d["sample"]), 200))
        keep("grid", _pick(rng, len(d["grid"]), 200))
        for k in [k for k in d if k.startswith("weights_") and not k.endswith("_idx")]:
            keep(k, _pick(rng, len(d[k]), 4, always=np.arange(30, 34)))  # (+ the four corners)
    elif name == "cameras":
        n = d["unproject"].shape[1]
        keep("unproject", _pick(rng, n, 60, always=np.arange(n - 3, n)), axis=1)  # (+ the three pixel centres)
        keep("project_xy", _pick(rng, d["project_xy"].shape[1], 300), axis=1, also=("project_ok",))
    elif name.startswith(("mvs_", "two_")):
        before = np.asarray(d["before"]).reshape(len(d["before"]), -1)
        idx = _pick(rng, before.shape[1], 192 if name.startswith("mvs_") else 384)
        d["before"] = before[:, idx]
        d["after"] = np.asarray(d["after"]).reshape(before.shape)[:, idx]
        d["before_idx"] = d["after_idx"] = idx
        if name.startswith("mvs_"):
            sel = [np.sort(rng.choice(len(p), 12, replace=False)) for p in d["peak_pix"]]
            d["peak_pix"] = np.array([p[s] for p, s in zip(d["peak_pix"], sel)])
            d["peaks"] = np.array([k[s] for k, s in zip(d["peaks"], sel)])
            d["curve_points"] = d["curve_points"].astype(np.int16)
    return d


def main():
    live = V.REF is not None
    os.makedirs(OUT, exist_ok=True)
    jobs = [("lines", V.ref_lines, lines), ("rays", V.ref_rays, rays), ("samples", V.ref_samples, samples),
            ("cameras", V.ref_cameras, cameras), ("label_mvs", V.ref_label_mvs, label_mvs),
            ("label_two", V.ref_label_two, label_two)]
    jobs += [(V.mvs_name(*k), lambda k=k: V.ref_mvs(*k), lambda k=k: mvs(*k)) for k in V.MVS_COMBOS]
    jobs += [(V.two_name(*k), lambda k=k: V.ref_two(*k), lambda k=k: two(*k)) for k in V.TWO_COMBOS]
    jobs += [("host_cameras", host_cameras, host_cameras)]
    for i, (name, from_ref, pinned) in enumerate(jobs):
        d = shrink(name, from_ref() if live else pinned(), i)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **d)
        print(f"{name}: {os.path.getsize(path) / 1e3:.0f} kB")
    with open(os.path.join(OUT, "SOURCE.json"), "w") as f:
        json.dump({"from": "oracle/_ref (the reference itself)" if live else
                   "the oracle and the C++ Camera class, pinned to the reference on these inputs (DESIGN.md section 2)"},
                  f, indent=1)


if __name__ == "__main__":
    main()
