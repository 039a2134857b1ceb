#!/usr/bin/env python
"""Full-size (1024 x 768) `bunny` golden vectors from THE REFERENCE ITSELF (BASELINE configs[0], [1]).

  REF=<reference source tree> python tests/golden/make_bunny_full.py     (reads $REF/example and needs
                                              oracle/_ref = the reference compiled where it lies)

The reference's own example data at its own size: real calibrated, lens-distorted cameras, real object
masks, flat regions.  11 MB of PNGs do not belong in the history and the reference needs minutes per full
view on the host, so the fixture is a REGION of the job, chosen so that the reference and the code under
test read exactly the same pixels as they would on the full images:

  mvs   reference view 7310089 (index 2) against the three neighbours the class's own rule selects, rows
        [R0, R1) of the reference view only (the class skips pixels outside its mask: the reference view's
        mask is reduced to the band).  Neighbour masks are the ORIGINAL ones.  RGB is kept where it can be
        read: around the band in the reference view, and inside the bounding box (+ margin) of every
        depth level's projection of the band in each neighbour; zero elsewhere (PNG shrinks 10x).
  two   cameras 7310085 + 7310087 (cfg1), TwoViewStereo's constants (r = 5, GeodesicWeight, NCC): the left
        mask reduced to a band, the right mask to the box the band's depth range projects into; both
        directions of the live search, before the cross-check.

Outputs of the reference (depth maps before the cross-check, rows of the band / box only) for the shipped
GeodesicWeight typedef and for the AdaptiveWeight build of the same file (BASELINE configs[1]), with the
injected interface of SURVEY §8d cfg1/cfg2 ((px,py) = principal point + (40,25) px, dist = 10, n = 1.333):
tests/golden/bunny_full/golden.npz; inputs: tests/golden/bunny_full/*.png + cameras in the npz (settled
through the reference's own Camera::set).  tests/test_bunny_full.py replays them on the GPU (curve mode).
"""
import json
import os
import sys

import numpy as np
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle_api as O  # noqa: E402
from stereoreconstruction_b200 import types as T  # noqa: E402
import golden_cases as G  # noqa: E402

REF = os.path.join(os.environ.get("REF", ""), "example")
OUT = os.path.join(HERE, "bunny_full")
MIN_D, MAX_D, LEVELS = 30.0, 55.0, 100     # brackets the object for the cameras of example/project.xml (golden_cases.py)
MVS_REF, BAND = 2, (396, 428)              # 32 rows through the middle of the object
TWO = (0, 1)
MARGIN = 8


def load_full():
    meta = json.load(open(os.path.join(HERE, "bunny", "cameras.json")))
    cams, imgs = [], []
    for c in meta["cameras"]:
        cam = T.camera_from_P(c["P"], dist=c["dist"])
        T.set_interface_px(cam, cam.K[2] + 40.0, cam.K[5] + 25.0, 10.0, 1.333)
        cams.append(cam)
        imgs.append(np.asarray(Image.open(os.path.join(REF, "images", "bunny", c["id"] + ".png")).convert("RGBA")).copy())
    return [c["id"] for c in meta["cameras"]], G.settled_cameras(cams), imgs


def mask_of(im):
    return np.where(im[..., 3] == 255, 255, 0).astype(np.uint8)


def dilate(m, r):
    out = m.copy()
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            out |= np.roll(np.roll(m, dy, 0), dx, 1)
    return out


def projected_box(sc, cams, ref, nbr, region_mask, h, w):
    """Bounding box in view `nbr` of the projections of the region's pixels at every depth level."""
    rays = sc.unproject_grid(ref)
    ys, xs = np.where(region_mask)
    sel = slice(None, None, 3)
    src, dr = rays[ys[sel], xs[sel], :3], rays[ys[sel], xs[sel], 3:]
    Cc, prin = np.array(cams[ref].C[:]), np.array(cams[ref].prin_dir[:])
    nrm = prin / np.linalg.norm(prin)
    lo = np.array([1e9, 1e9])
    hi = -lo
    for d in np.linspace(MIN_D, MAX_D, 26):
        x0 = Cc + d * prin
        t = ((x0 - src) @ nrm) / (dr @ nrm)
        xy, ok = sc.project_points(nbr, src + t[:, None] * dr)
        good = (ok != 0) & np.isfinite(xy).all(axis=1)
        if good.any():
            lo = np.minimum(lo, xy[good].min(axis=0))
            hi = np.maximum(hi, xy[good].max(axis=0))
    x0, y0 = max(0, int(lo[0]) - MARGIN), max(0, int(lo[1]) - MARGIN)
    x1, y1 = min(w, int(hi[0]) + MARGIN + 1), min(h, int(hi[1]) + MARGIN + 1)
    return x0, y0, x1, y1


def keep_rgb(im, keep):
    out = im.copy()
    out[..., :3][~keep] = 0
    return out


def main():
    O.build()
    assert O.ref_lib() is not None, "oracle/_ref is needed (the reference compiled where it lies)"
    ids, cams, imgs = load_full()
    h, w = imgs[0].shape[:2]
    masks = [mask_of(im) for im in imgs]
    sc = O.Scene(cams, imgs, masks)
    os.makedirs(OUT, exist_ok=True)
    out = {"ids": np.array(ids), "band": np.array(BAND), "depth_range": np.array([MIN_D, MAX_D, LEVELS])}

    # ------------------------------------------------------------------ multi-view (cfg2)
    nb = sc.select_neighbours(3)[MVS_REF]
    views = [MVS_REF] + list(nb)
    r0, r1 = BAND
    band_mask = np.zeros((h, w), bool)
    band_mask[r0:r1] = masks[MVS_REF][r0:r1] == 255
    mvs_imgs, mvs_masks = [], []
    for k, v in enumerate(views):
        if k == 0:
            keep = np.zeros((h, w), bool)
            keep[max(0, r0 - MARGIN):r1 + MARGIN] = True
            m = np.where(band_mask, 255, 0).astype(np.uint8)  # the reference view: band only
        else:
            x0, y0, x1, y1 = projected_box(sc, cams, MVS_REF, v, band_mask, h, w)
            keep = np.zeros((h, w), bool)
            keep[y0:y1, x0:x1] = True
            m = masks[v]
        im = keep_rgb(imgs[v], keep)
        im[..., 3] = m
        mvs_imgs.append(im)
        mvs_masks.append(m)
        Image.fromarray(im, "RGBA").save(os.path.join(OUT, f"mvs_{ids[v]}.png"), optimize=True)
    mvs_cams = [cams[v] for v in views]
    out["mvs_views"] = np.array(views)
    out["mvs_cams"] = G.cams_to_bytes(mvs_cams)
    for tag, ada in (("geo", False), ("ada", True)):
        ref = O.RefMVS(mvs_cams, mvs_imgs, mvs_masks, MIN_D, MAX_D, LEVELS, 5.0, image_scale=1.0, adaptive=ada)
        for v in range(len(views)):
            ref.set_neighbours(v, [u for u in range(len(views)) if u != v][:3])
        d, _ = ref.initial_estimate(0)
        ref.close()
        out[f"mvs_{tag}_before"] = d[r0:r1].copy()
        print("mvs", tag, "finite in band:", float(np.isfinite(d[r0:r1])[band_mask[r0:r1]].mean()),
              "with depth:", float((d[r0:r1][band_mask[r0:r1]] > 0).mean()))

    # ------------------------------------------------------------------ two-view (cfg1)
    a, b = TWO
    band_a = np.zeros((h, w), bool)
    band_a[r0:r1] = masks[a][r0:r1] == 255
    x0, y0, x1, y1 = projected_box(sc, cams, a, b, band_a, h, w)
    box_b = np.zeros((h, w), bool)
    box_b[y0:y1, x0:x1] = masks[b][y0:y1, x0:x1] == 255
    two_imgs, two_masks = [], []
    for v, reg in ((a, band_a), (b, box_b)):
        m = np.where(reg, 255, 0).astype(np.uint8)
        im = keep_rgb(imgs[v], dilate(reg, MARGIN))
        im[..., 3] = m
        two_imgs.append(im)
        two_masks.append(m)
        Image.fromarray(im, "RGBA").save(os.path.join(OUT, f"two_{ids[v]}.png"), optimize=True)
    two_cams = [cams[a], cams[b]]
    out["two_cams"] = G.cams_to_bytes(two_cams)
    out["two_box"] = np.array([x0, y0, x1, y1])
    ref = O.RefTwoView(two_cams[0], two_cams[1], two_imgs[0], two_imgs[1], two_masks[0], two_masks[1], MIN_D, MAX_D, LEVELS,
                       image_scale=1.0)
    bl, br = ref.search()
    ref.close()
    out["two_before_left"] = bl[r0:r1].copy()
    out["two_before_right"] = br[y0:y1].copy()
    print("two: left with depth", float(np.isfinite(bl[r0:r1])[band_a[r0:r1]].mean()),
          "right with depth", float(np.isfinite(br[y0:y1])[box_b[y0:y1]].mean()))

    np.savez_compressed(os.path.join(OUT, "golden.npz"), **out)
    tot = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT))
    print("fixture:", sorted(os.listdir(OUT)), tot // 1024, "KiB")


if __name__ == "__main__":
    main()
