#!/usr/bin/env python
"""Derives the small `bunny` fixture of tests/golden/bunny/ from the reference's example data.

  REF=<reference source tree> python tests/golden/make_bunny.py      (reads $REF/example)

BASELINE.json configs[0] and [1] are the reference's `example/project.xml` 'bunny' image set (8
calibrated, lens-distorted cameras, 1024x768 RGBA PNGs whose alpha channel is the object mask).
The tests must run without the reference's sources, and 11 MB of PNGs do not belong in the history, so the
fixture is: the 8 camera entries of the XML verbatim as JSON (projection matrix + distortion),
and the images reduced to 1/4 size (256x192, PIL LANCZOS on RGB, alpha thresholded so the mask
stays binary).  Both the oracle and the GPU path read these identically pre-scaled images with
image_scale = 0.25, which is how SURVEY §7 (hard part 6) says scaled runs must be compared.
"""
import json
import os
import re

import numpy as np
from PIL import Image

REF = os.path.join(os.environ.get("REF", ""), "example")
HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "bunny")
SCALE = 0.25


def main():
    xml = open(os.path.join(REF, "project.xml")).read()
    cams = []
    for m in re.finditer(r'<camera id="(\d+)">(.*?)</camera>', xml, re.S):
        cid, body = m.group(1), m.group(2)
        pm = dict(re.findall(r'(m\d\d)="([^"]+)"', re.search(r"<projectionMatrix ([^>]*)/>", body).group(1)))
        ld = re.search(r"<lensDistortion ([^>]*)/>", body)
        dist = dict(re.findall(r'(\w+)="([^"]+)"', ld.group(1))) if ld else {}
        cams.append({"id": cid, "P": [float(pm.get(f"m{r}{c}", 0)) for r in (1, 2, 3) for c in (1, 2, 3, 4)],
                     "dist": [float(dist.get(k, 0)) for k in ("k1", "k2", "p1", "p2", "k3")]})
    ids = re.findall(r'<image for="(\d+)"[^>]*file="(\d+\.png)"', re.search(r'<imageSet root="images/bunny".*?</imageSet>', xml, re.S).group(0))
    os.makedirs(HERE, exist_ok=True)
    keep = []
    for cid, fname in ids:
        im = Image.open(os.path.join(REF, "images", "bunny", fname)).convert("RGBA")
        w, h = im.size
        nw, nh = int(w * SCALE), int(h * SCALE)
        rgb = im.convert("RGB").resize((nw, nh), Image.LANCZOS)
        alpha = im.getchannel("A").resize((nw, nh), Image.BOX)
        a = np.where(np.asarray(alpha) == 255, 255, 0).astype(np.uint8)  # only fully opaque pixels stay in the mask
        out = np.dstack([np.asarray(rgb), a])
        Image.fromarray(out, "RGBA").save(os.path.join(HERE, fname), optimize=True)
        keep.append(cid)
    cams = [c for c in cams if c["id"] in keep]
    json.dump({"scale": SCALE, "full_size": [1024, 768], "cameras": cams,
               "source": "thegedge/StereoReconstruction example/project.xml + example/images/bunny (reduced to 1/4)"},
              open(os.path.join(HERE, "cameras.json"), "w"), indent=1)
    print(len(cams), "cameras;", sum(os.path.getsize(os.path.join(HERE, f)) for f in os.listdir(HERE)) // 1024, "KiB")


if __name__ == "__main__":
    main()
