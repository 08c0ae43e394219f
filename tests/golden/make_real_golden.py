"""Regenerates tests/golden/real_building.npz: REAL descriptors of the reference's own test pair.

The reference's e2e case (src/automatic.cpp:81-160 on build/left_building.jpg + right_building.jpg) needs SURF from
OpenCV's non-free xfeatures2d, which no OpenCV in this image has.  cv2.SIFT (128-D float descriptors, integer valued) is
the closest detector available, so this script runs the reference's strip pipeline with it:

    spherical_surf::do_all (src/spherical_surf.cpp:66-150): four strips per image (crop_rotated_image at 45, 0, -45, -90
    degrees), detect + describe per strip, rotate_keypoint back to ERP pixels, concatenate in strip order

using the ORACLE's restatement of crop_rotated_image / rotate_keypoint (oracle/erp_oracle.c), and pins the third-party
matcher on the result: cv2.BFMatcher(NORM_L2).knnMatch(k=2) and the crossCheck match.  Real facade structure (repeated
windows) produces the near-ties and low-contrast ratio tests that Gaussian synthetic descriptors never do.

Run from the repo root with a checkout of the reference:  python tests/golden/make_real_golden.py <reference checkout>
The archive is written with LZMA members (np.load reads them) to keep the fixture under 1 MB.
"""
import os
import sys
import zipfile

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle as O  # noqa: E402

PER_STRIP = 1200          # strongest SIFT features kept per strip (fixture size: 2 x 4 x 1200 x 128 bytes)
SCALE = 0.5               # the 5376 x 2688 originals are halved: 2688 x 1344 (a 4K-class ERP pair keeps the fixture small)


def strips(im):
    h, w = im.shape[:2]
    roi = im[h * 3 // 8: h * 3 // 8 + h // 4]
    return [O.crop_rotated_image(im, 45.0), np.ascontiguousarray(roi), O.crop_rotated_image(im, -45.0), O.crop_rotated_image(im, -90.0)]


def describe(im):
    h, w = im.shape[:2]
    sift = cv2.SIFT_create(nfeatures=PER_STRIP)
    keys, descs = [], []
    for n, (strip, pitch) in enumerate(zip(strips(im), (45.0, None, -45.0, -90.0))):
        kp, d = sift.detectAndCompute(cv2.cvtColor(strip, cv2.COLOR_BGR2GRAY), None)
        xy = np.array([k.pt for k in kp], np.float32).reshape(-1, 2)
        if pitch is None:
            xy[:, 1] += h * 3 // 8                                  # src/spherical_surf.cpp:122-124
        else:
            xy = O.rotate_keypoints(xy, pitch, w, h)                # src/spherical_surf.cpp:50-63
        keys.append(xy)
        descs.append(d)
    return np.concatenate(keys).astype(np.float32), np.concatenate(descs).astype(np.float32)


def main(ref):
    out = {}
    ims = {}
    for side in ("left", "right"):
        im = cv2.imread(os.path.join(ref, "build", side + "_building.jpg"), cv2.IMREAD_COLOR)
        im = cv2.resize(im, None, fx=SCALE, fy=SCALE, interpolation=cv2.INTER_AREA)
        ims[side] = im
        xy, d = describe(im)
        assert np.array_equal(d, np.round(d)) and d.min() >= 0 and d.max() <= 255        # SIFT descriptors are byte valued
        out[side + "_xy"] = xy
        out[side + "_desc_u8"] = d.astype(np.uint8)
    out["width"], out["height"] = np.int32(ims["left"].shape[1]), np.int32(ims["left"].shape[0])
    q, t = out["left_desc_u8"].astype(np.float32), out["right_desc_u8"].astype(np.float32)
    kn = cv2.BFMatcher(cv2.NORM_L2).knnMatch(q, t, k=2)
    out["bf_idx"] = np.array([[m[0].trainIdx, m[1].trainIdx] for m in kn], np.int32)
    out["bf_dist"] = np.array([[m[0].distance, m[1].distance] for m in kn], np.float32)
    cc = cv2.BFMatcher(cv2.NORM_L2, crossCheck=True).match(q, t)
    out["bf_cross"] = np.array(sorted((m.queryIdx, m.trainIdx) for m in cc), np.int32)
    with zipfile.ZipFile(os.path.join(HERE, "real_building.npz"), "w", compression=zipfile.ZIP_LZMA) as z:
        for k, v in out.items():
            with z.open(k + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(v))
    print({k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items()})


if __name__ == "__main__":
    main(sys.argv[1])
