"""Writes tests/golden/binary.npz: cv2.BFMatcher(NORM_HAMMING) results that the Hamming matcher is pinned against.

    python tests/golden/make_binary_golden.py      (needs cv2 with ORB; run once, the output is committed)

Two input sets:
  - synth.binary_pair(20000, 20000, 32): knnMatch(k=2) indices / distances, crossCheck=True match pairs, and the sha1 of
    the inputs (the tests regenerate them and check the digests instead of storing 1.3 MB of random bytes);
  - real ORB descriptors (cv2.ORB_create, 32 bytes) with their keypoints, from a seeded procedural equirectangular
    texture and a copy of it turned by 40 degrees of yaw (a horizontal roll of the ERP image).  Building photographs
    are not shipped with the project, so the image pair is procedural.
Tests never import cv2.
"""
from __future__ import annotations

import hashlib
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from erp_match_eightpoint_test_b200 import synth  # noqa: E402

W, H = 2048, 1024
YAW_DEG = 40


def sha1(a: np.ndarray) -> str:
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def texture(seed: int = 7) -> np.ndarray:
    """Gray ERP texture: blurred noise at a few scales plus random rectangles and discs (corners and blobs for ORB)."""
    rng = np.random.Generator(np.random.Philox(seed))
    img = np.zeros((H, W), np.float32)
    for s, a in ((4, 60.0), (16, 50.0), (64, 40.0)):
        n = rng.standard_normal((H // s, W // s)).astype(np.float32)
        img += a * cv2.resize(n, (W, H), interpolation=cv2.INTER_CUBIC)
    for _ in range(900):
        x, y = int(rng.integers(0, W)), int(rng.integers(0, H))
        w, h = int(rng.integers(6, 60)), int(rng.integers(6, 60))
        v = float(rng.uniform(-120, 120))
        if rng.random() < 0.5:
            cv2.rectangle(img, (x, y), (x + w, y + h), v, -1)
        else:
            cv2.circle(img, (x, y), w // 2, v, -1)
    img = img - img.min()
    return np.clip(img * (255.0 / img.max()), 0, 255).astype(np.uint8)


def knn_arrays(q: np.ndarray, t: np.ndarray):
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    knn = bf.knnMatch(q, t, k=2)
    idx = np.array([[m.trainIdx for m in r] for r in knn], np.int32)
    dist = np.array([[m.distance for m in r] for r in knn], np.float32)
    cc = cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True).match(q, t)
    pairs = np.array(sorted((m.queryIdx, m.trainIdx) for m in cc), np.int32).reshape(-1, 2)
    cc_dist = np.array([m.distance for m in sorted(cc, key=lambda m: m.queryIdx)], np.float32)
    return idx, dist, pairs, cc_dist


def main():
    out = {}
    q, t, _ = synth.binary_pair(20000, 20000, 32)
    idx, dist, pairs, cc_dist = knn_arrays(q, t)
    out.update(syn_q_sha1=sha1(q), syn_t_sha1=sha1(t), syn_idx=idx, syn_dist=dist, syn_cc=pairs, syn_cc_dist=cc_dist)

    left = texture()
    right = np.roll(left, -int(W * YAW_DEG / 360), axis=1)
    orb = cv2.ORB_create(nfeatures=5000)
    kl, dl = orb.detectAndCompute(left, None)
    kr, dr = orb.detectAndCompute(right, None)
    idx, dist, pairs, cc_dist = knn_arrays(dl, dr)
    out.update(orb_q=dl, orb_t=dr,
               orb_q_xy=np.array([k.pt for k in kl], np.float32), orb_t_xy=np.array([k.pt for k in kr], np.float32),
               orb_idx=idx, orb_dist=dist, orb_cc=pairs, orb_cc_dist=cc_dist,
               orb_width=np.int32(W), orb_height=np.int32(H), orb_yaw_deg=np.float32(YAW_DEG))
    path = os.path.join(HERE, "binary.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {os.path.getsize(path)} bytes, ORB {len(dl)} x {len(dr)}, cv2 {cv2.__version__}")


if __name__ == "__main__":
    main()
