"""Regenerates tests/golden/*.npz from the in-container Python OpenCV (cv2 4.13).

The reference (C++/OpenCV 3.4 + xfeatures2d) ships no golden vectors and cannot be
built here, so the oracle is pinned against the same third-party functions the
reference calls, as exposed by cv2:
  cv2.BFMatcher(NORM_L2).knnMatch(k=2) / crossCheck  <-> feature_matcher.cpp:45 (exact limit of FLANN)
  cv2.SVDecomp                                       <-> eight_point.cpp:39,46
  cv2.decomposeEssentialMat                          <-> eight_point.cpp:54
  cv2.invert on 3x3 CV_64F                           <-> erp_rotation.cpp:103 (cv::Mat::inv)
cv2 4.13 is built with LAPACK, so singular vectors can differ from OpenCV's own
Jacobi SVD by per-vector sign; consumers compare up to those signs.

Run from the repo root:  python tests/golden/make_golden.py
"""
import hashlib
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from erp_match_eightpoint_test_b200 import synth  # noqa: E402


def matching():
    out = {}
    for name, (nq, nt, dim) in {"m64": (700, 900, 64), "m128": (300, 500, 128)}.items():
        q, t, planted = synth.descriptor_pair(nq, nt, dim, seed=synth.SEED_BASE + dim)
        # exact duplicates in the train set exercise the lowest-trainIdx tie rule
        t[37] = t[12]; t[5] = t[12]
        q[3] = t[12]
        kn = cv2.BFMatcher(cv2.NORM_L2).knnMatch(q, t, k=2)
        out[name + "_q"], out[name + "_t"] = q, t
        out[name + "_idx"] = np.array([[m[0].trainIdx, m[1].trainIdx] for m in kn], np.int32)
        out[name + "_dist"] = np.array([[m[0].distance, m[1].distance] for m in kn], np.float32)
        cc = cv2.BFMatcher(cv2.NORM_L2, crossCheck=True).match(q, t)
        out[name + "_cross"] = np.array(sorted((m.queryIdx, m.trainIdx) for m in cc), np.int32)
    np.savez_compressed(os.path.join(HERE, "matching.npz"), **out)


def svd_and_decompose():
    rng = np.random.Generator(np.random.Philox(7))
    out = {}
    for i, rows in enumerate([8, 9, 12, 50]):
        A = rng.standard_normal((rows, 9))
        w, u, vt = cv2.SVDecomp(A)
        out[f"A{i}"], out[f"w{i}"], out[f"vt{i}"] = A, w.ravel(), vt
    Es, R1s, R2s, ts = [], [], [], []
    for k in range(6):
        kp = synth.keypoint_pair(64, 4096, 2048, euler_deg=(5 * k, -3 * k, 2 * k + 1),
                                 t=(0.3 + 0.1 * k, -0.9, 0.1 * k), noise_px=0.0, outlier_frac=0.0, seed=900 + k)
        E = kp["E"] / np.linalg.norm(kp["E"])
        R1, R2, t = cv2.decomposeEssentialMat(E)
        Es.append(E); R1s.append(R1); R2s.append(R2); ts.append(t.ravel())
    out.update(E=np.array(Es), R1=np.array(R1s), R2=np.array(R2s), t=np.array(ts))
    np.savez_compressed(os.path.join(HERE, "svd_decompose.npz"), **out)


def eight_point_cases():
    """Reference-form hypothesis solved with cv2 exactly as eight_point.cpp:22-61 does."""
    out = {}
    for k, (n, noise) in enumerate([(9, 0.0), (40, 0.5), (250, 0.5)]):
        kp = synth.keypoint_pair(n, 4096, 2048, noise_px=noise, outlier_frac=0.0, seed=700 + k)
        out[f"lxy{k}"], out[f"rxy{k}"] = kp["left_xy"], kp["right_xy"]

        def bearing(xy):
            lon = 2 * np.pi * (xy[:, 0] / np.float32(4096)).astype(np.float64)
            lat = np.pi * (xy[:, 1] / np.float32(2048)).astype(np.float64)
            return np.stack([-np.sin(lat) * np.cos(lon), np.sin(lat) * np.sin(lon), np.cos(lat)], 1)

        l, r = bearing(kp["left_xy"]), bearing(kp["right_xy"])
        A = np.einsum("na,nb->nab", l, r).reshape(n, 9)
        _, _, vt = cv2.SVDecomp(A)
        E = vt[-1].reshape(3, 3)
        w, u, vt3 = cv2.SVDecomp(E)
        w = w.ravel(); w[2] = 0
        Ec = u @ np.diag(w) @ vt3
        R1, R2, t = cv2.decomposeEssentialMat(Ec)
        out[f"l{k}"], out[f"r{k}"], out[f"e{k}"], out[f"Ec{k}"] = l, r, E, Ec
        out[f"R1_{k}"], out[f"R2_{k}"], out[f"t{k}"] = R1, R2, t.ravel()
    np.savez_compressed(os.path.join(HERE, "eight_point.npz"), **out)


def cfg2_matching():
    """configs[1] at full size (20k x 20k SURF-64, the inputs of tests/test_gpu_parity.py's cv2 comparison):
    cv2.BFMatcher(NORM_L2).knnMatch(k=2) indices and fp32 distances, and digests of the inputs they belong to."""
    q, t, _ = synth.descriptor_pair(20000, 20000, 64, seed=synth.SEED_BASE + 1)
    t[137] = t[12]; t[5] = t[12]; q[3] = t[12]
    kn = cv2.BFMatcher(cv2.NORM_L2).knnMatch(q, t, k=2)
    np.savez_compressed(os.path.join(HERE, "cfg2_bfmatcher.npz"),
                        idx=np.array([[m[0].trainIdx, m[1].trainIdx] for m in kn], np.int32),
                        dist=np.array([[m[0].distance, m[1].distance] for m in kn], np.float32),
                        q_sha1=hashlib.sha1(q.tobytes()).hexdigest(), t_sha1=hashlib.sha1(t.tobytes()).hexdigest())


def inverse3():
    """cv2.invert of the 3x3 matrices tests/test_oracle.py inverts: 20 normal draws and the oracle's eular2rot([0.3, -1.1, 2])."""
    import oracle as O

    rng = np.random.default_rng(0)
    A = np.stack([rng.normal(size=(3, 3)) for _ in range(20)])
    R = O.eular2rot([0.3, -1.1, 2.0])
    np.savez_compressed(os.path.join(HERE, "inv3.npz"), A=A, A_inv=np.stack([cv2.invert(a)[1] for a in A]),
                        R=R, R_inv=cv2.invert(R)[1])


if __name__ == "__main__":
    matching()
    svd_and_decompose()
    eight_point_cases()
    cfg2_matching()
    inverse3()
    print("golden fixtures written to", HERE)
