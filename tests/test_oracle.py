"""CPU tests: the oracle against the committed cv2 golden vectors and against the
known-answer designs of the reference's own test mains (SURVEY.md section 8(c))."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle as O
from conftest import GOLDEN, e_dist
from erp_match_eightpoint_test_b200 import synth


# ---- matching (feature_matcher.cpp:42-59 as exact brute force) -------------------------
@pytest.mark.parametrize("name", ["m64", "m128"])
def test_knn2_matches_cv2_bfmatcher(golden, name):
    g = golden["matching"]
    idx, dist, _ = O.knn2(g[name + "_q"], g[name + "_t"])
    assert np.array_equal(idx, g[name + "_idx"])
    # cv2 accumulates in fp32 SIMD lanes; ours is fp64 -> distances agree to ~1e-6 relative
    assert np.allclose(dist, g[name + "_dist"], rtol=2e-6, atol=1e-7)
    # tie rule: rows 5, 12, 37 of train are identical; query 3 equals them -> lowest two indices
    assert idx[3].tolist() == [5, 12] and dist[3, 0] == 0.0


@pytest.mark.parametrize("name", ["m64", "m128"])
def test_cross_check_matches_cv2(golden, name):
    g = golden["matching"]
    m = O.match(g[name + "_q"], g[name + "_t"], ratio=-1.0, cross_check=True)
    got = np.stack([m["queryIdx"], m["trainIdx"]], 1)
    assert np.array_equal(got, g[name + "_cross"])


def test_ratio_test_semantics():
    q, t, planted = synth.descriptor_pair(500, 600, 64, seed=11)
    idx, dist, _ = O.knn2(q, t)
    m = O.match(q, t, ratio=0.3)
    keep = dist[:, 0] < np.float32(0.3) * dist[:, 1]          # strict <, fp32 product
    assert np.array_equal(m["queryIdx"], np.nonzero(keep)[0])  # ascending queryIdx
    assert np.array_equal(m["trainIdx"], idx[keep, 0])
    assert np.array_equal(m["distance"], dist[keep, 0]) and (m["imgIdx"] == 0).all()
    # planted matches are what survives (one_image_test's "match error ~ 0" design)
    assert (planted[m["queryIdx"]] == m["trainIdx"]).all() and len(m) == (planted >= 0).sum()


def test_match_empty_and_ragged():
    q, t, _ = synth.descriptor_pair(7, 2, 64, seed=3)
    assert len(O.match(q[:0], t)) == 0
    idx, _, _ = O.knn2(q, t)                                   # nt == 2: both rows returned
    assert np.array_equal(np.sort(idx, 1), np.tile([0, 1], (7, 1)))


# ---- OpenCV SVD / decomposeEssentialMat restatement ------------------------------------
def test_svd_matches_cv2(golden):
    g = golden["svd_decompose"]
    for i in range(4):
        A = g[f"A{i}"]
        w, u, vt = O.svd(A)
        assert vt.shape == g[f"vt{i}"].shape               # 8x9 -> vt is 8x9 (SURVEY D7)
        assert np.allclose(w, g[f"w{i}"], atol=1e-13)
        assert np.allclose(u @ np.diag(w) @ vt, A, atol=1e-13)
        for a, b in zip(vt, g[f"vt{i}"]):                   # LAPACK vs Jacobi: per-vector sign
            assert min(np.abs(a - b).max(), np.abs(a + b).max()) < 1e-12


def test_decompose_essential_matches_cv2(golden):
    g = golden["svd_decompose"]
    for E, c1, c2, ct in zip(g["E"], g["R1"], g["R2"], g["t"]):
        R1, R2, t = O.decompose_essential(E)
        d = min(np.abs(R1 - c1).max() + np.abs(R2 - c2).max(), np.abs(R1 - c2).max() + np.abs(R2 - c1).max())
        assert d < 1e-12
        assert min(np.abs(t - ct).max(), np.abs(t + ct).max()) < 1e-12
        assert abs(np.linalg.det(R1) - 1) < 1e-12 and abs(np.linalg.norm(t) - 1) < 1e-12


def test_eight_point_matches_cv2_pipeline(golden):
    g = golden["eight_point"]
    for k in range(3):
        l = O.bearings(g[f"lxy{k}"], 4096, 2048)
        r = O.bearings(g[f"rxy{k}"], 4096, 2048)
        assert np.abs(l - g[f"l{k}"]).max() < 1e-15 and np.abs(r - g[f"r{k}"]).max() < 1e-15
        res = O.eight_point(l, r, null_mode=0)
        assert e_dist(res["e"], g[f"e{k}"]) < 1e-9
        assert e_dist(res["E"], g[f"Ec{k}"]) < 1e-9
        R1, R2, _ = O.decompose_essential(res["E"])
        c1, c2 = g[f"R1_{k}"], g[f"R2_{k}"]
        assert min(np.abs(R1 - c1).max() + np.abs(R2 - c2).max(),
                   np.abs(R1 - c2).max() + np.abs(R2 - c1).max()) < 1e-8
        # null_mode only differs for fewer than 9 rows
        assert e_dist(O.eight_point(l, r, null_mode=1)["e"], res["e"]) < 1e-9


def test_n8_trap_documented():
    """SURVEY D7: for exactly 8 points the reference's vt.row(7) is not the null vector."""
    kp = synth.keypoint_pair(8, 4096, 2048, noise_px=0.0, outlier_frac=0.0, seed=5)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    A = np.einsum("na,nb->nab", l, r).reshape(8, 9)
    faithful = O.eight_point(l, r, null_mode=0)["e"].reshape(9)
    null = O.eight_point(l, r, null_mode=1)["e"].reshape(9)
    assert np.linalg.norm(A @ null) < 1e-12 < 1e-3 < np.linalg.norm(A @ faithful)
    assert e_dist(O.eight_point(l, r, null_mode=1)["E"], kp["E"]) < 1e-4


# ---- geometry known answers (one_image_test/main.cpp:73-91 design) ---------------------
def test_euler_round_trip():
    for x in (0, 5, 10, 15, 20):
        for y in (0, 5, 10, 15, 20):
            for z in (0, 5, 10, 15, 20):
                th = np.deg2rad([x, y, z])
                assert np.allclose(O.rot2eular(O.eular2rot(th)), th, atol=1e-12)
                assert np.allclose(O.eular2rot(th), synth.eular2rot(th), atol=1e-15)


@pytest.mark.parametrize("euler", [(0, 0, 0), (5, 10, 15), (20, 20, 20), (-15, 5, 0)])
def test_known_pose_recovery(euler):
    """two_synthesis_image_test/main.cpp:132-135: mean abs Euler error must stay below 1 degree."""
    kp = synth.keypoint_pair(400, 4096, 2048, euler_deg=euler, noise_px=0.3, outlier_frac=0.0, seed=21)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    ig = O.initial_guess(l, r, O.ref_sample_table(400))
    assert ig["rc"] == 0
    want = O.rot2eular(kp["R"].T)   # l^T E r = 0 with E = [t]x R^T  ->  decomposition yields R^T
    assert np.rad2deg(np.abs(ig["R"] - want)).mean() < 1.0
    assert min(np.abs(ig["T"] - kp["t"]).max(), np.abs(ig["T"] + kp["t"]).max()) < 0.05


@pytest.mark.parametrize("m", [100, 50, 40, 30, 20])
def test_truncated_match_counts(m):
    """two_real_image_test/main.cpp:240,278-286 truncates the matches to these sizes."""
    kp = synth.keypoint_pair(m, 4096, 2048, noise_px=0.1, outlier_frac=0.0, seed=33)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    ig = O.initial_guess(l, r, O.ref_sample_table(m))
    assert ig["rc"] == 0 and np.isfinite(ig["R"]).all()


# ---- sampling -------------------------------------------------------------------------
def test_random_array_replays_libstdcxx():
    """eight_point.hpp:54-58 compiled as written (g++, std::random_shuffle, unseeded rand())."""
    src = r"""
    #include <algorithm>
    #include <numeric>
    #include <vector>
    #include <cstdio>
    int main(){ for(int rep=0;rep<3;rep++){ std::vector<int> a(37); std::iota(a.begin(),a.end(),0);
      std::random_shuffle(a.begin(),a.end()); for(int v:a) std::printf("%d ",v);} return 0; }
    """
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "a.cpp"), "w") as f:
            f.write(src)
        subprocess.run(["/usr/bin/g++", "-std=gnu++11", "-w", "-o", os.path.join(d, "a"), os.path.join(d, "a.cpp")], check=True)
        out = subprocess.run([os.path.join(d, "a")], check=True, capture_output=True, text=True).stdout.split()
    want = np.array(out, np.int32).reshape(3, 37)
    got = O.ref_sample_table(37, H=3, S=37, reseed=1)
    assert np.array_equal(got, want)
    assert sorted(got[0].tolist()) == list(range(37))


def test_philox_samples_distinct_and_deterministic():
    for hyp in range(200):
        s = O.philox_samples(99, hyp, 50, 8)
        assert len(set(s.tolist())) == 8 and s.min() >= 0 and s.max() < 50
    assert np.array_equal(O.philox_samples(1, 2, 1000, 8), O.philox_samples(1, 2, 1000, 8))
    assert not np.array_equal(O.philox_samples(1, 2, 1000, 8), O.philox_samples(1, 3, 1000, 8))
    assert sorted(O.philox_samples(5, 0, 8, 8).tolist()) == list(range(8))   # M == S still terminates


# ---- consensus pick (eight_point.cpp:131-149) ------------------------------------------
def test_consensus_pick_numpy():
    rng = np.random.default_rng(4)
    for C in (1, 2, 5, 37, 160):
        R = rng.standard_normal((C, 3)).astype(np.float32) * 0.1
        R[: C // 2] *= 0.01
        got, tm = O.consensus_pick(R)
        d = np.sqrt(((R[:, None, :] - R[None, :, :]) ** 2).sum(-1, dtype=np.float32)).astype(np.float64)
        d.sort(axis=1)
        lo, hi = int(C * 0.2), int(C * 0.8)
        if hi > lo:
            want = np.array([np.add.reduce(row[lo:hi]) / (hi - lo) for row in d])
            assert np.allclose(tm, want, rtol=1e-12)
            assert got == int(np.argmin(want))
        else:
            assert got == 0


# ---- scoring / RANSAC -------------------------------------------------------------------
def test_score_against_numpy_and_mask():
    kp = synth.keypoint_pair(3000, 4096, 2048, seed=8)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    E = np.stack([kp["E"], kp["E"] * -3.0, np.eye(3)])
    c = O.score(E, l, r)
    res = np.abs(np.einsum("na,ab,nb->n", l, kp["E"] / np.linalg.norm(kp["E"]) * np.sqrt(2), r))
    near = np.abs(res - 0.002) < 1e-5                      # fp32 vs fp64 can differ only at the threshold
    assert abs(int(c[0]) - int((res < 0.002).sum())) <= near.sum()
    assert c[0] == c[1]                                     # scale and sign invariant
    assert c[0] > 0.6 * 3000 > c[2]
    mask = O.inlier_mask(kp["E"], l, r)
    assert mask.sum() == c[0]
    for metric in (O.METRIC_SAMPSON, O.METRIC_ANGULAR):
        cm = O.score(E, l, r, metric=metric, tau=0.002)
        assert cm[0] > 0.6 * 3000 > cm[2]


def test_ransac_recovers_pose_and_shards_agree():
    kp = synth.keypoint_pair(1500, 4096, 2048, seed=9)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    full = O.ransac(l, r, seed=7, hyp0=0, H=600)
    assert e_dist(full["E"], kp["E"]) < 0.02 and full["count"] > 0.5 * 1500
    a = O.ransac(l, r, seed=7, hyp0=0, H=300)
    b = O.ransac(l, r, seed=7, hyp0=300, H=300)
    assert max(a["packed"], b["packed"]) == full["packed"]     # the allreduce(max) contract
    assert np.array_equal(np.concatenate([a["counts"], b["counts"]]), full["counts"])


def test_inv3_is_opencv_closed_form():
    """cv::Mat::inv() on 3x3 CV_64F (erp_rotation.cpp:103): the oracle's closed form is bit-identical to cv2.invert
    (tests/golden/inv3.npz, written by tests/golden/make_golden.py)."""
    g = np.load(os.path.join(GOLDEN, "inv3.npz"))
    for A, A_inv in zip(g["A"], g["A_inv"]):
        assert np.array_equal(O.inv3(A), A_inv)
    R = g["R"]                                          # O.eular2rot([0.3, -1.1, 2.0])
    assert np.array_equal(O.inv3(R), g["R_inv"]) and np.abs(O.inv3(R) - R.T).max() < 1e-15


def test_rotate_pixel_round_trip_and_image_identity():
    """rotate_pixel with R then R^-1 returns to the start within a pixel (one_image_test-style known answer),
    and rotating an image by a rotation and back reproduces most of it."""
    R = O.eular2rot([0.2, 0.1, -0.4])
    rng = np.random.default_rng(1)
    W, H = 2048, 1024
    rc = np.stack([rng.integers(H // 3, 2 * H // 3, 5000), rng.integers(0, W, 5000)], 1).astype(np.int32)      # away from the poles
    back = O.rotate_pixels(O.rotate_pixels(rc, R, W, H), R.T, W, H)
    d = np.abs(back - rc)
    d[:, 1] = np.minimum(d[:, 1], W - d[:, 1])
    assert d.max() <= 3
    kp = O.rotate_keypoints([[100.0, 40.0], [2000.5, 200.25]], 0.0, W, H)     # pitch 0: only the strip offset H*3/8
    assert np.array_equal(kp[:, 1], [40 + H * 3 // 8, 200 + H * 3 // 8]) and np.abs(kp[:, 0] - [100, 2000]).max() <= 1
