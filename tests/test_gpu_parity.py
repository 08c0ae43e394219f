"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU
oracle on the same seeded inputs, against the committed cv2 golden vectors, and -- at
BASELINE.json's full sizes -- through size-independent properties.

Bars (north_star): match indices and distances bit-exact (the oracle and the device spell
the same fp64 chain); inlier counts and masks bit-exact (same fp32 fma chain); E within 1e-5
Frobenius after sign/scale normalisation given the same samples; poses within 1e-5.
"""
import hashlib
import os

import numpy as np
import pytest

import erp_match_eightpoint_test_b200 as erp
import oracle as O
from conftest import GOLDEN, e_dist
from erp_match_eightpoint_test_b200 import binding, synth
from test_gpu_geometry_edges import planted_reference, rank2_bar

pytestmark = pytest.mark.gpu

E_TOL = 1e-5        # north_star: ||E_dev - E_ref||_F after sign and scale normalisation
POSE_TOL = 1e-5


@pytest.fixture(scope="module")
def ctx():
    c = erp.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def scene():
    kp = synth.keypoint_pair(3000, 4096, 2048, seed=9)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    return kp, l, r


def engines():
    return [binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X, binding.ENGINE_AUTO]


# ------------------------------------------------------------------ matching
@pytest.mark.parametrize("engine", engines())
@pytest.mark.parametrize("nq,nt,dim", [(1000, 1500, 64), (517, 733, 128), (64, 2, 64), (1, 300, 64),
                                        (333, 4097, 64), (200, 300, 4), (130, 140, 100)])
def test_knn2_bit_exact_vs_oracle(ctx, engine, nq, nt, dim):
    ctx.set_engine(engine)
    q, t, _ = synth.descriptor_pair(nq, nt, dim, seed=nq + nt)
    if nt > 40:
        t[37] = t[12]; t[5] = t[12]; q[0] = t[12]            # exact ties -> lowest trainIdx first
    idx, dist = ctx.knn2_raw(q, t)
    oidx, odist, _ = O.knn2(q, t)
    assert np.array_equal(idx, oidx)
    assert np.array_equal(dist.view(np.uint32), odist.view(np.uint32))   # bit-exact distances
    ctx.set_engine(binding.ENGINE_AUTO)


@pytest.mark.parametrize("engine", engines())
@pytest.mark.parametrize("name", ["m64", "m128"])
def test_knn2_matches_cv2_golden(ctx, golden, engine, name):
    ctx.set_engine(engine)
    g = golden["matching"]
    idx, dist = ctx.knn2_raw(g[name + "_q"], g[name + "_t"])
    assert np.array_equal(idx, g[name + "_idx"])
    assert np.allclose(dist, g[name + "_dist"], rtol=2e-6, atol=1e-7)     # cv2 sums in fp32 lanes
    m = ctx.knn2_match(g[name + "_q"], g[name + "_t"], ratio=-1.0, cross_check=True)
    assert np.array_equal(np.stack([m["queryIdx"], m["trainIdx"]], 1), g[name + "_cross"])
    ctx.set_engine(binding.ENGINE_AUTO)


@pytest.mark.parametrize("engine", engines())
@pytest.mark.parametrize("ratio,cross", [(0.3, False), (-1.0, False), (0.3, True), (0.8, True)])
def test_match_two_image_records(ctx, engine, ratio, cross):
    ctx.set_engine(engine)
    q, t, planted = synth.descriptor_pair(2500, 2200, 64, seed=5)
    got = ctx.knn2_match(q, t, ratio=ratio, cross_check=cross)
    want = O.match(q, t, ratio=ratio, cross_check=cross)
    assert got.dtype == binding.DMATCH and len(got) == len(want)
    assert got.tobytes() == want.tobytes()                                 # every field, bit for bit
    assert (np.diff(got["queryIdx"]) > 0).all()                            # ascending queryIdx
    if ratio == 0.3 and not cross:
        assert (planted[got["queryIdx"]] == got["trainIdx"]).all()
    ctx.set_engine(binding.ENGINE_AUTO)


@pytest.mark.parametrize("tc_engine,kappa", [(binding.ENGINE_TCGEN05, 2.0 ** -14), (binding.ENGINE_TCGEN05_1X, 2.0 ** -10)])
@pytest.mark.parametrize("nq,nt,dim", [(5000, 7000, 64), (3000, 4000, 128), (2000, 2500, 32), (1500, 1500, 96),
                                        (700, 900, 100), (129, 257, 64), (128, 256, 64), (4000, 300, 64), (257, 5000, 64)])
def test_tcgen05_engine_certifies_and_matches_exact(ctx, nq, nt, dim, tc_engine, kappa):
    """The tensor-core engine must (1) return exactly what the fp64 SIMT engine returns, (2) certify
    nearly every query itself (a broken tile layout would push everything through the re-scan and
    still pass (1)), (3) stay far inside the certificate's error budget KAPPA = 2^-14."""
    q, t, _ = synth.descriptor_pair(nq, nt, dim, seed=3 * nq + nt)
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    eidx, edist = ctx.knn2_raw(q, t)
    ctx.set_engine(tc_engine)
    idx, dist = ctx.knn2_raw(q, t)
    st = ctx.last_knn_stats()
    ctx.set_engine(binding.ENGINE_AUTO)
    assert st["engine"] == tc_engine
    assert np.array_equal(idx, eidx)
    assert np.array_equal(dist.view(np.uint32), edist.view(np.uint32))
    assert st["rescanned"] <= max(2, nq // 100), st
    assert 0 < st["deviation"] < kappa / 2, st


@pytest.mark.parametrize("tc_engine", [binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X])
def test_tcgen05_engine_adversarial_inputs(ctx, tc_engine):
    """Duplicated rows (more duplicates than the candidate list holds), un-normalised and widely
    scaled descriptors, zero rows: everything the certificate cannot prove must be re-scanned."""
    rng = np.random.default_rng(5)
    q = rng.normal(size=(600, 64)).astype(np.float32) * rng.uniform(0.01, 50.0, (600, 1)).astype(np.float32)
    t = rng.normal(size=(900, 64)).astype(np.float32) * rng.uniform(0.01, 50.0, (900, 1)).astype(np.float32)
    t[100:110] = t[7]            # 11 identical train rows
    q[3] = t[7]
    q[4] = 0
    t[50] = 0
    t[51] = 0
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    eidx, edist = ctx.knn2_raw(q, t)
    ctx.set_engine(tc_engine)
    idx, dist = ctx.knn2_raw(q, t)
    ctx.set_engine(binding.ENGINE_AUTO)
    assert np.array_equal(idx, eidx)
    assert np.array_equal(dist.view(np.uint32), edist.view(np.uint32))
    oidx, odist, _ = O.knn2(q, t)
    assert np.array_equal(idx, oidx)


@pytest.mark.parametrize("engine", [binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X])
@pytest.mark.parametrize("shape", [(300, 400), (5000, 6000)])
def test_nan_descriptors_never_match(ctx, engine, shape):
    """A descriptor row holding a NaN compares false against everything (src/feature_matcher.cpp:52 on a NaN distance):
    such a query has no neighbours (index -1) and emits no record, such a train row is never anyone's neighbour, with
    and without cross-check, and every other row is unaffected.  Same as the oracle."""
    nq, nt = shape
    q, t, _ = synth.descriptor_pair(nq, nt, 64, seed=3)
    q[5, 7] = np.nan; q[9, :] = np.nan; t[11, 3] = np.nan
    oidx, _, _ = O.knn2(q, t)
    assert (oidx[[5, 9]] == -1).all() and not (oidx == 11).any()
    ctx.set_engine(engine)
    try:
        idx, _ = ctx.knn2_raw(q, t)
        assert np.array_equal(idx, oidx)
        for ratio, cross in ((0.8, False), (-1.0, True), (0.8, True)):
            assert ctx.knn2_match(q, t, ratio, cross).tobytes() == O.match(q, t, ratio, cross).tobytes(), (ratio, cross)
    finally:
        ctx.set_engine(binding.ENGINE_AUTO)


def test_match_edge_cases(ctx):
    q, t, _ = synth.descriptor_pair(10, 5, 64, seed=1)
    assert len(ctx.knn2_match(q[:0], t)) == 0                              # empty query set
    with pytest.raises(erp.ErpError) as ei:                                # knnMatch(k=2) on one row
        ctx.knn2_match(q, t[:1])
    assert ei.value.status == binding.E_TOO_FEW_TRAIN
    with pytest.raises(erp.ErpError) as ei:
        ctx.knn2_match(q[:, :63], t[:, :63])
    assert ei.value.status == binding.E_DIM
    # cv::Mat with a row step larger than the row (a column range of a wider matrix)
    wide = np.zeros((10, 96), np.float32)
    wide[:, :64] = q
    sub = wide[:, :64]
    lib = erp.lib()
    out = np.empty(10, binding.DMATCH)
    n = np.zeros(1, np.int32)
    import ctypes
    st = lib.erp_knn2_match(ctx._h, sub.ctypes.data, 10, sub.strides[0], t.ctypes.data, 5, t.strides[0], 64,
                            -1.0, 0, out.ctypes.data, n.ctypes.data_as(ctypes.POINTER(ctypes.c_int)))
    assert st == 0 and out[: n[0]].tobytes() == O.match(q, t, ratio=-1.0).tobytes()


# ------------------------------------------------------------------ geometry
def test_bearings(ctx):
    kp = synth.keypoint_pair(5000, 8192, 4096, seed=2)
    for xy in (kp["left_xy"], kp["right_xy"]):
        got, want = ctx.bearings(xy, 8192, 4096), O.bearings(xy, 8192, 4096)
        assert np.abs(got - want).max() < 1e-14           # CUDA sincos vs glibc: a few ulp
        assert np.abs(np.linalg.norm(got, axis=1) - 1).max() < 1e-14
    assert ctx.bearings(kp["left_xy"][:0], 8192, 4096).shape == (0, 3)


def test_philox_table_matches_oracle(ctx):
    for (seed, off, H, S, m) in [(7, 0, 500, 8, 3000), (2**40 + 3, 10**6, 64, 8, 9), (1, 5, 33, 12, 40), (9, 0, 10, 8, 8)]:
        got = ctx.philox_samples(seed, off, H, S, m)
        want = np.stack([O.philox_samples(seed, off + h, m, S) for h in range(H)])
        assert np.array_equal(got, want)


def _pose_close(pose, ref):
    """pose: 12 floats (R1e, R2e, T, v1, v2).  {R1,R2} compared as a set: which rotation is
    called R1 depends on the sign of a numerically-zero singular vector (DESIGN.md)."""
    a = np.abs(pose[0:3] - ref["R1"]).max() + np.abs(pose[3:6] - ref["R2"]).max()
    b = np.abs(pose[0:3] - ref["R2"]).max() + np.abs(pose[3:6] - ref["R1"]).max()
    swapped = b < a
    v = (bool(pose[9]), bool(pose[10]))
    vref = (ref["R1_valid"], ref["R2_valid"])
    if swapped:
        vref = vref[::-1]
    return min(a, b), np.abs(pose[6:9] - ref["T"]).max(), v == vref


@pytest.mark.parametrize("S", [8, 9, 16, 32])
def test_eight_point_batch_minimal_samples(ctx, scene, S):
    kp, l, r = scene
    H = 400
    samples = ctx.philox_samples(11, 0, H, S, len(l))
    E, pose = ctx.eight_point_batch(l, r, samples=samples)
    Ephi, _ = ctx.eight_point_batch(l, r, H=H, S=S, seed=11, hyp_offset=0, want_pose=False)
    assert np.array_equal(E, Ephi)                         # device-drawn samples == replayed table
    # every sample against the 50-digit projection of its 50-digit null vector, within the conditioning-aware bar of
    # test_gpu_geometry_edges (kappa or kappa^2 of the S x 9 system, s1 / (s2 - s3) of the projected matrix)
    A = np.einsum("hna,hnb->hnab", l[samples], r[samples]).reshape(H, S, 9)
    sv, vt = np.linalg.svd(A)[1:]
    worst = 0.0
    for h in range(H):
        ref = planted_reference(l[samples[h]], r[samples[h]], {S: (sv[h], vt[h, -1])}, sizes=(S,))[S]
        d, bar = e_dist(E[h], ref["Ec"]), rank2_bar(ref)
        assert d <= bar, (h, d, bar, ref["kappa"], ref["sigma"])
        worst = max(worst, d / bar)
        if sv[h, 7] / sv[h, 0] > 1e-5:                     # the oracle and the pose are checked where the oracle's SVD is
            oref = O.eight_point(l[samples[h]], r[samples[h]], null_mode=1)
            assert e_dist(E[h], oref["E"]) < E_TOL
            dr, dt, vok = _pose_close(pose[h], oref)
            assert dr < POSE_TOL * 10 and dt < POSE_TOL and vok, (h, dr, dt)
    print("S=%d: worst error / bar %.2e" % (S, worst))


def test_eight_point_estimation_and_golden(ctx, golden, scene):
    g = golden["eight_point"]
    for k in range(3):
        l, r = g[f"l{k}"], g[f"r{k}"]
        res = ctx.eight_point_estimation(l, r)
        assert e_dist(res["E"], g[f"Ec{k}"]) < E_TOL       # cv2.SVDecomp pipeline (eight_point.cpp:22-50)
        ref = O.eight_point(l, r, null_mode=0)
        assert e_dist(res["E"], ref["E"]) < 1e-8
    kp, l, r = scene
    inl = kp["inlier"]
    res = ctx.eight_point_estimation(l[inl], r[inl])
    ref = O.eight_point(l[inl], r[inl])
    assert e_dist(res["E"], ref["E"]) < 1e-8 and e_dist(res["E"], kp["E"]) < 5e-3
    pose = np.concatenate([res["R1"], res["R2"], res["T"], [res["R1_valid"], res["R2_valid"], 0]]).astype(np.float32)
    dr, dt, vok = _pose_close(pose, ref)
    assert dr < POSE_TOL and dt < POSE_TOL and vok
    with pytest.raises(erp.ErpError) as ei:
        ctx.eight_point_estimation(l[:7], r[:7])
    assert ei.value.status == binding.E_TOO_FEW_POINTS


# ------------------------------------------------------------------ scoring / RANSAC
@pytest.mark.parametrize("metric,tau", [(0, 0.002), (1, 0.002), (2, 0.002), (0, 0.01)])
@pytest.mark.parametrize("m", [3000, 777, 1])
def test_score_counts_bit_exact(ctx, scene, metric, tau, m):
    kp, l, r = scene
    E, _ = ctx.eight_point_batch(l, r, H=300, S=8, seed=5, want_pose=False)
    E = np.concatenate([E, kp["E"][None], -2.5 * kp["E"][None], np.zeros((1, 3, 3))])
    got = ctx.score(E, l[:m], r[:m], metric, tau)
    want = O.score(E, l[:m], r[:m], metric, tau)
    assert np.array_equal(got, want)
    mask, n = ctx.inlier_mask(kp["E"], l[:m], r[:m], metric, tau)
    assert np.array_equal(mask, O.inlier_mask(kp["E"], l[:m], r[:m], metric, tau)) and n == mask.sum() == got[300]


@pytest.mark.parametrize("tc_engine", [binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X])
def test_tcgen05_engine_ties_beyond_list_capacity(ctx, tc_engine):
    """Several train tiles with far more exact ties than a candidate list holds (40 copies of one row, 30 of a zero
    row), queries on and next to them, one all-zero query (every score equal): the list floor must bound what was
    pushed out and everything it cannot prove must come back through the exact re-scan."""
    rng = np.random.default_rng(11)
    t = synth.surf_like(3000, 64, rng)
    q = synth.surf_like(700, 64, rng)
    copies = rng.permutation(3000)[:40]
    t[copies] = t[copies[0]]
    zeros = rng.permutation(np.setdiff1d(np.arange(3000), copies))[:30]
    t[zeros] = 0
    q[0] = t[copies[0]]
    q[1] = t[copies[0]] + np.float32(1e-4) * rng.standard_normal(64).astype(np.float32)
    q[2] = 0
    q[3:40] = t[copies[0]] * rng.uniform(0.5, 1.5, (37, 1)).astype(np.float32)
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    eidx, edist = ctx.knn2_raw(q, t)
    ctx.set_engine(tc_engine)
    idx, dist = ctx.knn2_raw(q, t)
    ctx.set_engine(binding.ENGINE_AUTO)
    assert np.array_equal(idx, eidx)
    assert np.array_equal(dist.view(np.uint32), edist.view(np.uint32))


def test_host_call_with_query_chunks_equals_single_call(tmp_path):
    """$ERP_B200_HOST_CHUNKS pipelines the upload of a host-buffer call over query chunks (read once per process):
    results and statistics must not depend on the cut."""
    import subprocess, sys, textwrap
    code = textwrap.dedent("""
        import sys, numpy as np
        sys.path.insert(0, ".")
        import erp_match_eightpoint_test_b200 as erp
        from erp_match_eightpoint_test_b200 import binding, synth
        ctx = erp.Context(0)
        # AUTO, first in the process (no earlier search left a train operand in scratch): at 7 chunks the first one has
        # 256 rows (2.56e6 pairs, below the tensor-core threshold of a search on its own), the later ones 512 rows
        qa, ta, _ = synth.descriptor_pair(3001, 10000, 64, seed=10)
        idx, dist = ctx.knn2_raw(qa, ta)
        np.save(sys.argv[1] + "_idx_auto.npy", idx); np.save(sys.argv[1] + "_dist_auto.npy", dist)
        q, t, _ = synth.descriptor_pair(3001, 2500, 64, seed=9)
        for eng in (binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X):
            ctx.set_engine(eng)
            idx, dist = ctx.knn2_raw(q, t)
            m = ctx.knn2_match(q, t, 0.3, True)
            st = ctx.last_knn_stats()
            np.save(sys.argv[1] + f"_idx{eng}.npy", idx); np.save(sys.argv[1] + f"_dist{eng}.npy", dist)
            np.save(sys.argv[1] + f"_m{eng}.npy", m)
            print(eng, st["rescanned"])
        qb, tb, _ = synth.binary_pair(3001, 2500, 32, seed=11)
        for eng in (binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05_1X):
            ctx.set_engine(eng)
            idx, dist = ctx.knn2_raw_bin(qb, tb)
            np.save(sys.argv[1] + f"_idx_bin{eng}.npy", idx); np.save(sys.argv[1] + f"_dist_bin{eng}.npy", dist)
            for cross in (False, True):
                np.save(sys.argv[1] + f"_m{int(cross)}_bin{eng}.npy", ctx.knn2_match_bin(qb, tb, 0.8, cross))
        # the whole pair through one host-buffer call: with more than one chunk the descriptors travel behind the search
        ctx.set_engine(binding.ENGINE_AUTO)
        rng = np.random.default_rng(3)
        left = (rng.uniform(0, 1, (3001, 2)) * [4096, 2047]).astype(np.float32)
        right = (rng.uniform(0, 1, (2500, 2)) * [4096, 2047]).astype(np.float32)
        for cross in (False, True):
            pm, res = ctx.pair_pose(q, t, left, right, 4096, 2048, ratio=0.8, cross_check=cross, seed=3, H=3000)
            np.save(sys.argv[1] + f"_pm{int(cross)}.npy", pm)
            np.save(sys.argv[1] + f"_pres{int(cross)}.npy", np.frombuffer(np.array([res["packed"], res["count"]], np.uint64).tobytes() + res["mask"].tobytes() + res["E_refit"].tobytes(), np.uint8))
        ctx.close()
    """)
    import os
    outs = {}
    for chunks in ("1", "3", "7"):                   # 3 and 7: a short first chunk, then even ones (api.cu: chunk_bounds)
        env = dict(os.environ, ERP_B200_HOST_CHUNKS=chunks)
        base = str(tmp_path / f"c{chunks}")
        r = subprocess.run([sys.executable, "-c", code, base], env=env, capture_output=True, text=True, timeout=300,
                           cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        assert r.returncode == 0, r.stderr[-2000:]
        outs[chunks] = base
    for eng in (binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X):
        for what in ("idx", "dist", "m"):
            a = np.load(outs["1"] + f"_{what}{eng}.npy")
            for chunks in ("3", "7"):
                assert a.tobytes() == np.load(outs[chunks] + f"_{what}{eng}.npy").tobytes(), (eng, what, chunks)
    bin_outs = [f"{what}_bin{eng}" for eng in (binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05_1X) for what in ("idx", "dist", "m0", "m1")]
    for what in ["idx_auto", "dist_auto"] + bin_outs + ["pm0", "pm1", "pres0", "pres1"]:
        a = np.load(outs["1"] + f"_{what}.npy")
        assert len(a) > 8
        for chunks in ("3", "7"):
            assert a.tobytes() == np.load(outs[chunks] + f"_{what}.npy").tobytes(), (what, chunks)


@pytest.mark.parametrize("H,m,tau", [(5000, 3000, 0.002), (129, 257, 0.002), (20000, 777, 0.01), (3000, 3000, 1e-5),
                                      (1500, 100, 0.002), (40000, 2500, 0.0005),
                                      # the power-of-two scaling of the counting epilogue at both ends of its range
                                      (3000, 3000, 0.5), (2000, 1000, 4.0), (3000, 3000, 1e-9)])
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_tensor_core_best_search_is_exact(ctx, scene, H, m, tau, metric):
    """score_tc.cu bounds every hypothesis' inlier count with a 3xTF32 residual GEMM and re-scores the
    contenders exactly: winner, count (the packed word) and inlier mask must equal the all-SIMT path
    and the oracle, also when residuals crowd the threshold or tau is below the band width.  Sampson (1) and
    angular (2) residuals go through a per-hypothesis bound (tau s1 sqrt(max(|l|^2 + |r|^2)), sin(tau) s1 max|r|)."""
    kp, l, r = scene
    rng = np.random.default_rng(H + m)
    ll = np.concatenate([l, l[rng.integers(0, len(l), max(0, m - len(l)))]])[:m]
    rr = np.concatenate([r, r[rng.integers(0, len(r), max(0, m - len(r)))]])[:m]
    if metric and tau > 1.0:
        tau = 1.0                                           # an angle: sin(tau) stops growing at pi / 2
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    simt = ctx.ransac(ll, rr, seed=4, hyp_offset=10, H=H, S=8, metric=metric, tau=tau)
    ctx.set_engine(binding.ENGINE_TCGEN05)
    tc = ctx.ransac(ll, rr, seed=4, hyp_offset=10, H=H, S=8, metric=metric, tau=tau)
    ctx.set_engine(binding.ENGINE_AUTO)
    assert tc["packed"] == simt["packed"]
    assert np.array_equal(tc["mask"], simt["mask"]) and tc["count"] == simt["count"]
    if H * m <= 2 * 10 ** 6:
        assert tc["packed"] == O.ransac(ll, rr, seed=4, hyp0=10, H=H, S=8, metric=metric, tau=tau)["packed"]


@pytest.mark.parametrize("m,outliers,H", [(20000, 0.3, 30000), (20000, 0.85, 30000), (6000, 0.5, 50000), (2048, 0.3, 20000)])
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_tensor_core_best_search_with_pruning(ctx, m, outliers, H, metric):
    """Three-pass progressive pruning (bounds on a prefix, exact L*, survivors only for the rest): the
    winner must not depend on it, for high and low inlier ratios (pruning switches itself off), for all three residuals."""
    kp = synth.keypoint_pair(m, 8192, 4096, outlier_frac=outliers, seed=m + H)
    l, r = O.bearings(kp["left_xy"], 8192, 4096), O.bearings(kp["right_xy"], 8192, 4096)
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    simt = ctx.ransac(l, r, seed=9, hyp_offset=0, H=H, S=8, metric=metric, tau=0.002)
    ctx.set_engine(binding.ENGINE_TCGEN05)
    tc = ctx.ransac(l, r, seed=9, hyp_offset=0, H=H, S=8, metric=metric, tau=0.002)
    print("metric %d: search stats %s" % (metric, ctx.last_score_stats()))
    ctx.set_engine(binding.ENGINE_AUTO)
    assert tc["packed"] == simt["packed"] and tc["count"] == simt["count"]
    assert np.array_equal(tc["mask"], simt["mask"])
    if outliers <= 0.5:
        assert e_dist(tc["E_refit"], kp["E"]) < 2e-2


def test_ransac_on_keypoints_equals_ransac_on_bearings(ctx):
    """erp_ransac_pixels = erp_bearings_from_pixels (both views) + erp_ransac without the round trip of the bearings."""
    kp = synth.keypoint_pair(5000, 8192, 4096, seed=77)
    l, r = ctx.bearings(kp["left_xy"], 8192, 4096), ctx.bearings(kp["right_xy"], 8192, 4096)
    a = ctx.ransac(l, r, seed=3, hyp_offset=5, H=20000, S=8, metric=0, tau=0.002)
    b = ctx.ransac_pixels(kp["left_xy"], kp["right_xy"], 8192, 4096, seed=3, hyp_offset=5, H=20000, S=8, metric=0, tau=0.002)
    assert a["packed"] == b["packed"] and a["count"] == b["count"] and np.array_equal(a["mask"], b["mask"])
    assert np.array_equal(a["E_refit"], b["E_refit"]) and np.array_equal(a["pose"], b["pose"])
    # cv::KeyPoint records (28 bytes, pt first)
    rec = np.zeros((5000, 7), np.float32)
    rec[:, :2] = kp["left_xy"]
    c = ctx.ransac_pixels(rec, np.concatenate([kp["right_xy"], np.zeros((5000, 5), np.float32)], axis=1), 8192, 4096,
                          seed=3, hyp_offset=5, H=20000)
    assert c["packed"] == a["packed"]


def test_pair_pose_equals_the_separate_calls(ctx):
    """erp_pair_pose = erp_knn2_match + the caller's gather of the matched keypoints + erp_ransac_pixels."""
    q, t, planted = synth.descriptor_pair(4000, 5000, 64, seed=21)
    n_pl = int((planted >= 0).sum())
    kp = synth.keypoint_pair(n_pl, 4096, 2048, seed=22)
    rng = np.random.default_rng(23)
    left = (rng.uniform(0, 1, (4000, 2)) * [4096, 2047]).astype(np.float32)
    right = (rng.uniform(0, 1, (5000, 2)) * [4096, 2047]).astype(np.float32)
    qi = np.nonzero(planted >= 0)[0]
    left[qi] = kp["left_xy"]
    right[planted[qi]] = kp["right_xy"]
    for cross in (False, True):
        m = ctx.knn2_match(q, t, 0.3, cross)
        want = ctx.ransac_pixels(left[m["queryIdx"]], right[m["trainIdx"]], 4096, 2048, seed=5, hyp_offset=0, H=8192)
        got_m, got = ctx.pair_pose(q, t, left, right, 4096, 2048, ratio=0.3, cross_check=cross, seed=5, H=8192)
        assert got_m.tobytes() == m.tobytes()
        assert got["packed"] == want["packed"] and np.array_equal(got["mask"], want["mask"])
        assert np.array_equal(got["E_refit"], want["E_refit"]) and np.array_equal(got["pose"], want["pose"])
    # too few matches: the records still come back, the status says why there is no pose
    with pytest.raises(erp.ErpError) as ei:
        ctx.pair_pose(q[:50], t, left[:50], right, 4096, 2048, ratio=1e-9, H=64)      # nothing passes such a ratio test
    assert ei.value.status == binding.E_TOO_FEW_POINTS


def test_two_contexts_on_two_host_threads(ctx):
    """One context per host thread (INTEGRATION.md): two threads with a context each, interleaving pairs on the same
    GPU, return exactly what a single context returns (cfg5: frame pairs of a video are sharded this way)."""
    import threading
    pairs = []
    for i in range(3):
        q, t, planted = synth.descriptor_pair(3000 + 64 * i, 3500, 64, seed=31 + i)
        rng = np.random.default_rng(100 + i)
        left = (rng.uniform(0, 1, (len(q), 2)) * [4096, 2047]).astype(np.float32)
        right = (rng.uniform(0, 1, (len(t), 2)) * [4096, 2047]).astype(np.float32)
        kp = synth.keypoint_pair(int((planted >= 0).sum()), 4096, 2048, seed=200 + i)
        qi = np.nonzero(planted >= 0)[0]
        left[qi] = kp["left_xy"]
        right[planted[qi]] = kp["right_xy"]
        pairs.append((q, t, left, right))
    want = [ctx.pair_pose(q, t, l, r, 4096, 2048, seed=2, H=4096) for q, t, l, r in pairs]
    got = [None] * 12
    errs = []

    def work(tid):
        try:
            c = erp.Context(0)
            for i in range(tid, 12, 2):
                q, t, l, r = pairs[i % 3]
                got[i] = c.pair_pose(q, t, l, r, 4096, 2048, seed=2, H=4096)
            c.close()
        except Exception as e:          # surfaced below: an exception in a thread would otherwise pass silently
            errs.append(e)

    ts = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
    for i in range(12):
        m, r = got[i]
        wm, wr = want[i % 3]
        assert m.tobytes() == wm.tobytes() and r["packed"] == wr["packed"] and np.array_equal(r["mask"], wr["mask"])


def test_refit_on_inliers(ctx, scene):
    kp, l, r = scene
    mask = O.inlier_mask(kp["E"], l, r)
    E, pose = ctx.refit(l, r, mask)
    ref = O.eight_point(l[mask > 0], r[mask > 0])
    assert e_dist(E, ref["E"]) < 1e-8
    dr, dt, vok = _pose_close(pose, ref)
    assert dr < POSE_TOL and dt < POSE_TOL and vok


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_ransac_same_winner_same_inliers(ctx, scene, metric):
    kp, l, r = scene
    H = 1500
    got = ctx.ransac(l, r, seed=42, hyp_offset=0, H=H, S=8, metric=metric, tau=0.002)
    want = O.ransac(l, r, seed=42, hyp0=0, H=H, S=8, metric=metric, tau=0.002)
    assert got["packed"] == want["packed"]                 # same hypothesis, same inlier count
    assert e_dist(got["E"], want["E"]) < E_TOL
    omask = O.inlier_mask(want["E"], l, r, metric, 0.002)
    assert np.array_equal(got["mask"], omask) and got["n_refit"] == got["count"] == omask.sum()
    ref = O.eight_point(l[omask > 0], r[omask > 0])
    assert e_dist(got["E_refit"], ref["E"]) < 1e-8
    assert e_dist(got["E_refit"], kp["E"]) < 5e-3          # and it is the right answer
    # sharded hypothesis ranges: max of the packed words == the single-range result
    a = ctx.ransac(l, r, seed=42, hyp_offset=0, H=700, S=8, metric=metric)
    b = ctx.ransac(l, r, seed=42, hyp_offset=700, H=800, S=8, metric=metric)
    assert max(a["packed"], b["packed"]) == got["packed"]


# ------------------------------------------------------------------ reference mode
@pytest.mark.parametrize("m", [2000, 400, 100, 50, 40])
def test_initial_guess_reference_mode(ctx, m):
    """eight_point::initial_guess with the libstdc++/glibc sample replay (H=80, S=m/4)."""
    kp = synth.keypoint_pair(m, 4096, 2048, noise_px=0.3, outlier_frac=0.0, seed=60 + m)
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    table = O.ref_sample_table(m)
    got = ctx.initial_guess(l, r)                          # samples=None -> in-library replay
    want = O.initial_guess(l, r, table, null_mode=1)
    assert len(got["cand_R"]) == len(want["cand_R"])
    # candidate lists agree as multisets of (R, T) (R1/R2 order inside one hypothesis may swap)
    key = lambda R, T: np.lexsort(np.round(np.concatenate([R, T], 1), 4).T[::-1])
    gi, wi = key(got["cand_R"], got["cand_T"]), key(want["cand_R"], want["cand_T"])
    assert np.abs(got["cand_R"][gi] - want["cand_R"][wi]).max() < 1e-4
    assert np.abs(got["R"] - want["R"]).max() < POSE_TOL and np.abs(got["T"] - want["T"]).max() < POSE_TOL
    assert np.rad2deg(np.abs(got["R"] - O.rot2eular(kp["R"].T))).mean() < 1.0   # two_synthesis_image_test bar


def test_find_end_to_end(ctx):
    kp = synth.keypoint_pair(1200, 4096, 2048, euler_deg=(10, 5, 20), noise_px=0.3, outlier_frac=0.0, seed=77)
    R, T = ctx.find(4096, 2048, kp["left_xy"], kp["right_xy"])
    l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
    want = O.initial_guess(l, r, O.ref_sample_table(1200))
    assert np.abs(R - want["R"]).max() < POSE_TOL and np.abs(T - want["T"]).max() < POSE_TOL
    # match_size smaller than the keypoint vectors (two_real_image_test/main.cpp:278-286)
    R2, T2 = ctx.find(4096, 2048, kp["left_xy"], kp["right_xy"], match_size=100)
    w2 = O.initial_guess(l[:100], r[:100], O.ref_sample_table(100))
    assert np.abs(R2 - w2["R"]).max() < POSE_TOL
    with pytest.raises(erp.ErpError) as ei:                # S = int(20*0.25) = 5 < 8
        ctx.find(4096, 2048, kp["left_xy"], kp["right_xy"], match_size=20)
    assert ei.value.status == binding.E_TOO_FEW_POINTS


# ------------------------------------------------------------------ BASELINE sizes, properties
def test_cfg2_full_size_properties(ctx):
    """configs[1]: 20k x 20k SURF-64 + 10k hypotheses on one GPU."""
    q, t, planted = synth.descriptor_pair(20000, 20000, 64, seed=synth.SEED_BASE + 1)
    m = ctx.knn2_match(q, t, ratio=0.3)
    assert len(m) == (planted >= 0).sum() and (planted[m["queryIdx"]] == m["trainIdx"]).all()
    # a 1/16 sub-sample of the queries checked exactly against the oracle
    sub = np.arange(0, 20000, 16)
    idx, dist = ctx.knn2_raw(q, t)
    oidx, odist, _ = O.knn2(q[sub], t)
    assert np.array_equal(idx[sub], oidx) and np.array_equal(dist[sub], odist)
    # cross-check is idempotent and symmetric: matching t->q gives the mirrored pairs
    a = ctx.knn2_match(q, t, ratio=-1.0, cross_check=True)
    b = ctx.knn2_match(t, q, ratio=-1.0, cross_check=True)
    assert set(zip(a["queryIdx"].tolist(), a["trainIdx"].tolist())) == set(zip(b["trainIdx"].tolist(), b["queryIdx"].tolist()))
    kp = synth.keypoint_pair(len(m), 4096, 2048, seed=synth.SEED_BASE + 2)
    l, r = ctx.bearings(kp["left_xy"], 4096, 2048), ctx.bearings(kp["right_xy"], 4096, 2048)
    res = ctx.ransac(l, r, seed=1, hyp_offset=0, H=10000)
    assert e_dist(res["E_refit"], kp["E"]) < 5e-3 and res["count"] > 0.55 * len(m)
    assert res["mask"].sum() == res["count"]
    assert (res["mask"][kp["inlier"]].mean() > 0.8) and (res["mask"][~kp["inlier"]].mean() < 0.1)


def test_cfg3_full_size_tensor_core_equals_exact_engine(ctx):
    """configs[2] at full size on one GPU: 100k x 100k SURF-64.  The tcgen05 engine must return
    exactly what the fp64 SIMT engine returns for every one of the 100k queries, certify (nearly) all
    of them itself, and the 1M-hypothesis RANSAC must find the planted geometry; a 1/64 sub-sample of
    the queries is also checked against the CPU oracle."""
    q, t, planted = synth.descriptor_pair(100000, 100000, 64, seed=synth.SEED_BASE + 3)
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    eidx, edist = ctx.knn2_raw(q, t)
    for eng, kappa in ((binding.ENGINE_TCGEN05, 2.0 ** -14), (binding.ENGINE_TCGEN05_1X, 2.0 ** -10)):
        ctx.set_engine(eng)
        idx, dist = ctx.knn2_raw(q, t)
        st = ctx.last_knn_stats()
        m = ctx.knn2_match(q, t, ratio=0.3)
        assert np.array_equal(idx, eidx) and np.array_equal(dist.view(np.uint32), edist.view(np.uint32))
        assert st["rescanned"] <= 100 and st["deviation"] < kappa / 2, st
    ctx.set_engine(binding.ENGINE_AUTO)
    assert len(m) == (planted >= 0).sum() and (planted[m["queryIdx"]] == m["trainIdx"]).all()
    assert (np.diff(m["queryIdx"]) > 0).all()
    # the host-buffer call cuts the queries differently for pageable (above: 1/8 + 3/8 + 1/2) and pinned sources (5/32 + 27/32)
    import torch
    pq, pt = torch.from_numpy(q).pin_memory().numpy(), torch.from_numpy(t).pin_memory().numpy()
    assert ctx.knn2_match(pq, pt, ratio=0.3).tobytes() == m.tobytes()
    del pq, pt
    sub = np.arange(0, 100000, 64)
    oidx, odist, _ = O.knn2(q[sub], t)
    assert np.array_equal(idx[sub], oidx) and np.array_equal(dist[sub], odist)
    kp = synth.keypoint_pair(len(m), 8192, 4096, seed=synth.SEED_BASE + 4)
    l, r = ctx.bearings(kp["left_xy"], 8192, 4096), ctx.bearings(kp["right_xy"], 8192, 4096)
    res = ctx.ransac(l, r, seed=1, hyp_offset=0, H=1000000)
    ps = ctx.last_score_stats()
    assert e_dist(res["E_refit"], kp["E"]) < 5e-3 and res["count"] > 0.6 * len(m)
    assert res["mask"].sum() == res["count"] == res["n_refit"]
    assert 0 < ps["survivors"] < ps["hyps"] // 4 and ps["lstar"] <= res["count"]      # pruning was active and sound
    # hypothesis sharding: the max of the packed words of two id ranges is the single-range winner
    a = ctx.ransac(l, r, seed=1, hyp_offset=0, H=400000)
    b = ctx.ransac(l, r, seed=1, hyp_offset=400000, H=600000)
    assert max(a["packed"], b["packed"]) == res["packed"]
    # the same million hypotheses scored one by one with the fp32 chain (SIMT engine, 5e10 residuals): same packed winner,
    # same mask -- the tensor-core search with exact pruning is checked at FULL size, not only through properties
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    full = ctx.ransac(l, r, seed=1, hyp_offset=0, H=1000000)
    ctx.set_engine(binding.ENGINE_AUTO)
    assert full["packed"] == res["packed"] and np.array_equal(full["mask"], res["mask"])
    assert np.array_equal(full["E_refit"], res["E_refit"])


def test_cfg2_full_size_against_cv2_bfmatcher_with_near_tie_report(ctx):
    """configs[1] at full size against the third-party matcher itself: cv2.BFMatcher(NORM_L2).knnMatch(k=2) computes
    and compares in fp32 (as src/feature_matcher.cpp:45,52 does); the device result is exact.  north_star: indices
    bit-exact except for documented fp32 distance ties.  Every query on which cv2 returns another index must be in the
    near-tie report (erp_knn2_near_ties); the report itself is checked against its definition on a sub-sample.
    cv2's output is tests/golden/cfg2_bfmatcher.npz (written by tests/golden/make_golden.py from these inputs)."""
    q, t, planted = synth.descriptor_pair(20000, 20000, 64, seed=synth.SEED_BASE + 1)
    t[137] = t[12]; t[5] = t[12]; q[3] = t[12]                          # exact ties: lowest trainIdx first, on both sides
    g = np.load(os.path.join(GOLDEN, "cfg2_bfmatcher.npz"))
    assert hashlib.sha1(q.tobytes()).hexdigest() == g["q_sha1"] and hashlib.sha1(t.tobytes()).hexdigest() == g["t_sha1"]
    cidx, cdist = g["idx"], g["dist"]
    idx, dist = ctx.knn2_raw(q, t)
    # fp32 accumulation of 64 terms: documented tolerance of the report = 64 * 2^-24 relative on the distance
    tol = 64 * 2.0 ** -24
    flags = ctx.knn2_near_ties(q, t, tol)
    bad = np.nonzero((idx != cidx).any(1))[0]
    print("cfg2 vs cv2.BFMatcher: %d of %d queries differ, %d flagged as near ties at rel_tol %.1e (%d at 1e-6)" %
          (len(bad), len(q), (flags != 0).sum(), tol, (ctx.knn2_near_ties(q, t, 1e-6) != 0).sum()))
    assert (flags[bad] != 0).all(), bad[flags[bad] == 0][:10]
    assert len(bad) <= 20
    ok = np.setdiff1d(np.arange(len(q)), bad)
    assert np.abs(dist[ok].astype(np.float64) - cdist[ok]).max() <= 4e-6 * dist.max()      # cv2's distances are fp32 sums
    # the report is what its definition says (numpy fp64, 256 queries incl. the planted ties)
    sub = np.concatenate([np.arange(0, 20000, 80), bad[:6]]).astype(np.int64)
    q64, t64 = q[sub].astype(np.float64), t.astype(np.float64)
    for j, i in enumerate(sub):
        d = np.sqrt(((t64 - q64[j]) ** 2).sum(1))
        d0, d1 = d[idx[i, 0]], d[idx[i, 1]]
        others = np.ones(len(t), bool)
        others[idx[i]] = False
        want = (1 if d1 - d0 <= tol * d1 else 0) | (2 if (d[others] <= d1 * (1 + tol)).any() else 0)
        assert flags[i] == want, (i, flags[i], want)
    assert flags[3] & 1 or flags[3] & 2                                                     # the planted triple tie is reported


def test_one_product_engine_worst_case_rounding(ctx):
    """Adversarial input for the 1xTF32 certificate (kappa = 1.05 * 2^-10): every component of every descriptor sits just
    below a tf32 rounding midpoint (v0 + 2^-11 - 2^-18 with v0 a tf32 value close to 1), all positive and of nearly equal
    norm, so BOTH operands of every product round down by almost 2^-11 and no error cancels; half of the queries are
    exact copies of train rows (q.t = |t|^2).  The observed deviation approaches 2^-10 (|q|^2 + max|t|^2); the result
    must still equal the fp64 engine bit for bit, with or without re-scans."""
    rng = np.random.default_rng(7)
    nq, nt = 3000, 5000
    for dim in (64, 128):
        def adversarial(n):
            # tf32 values 1 + m / 1024 with small m, plus just under half a tf32 ulp: cvt.rna rounds DOWN by ~2^-11 relative
            m = rng.integers(0, 64, size=(n, dim)).astype(np.float64)
            return np.ascontiguousarray((1.0 + m / 1024.0 + 2.0 ** -11 - 2.0 ** -18).astype(np.float32))
        t = adversarial(nt)
        q = adversarial(nq)
        q[: nq // 2] = t[rng.permutation(nt)[: nq // 2]]                 # exact copies: q.t = |t|^2, the error term is maximal
        ctx.set_engine(binding.ENGINE_EXACT_SIMT)
        eidx, edist = ctx.knn2_raw(q, t)
        ctx.set_engine(binding.ENGINE_TCGEN05_1X)
        idx, dist = ctx.knn2_raw(q, t)
        st = ctx.last_knn_stats()
        ctx.set_engine(binding.ENGINE_AUTO)
        assert np.array_equal(idx, eidx) and np.array_equal(dist.view(np.uint32), edist.view(np.uint32))
        print("worst-case rounding, D=%d: deviation %.3e = %.3f of 2^-10, %d re-scanned" % (dim, st["deviation"], st["deviation"] * 1024, st["rescanned"]))
        assert 0.8 * 2.0 ** -10 < st["deviation"] <= 1.05 * 2.0 ** -10, st


def test_cfg4_full_size_surf128_cross_check_properties(ctx):
    """configs[3] at full size: 200k x 200k SURF-128 with cross-check (4e10 dist-evals each way) through the host-buffer
    call.  Size-independent properties: every planted pair is found and nothing else passes ratio + cross-check;
    records ascend; matching t -> q gives the mirrored pairs; a sub-sample of the rows equals the fp64 SIMT engine
    bit for bit and a smaller one equals the oracle."""
    n = 200000
    q, t, planted = synth.descriptor_pair(n, n, 128, seed=synth.SEED_BASE + 5)
    m = ctx.knn2_match(q, t, ratio=0.3, cross_check=True)
    st = ctx.last_knn_stats()
    assert st["engine"] == binding.ENGINE_TCGEN05_1X and st["rescanned"] <= n // 100, st
    assert len(m) == (planted >= 0).sum() and (planted[m["queryIdx"]] == m["trainIdx"]).all()
    assert (np.diff(m["queryIdx"]) > 0).all() and (m["imgIdx"] == 0).all()
    a = ctx.knn2_match(q, t, ratio=-1.0, cross_check=True)
    b = ctx.knn2_match(t, q, ratio=-1.0, cross_check=True)
    assert len(a) == len(b)
    order = np.lexsort((b["queryIdx"], b["trainIdx"]))
    assert np.array_equal(a["queryIdx"], b["trainIdx"][order]) and np.array_equal(a["trainIdx"], b["queryIdx"][order])
    idx, dist = ctx.knn2_raw(q, t)
    sub = np.arange(0, n, 97)
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    eidx, edist = ctx.knn2_raw(q[sub], t)
    ctx.set_engine(binding.ENGINE_AUTO)
    assert np.array_equal(idx[sub], eidx) and np.array_equal(dist[sub].view(np.uint32), edist.view(np.uint32))
    tiny = sub[::32]
    oidx, odist, _ = O.knn2(q[tiny], t)
    assert np.array_equal(idx[tiny], oidx) and np.array_equal(dist[tiny], odist)


@pytest.mark.parametrize("engine", [binding.ENGINE_EXACT_SIMT, binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X])
def test_cfg4_style_surf128_cross_check(ctx, engine):
    """configs[3] reduced: extended 128-D descriptors with cross-check matching, both engines."""
    q, t, _ = synth.descriptor_pair(6000, 7000, 128, seed=41)
    ctx.set_engine(engine)
    got = ctx.knn2_match(q, t, ratio=-1.0, cross_check=True)
    got_r = ctx.knn2_match(q, t, ratio=0.3, cross_check=True)
    ctx.set_engine(binding.ENGINE_AUTO)
    assert got.tobytes() == O.match(q, t, ratio=-1.0, cross_check=True).tobytes()
    assert got_r.tobytes() == O.match(q, t, ratio=0.3, cross_check=True).tobytes()


def test_rotation_grid_known_answer(ctx):
    """The reference's own test design: a grid of XYZ Euler rotations (one_image_test/main.cpp:73-80 uses
    {0,5,10,15,20} deg per axis) and the only numeric bar in the repository, mean |Euler error| < 1 deg
    (two_synthesis_image_test/main.cpp:132-141), on synthetic two-view keypoints through eight_point::find."""
    worst = 0.0
    for k, euler in enumerate([(0, 0, 0), (5, 0, 0), (0, 10, 0), (0, 0, 15), (20, 5, 10), (10, 20, 5), (15, 15, 15), (20, 20, 20)]):
        kp = synth.keypoint_pair(800, 4096, 2048, euler_deg=euler, noise_px=0.3, outlier_frac=0.0, seed=900 + k)
        R, T = ctx.find(4096, 2048, kp["left_xy"], kp["right_xy"])
        l, r = O.bearings(kp["left_xy"], 4096, 2048), O.bearings(kp["right_xy"], 4096, 2048)
        want = O.initial_guess(l, r, O.ref_sample_table(800))
        assert np.abs(R - want["R"]).max() < POSE_TOL and np.abs(T - want["T"]).max() < POSE_TOL
        # E = [t]x R^T in synth, so find() returns the Euler vector of R^T (l^T E r = 0 convention)
        err = np.rad2deg(np.abs(R - O.rot2eular(kp["R"].T))).mean()
        worst = max(worst, err)
        assert abs(abs(float(np.dot(T, kp["t"]))) - 1.0) < 5e-3          # translation direction up to sign
    assert worst < 1.0, worst
