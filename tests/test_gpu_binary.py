"""Binary descriptors on the B200: the tcgen05 kind::i8 engine, the SIMT popcount engine and the CPU reference
(tests/binary_ref.py) return identical 2-NN lists and match records, equal to cv2.BFMatcher(NORM_HAMMING) on the stored
fixtures, for every k-chunk count, ragged shapes and adversarial ties; the pair-pose calls chain into the RANSAC unchanged."""
import os

import numpy as np
import pytest

import binary_ref as B
import oracle as O
from conftest import GOLDEN
from erp_match_eightpoint_test_b200 import binding, synth

pytestmark = pytest.mark.gpu

I8, POPC = binding.ENGINE_TCGEN05_1X, binding.ENGINE_EXACT_SIMT
ENGINES = (I8, POPC)


@pytest.fixture(scope="module")
def ctx():
    c = binding.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def fx():
    return np.load(os.path.join(GOLDEN, "binary.npz"))


def _raw(ctx, engine, q, t):
    ctx.set_engine(engine)
    try:
        return ctx.knn2_raw_bin(q, t)
    finally:
        ctx.set_engine(binding.ENGINE_AUTO)


def _same(ctx, q, t, engines=ENGINES):
    want = B.knn2(q, t)
    for e in engines:
        idx, dist = _raw(ctx, e, q, t)
        assert np.array_equal(idx, want[0]), (e, np.nonzero((idx != want[0]).any(1))[0][:10])
        assert np.array_equal(dist, want[1]), e
    return want


def test_small_shape_i8_equals_popc_and_reference(ctx):
    q, t, _ = synth.binary_pair(300, 700, 32, seed=11)
    _same(ctx, q, t)


@pytest.mark.parametrize("nbytes", [1, 3, 16, 17, 32, 48, 61, 64])
def test_every_k_chunk_count(ctx, nbytes):
    q, t, _ = synth.binary_pair(1003, 2003, nbytes, seed=100 + nbytes)
    _same(ctx, q, t)


@pytest.mark.parametrize("nq,nt", [(1, 2), (2, 255), (255, 256), (256, 257), (257, 3003), (3003, 257), (4099, 5003)])
def test_ragged_shapes(ctx, nq, nt):
    q, t, _ = synth.binary_pair(nq, nt, 32, seed=nq * 7 + nt)
    _same(ctx, q, t)


def test_adversarial_ties(ctx):
    rng = np.random.default_rng(5)
    q = rng.integers(0, 256, (600, 32), dtype=np.uint8)
    q[:10] = 0
    q[10:20] = 255
    # every train row equal: the two lowest indices win everywhere
    _same(ctx, q, np.repeat(rng.integers(0, 256, (1, 32), dtype=np.uint8), 1500, axis=0))
    # all-zero and all-ones train rows among random ones
    t = rng.integers(0, 256, (3000, 32), dtype=np.uint8)
    t[[5, 700, 2999]] = 0
    t[[6, 701, 2998]] = 255
    _same(ctx, q, t)
    # the best and second best of each query duplicated across column groups (128), train tiles (256) and segments
    t = rng.integers(0, 256, (9000, 32), dtype=np.uint8)
    src = rng.integers(0, 100, 600)
    q = t[src].copy()
    for off in (128, 256, 1000, 4500, 8800):
        t[src + off] = t[src]
    q[::3, 0] ^= 1
    _same(ctx, q, t)


@pytest.mark.parametrize("ratio", [-1.0, 0.7, 0.8])
@pytest.mark.parametrize("cross_check", [False, True])
def test_match_records(ctx, ratio, cross_check):
    q, t, _ = synth.binary_pair(3000, 3500, 32, seed=21)
    want = B.match(q, t, ratio, cross_check)
    for e in ENGINES:
        ctx.set_engine(e)
        got = ctx.knn2_match_bin(q, t, ratio, cross_check)
        ctx.set_engine(binding.ENGINE_AUTO)
        assert got.tobytes() == want.tobytes(), e


@pytest.mark.parametrize("prefix", ["orb", "syn"])
def test_equal_cv2_on_fixtures(ctx, fx, prefix):
    if prefix == "orb":
        q, t = fx["orb_q"], fx["orb_t"]
    else:
        q, t, _ = synth.binary_pair(20000, 20000, 32)
    for e in ENGINES:
        idx, dist = _raw(ctx, e, q, t)
        assert np.array_equal(idx, fx[prefix + "_idx"]) and np.array_equal(dist, fx[prefix + "_dist"]), e
        ctx.set_engine(e)
        cc = ctx.knn2_match_bin(q, t, -1.0, True)
        ctx.set_engine(binding.ENGINE_AUTO)
        assert np.array_equal(np.stack([cc["queryIdx"], cc["trainIdx"]], 1), fx[prefix + "_cc"]), e
        assert np.array_equal(cc["distance"], fx[prefix + "_cc_dist"]), e


def test_host_strides_pinned_pageable_and_device(ctx):
    import torch

    q, t, _ = synth.binary_pair(2500, 2700, 32, seed=31)
    want = B.match(q, t, 0.8, True)
    wide_q = np.zeros((len(q), 48), np.uint8)
    wide_q[:, 5:37] = q
    wide_t = np.zeros((len(t), 40), np.uint8)
    wide_t[:, :32] = t
    for e in ENGINES:
        ctx.set_engine(e)
        assert ctx.knn2_match_bin(wide_q[:, 5:37], wide_t[:, :32], 0.8, True).tobytes() == want.tobytes()
        pq, pt = torch.from_numpy(q).pin_memory().numpy(), torch.from_numpy(t).pin_memory().numpy()
        assert ctx.knn2_match_bin(pq, pt, 0.8, True).tobytes() == want.tobytes()
        dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
        out = torch.zeros(len(q) * 16, dtype=torch.uint8, device="cuda")
        n = torch.zeros(1, dtype=torch.int32, device="cuda")
        ctx.knn2_match_bin_dev(dq, len(q), dt, len(t), 32, 0.8, True, out, n)
        ctx.synchronize()
        got = out.cpu().numpy()[: 16 * int(n.item())].view(binding.DMATCH)
        assert got.tobytes() == want.tobytes()
        idx = torch.zeros((len(q), 2), dtype=torch.int32, device="cuda")
        dist = torch.zeros((len(q), 2), dtype=torch.float32, device="cuda")
        d2 = torch.zeros((len(q), 2), dtype=torch.float64, device="cuda")
        ctx.knn2_bin_dev(dq, len(q), dt, len(t), 32, idx, dist, d2)
        ctx.synchronize()
        ref = B.knn2(q, t)
        assert np.array_equal(idx.cpu().numpy(), ref[0]) and np.array_equal(d2.cpu().numpy(), ref[1].astype(np.float64))
    ctx.set_engine(binding.ENGINE_AUTO)


def test_diagnostics(ctx):
    q, t, _ = synth.binary_pair(2000, 2000, 32, seed=41)
    for e, ops in ((I8, binding.OPERANDS_I8), (POPC, binding.OPERANDS_NONE)):
        ctx.set_engine(e)
        ctx.knn2_raw_bin(q, t)
        st = ctx.last_knn_stats()
        assert st["engine"] == e and st["rescanned"] == 0
        assert ctx.last_knn_operands()["operands"] == ops
        assert ctx.last_knn_kernel_ms() > 0
    ctx.set_engine(binding.ENGINE_TCGEN05)
    ctx.knn2_raw_bin(q, t)
    assert ctx.last_knn_operands()["operands"] == binding.OPERANDS_I8
    ctx.set_engine(binding.ENGINE_AUTO)
    # a float search afterwards reports its own operands again
    fq, ft, _ = synth.descriptor_pair(3000, 3000, 64, seed=1)
    ctx.set_engine(binding.ENGINE_TCGEN05_1X)
    ctx.knn2_raw(fq, ft)
    assert ctx.last_knn_operands()["operands"] == binding.OPERANDS_F16
    ctx.set_engine(binding.ENGINE_AUTO)


def _scene(nq=4000, nt=4200, W=4096, H=2048, seed=51):
    q, t, planted = synth.binary_pair(nq, nt, 32, f_match=0.6, seed=seed)
    qi = np.nonzero(planted >= 0)[0]
    kp = synth.keypoint_pair(len(qi), W, H, euler_deg=(5.0, 10.0, 15.0), noise_px=0.3, outlier_frac=0.0, seed=seed + 1)
    rng = np.random.default_rng(seed)
    lxy = (rng.uniform(0, 1, (nq, 2)) * [W, H - 1]).astype(np.float32)
    rxy = (rng.uniform(0, 1, (nt, 2)) * [W, H - 1]).astype(np.float32)
    lxy[qi] = kp["left_xy"]
    rxy[planted[qi]] = kp["right_xy"]
    return q, t, lxy, rxy, W, H, kp


def test_pair_pose_bin_equals_match_then_ransac_and_recovers_pose(ctx):
    q, t, lxy, rxy, W, H, kp = _scene()
    for e in ENGINES:
        ctx.set_engine(e)
        m, res = ctx.pair_pose_bin(q, t, lxy, rxy, W, H, ratio=0.8, seed=3, H=4096)
        want = ctx.knn2_match_bin(q, t, 0.8, False)
        assert m.tobytes() == want.tobytes()
        ref = ctx.ransac_pixels(lxy[want["queryIdx"]], rxy[want["trainIdx"]], W, H, seed=3, hyp_offset=0, H=4096)
        assert res["packed"] == ref["packed"] and np.array_equal(res["mask"], ref["mask"])
        assert res["E_refit"].tobytes() == ref["E_refit"].tobytes()
        truth = O.rot2eular(kp["R"].T)
        err = min(np.rad2deg(np.abs(res["pose"][0:3] - truth)).mean(), np.rad2deg(np.abs(res["pose"][3:6] - truth)).mean())
        assert err < 1.0, err
    ctx.set_engine(binding.ENGINE_AUTO)


def test_pair_pose_bin_dev_replay_is_identical(ctx):
    import torch

    q, t, lxy, rxy, W, H, _ = _scene(seed=61)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
    dl, dr = torch.from_numpy(lxy).cuda(), torch.from_numpy(rxy).cuda()
    outs = []
    for _ in range(3):                       # direct, captured, replayed
        dm = torch.zeros(len(q) * 16, dtype=torch.uint8, device="cuda")
        dn = torch.zeros(1, dtype=torch.int32, device="cuda")
        dmask = torch.zeros(len(q), dtype=torch.uint8, device="cuda")
        dres = torch.zeros(binding.C.sizeof(binding.RansacResult), dtype=torch.uint8, device="cuda")
        ctx.pair_pose_bin_dev(dq, len(q), dt, len(t), 32, 0.8, True, dl, dr, 8, W, H, 3, 4096, 8, 0, 0.002, dm, dn, dmask, dres)
        ctx.synchronize()
        n = int(dn.item())
        outs.append((dm.cpu().numpy()[: 16 * n].tobytes(), dmask.cpu().numpy()[:n].tobytes(), dres.cpu().numpy().tobytes()))
    assert outs[0] == outs[1] == outs[2]
    assert outs[0][0] == B.match(q, t, 0.8, True).tobytes()


def test_host_dropin_norm_hamming(tmp_path, fx):
    import subprocess

    exe = B.build_hamming_main(tmp_path)
    q, t = fx["orb_q"], fx["orb_t"]
    inp, out = tmp_path / "in.bin", tmp_path / "out.bin"
    B.write_hamming_input(inp, q, t, 0.8, True)
    r = subprocess.run([str(exe), str(inp), str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert B.read_hamming_output(out).tobytes() == B.match(q, t, 0.8, True).tobytes()


def test_large_i8_equals_popc(ctx):
    import torch

    q, t, _ = synth.binary_pair(100000, 100000, 32, seed=71)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
    res = []
    for e in ENGINES:
        ctx.set_engine(e)
        idx = torch.zeros((len(q), 2), dtype=torch.int32, device="cuda")
        dist = torch.zeros((len(q), 2), dtype=torch.float32, device="cuda")
        ctx.knn2_bin_dev(dq, len(q), dt, len(t), 32, idx, dist)
        ctx.synchronize()
        res.append((idx.cpu().numpy(), dist.cpu().numpy()))
    ctx.set_engine(binding.ENGINE_AUTO)
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    # spot check against the CPU reference on a slice of the queries
    ref = B.knn2(q[:512], t)
    assert np.array_equal(res[0][0][:512], ref[0]) and np.array_equal(res[0][1][:512], ref[1])
