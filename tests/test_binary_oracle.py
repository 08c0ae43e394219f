"""Binary descriptors on the CPU: the Hamming reference (tests/binary_ref.py) equals cv2.BFMatcher(NORM_HAMMING) bit for
bit on the stored fixtures (tests/golden/binary.npz, written by tests/golden/make_binary_golden.py), the synthetic inputs
are the ones the fixture was made from, and without a GPU every binary entry point fails instead of falling back."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

import binary_ref as B
import erp_match_eightpoint_test_b200 as erp
from conftest import GOLDEN
from erp_match_eightpoint_test_b200 import binding, synth


@pytest.fixture(scope="module")
def fx():
    return np.load(os.path.join(GOLDEN, "binary.npz"))


@pytest.fixture(scope="module")
def syn():
    q, t, _ = synth.binary_pair(20000, 20000, 32)
    return q, t


def test_binary_pair_digests_match_the_fixture(fx, syn):
    q, t = syn
    assert hashlib.sha1(q.tobytes()).hexdigest() == str(fx["syn_q_sha1"])
    assert hashlib.sha1(t.tobytes()).hexdigest() == str(fx["syn_t_sha1"])


def test_binary_pair_has_ties_and_planted_matches():
    q, t, planted = synth.binary_pair(2000, 2000, 32, seed=3)
    idx, dist = B.knn2(q, t)
    assert (dist[:, 0] == dist[:, 1]).mean() > 0.1             # duplicated train rows tie at the first position
    pl = planted >= 0
    assert (B.distances(q[pl], t)[np.arange(pl.sum()), planted[pl]] == dist[pl, 0]).all()


def _check_set(fx, prefix, q, t):
    idx, dist = B.knn2(q, t)
    assert np.array_equal(idx, fx[prefix + "_idx"])
    assert np.array_equal(dist, fx[prefix + "_dist"])
    cc = B.match(q, t, ratio=-1.0, cross_check=True, knn=(idx, dist))
    assert np.array_equal(np.stack([cc["queryIdx"], cc["trainIdx"]], 1), fx[prefix + "_cc"])
    assert np.array_equal(cc["distance"], fx[prefix + "_cc_dist"])


def test_reference_equals_cv2_on_orb(fx):
    _check_set(fx, "orb", fx["orb_q"], fx["orb_t"])


def test_reference_equals_cv2_on_synthetic(fx, syn):
    _check_set(fx, "syn", *syn)


def test_reference_ratio_is_fp32_and_strict():
    q = np.zeros((3, 1), np.uint8)
    t = np.array([[0b1], [0b11], [0b111]], np.uint8)        # distances 1, 2, 3
    q[1] = 0b1111                                           # distances 3, 2, 1: nearest t[2], second t[1]
    m = B.match(q, t, ratio=0.5)
    assert list(m["queryIdx"]) == [] and len(B.match(q, t, ratio=0.51)) == 3


def test_binary_entry_points_fail_without_a_device():
    if erp.lib().erp_device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = erp.lib()
    q = np.zeros((4, 32), np.uint8)
    n = binding.C.c_int(0)
    out = np.zeros(4, binding.DMATCH)
    idx, dist = np.zeros((4, 2), np.int32), np.zeros((4, 2), np.float32)
    assert L.erp_knn2_match_bin(None, q.ctypes.data, 4, 32, q.ctypes.data, 4, 32, 32, 0.8, 0, out.ctypes.data,
                                binding.C.byref(n)) == binding.E_ARG
    with pytest.raises(erp.ErpError) as ei:
        erp.Context(0)
    assert ei.value.status == binding.E_NO_DEVICE
    assert L.erp_knn2_raw_bin(None, q.ctypes.data, 4, 32, q.ctypes.data, 4, 32, 32, idx.ctypes.data, dist.ctypes.data) == binding.E_ARG


def test_host_matcher_has_norm_type_and_refuses_to_run_without_a_gpu(tmp_path):
    exe = B.build_hamming_main(tmp_path)
    syms = subprocess.run(["nm", "-C", str(exe)], capture_output=True, text=True).stdout
    assert "erp_knn2_match_bin" in syms
    if erp.lib().erp_device_count() > 0:
        pytest.skip("a CUDA device is present: covered by the gpu test")
    q, t, _ = synth.binary_pair(50, 60, 32)
    inp, out = tmp_path / "in.bin", tmp_path / "out.bin"
    B.write_hamming_input(inp, q, t, 0.8, False)
    r = subprocess.run([str(exe), str(inp), str(out)], capture_output=True, text=True)
    # exit 1: the default L2 matcher refused the CV_8U rows (else 3 / 4), then NORM_HAMMING reached the library
    assert r.returncode == 1 and "no CPU fallback" in r.stderr and not out.exists()
