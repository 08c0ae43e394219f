"""The one-product engine's f16 operands (csrc/knn_tc1.cu): every case equals ERP_ENGINE_EXACT_SIMT bit for bit, and
erp_ctx_last_knn_operands shows which path ran -- the f16 products, the range guard (a finite input f16 cannot hold), or
the per-query check that sends norms too small for f16 subnormal rounding to the exact re-scan."""
import os

import numpy as np
import pytest

import erp_match_eightpoint_test_b200 as erp
from conftest import GOLDEN
from erp_match_eightpoint_test_b200 import binding, synth

pytestmark = pytest.mark.gpu

KAPPA = 1.05 * 2.0 ** -10


@pytest.fixture(scope="module")
def ctx():
    c = erp.Context(0)
    yield c
    c.close()


def one_product_vs_exact(ctx, q, t):
    """2-NN of the one-product engine, checked bit for bit against the fp64 engine; returns its statistics."""
    ctx.set_engine(binding.ENGINE_EXACT_SIMT)
    eidx, edist = ctx.knn2_raw(q, t)
    ctx.set_engine(binding.ENGINE_TCGEN05_1X)
    idx, dist = ctx.knn2_raw(q, t)
    st = ctx.last_knn_stats()
    st.update(ctx.last_knn_operands())
    ctx.set_engine(binding.ENGINE_AUTO)
    assert st["engine"] == binding.ENGINE_TCGEN05_1X and st["operands"] == binding.OPERANDS_F16, st
    assert np.array_equal(idx, eidx), st
    assert np.array_equal(dist.view(np.uint32), edist.view(np.uint32)), st
    return st


def test_out_of_range_inputs_take_the_guard(ctx):
    q, t, _ = synth.descriptor_pair(1000, 3000, 64, seed=11)
    # one train component of 1e5 (f16 tops out at 65504), then one query component of 4e4 (x(-2) = -8e4)
    for which in ("t", "q"):
        qq, tt = q.copy(), t.copy()
        if which == "t":
            tt[17, 5] = 1.0e5
        else:
            qq[3, 40] = 4.0e4
        st = one_product_vs_exact(ctx, qq, tt)
        assert st["guard"] and st["range_rescanned"] == len(q) and st["rescanned"] == len(q), (which, st)
    # every row scaled to 1e-6: nothing overflows, but subnormal rounding is outside the certificate for every query
    st = one_product_vs_exact(ctx, q * np.float32(1e-6), t * np.float32(1e-6))
    assert not st["guard"] and st["range_rescanned"] == len(q) and st["rescanned"] == len(q), st
    # the guard is per call: the next in-range call runs on the f16 products again
    st = one_product_vs_exact(ctx, q, t)
    assert not st["guard"] and st["range_rescanned"] == 0, st


@pytest.mark.parametrize("dim", [32, 64, 96, 100, 128])
@pytest.mark.parametrize("nq,nt", [(129, 257), (4000, 300)])
def test_subnormal_heavy_ragged_shapes(ctx, dim, nq, nt):
    """Unit-norm rows of which three quarters of the components lie in f16's subnormal range (|x| < 2^-14, many below
    2^-24): the absolute rounding of those stays inside the certificate, so no query is re-scanned for range."""
    rng = np.random.default_rng(dim * 7 + nq)

    def rows(n):
        x = rng.standard_normal((n, dim))
        tiny = rng.random((n, dim)) < 0.75
        x[tiny] *= 10.0 ** rng.uniform(-9, -4.5, size=tiny.sum())
        return np.ascontiguousarray((x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32))

    t = rows(nt)
    q = rows(nq)
    q[: nq // 4] = t[rng.integers(0, nt, nq // 4)]
    st = one_product_vs_exact(ctx, q, t)
    assert not st["guard"] and st["range_rescanned"] == 0, st
    assert st["deviation"] <= KAPPA, st


@pytest.mark.parametrize("exp", [-3, 4])
def test_worst_case_rounding_outside_one_to_two(ctx, exp):
    """test_gpu_parity's adversarial set moved to the binades [2^-3, 2^-2) and [16, 32): every component just below an f16
    rounding midpoint, all positive, half of the queries copies of train rows.  f16 midpoints scale with the binade, so
    the observed deviation must again approach 2^-10 (|q|^2 + max|t|^2) and stay within the certificate."""
    rng = np.random.default_rng(70 + exp)
    nq, nt = 3000, 5000
    for dim in (64, 128):
        def adversarial(n):
            m = rng.integers(0, 64, size=(n, dim)).astype(np.float64)
            return np.ascontiguousarray(((1.0 + m / 1024.0 + 2.0 ** -11 - 2.0 ** -18) * 2.0 ** exp).astype(np.float32))
        t = adversarial(nt)
        q = adversarial(nq)
        q[: nq // 2] = t[rng.permutation(nt)[: nq // 2]]
        st = one_product_vs_exact(ctx, q, t)
        print("f16 worst case, 2^%d, D=%d: deviation %.3f of 2^-10, %d re-scanned" % (exp, dim, st["deviation"] * 1024, st["rescanned"]))
        assert not st["guard"] and st["range_rescanned"] == 0, st
        assert 0.8 * 2.0 ** -10 < st["deviation"] <= KAPPA, st


# queries the tf32 operands of the same engine re-scanned on these three sets: 0 of 4774, 0 of 20000 and 0 of 20000
# (NVIDIA B200, 1000 W power limit, measured with 01dff16, the last build that had the tf32 operands)
TF32_RESCANNED = (0, 0, 0)


def test_real_and_synthetic_descriptors_run_on_f16(ctx):
    """Synthetic SURF-64 / SURF-128 and the real SIFT pair take the f16 products, and re-scan no more queries than the
    tf32 operands did on the same inputs."""
    z = np.load(os.path.join(GOLDEN, "real_building.npz"))
    sets = [(z["left_desc_u8"].astype(np.float32), z["right_desc_u8"].astype(np.float32))]
    for dim in (64, 128):
        q, t, _ = synth.descriptor_pair(20000, 20000, dim, seed=synth.SEED_BASE + 40 + dim)
        sets.append((q, t))
    for i, ((q, t), r32) in enumerate(zip(sets, TF32_RESCANNED)):
        st = one_product_vs_exact(ctx, q, t)
        print("set %d (%d x %d x %d): re-scanned f16 %d, tf32 %d; deviation %.3f of 2^-10" %
              (i, len(q), len(t), q.shape[1], st["rescanned"], r32, st["deviation"] * 1024))
        assert not st["guard"] and st["range_rescanned"] == 0, st
        assert st["rescanned"] <= r32 + max(5, r32 // 20), (i, st, r32)
