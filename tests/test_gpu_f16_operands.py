"""The one-product engine's f16 operands (csrc/knn_tc1.cu): every case equals ERP_ENGINE_EXACT_SIMT bit for bit, and
erp_ctx_last_knn_operands shows which path ran -- the f16 products, the range guard (a finite input f16 cannot hold), or
the per-query check that sends norms too small for f16 subnormal rounding to the exact re-scan."""
import os
import subprocess
import sys

import numpy as np
import pytest

import erp_match_eightpoint_test_b200 as erp
from conftest import GOLDEN
from erp_match_eightpoint_test_b200 import binding, synth

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(os.environ.get("ERP_B200_TC1_OPERANDS") == "tf32", reason="tf32 operands selected for this process"),
]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
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


TF32_RESCANS = """
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import erp_match_eightpoint_test_b200 as erp
from erp_match_eightpoint_test_b200 import binding
z = np.load(sys.argv[2])
with erp.Context(0) as ctx:
    ctx.set_engine(binding.ENGINE_TCGEN05_1X)
    out = []
    for k in sorted(z.files)[::2]:
        ctx.knn2_raw(z[k], z[k.replace("q", "t")])
        assert ctx.last_knn_operands()["operands"] == binding.OPERANDS_TF32
        out.append(ctx.last_knn_stats()["rescanned"])
print(" ".join(map(str, out)))
"""


def test_real_and_synthetic_descriptors_run_on_f16(ctx, tmp_path):
    """Synthetic SURF-64 / SURF-128 and the real SIFT pair take the f16 products, and re-scan no more queries than the
    tf32 operands do on the same inputs (measured in a child process: the operand choice is read once per process)."""
    z = np.load(os.path.join(GOLDEN, "real_building.npz"))
    sets = {"0q": z["left_desc_u8"].astype(np.float32), "0t": z["right_desc_u8"].astype(np.float32)}
    for i, dim in enumerate((64, 128), 1):
        q, t, _ = synth.descriptor_pair(20000, 20000, dim, seed=synth.SEED_BASE + 40 + dim)
        sets["%dq" % i], sets["%dt" % i] = q, t
    path = str(tmp_path / "sets.npz")
    np.savez(path, **sets)
    env = dict(os.environ, ERP_B200_TC1_OPERANDS="tf32")
    out = subprocess.run([sys.executable, "-s", "-c", TF32_RESCANS, ROOT, path], env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    tf32 = [int(x) for x in out.stdout.split()]
    for i, r32 in enumerate(tf32):
        q, t = sets["%dq" % i], sets["%dt" % i]
        st = one_product_vs_exact(ctx, q, t)
        print("set %d (%d x %d x %d): re-scanned f16 %d, tf32 %d; deviation %.3f of 2^-10" %
              (i, len(q), len(t), q.shape[1], st["rescanned"], r32, st["deviation"] * 1024))
        assert not st["guard"] and st["range_rescanned"] == 0, st
        assert st["rescanned"] <= r32 + max(5, r32 // 20), (i, st, r32)
