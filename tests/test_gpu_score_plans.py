"""The tcgen05 hypothesis search (score_tc.cu) checked bound by bound, not only through its winner.

The search is exact only if every count it keeps is an upper bound of the hypothesis' exact fp32-chain count over the
correspondences it covered: pass A and B bounds over the first ct1 tiles, pass C bounds of the survivors over the rest.
The public call shows only the winner, so an undercounted loser (a stream-K cut whose partial count is lost, a band
too narrow, a Sampson / angular row gain too tight) or an overcounted one (a tile counted twice, pads not subtracted)
goes unnoticed as long as the winner's own bound holds.

A small program linked against the library's own objects runs the production search (erp::ransac_search on a forced
TCGEN05 context) and dumps the last hypothesis chunk's E, both bound arrays, the survivor and contender lists and the
device words.  Each case then checks, against the CPU oracle:
  * soundness: bound >= exact count over the covered correspondences, for a sample and every hypothesis of rows that
    straddle a CTA boundary of the stream-K cut;
  * tightness: bound <= the count of residuals inside tau plus twice the band, in fp64 (catches double counting and
    pad errors);
  * the plan words: L*, ct1, the remaining correspondences, the survivor and contender lists, equal to a Python mirror of
    argmax_plan_kernel and the selection kernels;
and asserts which per-CTA pipeline state (ScoreShape + SegIter, mirrored here) the case exists for.  The public call
must also equal the SIMT engine bit for bit.  Then the RANSAC paths no other test reaches: two hypothesis chunks,
S > 8 (prep_e_kernel), non-finite correspondences and hypothesis ids at the top of the 32-bit range.
"""
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

import oracle as O
from erp_match_eightpoint_test_b200 import binding, build, synth
from test_gpu_pipeline_plans import CSRC, _constants, cdiv, seg_iter

gpu = pytest.mark.gpu

TC, SIMT = binding.ENGINE_TCGEN05, binding.ENGINE_EXACT_SIMT
TAU = 0.002
_C = {**_constants("score_tc.cu"), **_constants("score_common.cuh"), **_constants("common.cuh")}
HYP_ROWS = _C["SM_ROWS"] * _C["S_SUB"]          # hypotheses per tile pair (one row of the stream-K grid)
TILE = _C["SC_TILE"]                            # correspondences per tile
N0 = _C["SC_N0"]                                # tiles of pass A
RING = _C["S_NSLOT"]                            # correspondence ring slots, one tile each
CHUNK = _C["RANSAC_CHUNK"]
W = {k: int(v) for k, v in re.findall(r"\b(W_\w+) = (\d+)", open(os.path.join(CSRC, "score_common.cuh")).read())}
SLACK_DIV, SLACK_TILES = 16, 2                  # argmax_plan_kernel's pruning slack (score_tc_search defaults)

HARNESS = r"""
#include "common.cuh"
#include "score_common.cuh"
#include <cstdio>
#include <cstdlib>
#include <vector>
// argv[1]: cases, each int64 { m, seed, hyp_offset, H, S, metric }, float64 tau, float64 l3[m][3], r3[m][3]
// argv[2]: per case int64 { sm_count, first hypothesis of the last chunk h0, its size n, packed best }, int32 words[W_WORDS],
//          then of the last chunk: float64 E[n][9], int32 bounds[2n], int32 lists[2n]
#define CK(x) do { const int s_ = (int)(x); if (s_) { fprintf(stderr, "%s -> %d %s\n", #x, s_, erp_last_error()); exit(1); } } while (0)
#define CU(x) do { const cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s -> %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)
template <class T> static void down(erp_ctx* ctx, int id, std::vector<T>& v)
{
    if (!ctx->dev[id].p || ctx->dev[id].cap < v.size() * sizeof(T)) { fprintf(stderr, "scratch %d missing\n", id); exit(1); }
    CU(cudaMemcpyAsync(v.data(), ctx->dev[id].p, v.size() * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
}
int main(int argc, char** argv)
{
    if (argc != 3) return 2;
    FILE *in = fopen(argv[1], "rb"), *out = fopen(argv[2], "wb");
    if (!in || !out) return 2;
    erp_ctx* ctx = nullptr;
    CK(erp_ctx_create(0, &ctx));
    CK(erp_ctx_set_engine(ctx, ERP_ENGINE_TCGEN05));
    int64_t hd[6];
    double tau;
    while (fread(hd, 8, 6, in) == 6 && fread(&tau, 8, 1, in) == 1) {
        const int m = (int)hd[0], H = (int)hd[3], S = (int)hd[4], metric = (int)hd[5];
        std::vector<double> l3((size_t)m * 3), r3((size_t)m * 3);
        if (fread(l3.data(), 8, l3.size(), in) != l3.size() || fread(r3.data(), 8, r3.size(), in) != r3.size()) return 2;
        double *dl, *dr;
        float *dl4, *dr4;
        uint64_t* dp;
        CU(cudaMalloc(&dl, l3.size() * 8)); CU(cudaMalloc(&dr, r3.size() * 8));
        CU(cudaMalloc(&dl4, (size_t)m * 16)); CU(cudaMalloc(&dr4, (size_t)m * 16)); CU(cudaMalloc(&dp, 8));
        CU(cudaMemcpyAsync(dl, l3.data(), l3.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(dr, r3.data(), r3.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemsetAsync(dp, 0, 8, ctx->stream));
        CK(erp_pack_float4_dev(ctx, dl, m, dl4));
        CK(erp_pack_float4_dev(ctx, dr, m, dr4));
        CK(erp::ransac_search(ctx, dl, dr, dl4, dr4, m, nullptr, (uint64_t)hd[1], (uint64_t)hd[2], H, S, metric, (float)tau, false, dp));
        const int h0 = (H - 1) / erp::RANSAC_CHUNK * erp::RANSAC_CHUNK, n = H - h0;
        std::vector<double> E((size_t)n * 9);
        std::vector<int32_t> w(erp::W_WORDS), bounds((size_t)n * 2), lists((size_t)n * 2);
        int64_t oh[4] = {ctx->sm_count, h0, n, 0};
        down(ctx, erp::S_E, E); down(ctx, erp::S_SC_MISC, w); down(ctx, erp::S_SC_BOUNDS, bounds); down(ctx, erp::S_SC_LIST, lists);
        CU(cudaMemcpyAsync(&oh[3], dp, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        fwrite(oh, 8, 4, out); fwrite(w.data(), 4, w.size(), out); fwrite(E.data(), 8, E.size(), out);
        fwrite(bounds.data(), 4, bounds.size(), out); fwrite(lists.data(), 4, lists.size(), out);
        CU(cudaFree(dl)); CU(cudaFree(dr)); CU(cudaFree(dl4)); CU(cudaFree(dr4)); CU(cudaFree(dp));
    }
    erp_ctx_destroy(ctx);
    return fclose(out) == 0 ? 0 : 1;
}
"""


@pytest.fixture(scope="module")
def harness_exe(tmp_path_factory):
    if not os.path.exists(build.NVCC):
        pytest.skip("nvcc not found")
    build.build()
    d = tmp_path_factory.mktemp("score_dump")
    src, exe = d / "score_dump.cu", d / "score_dump"
    src.write_text(HARNESS)
    objs = [os.path.join(build.OUT_DIR, s.replace(".cu", ".o")) for s in build.SOURCES]
    r = subprocess.run([build.NVCC] + build.FLAGS + [str(src)] + objs + ["-cudart", "static", "-ldl", "-lpthread", "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return str(exe)


def test_harness_compiles_and_links_against_the_library_objects(harness_exe):
    assert os.access(harness_exe, os.X_OK)


@pytest.fixture(scope="module")
def search(harness_exe, tmp_path_factory):
    """search(cases) -> one dump per case; a case is dict(l, r, seed, hyp0, H, S, metric, tau)"""
    d = tmp_path_factory.mktemp("score_io")

    def run(cases):
        inp, out = d / "in.bin", d / "out.bin"
        with open(inp, "wb") as f:
            for c in cases:
                f.write(np.array([len(c["l"]), c["seed"], c["hyp0"], c["H"], c["S"], c["metric"]], np.int64).tobytes())
                f.write(np.array([c["tau"]], np.float64).tobytes())
                f.write(np.ascontiguousarray(c["l"], np.float64).tobytes() + np.ascontiguousarray(c["r"], np.float64).tobytes())
        r = subprocess.run([harness_exe, str(inp), str(out)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        buf, k, dumps = open(out, "rb").read(), 0, []
        for _ in cases:
            sms, h0, n, packed = np.frombuffer(buf, np.int64, 4, k).tolist()
            k += 32
            w = np.frombuffer(buf, np.int32, W["W_WORDS"], k)
            k += 4 * W["W_WORDS"]
            E = np.frombuffer(buf, np.float64, 9 * n, k).reshape(n, 9)
            k += 72 * n
            bounds = np.frombuffer(buf, np.int32, 2 * n, k)
            k += 8 * n
            lists = np.frombuffer(buf, np.int32, 2 * n, k)
            k += 8 * n
            dumps.append(dict(sms=sms, h0=h0, n=n, packed=packed & 0xFFFFFFFFFFFFFFFF, w=w, E=E, bounds=bounds, lists=lists))
        assert k == len(buf)
        return dumps

    return run


@pytest.fixture(scope="module")
def ctx():
    c = binding.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------- mirrors of score_tc.cu
def pass_plan(H, c0, c1, grid):
    """ScoreShape + SegIter of one launch: rows are tile pairs of hypotheses, columns correspondence tiles [c0, c1)."""
    n_ht, n_ct = cdiv(H, HYP_ROWS), max(c1 - c0, 0)
    total = n_ht * n_ct
    L = max(cdiv(total, grid), 1)
    walks = [list(seg_iter(n_ht, n_ct, L, c)) for c in range(grid)] if total else []
    # rows whose units two CTAs share: a CTA's range starts inside the row
    cuts = sorted({c * L // n_ct for c in range(1, grid) if c * L < total and c * L % n_ct})
    return dict(H=H, n_htiles=n_ht, n_ctiles=n_ct, L=L, max_segs=max((len(w) for w in walks), default=0),
                max_tiles=max((sum(s[2] - s[1] for s in w) for w in walks), default=0), cut_rows=cuts)


def plan_of(lstar, m, n0, nct):
    """argmax_plan_kernel: pass B's end tile ct1 and the correspondences left for pass C"""
    need = m - lstar
    need += need // SLACK_DIV + SLACK_TILES * TILE
    ct1 = max(cdiv(need, TILE), n0)
    if ct1 > nct or lstar * 4 < m:
        ct1 = nct
    return ct1, max(m - ct1 * TILE, 0)


def f32_of(word):
    return float(np.array([word], np.int32).view(np.float32)[0])


def scale_e(E):
    """scale_E: ||E||_F = sqrt(2) in fp64 (sequential sum), then to float"""
    E = np.asarray(E, np.float64).reshape(-1, 9)
    n = np.zeros(len(E))
    for i in range(9):
        n = n + E[:, i] * E[:, i]
    with np.errstate(divide="ignore", invalid="ignore"):
        s = np.where(n > 0, np.sqrt(2.0) / np.sqrt(n), 0.0)
    return (E * s[:, None]).astype(np.float32)


def row_gain(e, metric, tau, w):
    """score_common.cuh row_gain, in fp64 like the device"""
    if metric == O.METRIC_ALGEBRAIC:
        return np.ones(len(e), np.float32)
    d = e.astype(np.float64)
    mm = np.zeros((6, len(e)))
    for i in range(3):
        a, b, c = d[:, 3 * i], d[:, 3 * i + 1], d[:, 3 * i + 2]
        mm += np.stack([a * a, a * b, a * c, b * b, b * c, c * c])
    t = mm[0] + mm[3] + mm[5]
    c1 = (mm[0] * mm[3] - mm[1] * mm[1]) + (mm[0] * mm[5] - mm[2] * mm[2]) + (mm[3] * mm[5] - mm[4] * mm[4])
    disc = t * t - 4.0 * c1
    with np.errstate(invalid="ignore", over="ignore"):
        s1sq = 0.5 * (t + np.sqrt(np.where(disc > 0, disc, 0.0))) * (1.0 + 1e-6) + 1e-9 * t
        s1sq = np.where(s1sq < t, s1sq, t)
        R = f32_of(w[W["W_RMAX"] if metric == O.METRIC_SAMPSON else W["W_RRMAX"]])
        th = float(np.float32(tau)) if metric == O.METRIC_SAMPSON else float(np.float32(np.sin(np.float64(np.float32(tau)))))
        T = th * np.sqrt(s1sq * R) * (1.0 + 1e-5)
        g = np.where(T > float(np.float32(tau)), (float(np.float32(tau)) / T).astype(np.float32), np.float32(1))
    return np.where(np.isfinite(T), g, 0).astype(np.float32)


def band_counts(eg, l, r, thr):
    """#{c : |res64| < thr} per row of eg (float rows), res64 = eg . (l (x) r) in fp64 of the float bearings"""
    lf, rf = l.astype(np.float32).astype(np.float64), r.astype(np.float32).astype(np.float64)
    K = (lf[:, :, None] * rf[:, None, :]).reshape(len(l), 9)
    out = np.empty(len(eg), np.int64)
    for i in range(0, len(eg), 512):
        out[i: i + 512] = (np.abs(eg[i: i + 512].astype(np.float64) @ K.T) < thr).sum(1)
    return out


def packed_of(counts, ids):
    return max(((int(c) << 32) | (0xFFFFFFFF - int(h))) for c, h in zip(counts, ids)) if len(ids) else 0


def check_dump(d, l, r, S, metric, tau, hyp0, tight=True, label=""):
    """Plan words, lists, soundness and tightness of one dump (its last hypothesis chunk).  Returns the plan and the
    packed best of the chunk's contenders."""
    w, n, m = d["w"], d["n"], len(l)
    nct, n0, lstar, remain = int(w[W["W_NCT"]]), int(w[W["W_N0"]]), int(w[W["W_LSTAR"]]), int(w[W["W_REMAIN"]])
    ct1, n_surv, n_cont = int(w[W["W_DYN_B"] + 2]), int(w[W["W_DYN_C"]]), int(w[W["W_LENF"]])
    assert (int(w[W["W_M"]]), nct, n0) == (m, cdiv(m, TILE), min(cdiv(m, TILE), N0)), w
    assert list(w[W["W_DYN_A"]: W["W_DYN_A"] + 4]) == [n, 0, n0, m], w
    assert list(w[W["W_DYN_B"]: W["W_DYN_B"] + 4]) == [n, n0, ct1, m], w
    assert list(w[W["W_DYN_C"] + 1: W["W_DYN_C"] + 4]) == [ct1, nct, m], w
    assert (ct1, remain) == plan_of(lstar, m, n0, nct), (lstar, m, n0, nct, ct1, remain)
    upper, upper2 = d["bounds"][:n].astype(np.int64), d["bounds"][n:].astype(np.int64)
    surv, cont = d["lists"][:n_surv], d["lists"][n: n + n_cont]
    assert upper.min() >= 0 and upper2[:n_surv].min(initial=0) >= 0, "negative count"
    # the selection kernels, recomputed from the dumped arrays (list order is the order of block arrival)
    if remain > 0:
        assert np.array_equal(np.sort(surv), np.nonzero(upper + remain >= lstar)[0]), "survivors"
        want = surv[upper[surv] + upper2[:n_surv] >= lstar]
    else:
        assert n_surv == 0
        want = np.nonzero(upper >= lstar)[0]
    assert np.array_equal(np.sort(cont), np.sort(want)), "contenders"
    # L* is the exact count of a hypothesis (a sound bound keeps it a contender); the winner is the best contender
    E = d["E"]
    exact_cont = O.score(E[cont], l, r, metric, tau)
    assert lstar in set(exact_cont.tolist()), (lstar, np.sort(exact_cont)[-5:])
    chunk_best = packed_of(exact_cont, [hyp0 + d["h0"] + int(h) for h in cont])
    assert lstar <= chunk_best >> 32 and chunk_best <= d["packed"]

    passes = {"A": pass_plan(n, 0, n0, d["sms"]), "B": pass_plan(n, n0, ct1, d["sms"]), "C": pass_plan(n_surv, ct1, nct, d["sms"])}
    shape = "pass A only" if nct <= N0 else "weak model, no pass C" if lstar * 4 < m else \
        "pruned" if remain > 0 else "complete after pass B"
    print("%s metric %d H %d (chunk %d + %d) m %d S %d: %s, L* %d, ct1 %d of %d, remain %d, survivors %d, contenders %d" %
          (label, metric, d["h0"] + n, d["h0"], n, m, S, shape, lstar, ct1, nct, remain, n_surv, n_cont))
    for k, p in passes.items():
        print("    pass %s: %d x %d units, %d per CTA, per CTA up to %d segments and %d tiles, %d rows cut between CTAs %s" %
              (k, p["n_htiles"], p["n_ctiles"], p["L"], p["max_segs"], p["max_tiles"], len(p["cut_rows"]), p["cut_rows"][:6]))

    # soundness: a 1/16 sample, every contender, every hypothesis of up to four cut rows of passes A and B
    def some(rows):
        return rows if len(rows) <= 4 else [rows[0], rows[len(rows) // 3], rows[2 * len(rows) // 3], rows[-1]]

    rows = sorted(set(some(passes["A"]["cut_rows"])) | set(some(passes["B"]["cut_rows"])))
    hs = np.union1d(np.arange(0, n, 16), cont)
    for row in rows:
        hs = np.union1d(hs, np.arange(row * HYP_ROWS, min(row * HYP_ROWS + HYP_ROWS, n)))
    P = min(m, ct1 * TILE)
    exact_p = O.score(E[hs], l[:P], r[:P], metric, tau)
    bad = np.nonzero(upper[hs] < exact_p)[0]
    assert len(bad) == 0, ("bound below the exact count", hs[bad[:8]], upper[hs[bad[:8]]], exact_p[bad[:8]])
    # pass C: survivor slots of a 1/16 sample and of up to four cut rows; bound over all m
    slots = np.arange(0, n_surv, 16)
    for row in some(passes["C"]["cut_rows"]):
        slots = np.union1d(slots, np.arange(row * HYP_ROWS, min(row * HYP_ROWS + HYP_ROWS, n_surv)))
    total = upper[surv[slots]] + upper2[slots]
    exact_all = O.score(E[surv[slots]], l, r, metric, tau)
    bad = np.nonzero(total < exact_all)[0]
    assert len(bad) == 0, ("pass C bound below the exact count", surv[slots[bad[:8]]], total[bad[:8]], exact_all[bad[:8]])

    # tightness: nothing counted outside tau + 2 delta (the device's band plus its own operand error)
    kmax = f32_of(w[W["W_KMAX"]])
    if tight:
        assert np.isfinite(kmax)
        thr = float(np.float32(tau)) + 2 * 2.0 ** -16 * np.sqrt(2.0) * kmax
        if metric != O.METRIC_ALGEBRAIC:
            thr *= 1 + 1e-4
        e = scale_e(E)
        eg = (e * row_gain(e, metric, tau, w)[:, None]).astype(np.float32)
        hi = band_counts(eg[hs], l[:P], r[:P], thr)
        bad = np.nonzero(upper[hs] > hi)[0]
        assert len(bad) == 0, ("bound above the band count", hs[bad[:8]], upper[hs[bad[:8]]], hi[bad[:8]])
        if n_surv:
            hi = band_counts(eg[surv[slots]], l, r, thr)
            assert (total <= hi).all(), ("pass C bound above the band count", total[total > hi][:8], hi[total > hi][:8])
    return dict(passes=passes, ct1=ct1, nct=nct, remain=remain, survivors=n_surv, contenders=n_cont, lstar=lstar, kmax=kmax,
                chunk_best=chunk_best)


# ---------------------------------------------------------------- public calls
def scene(m, seed, outliers=0.3, noise=0.5):
    kp = synth.keypoint_pair(m, 8192, 4096, noise_px=noise, outlier_frac=outliers, seed=seed)
    return O.bearings(kp["left_xy"], 8192, 4096), O.bearings(kp["right_xy"], 8192, 4096)


def ransac_on(ctx, engine, *a, **k):
    ctx.set_engine(engine)
    try:
        return ctx.ransac(*a, **k)
    finally:
        ctx.set_engine(binding.ENGINE_AUTO)


def tc_equals_simt(ctx, l, r, seed, hyp0, H, S, metric, tau=TAU):
    tc = ransac_on(ctx, TC, l, r, seed=seed, hyp_offset=hyp0, H=H, S=S, metric=metric, tau=tau)
    simt = ransac_on(ctx, SIMT, l, r, seed=seed, hyp_offset=hyp0, H=H, S=S, metric=metric, tau=tau)
    assert tc["packed"] == simt["packed"] and tc["count"] == simt["count"]
    assert np.array_equal(tc["mask"], simt["mask"])
    assert np.array_equal(tc["E_refit"].view(np.uint64), simt["E_refit"].view(np.uint64))
    return tc


def case(l, r, seed, hyp0, H, S, metric, tau=TAU):
    return dict(l=l, r=r, seed=seed, hyp0=hyp0, H=H, S=S, metric=metric, tau=tau)


def dumped_e_is_the_solvers(ctx, d, c):
    """the dumped E of the last chunk = erp_eight_point_batch of the same ids; returns it"""
    E, _ = ctx.eight_point_batch(c["l"], c["r"], H=d["n"], S=c["S"], seed=c["seed"], hyp_offset=c["hyp0"] + d["h0"], want_pose=False)
    E = E.reshape(-1, 9)
    assert np.array_equal(E.view(np.uint64), d["E"].view(np.uint64))
    return E


def run(ctx, search, c, tight=True, label=""):
    """public TC = SIMT, harness dump = public winner, E = the solver's, bound checks"""
    tc = tc_equals_simt(ctx, c["l"], c["r"], c["seed"], c["hyp0"], c["H"], c["S"], c["metric"], c["tau"])
    d = search([c])[0]
    assert d["packed"] == tc["packed"]
    dumped_e_is_the_solvers(ctx, d, c)
    info = check_dump(d, c["l"], c["r"], c["S"], c["metric"], c["tau"], c["hyp0"], tight=tight, label=label)
    if d["h0"] == 0:
        assert info["chunk_best"] == d["packed"]
    return tc, d, info


def seed_of(*a):
    return zlib.crc32(repr(a).encode())


# ---------------------------------------------------------------- plan classes
METRICS = [O.METRIC_ALGEBRAIC, O.METRIC_SAMPSON, O.METRIC_ANGULAR]


@gpu
@pytest.mark.parametrize("metric", METRICS)
def test_deep_plan_reuses_both_query_buffers_wraps_the_ring_and_cuts_rows(ctx, search, sms, metric):
    """Pass A: a CTA walks >= 5 tile-pair rows (the two query buffers at both phases); pass B: a CTA consumes >= 2 ring
    depths of correspondence tiles; every pass: CTA boundaries inside a row (two CTAs add partial counts)."""
    H = (4 * sms + 7) * HYP_ROWS - 100          # pass A: about 4 rows of N0 tiles per CTA, and a partial last pair
    pa = pass_plan(H, 0, N0, sms)
    assert pa["max_segs"] >= 5 and pa["cut_rows"], pa
    l, r = scene(12000, seed_of("deep", metric))
    _, d, info = run(ctx, search, case(l, r, 7, 0, H, 8, metric), label="deep")
    assert d["sms"] == sms
    p = info["passes"]
    assert p["A"]["max_segs"] >= 5, p["A"]
    assert p["B"]["max_tiles"] >= 2 * RING, p["B"]
    assert info["remain"] > 0 and info["survivors"] > 0, info
    for k in "ABC":
        assert p[k]["cut_rows"], (k, p[k])


# (m, outlier share, noise px, H): each reaches one pass shape
SHAPES = {"pass_a_only": (2000, 0.3, 0.5, 20000), "weak": (6000, 0.85, 0.5, 30000), "pruned": (20000, 0.3, 0.5, 30000),
          "few_survivors": (20000, 0.5, 0.5, 30000), "outlier_free": (20000, 0.0, 0.1, 30000)}


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("metric", METRICS)
def test_pass_shapes(ctx, search, metric, shape):
    m, outliers, noise, H = SHAPES[shape]
    l, r = scene(m, seed_of(shape, metric), outliers, noise)
    _, d, info = run(ctx, search, case(l, r, 3, 11, H, 8, metric), label=shape)
    ct1, nct, remain, surv = info["ct1"], info["nct"], info["remain"], info["survivors"]
    if shape == "pass_a_only":
        assert nct <= N0 and ct1 == nct and remain == 0 and surv == 0, info
        assert info["passes"]["B"]["n_ctiles"] == 0
    elif shape == "weak":
        assert info["lstar"] * 4 < m and ct1 == nct and surv == 0, info
    elif shape == "pruned":
        assert 0 < surv < H and ct1 < nct and remain > 0, info
    elif shape == "few_survivors":
        # half the correspondences are outliers: nearly every sample holds one, and only the few clean samples (about
        # 0.5^8 of them) keep bound + remaining >= L*
        assert remain > 0 and 0 < surv < H // 50, info
        print("    reached: %d survivors of %d hypotheses, %d correspondences left for pass C" % (surv, H, remain))
    else:
        # outlier-free: L* = m, pass B has no tile at all (ct1 = n0) and pass C takes everything past pass A
        assert info["lstar"] == m and ct1 == N0 and remain == m - N0 * TILE and surv > 0, info
        assert info["passes"]["B"]["n_ctiles"] == 0


@gpu
@pytest.mark.parametrize("metric", METRICS)
def test_ragged_and_minimal_shapes(ctx, search, metric):
    """H in {1, 255, 256, 257}: the second sub-tile of a pair empty, partial or full; m around the tile and column-group
    edges and the end of pass A (2048 = N0 tiles): the pads in either column group and in pass A or B."""
    cases = []
    for H in (1, HYP_ROWS - 1, HYP_ROWS, HYP_ROWS + 1):
        for m in (8, TILE - 1, TILE, TILE + 1, N0 * TILE - 1, N0 * TILE, N0 * TILE + 1):
            l, r = scene(m, seed_of("ragged", H, m, metric), 0.2)
            cases.append(case(l, r, 5, 2, H, 8, metric))
    dumps = search(cases)
    for c, d in zip(cases, dumps):
        tc = tc_equals_simt(ctx, c["l"], c["r"], c["seed"], c["hyp0"], c["H"], 8, metric)
        assert d["packed"] == tc["packed"]
        assert tc["packed"] == O.ransac(c["l"], c["r"], c["seed"], c["hyp0"], c["H"], 8, metric, TAU, want_counts=False)["packed"]
        dumped_e_is_the_solvers(ctx, d, c)
        info = check_dump(d, c["l"], c["r"], 8, metric, TAU, c["hyp0"], label="ragged")
        pa = info["passes"]["A"]
        assert pa["n_htiles"] == cdiv(c["H"], HYP_ROWS) and pa["n_ctiles"] == min(cdiv(len(c["l"]), TILE), N0)
        assert info["chunk_best"] == d["packed"]


# ---------------------------------------------------------------- RANSAC paths no other test reaches
@gpu
@pytest.mark.parametrize("tail", [4099, 1])
@pytest.mark.parametrize("metric", METRICS)
def test_two_hypothesis_chunks(ctx, search, metric, tail):
    """H = 2^20 + tail: the second chunk resets the per-chunk words, works on a shorter bound array and offsets its ids."""
    H = CHUNK + tail
    l, r = scene(300, seed_of("chunks", metric, tail))
    c = case(l, r, 13, 6, H, 8, metric)
    tc, d, info = run(ctx, search, c, label="two chunks")
    assert (d["h0"], d["n"]) == (CHUNK, tail)
    a = ransac_on(ctx, TC, l, r, seed=13, hyp_offset=6, H=CHUNK, S=8, metric=metric, tau=TAU)
    b = ransac_on(ctx, TC, l, r, seed=13, hyp_offset=6 + CHUNK, H=tail, S=8, metric=metric, tau=TAU)
    assert max(a["packed"], b["packed"]) == tc["packed"]
    assert info["chunk_best"] == b["packed"]


@gpu
@pytest.mark.parametrize("S", [9, 16, 32])
@pytest.mark.parametrize("metric", METRICS)
def test_sample_sizes_above_eight(ctx, search, metric, S):
    """S > 8: Gram + Jacobi solver, hypothesis operand written by prep_e_kernel; the winner is the exact argmax."""
    l, r = scene(4000, seed_of("S", S, metric))
    c = case(l, r, 17, 0, 6000, S, metric)
    tc, d, _ = run(ctx, search, c, label="S %d" % S)
    counts = O.score(d["E"], l, r, metric, TAU)
    assert tc["packed"] == packed_of(counts, range(c["H"]))


@gpu
@pytest.mark.parametrize("metric", METRICS)
def test_non_finite_correspondences(ctx, search, metric):
    """Rows of NaN, +-inf and all-zero bearings in a real scene: the band becomes infinite (every finite residual is a
    candidate), Sampson / angular rows lose their gain, and the exact re-score still picks the oracle's winner."""
    l, r = scene(6000, seed_of("nonfinite", metric))
    l[100:120] = np.nan
    r[300:310, 1] = np.nan
    r[500:510] = np.inf
    l[700:705, 2] = -np.inf
    l[900:910] = 0.0
    r[910:920] = 0.0
    c = case(l, r, 19, 0, 20000, 8, metric)
    tc, d, info = run(ctx, search, c, tight=False, label="non-finite")
    assert not np.isfinite(info["kmax"])
    counts = O.score(d["E"], l, r, metric, TAU)
    assert tc["packed"] == packed_of(counts, range(c["H"]))
    nan_rows = np.isnan(l).any(1) | np.isnan(r).any(1)
    assert not tc["mask"][nan_rows].any()
    assert np.array_equal(tc["mask"], O.inlier_mask(tc["E"], l, r, metric, TAU))


@gpu
@pytest.mark.parametrize("metric", METRICS)
def test_hypothesis_ids_at_the_top_of_32_bits(ctx, search, metric):
    """The highest ids the API takes: hyp_offset + H = 2^32 - 1, so the last id is 0xFFFFFFFE and its packed low word 1
    (id 0xFFFFFFFF would pack like 'no hypothesis' and is refused)."""
    H = 5000
    hyp0 = (1 << 32) - 1 - H
    l, r = scene(3000, seed_of("top", metric))
    with pytest.raises(binding.ErpError) as ei:
        ransac_on(ctx, TC, l, r, seed=23, hyp_offset=hyp0 + 1, H=H, S=8, metric=metric, tau=TAU)
    assert ei.value.status == binding.E_LIMIT
    c = case(l, r, 23, hyp0, H, 8, metric)
    tc, d, _ = run(ctx, search, c, label="top ids")
    counts = O.score(d["E"], l, r, metric, TAU)
    want = packed_of(counts, [hyp0 + h for h in range(H)])
    assert tc["packed"] == want
    hyp = 0xFFFFFFFF - (tc["packed"] & 0xFFFFFFFF)
    assert hyp0 <= hyp < 1 << 32 and tc["hyp"] == hyp and counts[hyp - hyp0] == tc["count"]
