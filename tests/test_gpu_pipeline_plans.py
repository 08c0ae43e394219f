"""Every tcgen05 distance-kernel instantiation through the pipeline state that only shows after many train tiles, or after
a CTA moves from one query row to the next: the T-ring slot and phase, the parity of the two TMEM accumulators, the phase
of the query barriers across segments, the norm operand's double buffer, and the per-row threshold reset at each segment.

Each case first computes its stream-K plan with the Python copy of stream_k_plan / SegIter below (tc_common.cuh;
tests/test_plan_host.py holds it equal to the C++ planner), asserts that the library ran that plan, and asserts the
property the case exists for: many ring turns in one CTA (class A), several query rows in one CTA (B), the largest
number of segments per row (C), minimal and ragged shapes (D).  A change of the SM count, of a segment limit or of the
planner then fails here instead of quietly shrinking what the tests reach.  Exact ties are planted across column-group,
tile and segment boundaries; results are compared with the fp64 oracle and the CPU Hamming reference.
"""
import os
import re
import zlib
from typing import NamedTuple

import numpy as np
import pytest

import binary_ref as B
import oracle as O
from erp_match_eightpoint_test_b200 import binding, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "erp_match_eightpoint_test_b200", "csrc")

TC3, TC1, SIMT = binding.ENGINE_TCGEN05, binding.ENGINE_TCGEN05_1X, binding.ENGINE_EXACT_SIMT
KAPPA = {TC3: 2.0 ** -14, TC1: 1.05 * 2.0 ** -10}      # certificate slack of the 3xTF32 and f16 engines


# ---------------------------------------------------------------- the planner, as tc_common.cuh spells it
TILE_N = 256                                    # train rows per tile of every engine (BN, F_BN, B_BN)
MAX_SEG = {"f16": 8, "tf32": 8, "i8": 16}       # F_MAX_SEG, MAX_SEG, B_MAX_SEG


def cdiv(a, b):
    return -(-a // b)


def stream_k_plan(n_rows, n_ttiles, sms, max_seg):
    """(units per CTA L, segments per row n_seg, grid)"""
    total = n_rows * n_ttiles
    lmin = cdiv(n_ttiles, max_seg - 2) if max_seg > 2 else n_ttiles
    L = max(cdiv(total, sms), lmin, 1)
    return L, min(cdiv(n_ttiles, L) + 1, max_seg), cdiv(total, L)


def seg_iter(n_rows, n_ttiles, L, cta):
    """The segments (query row, t0, t1, list slot) of one CTA."""
    u, end = cta * L, min(cta * L + L, n_rows * n_ttiles)
    while u < end:
        row = u // n_ttiles
        row0 = row * n_ttiles
        t0 = u - row0
        t1 = min(t0 + end - u, n_ttiles)
        yield row, t0, t1, u // L - row0 // L
        u += t1 - t0


def seg_of(row, tile, n_ttiles, L):
    """List slot of the segment that scans train tile `tile` of query row `row`."""
    return (row * n_ttiles + tile) // L - (row * n_ttiles) // L


# ---------------------------------------------------------------- unit geometry of the three engines
def b_sub(kch):
    return 2 if kch <= 3 else 1                 # knn_bin.cu b_sub: resident query sub-tiles


def _constants(src):
    """The integer constexprs of tc_common.cuh and one kernel source that need no template parameter."""
    env = {}
    for f in ("tc_common.cuh", src):
        for name, expr in re.findall(r"constexpr int (\w+) = ([^;,]+);", open(os.path.join(CSRC, f)).read()):
            try:
                env[name] = eval(expr.replace("/", "//"), {}, dict(env))
            except NameError:
                pass
    return env


def ring_depth(kind, kch):
    """T-ring slots (k chunks of 32 KB) of an instantiation: f_slots, n_slots and b_slots of the kernel sources."""
    if kind == "f16":
        c = _constants("knn_tc1.cu")
        return (c["TC_SMEM_LIMIT"] - c["F_SUB"] * kch * c["F_QCH"] - c["F_TAIL"]) // c["F_TCH"]
    if kind == "tf32":
        c = _constants("knn_tc.cu")
        return (c["SMEM_LIMIT"] - 2 * kch * c["Q_CHUNK_BYTES"] - c["SMEM_TAIL"]) // c["T_CHUNK_BYTES"]
    c = _constants("knn_bin.cu")
    return (c["TC_SMEM_LIMIT"] - b_sub(kch) * kch * c["B_QCH"] - c["B_BARS"]) // c["B_TCH"]


class Geo(NamedTuple):
    kind: str       # f16, tf32 or i8
    width: int      # D, or bytes per binary row
    kch: int        # template parameter: 128-byte k chunks (f16, i8) or 32-float k chunks per half (tf32)
    rows: int       # query rows per unit
    max_seg: int
    ring: int


def geometry(kind, width):
    kch = cdiv(width, {"f16": 64, "tf32": 32, "i8": 16}[kind])
    rows = {"f16": 256, "tf32": 128, "i8": 128 * b_sub(kch)}[kind]
    return Geo(kind, width, kch, rows, MAX_SEG[kind], ring_depth(kind, kch))


def plan(geo, nq, nt, sms):
    n_rows, n_tt = cdiv(nq, geo.rows), cdiv(nt, TILE_N)
    L, n_seg, grid = stream_k_plan(n_rows, n_tt, sms, geo.max_seg)
    walks = [list(seg_iter(n_rows, n_tt, L, c)) for c in range(grid)]
    return dict(L=L, n_seg=n_seg, grid=grid, n_ttiles=n_tt, max_tiles=max(sum(s[2] - s[1] for s in w) for w in walks),
                max_segs=max(len(w) for w in walks))


# ---------------------------------------------------------------- the cases
# every instantiation: f16 <1> <2>, 3xTF32 <1>..<4>, i8 <1>..<4> (D and bytes per row), plus ragged widths
FLOAT = [(TC1, 64), (TC1, 128), (TC1, 4), (TC1, 68), (TC1, 100),
         (TC3, 32), (TC3, 64), (TC3, 96), (TC3, 128), (TC3, 4), (TC3, 68), (TC3, 100)]
BINARY = [16, 32, 48, 64, 1, 17, 61]


def shapes(geo, cls):
    if cls == "A":          # deep: at least three ring depths of train tiles in one CTA
        return [(20000, 20000)]
    if cls == "B":          # a CTA walks several query rows of 2 or 3 tiles
        return [(40000, 300)] + ([(120000, 520)] if (geo.kind, geo.width) == ("f16", 64) else [])
    if cls == "C":          # one or two query rows cut into the largest number of segments
        return [(geo.rows, 60000)] + ([(geo.rows + 1, 60000)] if geo.rows == 128 else [])
    r = geo.rows            # minimal, one padded tile, an empty or partial last sub-tile
    return [(1, 2), (1, 257), (r + 1, 300), (r + 128, 300), (r + 129, 300)]


def check_plan(geo, cls, nq, nt, p):
    print("%s %3d class %s %6d x %5d: L %3d n_seg %2d grid %3d, per CTA up to %3d tiles and %2d segments (ring %d)" %
          (geo.kind, geo.width, cls, nq, nt, p["L"], p["n_seg"], p["grid"], p["max_tiles"], p["max_segs"], geo.ring))
    if cls == "A":
        assert p["max_tiles"] >= 3 * geo.ring, p
    elif cls == "B":
        assert p["max_segs"] >= 2, p
    elif cls == "C":
        assert p["n_seg"] == geo.max_seg - 1, p
    elif (nq, nt) == (1, 2):
        assert p["grid"] == 1, p


def check_stats(ctx, p, binary):
    st = ctx.last_knn_stats()
    assert st["segments"] == p["n_seg"] and st["units_per_cta"] == p["L"], (st, p)
    if binary:
        assert st["grid"] == p["grid"], (st, p)
    return st


def tie_groups(nt):
    """Groups of train rows that receive copies of one new row: the two sides of the column-group boundary (127/128), of
    the first and of a middle tile boundary, the last row with a row a third of the way in, and rows in three quarters of
    the train set (other segments of the same query row wherever the row is cut)."""
    n_tt = cdiv(nt, TILE_N)
    k = max(n_tt // 2, 2)
    cand = [[127, 128], [255, 256], [k * 256 - 1, k * 256], [nt // 3 + 5, nt - 1], [nt // 4 + 1, nt // 2 + 2, 3 * nt // 4 + 3]]
    used, groups = set(), []
    for c in cand:
        p = sorted({x for x in c if 0 <= x < nt} - used)
        if len(p) >= 2:
            groups.append(p)
            used |= set(p)
    return groups


def plant_ties(q, t, groups, new_row, near):
    """t[group] = one new row; queries at both ends of the query set become that row, exactly and slightly moved.  Every
    copy is at the same exact distance from them, so the two nearest are the two lowest indices of the group."""
    nq = len(q)
    planted = []
    for g, pos in enumerate(groups):
        v = new_row()
        t[pos] = v
        for j, exact in ((3 * g % nq, True), ((nq - 1 - 3 * g) % nq, False)):
            q[j] = v if exact else near(v)
            planted.append(j)
    return np.unique(np.array(planted, np.int64))


@pytest.fixture(scope="module")
def ctx():
    c = binding.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("cls", ["A", "B", "C", "D"])
@pytest.mark.parametrize("engine,dim", FLOAT)
def test_float_instantiation_plans(ctx, sms, engine, dim, cls):
    geo = geometry("f16" if engine == TC1 else "tf32", dim)
    for nq, nt in shapes(geo, cls):
        p = plan(geo, nq, nt, sms)
        check_plan(geo, cls, nq, nt, p)
        seed = zlib.crc32(b"%d %d %s %d %d" % (engine, dim, cls.encode(), nq, nt))
        q, t, _ = synth.descriptor_pair(nq, nt, dim, seed=seed)
        rng = np.random.default_rng(seed)
        ties = plant_ties(q, t, tie_groups(nt), lambda: synth.surf_like(1, dim, rng)[0],
                          lambda v: v + np.float32(1e-3) * rng.standard_normal(dim).astype(np.float32))
        if cls == "C":          # the spread group lies in three segments of the first query row
            spread = tie_groups(nt)[-1]
            assert len({seg_of(0, x // TILE_N, p["n_ttiles"], p["L"]) for x in spread}) == 3, spread
        ctx.set_engine(engine)
        try:
            idx, dist = ctx.knn2_raw(q, t)
            st = check_stats(ctx, p, binary=False)
        finally:
            ctx.set_engine(binding.ENGINE_AUTO)
        assert st["engine"] == engine
        if cls == "A":          # every query against the fp64 SIMT engine, a sub-sample and the tie queries against the oracle
            ctx.set_engine(SIMT)
            eidx, edist = ctx.knn2_raw(q, t)
            ctx.set_engine(binding.ENGINE_AUTO)
            assert np.array_equal(idx, eidx) and np.array_equal(dist.view(np.uint32), edist.view(np.uint32))
            sub = np.union1d(np.arange(0, nq, 64), ties)
        else:
            sub = np.arange(nq)
        oidx, odist, _ = O.knn2(q[sub], t)
        bad = np.nonzero((idx[sub] != oidx).any(1))[0]
        assert len(bad) == 0, (sub[bad[:10]], idx[sub[bad[:10]]], oidx[bad[:10]])
        assert np.array_equal(dist[sub].view(np.uint32), odist.view(np.uint32))
        # the kernel itself must have found (nearly) every answer: the exact re-scan would repair a broken tile.  At D = 4,
        # thousands of rows crowd the unit sphere so that most second neighbours sit within the certificate's margin of
        # a third one and the re-scan is the designed path; the k-chunk count of D = 4 is checked at D = 32 / 64 instead.
        # Four products average no rounding: the observed deviation reaches 0.7 of the f16 bound there.
        if dim >= 32:
            assert st["rescanned"] <= max(2, nq // 100), st
        assert st["deviation"] <= KAPPA[engine] / (2 if dim >= 32 else 1), st
        print("    re-scanned %d, deviation %.3f of kappa" % (st["rescanned"], st["deviation"] / KAPPA[engine]))


@pytest.mark.parametrize("cls", ["A", "B", "C", "D"])
@pytest.mark.parametrize("nbytes", BINARY)
def test_binary_instantiation_plans(ctx, sms, nbytes, cls):
    geo = geometry("i8", nbytes)
    for nq, nt in shapes(geo, cls):
        p = plan(geo, nq, nt, sms)
        check_plan(geo, cls, nq, nt, p)
        seed = zlib.crc32(b"i8 %d %s %d %d" % (nbytes, cls.encode(), nq, nt))
        q, t, _ = synth.binary_pair(nq, nt, nbytes, seed=seed)
        rng = np.random.default_rng(seed)

        def near(v):
            v = v.copy()
            v[0] ^= 1
            return v

        ties = plant_ties(q, t, tie_groups(nt), lambda: rng.integers(0, 256, nbytes, dtype=np.uint8), near)
        ctx.set_engine(TC1)
        try:
            idx, dist = ctx.knn2_raw_bin(q, t)
            check_stats(ctx, p, binary=True)
        finally:
            ctx.set_engine(binding.ENGINE_AUTO)
        ctx.set_engine(SIMT)
        eidx, edist = ctx.knn2_raw_bin(q, t)
        ctx.set_engine(binding.ENGINE_AUTO)
        assert np.array_equal(idx, eidx) and np.array_equal(dist, edist)
        sub = np.union1d(np.arange(0, nq, 64), ties) if cls == "A" else np.arange(nq)
        ridx, rdist = B.knn2(q[sub], t, chunk=64)
        bad = np.nonzero((idx[sub] != ridx).any(1))[0]
        assert len(bad) == 0, (sub[bad[:10]], idx[sub[bad[:10]]], ridx[bad[:10]])
        assert np.array_equal(dist[sub], rdist)
        if cls == "D" and nt == 300:
            # every train row at distance nbits: a padding column of the last tile (zero rows, nbits / 2) must never win
            ctx.set_engine(TC1)
            try:
                idx, dist = ctx.knn2_raw_bin(np.zeros((nq, nbytes), np.uint8), np.full((nt, nbytes), 255, np.uint8))
                check_stats(ctx, p, binary=True)
            finally:
                ctx.set_engine(binding.ENGINE_AUTO)
            assert (idx == [0, 1]).all() and (dist == 8 * nbytes).all()
        if cls == "B":          # match records; the reverse search of the cross-check is a class C shape
            ctx.set_engine(TC1)
            try:
                got = ctx.knn2_match_bin(q, t, 0.8, True)
                rp = plan(geo, nt, nq, sms)
                check_stats(ctx, rp, binary=True)
            finally:
                ctx.set_engine(binding.ENGINE_AUTO)
            assert rp["n_seg"] == geo.max_seg - 1, rp
            assert got.tobytes() == B.match(q, t, 0.8, True).tobytes()


@pytest.mark.parametrize("engine,dim", [(TC1, 64), (TC1, 128), (TC3, 64), (TC3, 128)])
def test_near_tie_clusters_beyond_list_capacity(ctx, sms, engine, dim):
    """Clusters of 27 to 40 train rows that differ by less than the engine's operand error: their exact distances differ,
    their approximate ranks scramble, and each cluster overflows the candidate lists of both column groups of one segment
    (the f16 list of 8, the 3xTF32 top-4) with different values.  Each cluster also has rows in every other segment of the
    query row, so the list floor and the threshold exchange between column groups and segments decide what is kept."""
    geo = geometry("f16" if engine == TC1 else "tf32", dim)
    nq, nt = geo.rows, 60000
    p = plan(geo, nq, nt, sms)
    check_plan(geo, "C", nq, nt, p)
    seed = zlib.crc32(b"clusters %d %d" % (engine, dim))
    q, t, _ = synth.descriptor_pair(nq, nt, dim, seed=seed)
    rng = np.random.default_rng(seed)
    rel = 3 * 2.0 ** -13 if engine == TC1 else 2.0 ** -16           # below each engine's operand rounding
    used = set()

    def draw(seg, k, upper=None):
        """k unused train rows in segment seg of the (single) query row, in the upper column group or either"""
        lo, hi, out = seg * p["L"] * TILE_N, min((seg + 1) * p["L"] * TILE_N, nt), []
        while len(out) < k:
            x = int(rng.integers(lo, hi))
            if x not in used and (upper is None or (x % TILE_N >= 128) == upper):
                used.add(x)
                out.append(x)
        return out

    for c in range(6):
        # 11 rows in each column group of one segment (more than a list holds), one row in each other segment, and the
        # rest anywhere
        pos = draw(c, 11, False) + draw(c, 11, True) + [draw(s, 1)[0] for s in range(6) if s != c]
        pos = np.sort(pos + [draw(int(rng.integers(6)), 1)[0] for _ in range(int(rng.integers(27, 41)) - len(pos))])
        n = len(pos)
        base = synth.surf_like(1, dim, rng)[0]
        t[pos] = base * (1 + rel * rng.uniform(-1, 1, (n, dim))).astype(np.float32)
        assert len({seg_of(0, x // TILE_N, p["n_ttiles"], p["L"]) for x in pos}) >= 3
        assert len({x % TILE_N >= 128 for x in pos}) == 2
        # on the base, on a member, and near the cluster
        q[4 * c] = base
        q[4 * c + 1] = t[pos[n // 2]]
        q[4 * c + 2] = base + np.float32(rel / 4) * rng.standard_normal(dim).astype(np.float32) * np.abs(base)
        q[4 * c + 3] = base + np.float32(1e-3) * rng.standard_normal(dim).astype(np.float32)
    ctx.set_engine(engine)
    try:
        idx, dist = ctx.knn2_raw(q, t)
        st = check_stats(ctx, p, binary=False)
    finally:
        ctx.set_engine(binding.ENGINE_AUTO)
    oidx, odist, _ = O.knn2(q, t)
    bad = np.nonzero((idx != oidx).any(1))[0]
    assert len(bad) == 0, (bad[:10], idx[bad[:10]], oidx[bad[:10]])
    assert np.array_equal(dist.view(np.uint32), odist.view(np.uint32))
    assert st["deviation"] <= KAPPA[engine], st
    print("    near-tie clusters: re-scanned %d of %d, deviation %.3f of kappa" % (st["rescanned"], nq, st["deviation"] / KAPPA[engine]))
