"""The fp64 geometry of geometry.cu against a 50-digit reference, at the spectra where its fast paths stop being right.

Every hypothesis and every pose goes through three solvers: the Householder null vector of an 8 x 9 system (min8_kernel)
or the 9 x 9 Jacobi of a Gram matrix (solve_kernel, solve1_kernel), then the closed-form rank-2 projection
(rank2_project_fast, with the 3 x 3 SVD as its fallback); the RANSAC refit is inverse iteration on the inlier Gram matrix
(refit_inverse_iteration, with the one-warp Jacobi as its fallback).  The fast paths are exact only while the spectrum
they work on is well separated, so the inputs here are built to sit on both sides of every threshold:

  * planted spectra: correspondences whose null vector is E = U diag(1, s2, s3) V^T, from sigma3 = 0 to sigma3 = sigma2,
    and sigma2 down past the isolation test of the projection, through S = 8 (min8) and S = 9, 16, 32 (Gram + Jacobi);
  * refit scenes from a unit baseline down to 1 % of it and in a narrow field of view, where the two smallest
    eigenvalues of the inlier Gram matrix are both noise and within a factor of a few.

Every reference is built in mpmath at 50 digits from the fp64 values the device receives, not from the planted model, so
the only error measured is the device's.  Each bar is the rounding floor of the problem (a condition number times
2^-52) times a constant fixed below, plus 1e-8.
"""
import multiprocessing
import os

import mpmath as mp
import numpy as np
import pytest

import erp_match_eightpoint_test_b200 as erp
import oracle as O
from conftest import e_dist
from erp_match_eightpoint_test_b200 import synth

gpu = pytest.mark.gpu
mp.mp.dps = 50

EPS = 2.0 ** -52
# rank-2 bar: 1e-8 + C_RANK2 * eps * (cond + s1 / (s2 - s3)), cond = kappa = sigma1 / sigma8 of the S x 9 system for the
# Householder solve on that system (S = 8) and kappa^2 for the Jacobi solves on its Gram matrix (S > 8)
C_RANK2 = 1e3
C_REFIT = 1e3           # refit bar: 1e-8 + C_REFIT * sqrt(m) * eps * trace(G) / (lambda2 - lambda1)
FLOOR = 1e-8

# ------------------------------------------------------------------ planted spectra
S2_GRID = (1.0, 0.5, 0.1, 1e-2, 2e-3, 1.2e-3, 1e-3)          # the last three straddle the isolation test (nb)
RATIO_GRID = (0.0, 1e-9, 0.3, 0.9, 0.97, 0.99, 0.999, 0.99999, 1.0)
DRAWS = 32
S_GRID = (8, 9, 16, 32)
NB_REL = 1e-12          # rank2_project_fast: nb > 1e-12 tr^4
NEWTON_CAP = 12         # rank2_project_fast: Newton steps
STEP_REL = 1e-17        # rank2_project_fast: |step| <= 1e-17 tr


def _rotation(rng):
    q, r = np.linalg.qr(rng.standard_normal((3, 3)))
    q = q * np.sign(np.diag(r))
    return q if np.linalg.det(q) > 0 else -q


def planted_draw(s2, ratio, rng, n=32):
    """n correspondences (l_i, r_i) with l_i^T E r_i = 0 for E = U diag(1, s2, s2 ratio) V^T (Frobenius-normalised)."""
    E = _rotation(rng) @ np.diag([1.0, s2, s2 * ratio]) @ _rotation(rng).T
    E /= np.linalg.norm(E)
    r = rng.standard_normal((n, 3))
    r /= np.linalg.norm(r, axis=1, keepdims=True)
    l = np.cross(r @ E.T, rng.standard_normal((n, 3)))
    l /= np.linalg.norm(l, axis=1, keepdims=True)
    return l, r, E


def planted_inputs():
    """All draws of the grid: l, r (cells x DRAWS x 32 x 3) and the planted E (cells x DRAWS x 3 x 3)."""
    cells = [(s2, q) for s2 in S2_GRID for q in RATIO_GRID]
    L = np.empty((len(cells), DRAWS, 32, 3))
    R = np.empty_like(L)
    E = np.empty((len(cells), DRAWS, 3, 3))
    for c, (s2, q) in enumerate(cells):
        rng = np.random.default_rng([17, c])
        for d in range(DRAWS):
            L[c, d], R[c, d], E[c, d] = planted_draw(s2, q, rng)
    return cells, L, R, E


def _mp_rows(l, r):
    """rows kron(l_i, r_i) of the S x 9 system, each product exact at 50 digits"""
    return [[mp.mpf(float(l[i, p])) * mp.mpf(float(r[i, q])) for p in range(3) for q in range(3)] for i in range(len(l))]


def _gram_add(G, rows):
    for a in rows:
        for j in range(9):
            for k in range(j, 9):
                G[j][k] += a[j] * a[k]


def _null_vector(G, x0):
    """smallest eigenvector of the Gram matrix G (upper triangle, 50 digits): one step of inverse iteration with a
    1e-30 trace shift from the fp64 estimate x0.  The second smallest eigenvalue of every planted system is above
    1e-17 trace (kappa < 1e8), so the step shrinks the error of x0 (below 1e-7) by 1e-13 or more."""
    tr = sum(G[j][j] for j in range(9))
    L = [[mp.mpf(0)] * 9 for _ in range(9)]
    for j in range(9):                                  # Cholesky of G + 1e-30 tr I
        d = G[j][j] + tr * mp.mpf("1e-30") - mp.fsum(L[j][k] ** 2 for k in range(j))
        L[j][j] = mp.sqrt(d)
        for i in range(j + 1, 9):
            L[i][j] = (G[j][i] - mp.fsum(L[i][k] * L[j][k] for k in range(j))) / L[j][j]
    y = [mp.mpf(float(v)) for v in x0]
    for i in range(9):
        y[i] = (y[i] - mp.fsum(L[i][k] * y[k] for k in range(i))) / L[i][i]
    for i in reversed(range(9)):
        y[i] = (y[i] - mp.fsum(L[k][i] * y[k] for k in range(i + 1, 9))) / L[i][i]
    n = mp.sqrt(mp.fsum(v * v for v in y))
    return [v / n for v in y]


def _spectrum3(En):
    """eigen-decomposition of En^T En at 50 digits: (l1 >= l2 >= l3, v3)"""
    ev, Q = mp.eigsy(En.T * En)
    order = sorted(range(3), key=lambda i: ev[i], reverse=True)
    lam = [ev[i] for i in order]
    v3 = mp.matrix([Q[k, order[2]] for k in range(3)])
    return lam, v3


def _path_state(En, lam, v3):
    """Which branch of rank2_project_fast the reference spectrum sits on:
    'fast'  isolated (nb above its threshold by 0.1 %), Newton from 0 meets its step test within 10 steps in exact
            arithmetic, and the rounding noise of a step is a tenth of that test;
    'svd'   nb below its threshold by 0.1 %, or Newton in exact arithmetic needs 14 or more steps (the device, whose
            steps are no larger, then ends at its cap of 12 and falls back);
    'either' anything in between."""
    l1, l2, l3 = lam
    tr = l1 + l2 + l3
    nb = ((l1 - l3) * (l2 - l3)) ** 2 * max(v3[k] ** 2 for k in range(3))
    if nb < (1 - 1e-3) * NB_REL * tr ** 4:
        return "svd"
    c2, c1, c0 = tr, l1 * l2 + l1 * l3 + l2 * l3, l1 * l2 * l3
    x, steps = mp.mpf(0), None
    for it in range(40):
        f, df = ((x - c2) * x + c1) * x - c0, (3 * x - 2 * c2) * x + c1
        if df <= 0:
            break
        step = f / df
        x -= step
        if abs(step) <= STEP_REL * tr:
            steps = it + 1
            break
    if steps is None or steps >= NEWTON_CAP + 2:
        return "svd"
    df = (l1 - l3) * (l2 - l3)
    noise = EPS * (l3 ** 3 + c2 * l3 ** 2 + c1 * l3 + c0) / df
    if nb > (1 + 1e-3) * NB_REL * tr ** 4 and steps <= NEWTON_CAP - 2 and noise <= 0.1 * STEP_REL * tr:
        return "fast"
    return "either"


def _np(M):
    return np.array([[float(M[i, j]) for j in range(M.cols)] for i in range(M.rows)])


def planted_reference(l, r, svd, sizes=S_GRID):
    """For the first S correspondences of one draw, S in sizes (ascending): the 50-digit null vector En (3 x 3, unit Frobenius
    norm), its rank-2 projection Ec, sigma(En), the path state, kappa = sigma1 / sigma8 and sigma9 / sigma1 of the
    S x 9 system.  svd[S]: the fp64 singular values and null vector of that system."""
    rows = _mp_rows(l, r)
    G = [[mp.mpf(0)] * 9 for _ in range(9)]
    out, done = {}, 0
    for S in sizes:
        _gram_add(G, rows[done:S])
        done = S
        sv, x0 = svd[S]
        x = _null_vector(G, x0)
        En = mp.matrix(3, 3)
        for k in range(9):
            En[k // 3, k % 3] = x[k]
        lam, v3 = _spectrum3(En)
        Ec = En - (En * v3) * v3.T
        kappa = sv[0] / sv[7]
        out[S] = dict(En=_np(En), Ec=_np(Ec), sigma=[float(mp.sqrt(max(v, 0))) for v in lam], kappa=kappa,
                      cond=kappa if S == 8 else kappa ** 2,
                      rank_gap=sv[8] / sv[0] if S > 8 else 0.0, state=_path_state(En, lam, v3))
    return out


_PLANTED = {}


def planted():
    """inputs and references of the whole grid, computed once per process (the 50-digit part on all CPUs)"""
    if not _PLANTED:
        cells, L, R, E = planted_inputs()
        n = len(cells) * DRAWS
        Lf, Rf = L.reshape(n, 32, 3), R.reshape(n, 32, 3)
        svd = {}
        for S in S_GRID:
            _, sv, vt = np.linalg.svd(np.einsum("hna,hnb->hnab", Lf[:, :S], Rf[:, :S]).reshape(n, S, 9))
            svd[S] = (sv, vt[:, -1])
        jobs = [(Lf[h], Rf[h], {S: (svd[S][0][h], svd[S][1][h]) for S in S_GRID}) for h in range(n)]
        with multiprocessing.get_context("fork").Pool(max(1, min(os.cpu_count() or 1, 32))) as pool:
            ref = pool.starmap(planted_reference, jobs, chunksize=8)
        _PLANTED.update(cells=cells, L=L, R=R, E=E, ref=[ref[c * DRAWS:(c + 1) * DRAWS] for c in range(len(cells))])
    return _PLANTED


def rank2_bar(ref):
    s1, s2, s3 = ref["sigma"]
    return FLOOR + C_RANK2 * EPS * (ref["cond"] + s1 / (s2 - s3))


def exact_tie_tol(ref):
    return FLOOR + C_RANK2 * EPS * ref["cond"]


def _cell(cells, s2, q):
    return cells.index((s2, q))


# Each cell asserts the state it exists for: every draw of the cell sits on that side of the thresholds.
EXPECTED_STATE = {
    (1.0, 0.0): "fast", (1.0, 1e-9): "fast", (0.1, 0.3): "fast", (1e-2, 0.9): "fast", (2e-3, 0.0): "fast",
    (0.1, 0.0): "fast", (1e-2, 0.3): "fast",
    (1.0, 0.99): "svd", (1.0, 0.999): "svd", (0.5, 0.999): "svd", (0.1, 0.999): "svd", (1.0, 0.99999): "svd",
    (1e-3, 0.0): "svd", (1e-3, 0.3): "svd", (1.2e-3, 0.9): "svd", (1.0, 1.0): "svd", (1e-2, 1.0): "svd",
}


def check_planted_states(P):
    cells, ref = P["cells"], P["ref"]
    for S in S_GRID:
        for cell, want in EXPECTED_STATE.items():
            got = [ref[_cell(cells, *cell)][d][S]["state"] for d in range(DRAWS)]
            assert all(g == want for g in got), (S, cell, want, got)
    # both sides of each threshold: the isolation test along sigma2 (ratio 0) and Newton's cap along sigma3 / sigma2
    assert EXPECTED_STATE[(2e-3, 0.0)] == "fast" and EXPECTED_STATE[(1e-3, 0.0)] == "svd"
    assert EXPECTED_STATE[(0.1, 0.3)] == "fast" and EXPECTED_STATE[(0.1, 0.999)] == "svd"
    assert EXPECTED_STATE[(1.0, 1e-9)] == "fast" and EXPECTED_STATE[(1.0, 0.99)] == "svd"


# ------------------------------------------------------------------ refit scenes
W_IMG, H_IMG = 4096, 2048
# name: (baseline, depth range, cone half-angle or None, noise px, outlier fraction, seed,
#        lambda1 / lambda2 band of the inlier Gram matrix for metric 0, 1, 2)
# With a small baseline the winning model depends on the residual, and with it the inlier set and its spectrum.
SCENES = {
    "wide": (1.0, (2.0, 20.0), None, 1.0, 0.3, 1, ((0, 1e-3), (0, 1e-3), (0, 1e-3))),
    "b0.05": (0.05, (2.0, 20.0), None, 1.0, 0.3, 2, ((1e-2, 0.1), (1e-2, 0.1), (1e-2, 0.1))),
    "b0.02": (0.02, (2.0, 20.0), None, 1.5, 0.3, 1, ((0.1, 0.3), (0.1, 0.3), (0.1, 0.3))),
    "b0.01": (0.01, (2.0, 20.0), None, 1.0, 0.3, 4, ((0.3, 0.9), (0.3, 0.9), (0.2, 0.3))),
    "b0.005": (0.005, (2.0, 20.0), None, 1.0, 0.3, 2, ((0.3, 0.9), (0.3, 0.9), (0, 1e-2))),
    # metric 1: the ratio where inverse iteration does not converge within its cap and the one-warp Jacobi finishes
    "b0.005j": (0.005, (2.0, 20.0), None, 1.0, 0.3, 20, ((0.1, 0.3), (0.5, 0.9), (0.1, 0.3))),
    "cone": (1.0, (2.0, 20.0), 0.15, 0.5, 0.3, 1, ((1e-2, 0.1), (1e-2, 0.1), (1e-2, 0.1))),
}
RANSAC_H = 4000
TAU = 0.002


def refit_scene(baseline, depth, cone, noise_px, outlier_frac, seed, m=1500, W=W_IMG, H=H_IMG):
    """Two ERP views of a random point cloud: depths in `depth`, directions uniform on the sphere or inside a cone of
    half-angle `cone` (the field of view), the second camera at distance `baseline` in a random direction and rotated a
    few degrees, pixel noise `noise_px`, a fraction of the right keypoints replaced by uniform ones."""
    rng = np.random.default_rng([29, seed])
    R = synth.eular2rot(np.deg2rad(rng.uniform(-5, 5, 3)))
    t = rng.standard_normal(3)
    t *= baseline / np.linalg.norm(t)
    if cone is None:
        d = rng.standard_normal((m, 3))
    else:
        axis = rng.standard_normal(3)
        axis /= np.linalg.norm(axis)
        e1 = np.cross(axis, [1.0, 0.0, 0.0] if abs(axis[0]) < 0.9 else [0.0, 1.0, 0.0])
        e1 /= np.linalg.norm(e1)
        e2 = np.cross(axis, e1)
        ct = rng.uniform(np.cos(cone), 1.0, m)                      # uniform on the spherical cap
        ph = rng.uniform(0, 2 * np.pi, m)
        st = np.sqrt(1 - ct ** 2)
        d = ct[:, None] * axis + st[:, None] * (np.cos(ph)[:, None] * e1 + np.sin(ph)[:, None] * e2)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    X = d * rng.uniform(depth[0], depth[1], (m, 1))
    Xr = (X - t) @ R.T
    lp = synth.bearing_to_pixel(X / np.linalg.norm(X, axis=1, keepdims=True), W, H) + noise_px * rng.standard_normal((m, 2))
    rp = synth.bearing_to_pixel(Xr / np.linalg.norm(Xr, axis=1, keepdims=True), W, H) + noise_px * rng.standard_normal((m, 2))
    out = rng.permutation(m)[: int(m * outlier_frac)]
    rp[out] = rng.uniform(0, 1, (len(out), 2)) * [W, H]
    for p in (lp, rp):
        p[:, 0] = np.mod(p[:, 0], W)
        p[:, 1] = np.clip(p[:, 1], 0, H - 1e-3)
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    return dict(left_xy=lp.astype(np.float32), right_xy=rp.astype(np.float32), E=tx @ R.T)


def scene_bearings(name):
    kp = refit_scene(*SCENES[name][:6])
    return kp, O.bearings(kp["left_xy"], W_IMG, H_IMG), O.bearings(kp["right_xy"], W_IMG, H_IMG)


def refit_reference(l, r, mask):
    """50-digit Gram matrix of the masked rows, its smallest eigenvector and that vector's rank-2 projection.
    Returns (Ec, bar, lambda1 / lambda2, m)."""
    idx = np.nonzero(mask)[0]
    rows = _mp_rows(l[idx], r[idx])
    cols = list(zip(*rows))
    G = mp.matrix(9, 9)
    for j in range(9):
        for k in range(j, 9):
            G[j, k] = G[k, j] = mp.fdot(cols[j], cols[k])
    ev, Q = mp.eigsy(G)
    order = sorted(range(9), key=lambda i: ev[i])
    lam1, lam2 = ev[order[0]], ev[order[1]]
    En = mp.matrix(3, 3)
    for k in range(9):
        En[k // 3, k % 3] = Q[k, order[0]]
    _, v3 = _spectrum3(En)
    Ec = _np(En - (En * v3) * v3.T)
    trace = sum(ev[i] for i in range(9))
    bar = FLOOR + C_REFIT * np.sqrt(len(idx)) * EPS * float(trace / (lam2 - lam1))
    return Ec, bar, float(lam1 / lam2), len(idx)


def gram_ratio(l, r, mask):
    A = np.einsum("na,nb->nab", l[mask > 0], r[mask > 0]).reshape(-1, 9)
    w = np.linalg.eigvalsh(A.T @ A)
    return w[0] / w[1]


# ------------------------------------------------------------------ CPU checks of the inputs
def test_planted_systems_have_rank_8_and_the_planted_null_vector():
    P = planted()
    for c in range(len(P["cells"])):
        for d in range(DRAWS):
            for S in S_GRID:
                ref = P["ref"][c][d][S]
                assert ref["rank_gap"] < 1e-14 and ref["kappa"] < 1e8, (P["cells"][c], d, S, ref["rank_gap"], ref["kappa"])
                En = ref["En"]
                assert e_dist(En, P["E"][c, d]) < 1e-12 * ref["kappa"], (P["cells"][c], d, S)
                assert abs(np.linalg.norm(En) - 1) < 1e-15


def test_planted_cells_sit_where_they_claim():
    check_planted_states(planted())


def test_tolerances_are_finite_and_positive():
    P = planted()
    for c, (s2, q) in enumerate(P["cells"]):
        for d in range(DRAWS):
            for S in S_GRID:
                ref = P["ref"][c][d][S]
                tol = exact_tie_tol(ref) if q == 1.0 else rank2_bar(ref)
                assert np.isfinite(tol) and tol > 0, (s2, q, S, tol)
    for name in SCENES:
        kp, l, r = scene_bearings(name)
        want = O.ransac(l, r, seed=7, hyp0=0, H=RANSAC_H, metric=0, tau=TAU)
        mask = O.inlier_mask(want["E"], l, r, 0, TAU)
        Ec, bar, ratio, m = refit_reference(l, r, mask)
        assert np.isfinite(bar) and 0 < bar < 1e-3 and m >= 8, (name, bar, m)


def test_refit_scenes_sit_in_their_bands():
    ratios = {}
    for name, spec in SCENES.items():
        kp, l, r = scene_bearings(name)
        for metric in (0, 1, 2):
            want = O.ransac(l, r, seed=7, hyp0=0, H=RANSAC_H, metric=metric, tau=TAU)
            mask = O.inlier_mask(want["E"], l, r, metric, TAU)
            ratios[name, metric] = gram_ratio(l, r, mask)
            lo, hi = spec[6][metric]
            assert lo <= ratios[name, metric] <= hi, (name, metric, ratios[name, metric], (lo, hi))
    assert sum(0.3 <= v <= 0.9 for v in ratios.values()) >= 2, ratios


# ------------------------------------------------------------------ device
@pytest.fixture(scope="module")
def ctx():
    c = erp.Context(0)
    yield c
    c.close()


def _batch(P, S):
    """the whole grid as one sample table: hypothesis h = draw h of the flattened (cell, draw) list, its first S rows"""
    n = len(P["cells"]) * DRAWS
    l = P["L"][:, :, :S].reshape(n * S, 3)
    r = P["R"][:, :, :S].reshape(n * S, 3)
    samples = np.arange(n * S, dtype=np.int32).reshape(n, S)
    return l, r, samples


@gpu
@pytest.mark.parametrize("S", S_GRID)
def test_planted_spectra_through_every_solver_path(ctx, S):
    """min8_kernel (S = 8) or gram_small_kernel + solve_kernel (S > 8), then the rank-2 projection, at every cell of
    the grid, against the 50-digit projection of the 50-digit null vector."""
    P = planted()
    check_planted_states(P)
    l, r, samples = _batch(P, S)
    E, pose = ctx.eight_point_batch(l, r, samples=samples)
    E0, _ = ctx.eight_point_batch(l, r, samples=samples, want_pose=False)
    assert E.tobytes() == E0.tobytes()
    assert np.isfinite(E).all() and np.isfinite(pose).all()
    worst = {}
    for c, (s2, q) in enumerate(P["cells"]):
        for d in range(DRAWS):
            ref = P["ref"][c][d][S]
            Ed = E[c * DRAWS + d]
            if q == 1.0:
                # sigma2 == sigma3: no unique projection, check the best approximation instead
                tol = exact_tie_tol(ref)
                sd = np.linalg.svd(Ed, compute_uv=False)
                En = ref["En"] if np.linalg.norm(ref["En"] - Ed) < np.linalg.norm(ref["En"] + Ed) else -ref["En"]
                err = max(sd[2], abs(np.linalg.norm(En - Ed) - ref["sigma"][2]),
                          abs(sd[0] - ref["sigma"][0]), abs(sd[1] - ref["sigma"][1]))
            else:
                tol = rank2_bar(ref)
                err = e_dist(Ed, ref["Ec"])
            worst[(s2, q)] = max(worst.get((s2, q), 0.0), err / tol)
            assert err <= tol, (S, s2, q, d, ref["state"], err, tol)
    print("S=%d worst error / bar per cell:" % S, {k: "%.1e" % v for k, v in worst.items()})


@gpu
@pytest.mark.parametrize("S", [9, 16, 32])
def test_one_warp_and_batched_jacobi_agree_bit_for_bit(ctx, S):
    """solve1_kernel (H = 1) and solve_kernel (H >= 2) apply the same rotations in the same order: the same sample row
    must give the same E and pose words, also on the rows that take the SVD fallback of the projection."""
    P = planted()
    l, r, samples = _batch(P, S)
    E, pose = ctx.eight_point_batch(l, r, samples=samples)
    picks = [_cell(P["cells"], *cell) * DRAWS + d for cell in [(1.0, 0.0), (0.1, 0.3), (1.0, 0.999), (1e-3, 0.0), (1.0, 1.0),
                                                               (2e-3, 0.99999), (0.5, 0.97)] for d in (0, 7)]
    for h in picks:
        E1, p1 = ctx.eight_point_batch(l, r, samples=samples[h:h + 1])
        E3, p3 = ctx.eight_point_batch(l, r, samples=np.repeat(samples[h:h + 1], 3, axis=0))
        assert E1[0].tobytes() == E[h].tobytes() and p1[0].tobytes() == pose[h].tobytes(), h
        for k in range(3):
            assert E3[k].tobytes() == E1[0].tobytes() and p3[k].tobytes() == p1[0].tobytes(), (h, k)


@gpu
@pytest.mark.parametrize("metric", [0, 1, 2])
@pytest.mark.parametrize("name", list(SCENES))
def test_ransac_refit_conditioning_sweep(ctx, name, metric):
    """The refit of erp_ransac (inverse iteration, Jacobi when it does not converge), erp_refit (one-warp Jacobi) and
    the oracle's eight-point on the device's inlier set, against the 50-digit smallest eigenvector of that set's Gram
    matrix, from a unit baseline down to 1 % of it and in a narrow field of view."""
    kp, l, r = scene_bearings(name)
    got = ctx.ransac(l, r, seed=7, hyp_offset=0, H=RANSAC_H, S=8, metric=metric, tau=TAU)
    mask = got["mask"]
    assert np.array_equal(mask, O.inlier_mask(got["E"], l, r, metric, TAU)) and got["n_refit"] == mask.sum()
    Ec, bar, ratio, m = refit_reference(l, r, mask)
    lo, hi = SCENES[name][6][metric]
    assert lo <= ratio <= hi, (name, metric, ratio)
    d_ransac = e_dist(got["E_refit"], Ec)
    E_jac, _ = ctx.refit(l, r, mask)
    d_jac = e_dist(E_jac, Ec)
    d_orc = e_dist(O.eight_point(l[mask > 0], r[mask > 0])["E"], Ec)
    print("%s metric %d: m=%d lambda1/lambda2=%.3g bar=%.2e  ransac %.2e  refit %.2e  oracle %.2e"
          % (name, metric, m, ratio, bar, d_ransac, d_jac, d_orc))
    assert d_ransac <= bar and d_jac <= bar and d_orc <= bar, (d_ransac, d_jac, d_orc, bar)
    assert e_dist(got["E_refit"], E_jac) <= 2 * bar
    if SCENES[name][0] >= 1.0 and SCENES[name][2] is None:
        assert e_dist(got["E_refit"], kp["E"]) < 2e-2


@gpu
def test_ransac_pixels_refit_low_parallax(ctx):
    """erp_ransac_pixels computes the bearings on the device: the reference uses the device's bearings."""
    kp = refit_scene(*SCENES["b0.005"][:6])
    got = ctx.ransac_pixels(kp["left_xy"], kp["right_xy"], W_IMG, H_IMG, seed=7, hyp_offset=0, H=RANSAC_H, metric=0, tau=TAU)
    l, r = ctx.bearings(kp["left_xy"], W_IMG, H_IMG), ctx.bearings(kp["right_xy"], W_IMG, H_IMG)
    mask = got["mask"]
    assert np.array_equal(mask, O.inlier_mask(got["E"], l, r, 0, TAU))
    Ec, bar, ratio, m = refit_reference(l, r, mask)
    assert 0.3 <= ratio <= 0.9, ratio
    assert e_dist(got["E_refit"], Ec) <= bar, (e_dist(got["E_refit"], Ec), bar)
