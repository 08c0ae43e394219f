"""Deterministic synthetic inputs for the hot path (SURVEY.md section 8(d)).

Descriptors mimic OpenCV SURF-64/128 rows (4x4 cells x (sum dx, sum dy, sum|dx|, sum|dy|),
L2-normalised); keypoints are ERP pixels of a two-view scene with a known relative
pose, the inverse of the pixel->bearing map in /root/reference/src/eight_point.cpp:164-185.
numpy's Philox bit generator makes every array identical on every machine.
"""
from __future__ import annotations

import numpy as np

SEED_BASE = 0xE8B0


def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.Philox(seed))


def surf_like(n: int, dim: int, rng: np.random.Generator) -> np.ndarray:
    d = rng.standard_normal((n, dim), dtype=np.float32)
    d[:, 2::4] = np.abs(d[:, 2::4])
    d[:, 3::4] = np.abs(d[:, 3::4])
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.ascontiguousarray(d, dtype=np.float32)


def descriptor_pair(nq: int, nt: int, dim: int = 64, f_match: float = 0.5, seed: int = SEED_BASE):
    """Returns (query, train, planted) where planted[i] is the train row query i was
    derived from (-1 for fresh rows).  Planted rows pass the 0.3 ratio test."""
    rng = _rng(seed)
    train = surf_like(nt, dim, rng)
    n_pl = min(int(nq * f_match), nt)
    src = rng.permutation(nt)[:n_pl]
    sigma = rng.uniform(0.002, 0.08, size=(n_pl, 1)).astype(np.float32) / np.sqrt(dim).astype(np.float32)
    noisy = train[src] + sigma * rng.standard_normal((n_pl, dim), dtype=np.float32)
    noisy /= np.linalg.norm(noisy, axis=1, keepdims=True)
    fresh = surf_like(nq - n_pl, dim, rng)
    query = np.concatenate([noisy, fresh], axis=0).astype(np.float32)
    planted = np.concatenate([src, -np.ones(nq - n_pl, dtype=np.int64)])
    perm = rng.permutation(nq)
    return np.ascontiguousarray(query[perm]), train, planted[perm]


def eular2rot(theta) -> np.ndarray:
    """R = Rx*Ry*Rz, /root/reference/src/erp_rotation.cpp:14-40."""
    x, y, z = [float(v) for v in theta]
    Rx = np.array([[1, 0, 0], [0, np.cos(x), -np.sin(x)], [0, np.sin(x), np.cos(x)]])
    Ry = np.array([[np.cos(y), 0, np.sin(y)], [0, 1, 0], [-np.sin(y), 0, np.cos(y)]])
    Rz = np.array([[np.cos(z), -np.sin(z), 0], [np.sin(z), np.cos(z), 0], [0, 0, 1]])
    return Rx @ Ry @ Rz


def bearing_to_pixel(b: np.ndarray, W: int, H: int) -> np.ndarray:
    """Inverse of eight_point.cpp:164-185: b = (-sin lat cos lon, sin lat sin lon, cos lat)."""
    lat = np.arccos(np.clip(b[:, 2], -1, 1))
    lon = np.arctan2(b[:, 1], -b[:, 0])
    lon = np.where(lon < 0, lon + 2 * np.pi, lon)
    return np.stack([lon / (2 * np.pi) * W, lat / np.pi * H], axis=1)


def keypoint_pair(m: int, W: int, H: int, euler_deg=(5.0, 10.0, 15.0), t=(0.3, -0.9, 0.1),
                  noise_px: float = 0.5, outlier_frac: float = 0.3, seed: int = SEED_BASE + 100):
    """Two-view ERP keypoints with l^T E r = 0 for E = [t]x R^T (r = R (X - t) direction).

    Returns dict(left_xy, right_xy float32 (m,2), R, t, E, inlier bool mask)."""
    rng = _rng(seed)
    R = eular2rot(np.deg2rad(euler_deg))
    t = np.asarray(t, dtype=np.float64)
    t = t / np.linalg.norm(t)
    d = rng.standard_normal((m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    X = d * rng.uniform(2.0, 20.0, size=(m, 1))
    l = X / np.linalg.norm(X, axis=1, keepdims=True)
    Xr = (X - t) @ R.T
    r = Xr / np.linalg.norm(Xr, axis=1, keepdims=True)
    lp = bearing_to_pixel(l, W, H) + noise_px * rng.standard_normal((m, 2))
    rp = bearing_to_pixel(r, W, H) + noise_px * rng.standard_normal((m, 2))
    n_out = int(m * outlier_frac)
    out_idx = rng.permutation(m)[:n_out]
    rp[out_idx] = rng.uniform(0, 1, size=(n_out, 2)) * np.array([W, H])
    lp[:, 0] = np.mod(lp[:, 0], W)
    rp[:, 0] = np.mod(rp[:, 0], W)
    lp[:, 1] = np.clip(lp[:, 1], 0, H - 1e-3)
    rp[:, 1] = np.clip(rp[:, 1], 0, H - 1e-3)
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    E = tx @ R.T
    inl = np.ones(m, bool)
    inl[out_idx] = False
    return dict(left_xy=lp.astype(np.float32), right_xy=rp.astype(np.float32), R=R, t=t, E=E, inlier=inl)


def binary_pair(nq: int, nt: int, nbytes: int = 32, f_match: float = 0.5, seed: int = SEED_BASE + 200):
    """Binary descriptors (ORB-like uint8 rows) for Hamming matching.  Returns (query, train, planted): a share f_match of
    the queries are train rows with a few flipped bits (planted[i] = that row, -1 for fresh random rows), and the last
    nt // 16 train rows duplicate earlier ones, so that exact distance ties are certain."""
    rng = _rng(seed)
    nbits = 8 * nbytes
    train = rng.integers(0, 256, size=(nt, nbytes), dtype=np.uint8)
    n_dup = nt // 16
    if n_dup:
        train[nt - n_dup:] = train[rng.integers(0, nt - n_dup, size=n_dup)]
    n_pl = min(int(nq * f_match), nt)
    src = rng.permutation(nt)[:n_pl]
    bits = np.unpackbits(train[src], axis=1)
    k_max = max(1, nbits // 16)
    pos = rng.integers(0, nbits, size=(n_pl, k_max))
    keep = np.arange(k_max)[None, :] < rng.integers(1, k_max + 1, size=(n_pl, 1))
    rows = np.broadcast_to(np.arange(n_pl)[:, None], pos.shape)
    bits[rows[keep], pos[keep]] ^= 1
    noisy = np.packbits(bits, axis=1)
    fresh = rng.integers(0, 256, size=(nq - n_pl, nbytes), dtype=np.uint8)
    query = np.concatenate([noisy, fresh], axis=0)
    planted = np.concatenate([src, -np.ones(nq - n_pl, dtype=np.int64)])
    perm = rng.permutation(nq)
    return np.ascontiguousarray(query[perm]), train, planted[perm]
