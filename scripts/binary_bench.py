"""Hamming 2-NN of binary descriptors on the B200: the tcgen05 kind::i8 engine against the SIMT popcount engine.

    python scripts/binary_bench.py [--steps 10] [--out binary_bench.jsonl]

Device-resident inputs (synth.binary_pair), the L2 overwritten (256 MB) before every timed step, CUDA events around the
whole call (step ms) and the library's own events around the distance kernel (kernel ms).  Both engines' outputs are
compared at every size.  Rows: a crossover sweep for ERP_ENGINE_AUTO, 20k x 20k and 100k x 100k at 32 and 64 bytes,
the erp_pair_pose_bin_dev step, and cv2.BFMatcher(NORM_HAMMING) on a host sample when cv2 is importable.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from erp_match_eightpoint_test_b200 import binding, synth  # noqa: E402

ENGINES = {"i8": binding.ENGINE_TCGEN05_1X, "popc": binding.ENGINE_EXACT_SIMT}


def gpu_line() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown"
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def timed(ctx, fn, flush, steps):
    """Host clock around a call that ends in a synchronise of the library's stream; fn returns the kernel ms (or 0)."""
    ms = []
    for _ in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        kern = fn()
        ctx.synchronize()
        ms.append(((time.perf_counter() - t0) * 1e3, kern))
    step = np.array([m[0] for m in ms])
    kern = np.array([m[1] for m in ms])
    return float(np.median(step)), float(np.median(kern)), float(step.min()), float(step.max())


def knn_row(ctx, nq, nt, nbytes, steps, flush, emit):
    q, t, _ = synth.binary_pair(nq, nt, nbytes, seed=nq + nbytes)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
    out = {}
    for name, e in ENGINES.items():
        ctx.set_engine(e)
        idx = torch.empty((nq, 2), dtype=torch.int32, device="cuda")
        dist = torch.empty((nq, 2), dtype=torch.float32, device="cuda")

        def call():
            ctx.knn2_bin_dev(dq, nq, dt, nt, nbytes, idx, dist)
            return 0.0

        call()
        ctx.synchronize()

        def call_k():
            ctx.knn2_bin_dev(dq, nq, dt, nt, nbytes, idx, dist)
            return ctx.last_knn_kernel_ms()
        step, kern, lo, hi = timed(ctx, call_k, flush, steps)
        out[name] = (idx.cpu().numpy(), dist.cpu().numpy())
        emit(dict(row="knn2_bin", engine=name, nq=nq, nt=nt, nbytes=nbytes, step_ms=step, step_ms_min=lo, step_ms_max=hi,
                  kernel_ms=kern, dist_evals_per_s=nq * nt / (kern * 1e-3) if kern > 0 else None,
                  bit_ops_per_s=2.0 * nq * nt * 8 * nbytes / (kern * 1e-3) if kern > 0 else None))
    ctx.set_engine(binding.ENGINE_AUTO)
    same = all(np.array_equal(out["i8"][k], out["popc"][k]) for k in (0, 1))
    emit(dict(row="knn2_bin_equal", nq=nq, nt=nt, nbytes=nbytes, identical=same))
    return same


def pair_row(ctx, steps, flush, emit, nq=20000, nt=20000, W=4096, H=2048):
    q, t, planted = synth.binary_pair(nq, nt, 32, f_match=0.6, seed=9)
    qi = np.nonzero(planted >= 0)[0]
    kp = synth.keypoint_pair(len(qi), W, H, noise_px=0.3, outlier_frac=0.0, seed=10)
    rng = np.random.default_rng(9)
    lxy = (rng.uniform(0, 1, (nq, 2)) * [W, H - 1]).astype(np.float32)
    rxy = (rng.uniform(0, 1, (nt, 2)) * [W, H - 1]).astype(np.float32)
    lxy[qi] = kp["left_xy"]
    rxy[planted[qi]] = kp["right_xy"]
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
    dl, dr = torch.from_numpy(lxy).cuda(), torch.from_numpy(rxy).cuda()
    dm = torch.empty(nq * 16, dtype=torch.uint8, device="cuda")
    dn = torch.empty(1, dtype=torch.int32, device="cuda")
    dmask = torch.empty(nq, dtype=torch.uint8, device="cuda")
    dres = torch.empty(binding.C.sizeof(binding.RansacResult), dtype=torch.uint8, device="cuda")
    for cc in (False, True):
        def call():
            ctx.pair_pose_bin_dev(dq, nq, dt, nt, 32, 0.8, cc, dl, dr, 8, W, H, 3, 4096, 8, 0, 0.002, dm, dn, dmask, dres)
            return 0.0
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        step, _, lo, hi = timed(ctx, call, flush, steps)
        match_ms, gather_ms, ransac_ms = ctx.last_stage_ms()
        emit(dict(row="pair_pose_bin_dev", nq=nq, nt=nt, nbytes=32, cross_check=cc, step_ms=step, step_ms_min=lo, step_ms_max=hi,
                  stage_ms=[match_ms, gather_ms, ransac_ms], device_ms=match_ms + gather_ms + ransac_ms, matches=int(dn.item()), hypotheses=4096))


def cv2_row(emit, n=20000, nbytes=32):
    try:
        import cv2
    except ImportError:
        emit(dict(row="cv2_bfmatcher", available=False))
        return
    q, t, _ = synth.binary_pair(n, n, nbytes, seed=n + nbytes)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    bf.knnMatch(q[:100], t, k=2)
    t0 = time.perf_counter()
    bf.knnMatch(q, t, k=2)
    s = time.perf_counter() - t0
    emit(dict(row="cv2_bfmatcher", available=True, nq=n, nt=n, nbytes=nbytes, ms=s * 1e3, threads=cv2.getNumThreads(),
              dist_evals_per_s=n * n / s))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="skip the 100k x 100k rows")
    a = ap.parse_args()
    f = open(a.out, "w") if a.out else None
    gpu = gpu_line()

    def emit(d):
        d["gpu"] = gpu
        line = json.dumps(d)
        print(line, flush=True)
        if f:
            f.write(line + "\n")

    ctx = binding.Context(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ok = True
    for n in (1000, 2000, 5000, 10000):
        ok &= knn_row(ctx, n, n, 32, a.steps, flush, emit)
    sizes = [(20000, 32), (20000, 64)] + ([] if a.quick else [(100000, 32), (100000, 64)])
    for n, nb in sizes:
        ok &= knn_row(ctx, n, n, nb, a.steps, flush, emit)
    pair_row(ctx, a.steps, flush, emit)
    cv2_row(emit)
    ctx.close()
    if f:
        f.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
