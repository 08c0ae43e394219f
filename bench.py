#!/usr/bin/env python
"""bench.py -- the hot path's headline benchmark (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3|cfg2|cfg4|cfg5] [--scaling strong|weak]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference's CPU path (oracle port) on host cores

One step = one pass of the hot path over one batch of synthetic input:
    cfg3 / cfg2   one ERP pair: 2-NN matching (+0.3 ratio test, ordered compaction) -> gather of the matched keypoints
                  -> bearings -> minimal-sample eight-point RANSAC (Philox samples, solve, score, best) -> mask -> refit,
                  ONE library call (erp_pair_pose_dev / erp_pair_pose_dist_dev), no host synchronisation inside
    cfg4          200k x 200k SURF-128 matching with cross-check (BASELINE configs[3]; matching only)
    cfg5          a sequence of 1024 ERP frame pairs x 20k keypoints (configs[4]), pairs sharded over the ranks
Default workload: cfg3 = BASELINE.json configs[2] "synthetic 8K ERP pair: 100k x 100k SURF-64 2-NN + 1M-hyp RANSAC sharded
1/2/4/8 B200" -- the configuration north_star's target is quoted on; it fits one GPU.

Scaling (`--scaling`, default "strong"): north_star's split of ONE pair -- query rows and hypothesis ids partitioned per
rank inside liberp_b200.so, match lists all-gathered in rank order, ONE 8-byte NCCL max all-reduce of the packed best
model (+ a min all-reduce for cross-check).  The total work is fixed as N grows.  "weak" = one whole pair per rank with
no data-path collective (N independent replicas; the frame-pair sharding of cfg5 without the fixed total).

`value` is BASELINE.json's first metric, 2-NN dist-evals/s, over the matching stage of the step (device-resident inputs,
device time from the library's own CUDA events, max over ranks); the second metric, RANSAC hyps/s, is reported beside it
(`ransac_hyps_per_s`) and `ms_per_step` is the whole step.  `e2e` is the same metric through the host-buffer C ABI call
the reference-facing wrappers make (H2D / D2H inside the timed region), over all --steps.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg2": dict(kind="pair", nq=20000, nt=20000, dim=64, W=4096, H=2048, hyps=10000, cross=False,
                 desc="synthetic 4K ERP pair: 20k x 20k SURF-64 2-NN + 8-pt RANSAC 10k hyps"),
    "cfg3": dict(kind="pair", nq=100000, nt=100000, dim=64, W=8192, H=4096, hyps=1000000, cross=False,
                 desc="synthetic 8K ERP pair: 100k x 100k SURF-64 2-NN + 1M-hyp RANSAC"),
    "cfg4": dict(kind="match", nq=200000, nt=200000, dim=128, W=8192, H=4096, hyps=0, cross=True,
                 desc="extended SURF-128 descriptors 200k x 200k with cross-check matching"),
    "cfg5": dict(kind="video", nq=20000, nt=20000, dim=64, W=4096, H=2048, hyps=10000, cross=False, pairs=1024, distinct=8,
                 desc="batched ERP video sequence: 1024 consecutive frame pairs x 20k kpts, pairs sharded across the GPUs"),
}
RATIO, TAU, METRIC, SAMPLE = 0.3, 0.002, 0, 8
CPU_Q_ROWS, CPU_HYPS = 32768, 65536          # the bounded CPU sample, the same in both arms (>= 1/16 of cfg3)


def make_pair(cfg, seed):
    """Descriptors with 50 % planted matches, and keypoints such that planted pairs are
    geometric correspondences of a known relative pose (30 % of them gross outliers)."""
    from erp_match_eightpoint_test_b200 import synth

    q, t, planted = synth.descriptor_pair(cfg["nq"], cfg["nt"], cfg["dim"], seed=seed)
    n_pl = int((planted >= 0).sum())
    kp = synth.keypoint_pair(n_pl, cfg["W"], cfg["H"], seed=seed + 100)
    rng = np.random.Generator(np.random.Philox(seed + 200))
    left = (rng.uniform(0, 1, (cfg["nq"], 2)) * [cfg["W"], cfg["H"] - 1]).astype(np.float32)
    right = (rng.uniform(0, 1, (cfg["nt"], 2)) * [cfg["W"], cfg["H"] - 1]).astype(np.float32)
    qi = np.nonzero(planted >= 0)[0]
    left[qi] = kp["left_xy"]
    right[planted[qi]] = kp["right_xy"]
    return dict(q=q, t=t, planted=planted, left=left, right=right, E=kp["E"], inlier=kp["inlier"])


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region.  The sampler is started
    before the warm-up (nvidia-smi needs ~100 ms to come up, a step takes a few ms) and every sample is
    time-stamped; mark() brackets the timed region and stop() keeps the samples inside it."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        self.t0 = self.t1 = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime

        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
            out, _ = self.p.communicate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), float(f[3]), [n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        if not rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.02 <= r[0] <= self.t1 + 0.02]
        where = "timed region"
        if not inside:      # region shorter than the sampling period: the warm-up ran the same kernels
            inside, where = rows, "warm-up + timed region"
        reasons = sorted({n for r in inside for n in r[4]})
        return dict(sm_mhz=float(np.median([r[1] for r in inside])), sm_max_mhz=float(max(r[2] for r in inside)),
                    power_w_max=float(max(r[3] for r in inside)), samples=len(inside), window=where, reasons=reasons)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(src="measured", hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sus=p.get("bf16_tflops_sustained", p["bf16_tflops"]))
    return dict(src="fallback", hbm=6650.0, bf16=1590.0, bf16_sus=1400.0)   # B200_PROFILING.md fallback


def tf32_measured():
    """The kept artefact of scripts/tf32_peak.py: a bare tcgen05.mma kind::tf32 loop at the sampled clock."""
    path = os.path.join(ROOT, "profiles", "r2_tf32_peak.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except ValueError:
            return None
    return None


def sass_stamp(kernel_substr, variant="ILi2"):
    """sha1 of the kernel's SASS in the shipped library (D = 64 instantiation): roofline.traffic is an ncu constant taken
    for ONE build of the kernel; a different stamp in profiles/roofline_traffic.json means the constant is stale."""
    import re

    lib = os.path.join(ROOT, "erp_match_eightpoint_test_b200", "lib", "liberp_b200.so")
    try:
        out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, timeout=120).stdout
    except (OSError, subprocess.TimeoutExpired):
        return None
    code, on = [], False
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            on = kernel_substr in m.group(1) and variant in m.group(1)
            continue
        if on and "/*0" in line:
            code.append(re.sub(r"/\*[0-9a-fx ]+\*/", "", line).strip())       # opcode text only: addresses and encodings dropped
    return hashlib.sha1("\n".join(code).encode()).hexdigest()[:12] if code else None


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle port; the reference itself needs
# OpenCV 3.4 C++ + xfeatures2d, which this image does not have -- DESIGN.md)
# --------------------------------------------------------------------------------------------
def cpu_sample(cfg, pair, q_rows=CPU_Q_ROWS, hyps=CPU_HYPS):
    """A bounded sample of the workload: q_rows queries against the full train set (+ cross-check where the workload
    has it), and `hyps` RANSAC hypotheses scored over the planted correspondences."""
    # all host cores: torchrun exports OMP_NUM_THREADS=1, which would throttle the CPU arm
    import oracle as O

    O.set_num_threads(len(os.sched_getaffinity(0)))
    q = pair["q"][:min(q_rows, cfg["nq"])]
    t0 = time.perf_counter()
    m = O.match(q, pair["t"], RATIO, cfg["cross"])
    t_match = time.perf_counter() - t0
    evals = len(q) * cfg["nt"] * (2 if cfg["cross"] else 1)
    out = dict(evals_per_s=evals / t_match, t_match=t_match, n_matches=len(m), cores=O.num_threads(), evals=evals,
               hyps_per_s=None, t_ransac=0.0, hyps=0)
    sample = f"{len(q)} of {cfg['nq']} queries x {cfg['nt']} train (exact brute-force 2-NN + ratio" + \
             (" + cross-check" if cfg["cross"] else "") + ", fp64 accumulate)"
    if cfg["hyps"] > 0:
        hyps = min(hyps, cfg["hyps"])
        qi = np.nonzero(pair["planted"] >= 0)[0]
        l = O.bearings(pair["left"][qi], cfg["W"], cfg["H"])
        r = O.bearings(pair["right"][pair["planted"][qi]], cfg["W"], cfg["H"])
        t0 = time.perf_counter()
        O.ransac(l, r, seed=1, hyp0=0, H=hyps, S=SAMPLE, metric=METRIC, tau=TAU, want_counts=False)
        out["t_ransac"] = time.perf_counter() - t0
        out["hyps_per_s"] = hyps / out["t_ransac"]
        out["hyps"] = hyps
        sample += f"; {hyps} of {cfg['hyps']} hypotheses x {len(l)} correspondences"
    out["sample"] = sample
    return out


def cv2_context(cfg, pair, q_rows=4096):
    """What the reference's own third-party matcher does on these cores (context, not the parity target): cv2 brute force
    on a query sample, and FLANN KD-trees (src/feature_matcher.cpp:16,45: approximate, sub-linear) on the same sample."""
    try:
        import cv2
    except ImportError:
        return None
    cv2.setNumThreads(len(os.sched_getaffinity(0)))
    q = np.ascontiguousarray(pair["q"][:q_rows])
    t = pair["t"]
    out = {"cv2": cv2.__version__, "queries": len(q), "train": len(t), "cores": cv2.getNumThreads()}
    t0 = time.perf_counter()
    bf = cv2.BFMatcher(cv2.NORM_L2).knnMatch(q, t, k=2)
    dt = time.perf_counter() - t0
    out["bf_dist_evals_per_s"] = len(q) * len(t) / dt
    t0 = time.perf_counter()
    fl = cv2.FlannBasedMatcher()          # KD-tree, 4 trees, 32 checks: what DescriptorMatcher::create(FLANNBASED) builds
    fm = fl.knnMatch(q, t, k=2)
    dt = time.perf_counter() - t0
    out["flann_equiv_dist_evals_per_s"] = len(q) * len(t) / dt          # brute-force-equivalent rate (index build included)
    out["flann_queries_per_s"] = len(q) / dt
    agree = sum(1 for a, b in zip(bf, fm) if a[0].trainIdx == b[0].trainIdx)
    out["flann_nn_agreement"] = agree / max(len(q), 1)
    return out


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pair = make_pair(cfg, 0xE8B0 + 3)
    for _ in range(args.warmup):
        cpu_sample(cfg, pair, 512, 1024)
    tm = tr = 0.0
    ev = hy = 0
    s = None
    for _ in range(args.steps):
        s = cpu_sample(cfg, pair)
        tm += s["t_match"]; tr += s["t_ransac"]; ev += s["evals"]; hy += s["hyps"]
    value = ev / tm
    hyps_s = hy / tr if tr > 0 else None
    line = {
        "impl": "reference", "metric": "2nn_dist_evals_per_s", "value": value, "unit": "dist-evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * (tm + tr) / args.steps, "higher_is_better": True,
        "scaling": scaling_of(args), "vs_baseline": None, "dtype": "f32 data, f64 accumulate", "data": "synthetic",
        "config": workload_config(cfg), "run": {"engine": "CPU oracle port of the reference path (OpenMP)", "sample": s["sample"]},
        "ransac_hyps_per_s": hyps_s,
        "cpu_baseline": {"value": value, "unit": "dist-evals/s", "cores": s["cores"], "kind": "port", "sample": s["sample"],
                         "ransac_hyps_per_s": hyps_s},
        "e2e": {"value": value, "unit": "dist-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def scaling_of(args):
    return args.scaling or "strong"


def workload_config(cfg):
    """What defines the workload -- identical in both arms (the driver compares `config`); how an arm ran it (engine,
    sharding, the CPU arm's bounded sample) goes under `run`."""
    c = {"workload": cfg["desc"], "nq": cfg["nq"], "nt": cfg["nt"], "dim": cfg["dim"], "hyps": cfg["hyps"], "cross_check": cfg["cross"],
         "ratio": RATIO, "tau": TAU, "sample_size": SAMPLE, "image": [cfg["W"], cfg["H"]]}
    if "pairs" in cfg:
        c["pairs"] = cfg["pairs"]
    return c


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
class Rig:
    """torch.distributed for the plumbing (rendezvous, barriers, max over ranks), liberp_b200.so for everything timed."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        import erp_match_eightpoint_test_b200 as erp

        self.torch, self.dist, self.erp = torch, dist, erp
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.ctx = erp.Context(self.local)
        if args.engine is not None:
            self.ctx.set_engine(args.engine)
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)
        self.strong = scaling_of(args) == "strong" and self.world > 1
        if self.strong:
            # the library's own NCCL clique: rank 0 makes the id, torch only carries the 128 bytes
            box = [erp.comm_unique_id() if self.rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            self.ctx.comm_init(self.world, self.rank, box[0])
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)                 # > 126 MB L2

    def flush_l2(self):
        with self.torch.cuda.stream(self.stream):
            self.flush.zero_()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def sum_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    def close(self):
        self.torch.cuda.synchronize()
        self.ctx.close()
        if self.world > 1:
            self.dist.destroy_process_group()


def distance_roofline(rig, cfg, stats, k_ms, nq_kernel, nt, dim, clocks, workload):
    """Roofline of the dominant kernel (distance tiles + fused top-k): algorithmic flops = 2*D per dist-eval.
    Two denominators: the driver-measured bf16 dense peak / 2 (tf32), and -- when scripts/tf32_peak.py has been run on
    this pool -- the measured tcgen05.mma kind::tf32 rate of a bare UMMA loop scaled to the sampled SM clock."""
    pk = peaks()
    engine = {1: "exact_simt_fp64", 2: "tcgen05_3xtf32", 3: "tcgen05_1xtf32"}.get(stats["engine"], str(stats["engine"]))
    k_s = k_ms * 1e-3
    achieved = nq_kernel * nt * 2.0 * dim / k_s / 1e12 if k_s > 0 else 0.0
    div = 1.0 if engine == "tcgen05_1xtf32" else 3.0
    peak = pk["bf16"] / 2.0 / div
    traffic = stamp = stamp_now = None
    tr_path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tr_path):
        tr = json.load(open(tr_path))
        traffic = tr.get(engine + ":" + workload)      # dram bytes per launch (ncu --set full)
        stamp = tr.get(engine + ":sass")
    if engine.startswith("tcgen05"):
        stamp_now = sass_stamp("knn2_tc1_kernelILi" if engine == "tcgen05_1xtf32" else "knn2_tc_kernelILi", "ILi%dE" % ((dim + 31) // 32))
    roof = {"bound": "tensor", "kernel": "distance tiles + fused top-k (" + engine + ")", "achieved": achieved,
            "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
            # the stamp belongs to the captured instantiation: compared only where a constant exists for this workload
            "traffic_sass_stamp": None if traffic is None else {"captured": stamp, "this_build": stamp_now,
                                   "stale": (stamp is not None and stamp_now is not None and stamp != stamp_now)},
            "kernel_ms": k_ms,
            "peak_from": f"{pk['src']} bf16 {pk['bf16']} TFLOP/s / 2 (tf32)" + ("" if div == 1.0 else " / 3 (3xTF32)")
                         + "; algorithmic 2*D flop per dist-eval", "rescanned_queries": stats["rescanned"]}
    tm = tf32_measured()
    if tm and tm.get("burst_tflops"):
        # a kernel timed alone in a short burst is compared with the burst figure (1965 MHz); the bare loop itself becomes
        # power capped after a few milliseconds (sustained figure)
        roof["peak_tcgen05_tf32_measured"] = {"burst_tflops": tm["burst_tflops"], "sustained_tflops": tm.get("sustained_tflops"),
                                              "frac_of_burst": achieved / (tm["burst_tflops"] / div),
                                              "issued_frac_of_burst": achieved * (dim + (8 if dim <= 64 and div == 1.0 else 0)) / dim / (tm["burst_tflops"] / div),
                                              "from": "profiles/r2_tf32_peak.json (scripts/tf32_peak.py: bare tcgen05.mma kind::tf32 loop)"}
    return engine, roof


def run_pair(args, cfg, rig):
    """cfg2 / cfg3: one ERP pair per step through ONE device-resident library call."""
    torch, erp = rig.torch, rig.erp
    from erp_match_eightpoint_test_b200 import binding

    rank, world, dev, ctx, stream, strong = rig.rank, rig.world, rig.dev, rig.ctx, rig.stream, rig.strong
    # ---- inputs.  weak: every rank owns a whole pair (own seed).  strong: one pair, query rows split.
    pair = make_pair(cfg, 0xE8B0 + 3 + (0 if (strong or world == 1) else rank))
    nq_all, nt, dim = cfg["nq"], cfg["nt"], cfg["dim"]
    qlo, qhi = erp.shard_range(nq_all, rank, world) if strong else (0, nq_all)
    nq = qhi - qlo
    hyps_rank = (erp.shard_range(cfg["hyps"], rank, world)[1] - erp.shard_range(cfg["hyps"], rank, world)[0]) if strong else cfg["hyps"]
    h_q = torch.from_numpy(pair["q"]).pin_memory()
    h_t = torch.from_numpy(pair["t"]).pin_memory()
    h_left = torch.from_numpy(pair["left"]).pin_memory()
    h_right = torch.from_numpy(pair["right"]).pin_memory()

    # device buffers live on torch's default stream (the library only borrows the pointers)
    d_q, d_t = h_q[qlo:qhi].to(dev), h_t.to(dev)
    d_left, d_right = h_left.to(dev), h_right.to(dev)
    d_matches = torch.empty((nq_all, 4), dtype=torch.int32, device=dev)          # erp_dmatch records
    d_n = torch.zeros(1, dtype=torch.int32, device=dev)
    d_mask = torch.empty(nq_all, dtype=torch.uint8, device=dev)
    d_res = torch.zeros(C_sizeof_result(), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def step():
        """One pass of the hot path with device-resident inputs: the call only enqueues."""
        with torch.cuda.stream(stream):
            ctx.pair_pose_dev(d_q, nq_all, d_t, nt, dim, RATIO, False, d_left, d_right, 8, cfg["W"], cfg["H"], 1, cfg["hyps"],
                              SAMPLE, METRIC, TAU, d_matches, d_n, d_mask, d_res, dist=strong)

    def result():
        buf = d_res.cpu().numpy().tobytes()
        res = binding.RansacResult.from_buffer_copy(buf)
        return int(d_n.item()), ctx._result(res)

    # ---- warm-up (the clock sampler is already running)
    sampler = ClockSampler(rig.local) if rank == 0 else None
    for _ in range(max(args.warmup, 0)):
        rig.flush_l2()
        step()
    rig.barrier()

    # ---- timed region: exactly K steps, L2 flushed between them (the flush is outside the library's stage events)
    if sampler:
        sampler.mark_start()
    launches0 = ctx.launch_count
    t_match = t_xchg = t_ransac = t_kernel = t_score = 0.0
    n_score = 0
    sc_stats = None
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        rig.flush_l2()
        step()
        a, b, c = ctx.last_stage_ms()                  # synchronises the library's stream
        t_match += a; t_xchg += b; t_ransac += c
        t_kernel += ctx.last_knn_kernel_ms()
        sc_ms, n_score = ctx.last_score_kernel_ms()
        t_score += sc_ms
    rig.barrier()
    if sampler:
        sampler.mark_end()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    m, res = result()
    if args.dump_outputs and rank == 0:
        # the outputs are identical on every rank of a strong-scaling clique; weak scaling dumps rank 0's own pair
        dump_outputs(args.dump_outputs, {"n_matches": m, **dmatch_arrays(d_matches[:m].cpu().numpy()),
                                         "inlier_mask": d_mask[:m].cpu().numpy(), **pose_arrays(res)})
    sc_stats = ctx.last_score_stats()
    stats = ctx.last_knn_stats()
    # max over ranks of the device-timed sums (the step of a rank ends when its pose is done; collectives inside)
    t_step = t_match + t_xchg + t_ransac
    t_match, t_xchg, t_ransac, t_kernel, t_score, t_step = rig.max_over_ranks([t_match, t_xchg, t_ransac, t_kernel, t_score, t_step])
    launches_all = rig.sum_over_ranks([launches])[0]

    # ---- end-to-end through the host-buffer C ABI (what the C++ class wrappers call), every step
    pq, pt = h_q.numpy(), h_t.numpy()
    pl, pr = h_left.numpy(), h_right.numpy()
    t_e2e_match = t_pair = 0.0
    mt = pm = pres = None
    for it in range(args.steps + 1):
        torch.cuda.synchronize()
        a = time.perf_counter()
        mt = ctx.knn2_match_dist(pq, pt, RATIO, False) if strong else ctx.knn2_match(pq, pt, RATIO, False)   # H2D q,t; D2H matches
        b = time.perf_counter()
        if strong:
            pm, pres = ctx.pair_pose_dist(pq, pt, pl, pr, cfg["W"], cfg["H"], ratio=RATIO, cross_check=False, seed=1, H=cfg["hyps"],
                                          S=SAMPLE, metric=METRIC, tau=TAU)
        else:
            pm, pres = ctx.pair_pose(pq, pt, pl, pr, cfg["W"], cfg["H"], ratio=RATIO, cross_check=False, seed=1, H=cfg["hyps"],
                                     S=SAMPLE, metric=METRIC, tau=TAU)
        c = time.perf_counter()
        if it > 0:
            t_e2e_match += b - a
            t_pair += c - b
    assert len(pm) == m and pres["packed"] == res["packed"], "host-buffer call disagrees with the device-resident call"
    # the same match call on PAGEABLE buffers (what a cv::Mat is): staged through pinned chunks by the library
    t_pageable = 0.0
    if not strong:
        gq, gt = np.array(pq), np.array(pt)
        for it in range(4):
            torch.cuda.synchronize()
            a = time.perf_counter()
            gm = ctx.knn2_match(gq, gt, RATIO, False)
            if it > 0:
                t_pageable += (time.perf_counter() - a) / 3
        assert gm.tobytes() == mt.tobytes()
    t_e2e_match, t_pair = rig.max_over_ranks([t_e2e_match, t_pair])
    share = 1.0 / world if strong else 1.0
    h2d = int(pq.nbytes * share + pt.nbytes * share)
    d2h = len(mt) * 16 + 4
    h2d_pair = int(pq.nbytes * share + pt.nbytes * share + pl.nbytes + pr.nbytes)
    d2h_pair = m * 16 + m + 4 + 216

    # the spec's arithmetic (3xTF32 tiles, knn_tc.cu) timed beside the default engine: same inputs, same results
    alt3 = None
    if stats["engine"] == 3 and rank == 0 and world == 1:
        d_idx = torch.empty((nq, 2), dtype=torch.int32, device=dev)
        d_dist = torch.empty((nq, 2), dtype=torch.float32, device=dev)
        ctx.set_engine(2)
        ms3 = []
        for it in range(6):
            rig.flush_l2()
            with torch.cuda.stream(stream):
                ctx.knn2_dev(d_q, nq, d_t, nt, dim, d_idx, d_dist)
            ms3.append(ctx.last_knn_kernel_ms())
        k3 = float(np.mean(ms3[3:])) * 1e-3
        pk3 = peaks()["bf16"] / 6.0
        alt3 = {"kernel": "knn2_tc_kernel (3xTF32, top-4)", "kernel_ms": k3 * 1e3, "dist_evals_per_s": nq * nt / k3,
                "achieved": nq * nt * 2.0 * dim / k3 / 1e12, "peak": pk3, "unit": "TFLOP/s", "frac": nq * nt * 2.0 * dim / k3 / 1e12 / pk3,
                "rescanned_queries": ctx.last_knn_stats()["rescanned"]}
        ctx.set_engine(0 if args.engine is None else args.engine)

    if rank != 0:
        return None

    # ---- sanity of the timed work (a number from a wrong result is not a number)
    n_pl = int((pair["planted"] >= 0).sum())
    assert m == n_pl, (m, n_pl)
    En = np.asarray(res["E_refit"]).reshape(9)
    Eg = pair["E"].reshape(9) / np.linalg.norm(pair["E"])
    En = En / np.linalg.norm(En)
    e_err = float(min(np.linalg.norm(En - Eg), np.linalg.norm(En + Eg)))
    assert e_err < 2e-2, e_err

    units = nq_all * nt * (1 if strong else world)
    hyps_total = cfg["hyps"] * (1 if strong else world)
    value = args.steps * units / (t_match * 1e-3)
    engine, roof = distance_roofline(rig, cfg, stats, t_kernel / args.steps, nq, nt, dim, clocks, args.workload)
    # the second kernel of the step: hypothesis scoring.  Algorithmic work = 2*9 flop per residual;
    # the tensor-core pass is followed by a 1.5-instruction-per-residual FP32 epilogue, which is what bounds it
    pk = peaks()
    peak3 = pk["bf16"] / 2.0 / 3.0
    sc_s = t_score * 1e-3 / args.steps
    residuals = float(hyps_rank) * m
    evaluated = residuals
    if sc_stats["hyps"] > 0 and sc_stats["tiles_total"] > 0:
        seen = min(sc_stats["tiles_all"] * 256, m)
        evaluated = residuals * (sc_stats["hyps"] * seen + sc_stats["survivors"] * (m - seen)) / float(sc_stats["hyps"] * m)
    score_roof = None
    if sc_s > 0:
        score_roof = {"kernel": "score_tc_kernel (3xTF32 residual GEMM + counting epilogue)" if n_score > 1 else "score_kernel (SIMT)",
                      "bound": "tensor (operands from shared memory) + issue", "launches_per_step": n_score,
                      "kernel_ms": t_score / args.steps, "problem_residuals_per_s": residuals / sc_s,
                      "evaluated_fraction": evaluated / residuals, "pruning": sc_stats, "residuals_per_s": evaluated / sc_s,
                      "achieved": evaluated * 18.0 / sc_s / 1e12, "unit": "TFLOP/s", "peak": peak3,
                      "frac": evaluated * 18.0 / sc_s / 1e12 / peak3,
                      "note": "EVALUATED residuals (exact progressive pruning skips the rest) x 18 algorithmic flop against the 3xTF32 "
                              "tensor peak (the padded K = 32 product issues 64 flop per residual: x 3.56); per rank"}
    cpu = cpu_ctx = None
    if world == 1 and not args.no_cpu_baseline:
        s = cpu_sample(cfg, pair)
        cpu = {"value": s["evals_per_s"], "unit": "dist-evals/s", "cores": s["cores"], "kind": "port", "sample": s["sample"],
               "ransac_hyps_per_s": s["hyps_per_s"], "seconds": s["t_match"] + s["t_ransac"]}
        cpu_ctx = cv2_context(cfg, pair)
    sharding = ("query rows + hypothesis ids per rank inside liberp_b200.so: all-gather of the match slots, one 8-byte max all-reduce "
                "of the packed best model -- both by the library's own kernels over NVLink peer-memory windows "
                "(ERP_B200_PEER=0: ncclAllGather / ncclAllReduce)") if strong else \
               ("one GPU" if world == 1 else "one ERP pair per rank, no collective")
    return {
        "metric": "2nn_dist_evals_per_s", "value": value, "unit": "dist-evals/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_step / args.steps, "higher_is_better": True,
        "scaling": scaling_of(args), "vs_baseline": None,
        "dtype": ("f32 data; TF32 tiles (certified) + f64 exact refine" if engine == "tcgen05_1xtf32" else
                  "f32 data; 3xTF32 tiles + f64 refine" if engine.startswith("tcgen05") else "f32 data; f64 direct-form accumulate"),
        "data": "synthetic",
        "config": workload_config(cfg),
        "run": {"engine": engine, "nq_per_gpu": nq, "hyps_per_gpu": hyps_rank, "correspondences": m,
                "l2": "flushed between timed steps (256 MiB write)", "sharding": sharding,
                "api": "erp_pair_pose_dist_dev" if strong else "erp_pair_pose_dev"},
        "match_ms": t_match / args.steps, "exchange_gather_ms": t_xchg / args.steps, "ransac_ms": t_ransac / args.steps,
        "ransac_hyps_per_s": args.steps * hyps_total / (t_ransac * 1e-3),
        "step_dist_evals_per_s": args.steps * units / (t_step * 1e-3),
        "roofline": roof, "roofline_3xtf32": alt3, "roofline_scoring": score_roof,
        "e2e": {"value": units * args.steps / t_e2e_match, "unit": "dist-evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h),
                "match_ms": 1e3 * t_e2e_match / args.steps, "steps": args.steps,
                "match_ms_pageable_source": 1e3 * t_pageable if t_pageable > 0 else None,
                "api": "erp_knn2_match_dist (host buffers, per rank: its query rows + 1/N of the train rows up, NVLink all-gather)" if strong
                       else "erp_knn2_match (host buffers)",
                "pair": {"ms": 1e3 * t_pair / args.steps, "dist_evals_per_s": units * args.steps / t_pair,
                         "h2d_bytes_per_step": h2d_pair, "d2h_bytes_per_step": int(d2h_pair),
                         "api": "erp_pair_pose_dist" if strong else "erp_pair_pose",
                         "what": "the whole pair in ONE host-buffer call: descriptors + keypoints up, match records + pose + mask back"}},
        "gpu_launches": int(launches_all), "gpu_launches_per_step_per_rank": launches / args.steps,
        "clocks": clocks, "cpu_baseline": cpu, "cpu_context": cpu_ctx,
        "check": {"matches": m, "planted": n_pl, "E_refit_err": e_err, "inliers": res["count"], "rescanned": stats["rescanned"]},
        "wall_s_timed_region": wall,
    }


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes what the timed path returned in its last step as <out_dir>/<name>.npy, so that two builds can be compared
    output for output on identical (seeded) inputs.  float32 results stay float32; everything else (indices, counts,
    fp64 matrices) is stored as float64, which holds every int32 exactly."""
    arrays = {k: (a if a.dtype == np.float32 else a.astype(np.float64)) for k, a in ((k, np.asarray(v)) for k, v in arrays.items())}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"dump of {total} bytes exceeds {DUMP_LIMIT}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dmatch_arrays(m, prefix="matches_"):
    """erp_dmatch records (cv::DMatch layout) as one array per field."""
    from erp_match_eightpoint_test_b200 import binding

    m = np.ascontiguousarray(m).view(binding.DMATCH).reshape(-1)
    return {prefix + "query_idx": m["queryIdx"], prefix + "train_idx": m["trainIdx"], prefix + "img_idx": m["imgIdx"],
            prefix + "distance": m["distance"]}


def pose_arrays(res):
    """The fields of erp_ransac_result a caller reads (`packed` is count and hyp_id together)."""
    return {"hyp_id": res["hyp"], "count": res["count"], "n_refit": res["n_refit"], "E_best": res["E"], "E_refit": res["E_refit"],
            "pose": res["pose"]}


def C_sizeof_result():
    import ctypes

    from erp_match_eightpoint_test_b200 import binding

    return ctypes.sizeof(binding.RansacResult)


def run_match(args, cfg, rig):
    """cfg4: 200k x 200k SURF-128 matching with cross-check; query rows per rank, per-train nearest query min-reduced."""
    torch, erp = rig.torch, rig.erp
    rank, world, dev, ctx, stream, strong = rig.rank, rig.world, rig.dev, rig.ctx, rig.stream, rig.strong
    from erp_match_eightpoint_test_b200 import synth

    seed = 0xE8B0 + 4 + (0 if (strong or world == 1) else rank)
    q, t, planted = synth.descriptor_pair(cfg["nq"], cfg["nt"], cfg["dim"], seed=seed)
    nq_all, nt, dim = cfg["nq"], cfg["nt"], cfg["dim"]
    qlo, qhi = erp.shard_range(nq_all, rank, world) if strong else (0, nq_all)
    nq = qhi - qlo
    h_q, h_t = torch.from_numpy(q).pin_memory(), torch.from_numpy(t).pin_memory()
    d_q, d_t = h_q[qlo:qhi].to(dev), h_t.to(dev)
    d_matches = torch.empty((nq + 1, 4), dtype=torch.int32, device=dev)
    d_n = torch.zeros(1, dtype=torch.int32, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()

    def step():
        e0, e1 = ev(), ev()
        with torch.cuda.stream(stream):
            e0.record(stream)
            ctx.knn2_match_dist_dev(d_q, nq_all, d_t, nt, dim, RATIO, True, d_matches, d_n)
            e1.record(stream)
        return e0, e1

    sampler = ClockSampler(rig.local) if rank == 0 else None
    for _ in range(max(args.warmup, 0)):
        rig.flush_l2()
        step()
    rig.barrier()
    if sampler:
        sampler.mark_start()
    launches0 = ctx.launch_count
    t_match = t_kernel = 0.0
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        rig.flush_l2()
        e0, e1 = step()
        torch.cuda.synchronize()
        t_match += e0.elapsed_time(e1)
        t_kernel += ctx.last_knn_kernel_ms()          # the reverse (cross-check) search is the last one: same shape class
    rig.barrier()
    if sampler:
        sampler.mark_end()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    n_local = int(d_n.item())
    if args.dump_outputs and rank == 0:
        # strong scaling: rank 0's query rows (global query ids) are what its caller receives
        dump_outputs(args.dump_outputs, {"n_matches": n_local, **dmatch_arrays(d_matches[:n_local].cpu().numpy())})
    stats = ctx.last_knn_stats()
    t_match, t_kernel = rig.max_over_ranks([t_match, t_kernel])
    n_total, launches_all = rig.sum_over_ranks([n_local if (strong or world == 1) else n_local / world, launches])

    pq, pt = h_q.numpy(), h_t.numpy()
    t_e2e = 0.0
    mt = None
    e2e_steps = args.steps
    for it in range(e2e_steps + 1):
        torch.cuda.synchronize()
        a = time.perf_counter()
        mt = ctx.knn2_match_dist(pq, pt, RATIO, True) if strong else ctx.knn2_match(pq, pt, RATIO, True)
        if it > 0:
            t_e2e += time.perf_counter() - a
    (t_e2e,) = rig.max_over_ranks([t_e2e])
    assert len(mt) == n_local
    if rank != 0:
        return None
    n_pl = int((planted >= 0).sum())
    assert abs(n_total - n_pl) <= n_pl * 1e-3, (n_total, n_pl)        # planted pairs are mutual nearest neighbours
    # forward + reverse search: 2 x nq x nt dist-evals per step
    units = 2.0 * nq_all * nt * (1 if strong else world)
    engine, roof = distance_roofline(rig, cfg, stats, t_kernel / args.steps, nt if True else nq, nq, dim, clocks, args.workload)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        s = cpu_sample(cfg, dict(q=q, t=t, planted=planted), q_rows=8192)
        cpu = {"value": s["evals_per_s"], "unit": "dist-evals/s", "cores": s["cores"], "kind": "port", "sample": s["sample"],
               "seconds": s["t_match"]}
    share = 1.0 / world if strong else 1.0
    return {
        "metric": "2nn_dist_evals_per_s", "value": args.steps * units / (t_match * 1e-3), "unit": "dist-evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_match / args.steps, "higher_is_better": True,
        "scaling": scaling_of(args), "vs_baseline": None, "dtype": "f32 data; TF32 tiles (certified) + f64 exact refine", "data": "synthetic",
        "config": workload_config(cfg),
        "run": {"engine": engine, "nq_per_gpu": nq, "l2": "flushed between timed steps (256 MiB write)",
                "sharding": ("query rows per rank; per-train nearest query: ncclAllReduce(min) of d2, then of the query id"
                             if strong else ("one GPU" if world == 1 else "one descriptor set pair per rank, no collective")),
                "dist_evals": "forward + reverse search = 2 x nq x nt per step", "api": "erp_knn2_match_dist_dev"},
        "match_ms": t_match / args.steps, "roofline": roof,
        "e2e": {"value": units * e2e_steps / t_e2e, "unit": "dist-evals/s", "h2d_bytes_per_step": int((pq.nbytes + pt.nbytes) * share),
                "d2h_bytes_per_step": int(len(mt) * 16 + 4), "match_ms": 1e3 * t_e2e / e2e_steps, "steps": e2e_steps,
                "api": "erp_knn2_match_dist (host buffers)" if strong else "erp_knn2_match (host buffers)"},
        "gpu_launches": int(launches_all), "clocks": clocks, "cpu_baseline": cpu,
        "check": {"matches": int(n_total), "planted": n_pl, "rescanned": stats["rescanned"]}, "wall_s_timed_region": wall,
    }


def run_video(args, cfg, rig):
    """cfg5: 1024 frame pairs, round-robin over the ranks; a rank runs TWO host threads with a context each so that the
    uploads of one pair overlap the kernels of the other.  No collective: pairs are independent."""
    torch, erp = rig.torch, rig.erp
    rank, world, dev = rig.rank, rig.world, rig.dev
    n_threads = args.threads
    mine = list(range(rank, cfg["pairs"], world))
    distinct = [make_pair(cfg, 0xE8B0 + 5 + i) for i in range(cfg["distinct"])]
    # pinned host copies (what a capture pipeline would hand over)
    host = []
    for p in distinct:
        host.append({k: torch.from_numpy(np.ascontiguousarray(p[k])).pin_memory().numpy() for k in ("q", "t", "left", "right")})
    ctxs = [rig.ctx] + [erp.Context(rig.local) for _ in range(n_threads - 1)]
    if args.engine is not None:
        for c in ctxs:
            c.set_engine(args.engine)
    first = [None] * cfg["distinct"]
    errs = []

    def batch(check, keep=None):
        def work(tid):
            try:
                c = ctxs[tid]
                for j in range(tid, len(mine), n_threads):
                    d = mine[j] % cfg["distinct"]
                    h = host[d]
                    m, r = c.pair_pose(h["q"], h["t"], h["left"], h["right"], cfg["W"], cfg["H"], ratio=RATIO, seed=1, H=cfg["hyps"],
                                       S=SAMPLE, metric=METRIC, tau=TAU)
                    if keep is not None:
                        keep[j] = (len(m), r, m if j < cfg["distinct"] else None)      # records of the first pairs only (size cap)
                    key = (len(m), r["packed"])
                    if check:
                        if first[d] is None:
                            first[d] = key
                        assert first[d] == key, (d, first[d], key)
            except Exception as e:      # surfaced below
                errs.append(e)
        ts = [threading.Thread(target=work, args=(k,)) for k in range(n_threads)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        if errs:
            raise errs[0]

    sampler = ClockSampler(rig.local) if rank == 0 else None
    for w in range(max(1, min(args.warmup, 2))):
        batch(True)
    rig.barrier()
    if sampler:
        sampler.mark_start()
    launches0 = sum(c.launch_count for c in ctxs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    wall0 = time.perf_counter()
    last = {} if args.dump_outputs else None
    for s in range(args.steps):
        batch(False, last if s == args.steps - 1 else None)
    e1.record()
    e1.synchronize()
    rig.barrier()
    if sampler:
        sampler.mark_end()
    wall = time.perf_counter() - wall0
    t_ms = e0.elapsed_time(e1)
    launches = sum(c.launch_count for c in ctxs) - launches0
    clocks = sampler.stop() if sampler else None
    k_ms = rig.ctx.last_knn_kernel_ms()
    stats = rig.ctx.last_knn_stats()
    (t_ms,) = rig.max_over_ranks([t_ms])
    (launches_all,) = rig.sum_over_ranks([launches])
    for c in ctxs[1:]:
        c.close()
    if rank != 0:
        return None
    if last is not None:
        # per pair of this rank (in `mine` order): match count and pose; match records and masks of its first `distinct` pairs
        # (one per distinct input; all of them would exceed the dump's size cap)
        rows = [pose_arrays(last[j][1]) for j in range(len(mine))]
        out = {k: np.stack([np.asarray(r[k]) for r in rows]) for k in rows[0]}
        out["pair"] = np.array(mine)
        out["n_matches"] = np.array([last[j][0] for j in range(len(mine))])
        first_pairs = range(min(cfg["distinct"], len(mine)))
        out.update(dmatch_arrays(np.concatenate([last[j][2] for j in first_pairs])))
        out["matches_pair"] = np.concatenate([np.full(last[j][0], mine[j]) for j in first_pairs])
        out["inlier_mask"] = np.concatenate([last[j][1]["mask"] for j in first_pairs])
        dump_outputs(args.dump_outputs, out)
    n_pl = int((distinct[0]["planted"] >= 0).sum())
    assert first[mine[0] % cfg["distinct"]][0] == int((distinct[mine[0] % cfg["distinct"]]["planted"] >= 0).sum())
    pairs = cfg["pairs"]
    units = float(pairs) * cfg["nq"] * cfg["nt"]
    value = args.steps * units / (t_ms * 1e-3)
    engine, roof = distance_roofline(rig, cfg, stats, k_ms, cfg["nq"], cfg["nt"], cfg["dim"], clocks, args.workload)
    h = host[0]
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        s = cpu_sample(cfg, distinct[0], q_rows=cfg["nq"], hyps=cfg["hyps"])
        cpu = {"value": s["evals_per_s"], "unit": "dist-evals/s", "cores": s["cores"], "kind": "port", "pairs_per_s": 1.0 / (s["t_match"] + s["t_ransac"]),
               "sample": "ONE of the %d pairs: " % pairs + s["sample"], "ransac_hyps_per_s": s["hyps_per_s"], "seconds": s["t_match"] + s["t_ransac"]}
    e2e = {"value": value, "unit": "dist-evals/s", "pairs_per_s": args.steps * pairs / (t_ms * 1e-3),
           "h2d_bytes_per_step": int((h["q"].nbytes + h["t"].nbytes + h["left"].nbytes + h["right"].nbytes) * pairs),
           "d2h_bytes_per_step": int((n_pl * 17 + 220) * pairs), "api": "erp_pair_pose (host buffers), one call per frame pair"}
    return {
        "metric": "2nn_dist_evals_per_s", "value": value, "unit": "dist-evals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 data; TF32 tiles (certified) + f64 exact refine", "data": "synthetic",
        "config": workload_config(cfg),
        "run": {"engine": engine, "pairs_per_gpu": len(mine), "distinct_pairs_cycled": cfg["distinct"], "host_threads_per_gpu": n_threads,
                "l2": "inputs stream from pinned host memory: every pair is a fresh 10.6 MB upload",
                "sharding": "frame pairs round-robin per rank, no collective; every call moves its inputs from host memory, so "
                            "value and e2e coincide"},
        "pairs_per_s": args.steps * pairs / (t_ms * 1e-3), "ms_per_pair": t_ms / args.steps / len(mine),
        "ransac_hyps_per_s": args.steps * pairs * cfg["hyps"] / (t_ms * 1e-3),
        "roofline": roof, "e2e": e2e, "gpu_launches": int(launches_all), "clocks": clocks, "cpu_baseline": cpu,
        "check": {"matches_pair0": first[0][0] if first[0] else None, "planted_pair0": n_pl}, "wall_s_timed_region": wall,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="strong (default): ONE workload split over the ranks inside the library; weak: a whole workload per rank")
    ap.add_argument("--engine", type=int, default=None, help="0 auto, 1 exact SIMT, 2 tcgen05 3xTF32, 3 tcgen05 1xTF32")
    ap.add_argument("--threads", type=int, default=2, help="cfg5: host threads (contexts) per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the product arm")
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, cfg)
        return
    rig = Rig(args)
    line = {"pair": run_pair, "match": run_match, "video": run_video}[cfg["kind"]](args, cfg, rig)
    if line is not None:
        print(json.dumps(line), flush=True)
    rig.close()


if __name__ == "__main__":
    sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)
    main()
