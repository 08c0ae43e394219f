"""A/B of the one-product engine's operand formats inside one build: runs bench.py alternately with
ERP_B200_TC1_OPERANDS=f16 and =tf32 and reports the median and spread of value, match_ms, roofline.kernel_ms and
ms_per_step per workload, with the card's name, power limit and the clocks bench.py sampled.

    python scripts/operands_ab.py [--runs 3] [--workloads cfg3,cfg4:1,cfg2] [--dump DIR] [--counters LIB] [--out FILE]

A workload written name:N runs N times per format instead of --runs.  --dump DIR also compares bench.py --dump-outputs of
the first run of each format byte for byte.  --counters LIB runs one short cfg3 bench per format against a library built
with scripts/build_variant.sh 1 and reports its per-tile clock64 phase timers."""
from __future__ import annotations

import argparse
import filecmp
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORMATS = ("f16", "tf32")


def bench(fmt, workload, extra=(), lib=None):
    env = dict(os.environ, ERP_B200_TC1_OPERANDS=fmt)
    if lib:
        # the instrumented build synchronises after every launch, which a captured CUDA graph does not allow
        env.update(ERP_B200_LIB=lib, ERP_B200_GRAPH="0")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", workload, *extra]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if p.returncode != 0:
        raise RuntimeError("%s %s failed:\n%s" % (fmt, workload, p.stderr[-4000:]))
    lines = p.stdout.strip().splitlines()
    return json.loads(lines[-1]), lines


def pick(r):
    roof = r.get("roofline") or {}
    return {"value": r["value"], "match_ms": r.get("match_ms"), "kernel_ms": roof.get("kernel_ms"), "ms_per_step": r["ms_per_step"]}


def summary(xs):
    xs = [x for x in xs if x is not None]
    if not xs:
        return None
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--workloads", default="cfg3")
    ap.add_argument("--dump", default=None)
    ap.add_argument("--counters", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    report = {"card": card[0] if card else None, "workloads": {}}
    for spec in args.workloads.split(","):
        workload, _, n = spec.partition(":")
        runs = int(n) if n else args.runs
        rows = {f: [] for f in FORMATS}
        clocks = {f: [] for f in FORMATS}
        for i in range(runs):
            for fmt in FORMATS:                 # alternate, so that drift of the shared machine hits both alike
                extra = []
                if args.dump and i == 0:
                    extra = ["--dump-outputs", os.path.join(args.dump, "%s_%s" % (workload, fmt))]
                r, _ = bench(fmt, workload, extra)
                rows[fmt].append(pick(r))
                clocks[fmt].append(r.get("clocks"))
                print(workload, fmt, i, json.dumps(pick(r)), flush=True)
        w = {}
        for fmt in FORMATS:
            w[fmt] = {k: summary([row[k] for row in rows[fmt]]) for k in rows[fmt][0]}
            w[fmt]["clocks"] = clocks[fmt]
        v16, v32 = w["f16"]["value"], w["tf32"]["value"]
        w["value_gain"] = v16["median"] / v32["median"] - 1.0
        w["value_spreads_disjoint"] = v16["min"] > v32["max"]
        if args.dump:
            a, b = (os.path.join(args.dump, "%s_%s" % (workload, f)) for f in FORMATS)
            names = sorted(os.listdir(a))
            w["dumps_identical"] = names == sorted(os.listdir(b)) and all(filecmp.cmp(os.path.join(a, n), os.path.join(b, n), shallow=False)
                                                                          for n in names)
        report["workloads"][workload] = w
        print(json.dumps({workload: {k: w[k] for k in w if k not in FORMATS}}), flush=True)
    if args.counters:
        report["counters"] = {}
        for fmt in FORMATS:
            _, lines = bench(fmt, "cfg3", ["--steps", "2", "--warmup", "1"], lib=args.counters)
            report["counters"][fmt] = [l for l in lines if l.startswith("epi:")][-1:]
            print(fmt, report["counters"][fmt], flush=True)
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
