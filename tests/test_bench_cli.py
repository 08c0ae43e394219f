"""bench.py's contract where it can be checked without a GPU: the CPU arm (`--impl reference` = the oracle port of the
reference path on the host cores) prints ONE JSON line with the keys the driver reads, its `config` is the product arm's
`config` for the same workload, ranks other than 0 stay silent, and the product arm fails loudly (no CPU fallback) when
there is no GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run_bench(*argv, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, timeout=600,
                          cwd=ROOT, env=dict(os.environ, **(env or {})))


@pytest.fixture(scope="module")
def reference_line():
    r = run_bench("--impl", "reference", "--workload", "cfg2", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_line_has_the_contract_keys(reference_line):
    d = reference_line
    assert d["impl"] == "reference"
    assert d["metric"] == "2nn_dist_evals_per_s" and d["unit"] == "dist-evals/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "queries" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_both_arms_describe_the_workload_identically(reference_line):
    import bench
    for name, cfg in bench.WORKLOADS.items():
        c = bench.workload_config(cfg)
        assert c["workload"] == cfg["desc"] and "engine" not in c and "sample" not in c, name     # how an arm ran goes under `run`
    assert reference_line["config"] == bench.workload_config(bench.WORKLOADS["cfg2"])
    # the CPU arm's sample is at least 1/16 of the workload in both dimensions (SURVEY 8d)
    assert "20000 of 20000 queries" in reference_line["cpu_baseline"]["sample"]


def test_reference_arm_runs_on_rank_zero_only():
    r = run_bench("--impl", "reference", "--workload", "cfg2", "--steps", "1", "--warmup", "0", "--gpus", "2",
                  env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_and_dump_arguments_are_checked():
    assert run_bench("--impl", "reference", "--workload", "cfg2", "--steps", "0").returncode == 2
    assert run_bench("--impl", "reference", "--workload", "cfg2", "--dump-outputs", "unused").returncode == 2


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_path_results(tmp_path):
    """--dump-outputs writes the last timed step's outputs (cfg2: match records, inlier mask, winner and pose) as float32 /
    float64 .npy files; they equal the oracle on the benchmark's seeded inputs, and a second run writes the same bytes."""
    import numpy as np

    import bench
    import oracle as O

    runs = []
    for k in range(2):
        out = tmp_path / str(k)
        r = run_bench("--workload", "cfg2", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == 3 and line["e2e"]["steps"] == 3
        runs.append({f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))})
    d = runs[0]
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert d.keys() == runs[1].keys() and all(d[k].tobytes() == runs[1][k].tobytes() for k in d)
    cfg = bench.WORKLOADS["cfg2"]
    pair = bench.make_pair(cfg, 0xE8B0 + 3)
    om = O.match(pair["q"], pair["t"], bench.RATIO, False)
    assert int(d["n_matches"]) == len(om)
    for key, field in (("query_idx", "queryIdx"), ("train_idx", "trainIdx"), ("img_idx", "imgIdx"), ("distance", "distance")):
        assert np.array_equal(d["matches_" + key], om[field]), key
    l = O.bearings(pair["left"][om["queryIdx"]], cfg["W"], cfg["H"])
    r = O.bearings(pair["right"][om["trainIdx"]], cfg["W"], cfg["H"])
    ref = O.ransac(l, r, seed=1, hyp0=0, H=cfg["hyps"], S=bench.SAMPLE, metric=bench.METRIC, tau=bench.TAU)
    assert int(d["hyp_id"]) == ref["hyp"] and int(d["count"]) == ref["count"] == int(d["inlier_mask"].sum())
    assert np.array_equal(d["inlier_mask"], O.inlier_mask(ref["E"], l, r, metric=bench.METRIC, tau=bench.TAU))
    assert d["E_best"].shape == d["E_refit"].shape == (3, 3) and d["pose"].shape == (12,)


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible: the product arm would run")
    r = run_bench("--workload", "cfg2", "--steps", "1", "--warmup", "0")
    assert r.returncode != 0
    assert not any(l.startswith("{") for l in r.stdout.splitlines())
