"""CPU suite: the bench.py contract that can be checked without a GPU -- the reference arm prints one JSON line with the
contract's keys, and the product arm refuses to run (no CPU fallback) instead of silently measuring something else.
GPU suite: the product arm's --dump-outputs and --steps."""
import json
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT

REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "e2e", "cpu_baseline", "impl"}


def run(*args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["metric"] == "warped frame-pairs/sec" and d["unit"] == "pairs/s"
    assert d["config"]["workload"] == "sintel_full" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_product_arm_refuses_to_run_without_a_gpu():
    if torch.cuda.is_available():
        import pytest
        pytest.skip("this check is for the GPU-less build container")
    r = run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_dump_outputs_repeat_and_steps_set_the_timed_steps(tmp_path):
    """--dump-outputs writes the last timed step's arrays (evaluate_sharded's dict) as float64 .npy; the seeded inputs make
    them identical from run to run, whatever the step count.  --steps K runs K timed steps: twice the steps, twice the
    library launches inside the timed region."""
    import numpy as np
    dumps, lines = [], []
    for steps in (3, 6):
        out = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--pairs", "16",
                            "--no-extras", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1]))
        dumps.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    assert [d["steps"] for d in lines] == [3, 6] and lines[1]["gpu_launches"] == 2 * lines[0]["gpu_launches"] > 0
    assert set(dumps[0]) == {"per_sequence_mean", "mean_over_sequences", "mean_over_pairs", "pooled_rmse", "n_pairs"}
    for k, a in dumps[0].items():
        assert a.dtype == np.float64 and np.array_equal(a, dumps[1][k]), k
    assert float(dumps[0]["n_pairs"]) == 16
    assert float(dumps[0]["mean_over_sequences"]) == float.fromhex(lines[0]["result_check"]["mean_over_sequences_rmse_hex"])


def test_committed_product_lines_carry_the_contract_and_are_self_consistent():
    """The JSON lines of `python bench.py` committed under profiles/ (taken on B200 boxes): every key the contract names, and the
    numbers agree with each other -- the kernel cannot take longer than the step that contains it, value = pairs / step time,
    roofline.achieved = algorithmic bytes / kernel time, frac = achieved / peak, e2e differs from the device-timed value."""
    import glob
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02_bench_line*.json")))
    # (a file is the captured stdout of the run: the JSON line is its last line that starts with a brace)
    lines = [json.loads([l for l in open(p).read().splitlines() if l.startswith("{")][-1]) for p in paths]
    product = [(p, d) for p, d in zip(paths, lines) if d.get("impl", "b200") != "reference"]
    assert len(product) >= 3
    for p, d in product:
        missing = (REQUIRED - {"impl", "cpu_baseline"}) | {"roofline", "clocks", "gpu_launches"}    # (cpu_baseline: N = 1 only)
        assert missing <= set(d), (p, missing - set(d))
        assert d["metric"] == "warped frame-pairs/sec" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
        assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"].startswith(("f32", "bf16")) and "workload" in d["config"]
        assert d["gpu_launches"] > 0 and d["warmup"] >= 3
        r, e, c = d["roofline"], d["e2e"], d["clocks"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert r["kernel_ms_per_launch"] <= d["ms_per_step"]
        assert abs(r["achieved"] - r["algorithmic_bytes_per_launch"] / r["kernel_ms_per_launch"] / 1e6) <= 1e-6 * r["achieved"]
        pairs = d["config"]["pairs_per_gpu_per_step"] * d["n_gpus"]
        assert abs(d["value"] - pairs / d["ms_per_step"] * 1e3) <= 1e-6 * d["value"]
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e) and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
        assert e["value"] < d["value"]
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c) and not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"]))
        if d["n_gpus"] == 1:
            cb = d["cpu_baseline"]
            assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] in ("port", "reference") and cb["value"] > 0
