"""bench.py's JSON contract, checked on the CPU: the reference arm (`--impl reference`, the restated CPU path) at a tiny
degree prints one line with every key the driver reads, and the product arm refuses to run without a CUDA device (there is
no CPU fallback to fall into silently)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_reference_arm_line_has_the_contract_keys():
    r = run("--impl", "reference", "--k", "10", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly ONE JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["unit"] == "s" and d["higher_is_better"] is False and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1000 * d["value"]) < 1e-6 * d["ms_per_step"] + 1e-9
    assert "wall-sec" in d["metric"] and d["config"]["workload"] and d["config"]["k"] == 10
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["unit"] == "s" and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["unit"] == "s" and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_product_arm_fails_loudly_without_a_gpu():
    try:
        import torch

        if torch.cuda.is_available():
            return  # on a GPU box the product arm runs; nothing to check here
    except Exception:
        pass
    r = run("--steps", "1", "--warmup", "0", "--k", "10", "--no-cpu-baseline")
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout) and not any(l.startswith("{") for l in r.stdout.splitlines())


def _bench_mod():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


class _Args:
    def __init__(self, k=0, shrink=0):
        self.k, self.shrink = k, shrink


def test_default_step_is_the_chunk_proof_of_configs_2():
    """BASELINE configs[2] (test-chunk-prove on the degree-26 SRS): inner k=20 + layer1 k=24 + layer2 k=25 in sequence;
    layer1 is the 28-column / 35-MSM replay, layer2 has the 11 MSMs of chunk.protocol and 12 coset NTTs; every unit of a
    layer lands on exactly one rank for 1/2/4/8 ranks."""
    b = _bench_mod()
    layers = b.layers_for(_Args())
    assert [(l.name, l.k) for l in layers] == [("inner", 20), ("layer1", 24), ("layer2", 25)]
    inner, l1, l2 = layers
    assert 300 <= inner.wit + inner.uni <= 1000  # "several hundred" columns (SURVEY.md §8(a) a5), stated in config
    j1 = b.make_jobs(l1)
    kinds = [j[0] for j in j1]
    assert kinds.count("lmsm") == 28 and kinds.count("ntt") == 28 and kinds.count("msm") == 7 and kinds.count("icoset") == 1
    msms = [j for j in j1 if j[0] in ("lmsm", "msm")]
    assert len(msms) == 35 and sum(1 for j in msms if j[1] == "w") == 19
    j2 = b.make_jobs(l2)
    k2 = [j[0] for j in j2]
    assert k2.count("lmsm") + k2.count("msm") == 11 and k2.count("ntt") == 5 and k2.count("ntt") + k2.count("coset") == 12
    assert k2.count("icoset") == 1
    c2 = b.op_counts(l2)
    assert c2["msm_w"] + c2["msm_u"] == 11 and c2["intt"] == 5 and c2["coset"] == 13
    w = b.workload_desc(_Args())
    assert "configs[2]" in w and "k=20" in w and "k=24" in w and "k=25" in w and "degree-26" in b.metric_name(_Args())
    assert "2^24" in b.workload_desc(_Args(k=24)) and "configs[1]" in b.workload_desc(_Args(k=24)) and "wall-sec" in b.metric_name(_Args(k=24))
    for layer in layers:
        jobs = b.make_jobs(layer)
        for world in (1, 2, 4, 8):
            plan = b.assign_jobs(jobs, world)  # per rank: the jobs themselves
            assert sorted(j for r in plan for j in r) == sorted(jobs)
            loads = [sum(j[2] for j in r) for r in plan]
            assert max(loads) <= 1.34 * max(sum(loads) / world, max(j[2] for j in jobs))


def test_reference_arm_of_the_chunk_step_is_built_from_full_size_samples_only():
    """--impl reference on the (shrunk) three-layer step: value = mean of the listed full-size samples, each the sum over
    layers of op time x op count; machine-readable `extrapolated_by_op_counts`; warm-up never feeds the value."""
    r = run("--impl", "reference", "--shrink", "14", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["extrapolated_by_op_counts"] is True and d["full_size_samples"] == len(d["sample_values_s"]) >= 1
    assert abs(d["value"] - sum(d["sample_values_s"]) / len(d["sample_values_s"])) < 1e-12
    det = d["cpu_baseline"]["detail"]
    assert set(det) == {"inner", "layer1", "layer2"} and [det[n]["k"] for n in ("inner", "layer1", "layer2")] == [6, 10, 11]
    total = 0.0
    for n in det:
        layer_s = sum(det[n]["op_counts"][o] * det[n]["op_s"][o] for o in det[n]["op_counts"])
        assert abs(layer_s - det[n]["layer_s"]) <= 0.02 * det[n]["layer_s"] + 1e-3  # op_s is rounded to 1 us
        total += det[n]["layer_s"]
    assert abs(total - d["sample_values_s"][-1]) < 1e-9
    assert "configs[2]" in d["config"]["workload"] and "shrunk" in d["metric"]


@pytest.mark.gpu
def test_dump_outputs_are_the_same_whatever_the_step_count(tmp_path):
    """--dump-outputs writes float arrays (64 MB at most) of the last timed step; the inputs are seeded, so 1 and 3 timed steps
    dump the same values, and --steps sets the number of timed steps (3 steps launch 3 times the kernels of 1)."""
    dumps, launches = [], []
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        r = run("--shrink", "8", "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--skip-e2e", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == steps
        launches.append(line["gpu_launches"])
        dumps.append({f.name: np.load(f) for f in sorted(d.iterdir())})
    a, b = dumps
    assert set(a) == {"inner_commitments.npy", "layer1_commitments.npy", "layer2_commitments.npy", "layer2_coefficients.npy",
                      "layer2_coefficient_rows.npy"}
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name, v in a.items():
        assert v.dtype in (np.float32, np.float64) and np.array_equal(v, b[name]), name
    assert a["inner_commitments.npy"].shape == (416 + 96 + 6 + 1, 2, 8) and a["layer2_commitments.npy"].any()
    assert a["layer2_coefficients.npy"].shape[0] == 5 and a["layer2_coefficients.npy"].any()
    assert launches[1] == 3 * launches[0] > 0
