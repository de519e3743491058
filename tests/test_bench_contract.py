"""The reference arm of bench.py (`--impl reference`): runs without a GPU, prints ONE JSON line with the keys the
driver reads, times the CPU restatement (never the CUDA library), and under a multi-rank launch only rank 0
works and prints.  The product arm: no number without a GPU; on one, --steps and --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, *args):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(env_extra or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-seconds", "1", *args], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.strip()]


def test_reference_arm_prints_the_contract_line():
    lines = _run()
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "pde_layer_fwd_bwd_cell_updates_per_s" and d["unit"] == "Gcell-updates/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert "fashion" in d["config"]["workload"] and "bounded sample" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "oracle/pde_oracle.c" in cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0           # nothing of the CUDA library runs on this arm


def test_reference_arm_other_ranks_exit_quietly():
    lines = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29591"},
                 "--gpus", "2")
    assert lines == []


def test_dump_outputs_is_refused_on_the_reference_arm(tmp_path):
    """--dump-outputs writes the GPU path's outputs; asked of the CPU arm it fails instead of leaving DIR empty."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    assert not (tmp_path / "d").exists() and r.stdout.strip() == ""


@pytest.mark.gpu
def test_product_arm_times_the_asked_steps_and_dumps_the_last_one(tmp_path):
    """--steps K is the number of timed passes: the measured window grows with K.  --dump-outputs writes what the
    last one returned: float32, 64 MB at most (here a seeded sample of the batch rows), the same arrays whatever
    K, and the layer's output and gradients on the seeded batch, as the oracle computes them."""
    import bench
    from . import cases as K
    from . import runners
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    B = 20000
    pnames = ("alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff")
    names = ["out", "grad_input"] + ["grad_" + n for n in pnames]
    dumps, window_ms = [], []
    for k in (10, 40):
        d = tmp_path / f"steps{k}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(k), "--warmup", "1",
                            "--batch", str(B), "--cpu-seconds", "1", "--all-layers", "0", "--train", "0",
                            "--dump-outputs", str(d)], capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.lstrip().startswith("{")][-1])
        assert line["steps"] == k and line["config"]["inner_repeats"] == 1
        window_ms.append(line["ms_per_step"] * k)          # the CUDA-event time of the whole timed region
        assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in names)
        assert sum(os.path.getsize(d / (n + ".npy")) for n in names) <= 64_000_000
        arrays = {n: np.load(d / (n + ".npy")) for n in names}
        assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
        assert arrays["out"].shape == arrays["grad_input"].shape and 1000 < arrays["out"].shape[0] < B
        assert arrays["out"].shape[1:] == (1, 28, 28) and arrays["grad_alpha_base"].shape == (28, 28)
        dumps.append(arrays)
    assert 2.5 <= window_ms[1] / window_ms[0] <= 6.0, window_ms
    for n, a in dumps[0].items():
        b = dumps[1][n]
        assert np.linalg.norm(a - b) <= 1e-6 * np.linalg.norm(b), n
    # the values: the oracle on the batch the timed path ran on, at the rows that were kept
    c = K.case("bench_fashion", "fashion", B=B, perturb=False)
    u, g, _ = bench.timed_inputs(B, c.shape, "cuda")
    want = runners.run_oracle(c, params=K.make_params(c), io=(u.cpu().numpy(), g.cpu().numpy()), dtype=np.float32)
    rows = bench.dump_rows(B, dumps[0]["out"].shape[0])
    got = {"y": dumps[0]["out"], "gin": dumps[0]["grad_input"], **{"g_" + n: dumps[0]["grad_" + n] for n in pnames}}
    errs = runners.compare(got, {"y": want["y"][rows], "gin": want["gin"][rows], **{"g_" + n: want["g_" + n] for n in pnames}})
    assert len(errs) == 6 and max(errs.values()) <= 1e-5, errs


def test_product_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: without a device the timed arm must fail, not print a number."""
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0
    assert not any(ln.lstrip().startswith("{") for ln in r.stdout.splitlines()), r.stdout[-500:]
