"""Step time of the training loop under eager, --graph and --compile, and the eager path's bench numbers against
another tree (the parent commit), alternated in one process tree.  One JSON line per measurement.

    python tools/compile_probe.py --out profiles/compile_probe.jsonl [--parent DIR] [--bench-steps 20]

The GPU's name and power limit are read in the same run and written into every line.  With --parent, bench.py
runs from DIR and from this tree, alternating, twice each; `script_batch_latency_us` and `value` of the four runs
are recorded with their spreads.  Where the compiled step is slower than the CUDA-graph step, a torch.profiler run
of the compiled step records the CUDA time per step and the kernel count, the launch-bound part of the difference.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (q.stdout.strip().splitlines() or [","])[0].split(",")[:2]
    return {"gpu": name.strip(), "power_limit": power.strip()}


def _bench(tree, steps, warmup):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup)],
                       cwd=tree, capture_output=True, text=True, timeout=3000)
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode or not line:
        raise RuntimeError(f"bench.py in {tree} failed:\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}")
    res = json.loads(line[-1])
    return {"value": res.get("value"), "script_batch_latency_us": res.get("script_batch_latency_us")}


def _steps(emit, meta):
    import torch
    from cnn_with_pde_b200.train import run
    cases = (("cifar10", 512, None), ("tiny", 64, 224))
    for model, batch, size in cases:
        ms = {}
        for mode in ("eager", "graph", "compile"):
            out = run(model, batch, 30, 5, graph=mode == "graph", compile=mode == "compile", quiet=True, image_size=size)
            ms[mode] = out["ms_per_step"]
            emit(dict(meta, kind="train_step", model=model, batch=batch, image_size=size or None, mode=mode,
                      ms_per_step=round(out["ms_per_step"], 4), img_per_s=round(out["img_per_s"], 1)))
        if ms["compile"] > ms["graph"]:
            emit(dict(meta, kind="compile_profile", model=model, batch=batch, image_size=size or None,
                      **_profile(model, batch, size), graph_ms_per_step=round(ms["graph"], 4),
                      compile_ms_per_step=round(ms["compile"], 4)))
        torch._dynamo.reset()


def _profile(model, batch, size):
    """CUDA time and kernel launches per compiled step (torch.profiler, in a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from cnn_with_pde_b200.train import run
    steps = 10
    run(model, batch, 1, 3, compile=True, quiet=True, image_size=size)   # compile outside the trace
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(model, batch, steps, 0, compile=True, quiet=True, image_size=size)
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kern = [e for e in evs if "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]
    total_us = sum(e.device_time for e in kern)
    pde_us = sum(e.device_time for e in kern if "pde" in e.name.lower() or "adi" in e.name.lower()
                 or "tiny" in e.name.lower() or "emo" in e.name.lower())
    # the run includes one warm-up step (compiled already) besides the timed ones
    return {"cuda_kernel_ms_per_step": round(total_us / 1e3 / (steps + 1), 4),
            "kernels_per_step": round(len(kern) / (steps + 1), 1),
            "pde_kernel_ms_per_step": round(pde_us / 1e3 / (steps + 1), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--parent", default=None, help="tree of the commit to compare bench.py against")
    ap.add_argument("--bench-steps", type=int, default=20)
    ap.add_argument("--bench-warmup", type=int, default=5)
    a = ap.parse_args()
    meta = _gpu()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    f = open(a.out, "a")

    def emit(rec):
        print(json.dumps(rec), flush=True)
        f.write(json.dumps(rec) + "\n")
        f.flush()

    if a.parent:
        runs = {"parent": [], "branch": []}
        for _ in range(2):
            for tag, tree in (("parent", a.parent), ("branch", ROOT)):
                res = _bench(tree, a.bench_steps, a.bench_warmup)
                runs[tag].append(res)
                emit(dict(meta, kind="bench", tree=tag, **res))
        for tag, rs in runs.items():
            emit(dict(meta, kind="bench_spread", tree=tag,
                      **{k: [min(r[k] for r in rs), max(r[k] for r in rs)] for k in ("value", "script_batch_latency_us")}))
    _steps(emit, meta)


if __name__ == "__main__":
    main()
