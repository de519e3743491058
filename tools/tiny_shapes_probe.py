#!/usr/bin/env python
"""Kernel times of tiny_imagenet's diffusion layer at plane shapes the tiled kernels serve (tiny_tiled.cu), next to
the whole-plane ring kernels at their own shapes, one JSON line per configuration.

    python tools/tiny_shapes_probe.py [--reps 20] [--out profiles/tiny_shapes_probe.jsonl]

Each pass is timed through the C ABI with CUDA events: three warm-up calls, then --reps timed windows of five
calls each, median per call.  The batch is chosen so that one input tensor is larger than twice the 126 MB L2.
Algorithmic bytes: forward 8 B per cell (read u, write out), backward 12 B per cell (read u and gout, write
grad_input), halved for bf16 I/O.  The share of peak is against the measured HBM copy rate DESIGN section 4.4 uses
(6551 GB/s on one B200).  The card name and power limit are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
from ctypes import byref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 1024 * 1024
HBM_COPY_GBS = 6551.0

# (label, C, H, W, steps, io): "ring" / "tiled" is the kernel family the dispatch picks for (forward, backward)
CASES = [
    ("yardstick 3x64^2 K=1", 3, 64, 64, 1, "fp32"),
    ("3x224^2 K=1", 3, 224, 224, 1, "fp32"),
    ("3x224^2 K=1", 3, 224, 224, 1, "bf16"),
    ("3x227^2 K=1", 3, 227, 227, 1, "fp32"),
    ("3x227^2 K=1", 3, 227, 227, 1, "bf16"),
    ("3x299^2 K=1", 3, 299, 299, 1, "fp32"),
    ("3x299^2 K=1", 3, 299, 299, 1, "bf16"),
    ("3x512^2 K=1", 3, 512, 512, 1, "fp32"),
    ("1x2048^2 K=1", 1, 2048, 2048, 1, "fp32"),
    ("3x64^2 K=11 (ring)", 3, 64, 64, 11, "fp32"),
    ("3x64^2 K=12 (tiled)", 3, 64, 64, 12, "fp32"),
    ("3x240^2 K=1 (ring forward, one stage)", 3, 240, 240, 1, "fp32"),
    ("3x241^2 K=1 (tiled)", 3, 241, 241, 1, "fp32"),
]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:   # noqa: BLE001 -- the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def time_case(P, C, H, W, steps, io, reps):
    import torch
    L = P._cabi.lib()
    dt = torch.bfloat16 if io == "bf16" else torch.float32
    es = 2 if io == "bf16" else 4
    B = max(1, -(-2 * L2_BYTES // (C * H * W * es)))
    d = P._cabi.TinyDesc(B, C, H, W, steps, 0.01, 1e-6, 0.15, 0.1)
    nws = L.pde_tiny_backward_workspace_bytes(byref(d))
    if nws == 0:
        raise RuntimeError(f"unsupported configuration {C}x{H}x{W} K={steps}")
    gen = torch.Generator(device="cuda").manual_seed(1)
    u = torch.randn(B, C, H, W, device="cuda", generator=gen).to(dt)
    g = torch.randn(B, C, H, W, device="cuda", generator=gen).to(dt)
    out, gin = torch.empty_like(u), torch.empty_like(u)
    al, sc = torch.full((C,), 0.05, device="cuda"), torch.ones(C, device="cuda")
    ga, gs = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    fwd = L.pde_tiny_forward_bf16 if io == "bf16" else L.pde_tiny_forward
    bwd = L.pde_tiny_backward_bf16 if io == "bf16" else L.pde_tiny_backward

    def f():
        P._cabi.check(fwd(byref(d), u.data_ptr(), al.data_ptr(), sc.data_ptr(), out.data_ptr(), st), "forward")

    def b():
        P._cabi.check(bwd(byref(d), u.data_ptr(), g.data_ptr(), al.data_ptr(), sc.data_ptr(), gin.data_ptr(),
                          ga.data_ptr(), gs.data_ptr(), ws.data_ptr(), ctypes.c_size_t(nws), st), "backward")

    res = {}
    for name, fn in (("fwd", f), ("bwd", b)):
        for _ in range(3):
            fn()
        times = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                fn()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) / 5)
        res[name] = sorted(times)[len(times) // 2]
    return B, res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tiny_shapes_probe.jsonl"))
    a = ap.parse_args()
    import torch
    import cnn_with_pde_b200 as P
    if not torch.cuda.is_available():
        raise SystemExit("tiny_shapes_probe needs a CUDA device")
    name, power = card()
    lines = []
    for label, C, H, W, steps, io in CASES:
        B, t = time_case(P, C, H, W, steps, io, a.reps)
        cells = B * C * H * W
        half = 0.5 if io == "bf16" else 1.0
        row = {"case": label, "io": io, "B": B, "C": C, "H": H, "W": W, "steps": steps, "gpu": name,
               "power_limit": power, "fwd_ms": round(t["fwd"], 4), "bwd_ms": round(t["bwd"], 4)}
        for k, bpc in (("fwd", 8.0), ("bwd", 12.0)):
            gbs = cells * bpc * half / (t[k] * 1e-3) / 1e9
            row[f"{k}_GBps"] = round(gbs, 1)
            row[f"{k}_of_hbm_copy_peak"] = round(gbs / HBM_COPY_GBS, 3)
        print(json.dumps(row), flush=True)
        lines.append(json.dumps(row))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
