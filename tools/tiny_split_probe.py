#!/usr/bin/env python
"""Kernel times of tiny_imagenet's dormant methods (pde_tiny_split) on planes beyond 64 x 64, where the
line-streaming kernels of tiny_split_tiled.cu serve them, next to tiny_split_kernel at 64 x 64; one JSON line per
configuration.

    python tools/tiny_split_probe.py [--reps 20] [--out profiles/tiny_split_probe.jsonl]

Each call is timed through the C ABI with CUDA events: three warm-up calls, then --reps timed windows of five calls
each, median per call.  The batch is chosen so that one input tensor is at least twice the 126 MB L2.  Algorithmic
bytes: 8 B per cell (read u, write out) for every mode; the share of peak is against the measured HBM copy rate
DESIGN section 4.4 uses (6551 GB/s on one B200).  The factorisation prologue is measured on one line of 4096
cells, once with bands whose pivots repeat after a few rows (the block copies the rest) and once with bands whose
pivots take thousands of rows to settle (r = 2e6: thread 0 computes that many rows serially); the row at which they
repeat is computed here in fp32 with the kernel's operations, and the difference over the difference in rows is the
serial cost of one row of the table.  The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
from ctypes import byref

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 1024 * 1024
HBM_COPY_GBS = 6551.0
METHODS = ("implicit_diffusion_step", "solve_implicit_x", "solve_implicit_y", "diffuse_x_explicit",
           "diffuse_y_explicit")
SHAPES = [(64, 64), (224, 224), (227, 227), (512, 512), (1000, 1003), (4096, 4096)]
COEFF_X, COEFF_Y, DT = 0.7, 1.9, 0.3


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:   # noqa: BLE001 -- the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def repeat_row(n, am, bmid, bend, eps):
    """The first middle row whose pivot repeats its predecessor's bit for bit (factorise_block), n if none does."""
    f = np.float32
    am, bmid, bend, eps = f(am), f(bmid), f(bend), f(eps)
    c, prev = f(am / bend), None
    for i in range(1, n - 1):
        d = f(bmid - f(am * c))
        d = eps if d < eps else d
        if i >= 2 and d == prev:
            return i
        prev, c = d, f(am / d)
    return n


def time_call(L, d, u, out, st, reps):
    import torch
    from cnn_with_pde_b200 import _cabi

    def call():
        _cabi.check(L.pde_tiny_split(byref(d), u.data_ptr(), out.data_ptr(), st), "pde_tiny_split")

    for _ in range(3):
        call()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            call()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / 5)
    return sorted(times)[len(times) // 2]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tiny_split_probe.jsonl"))
    a = ap.parse_args()
    import torch
    import cnn_with_pde_b200 as P
    import cnn_with_pde_b200.functional as F
    if not torch.cuda.is_available():
        raise SystemExit("tiny_split_probe needs a CUDA device")
    L = P._cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    name, power = card()
    lines = []

    def emit(row):
        row.update(gpu=name, power_limit=power)
        print(json.dumps(row), flush=True)
        lines.append(json.dumps(row))

    gen = torch.Generator(device="cuda").manual_seed(1)
    for H, W in SHAPES:
        B = max(1, -(-2 * L2_BYTES // (H * W * 4)))
        u = torch.randn(B, H, W, device="cuda", generator=gen)
        out = torch.empty_like(u)
        for mode, method in enumerate(METHODS):
            d = F._tiny_split_desc(mode, B, H, W, COEFF_X, COEFF_Y, DT, 1e-6)
            ms = time_call(L, d, u, out, st, a.reps)
            cells = B * H * W
            gbs = cells * 8.0 / (ms * 1e-3) / 1e9
            emit({"case": f"{method} {H}x{W}", "kernel": "tiny_split_kernel" if max(H, W) <= 64 else "tiled",
                  "mode": mode, "B": B, "H": H, "W": W, "ms": round(ms, 4), "GBps_at_8B_per_cell": round(gbs, 1),
                  "of_hbm_copy_peak": round(gbs / HBM_COPY_GBS, 3)})
        del u, out
    # the factorisation prologue at n = 4096: one line, so the time is prologue + one serial solve
    u = torch.randn(1, 1, 4096, device="cuda", generator=gen)
    out = torch.empty_like(u)
    for label, coeff, dt in (("pivots repeat early", COEFF_X, DT), ("pivots repeat late", 2.0e6, 1.0)):
        d = F._tiny_split_desc(1, 1, 1, 4096, coeff, 0.0, dt, 1e-6)
        ms = time_call(L, d, u, out, st, a.reps)
        emit({"case": f"prologue n=4096: solve_implicit_x 1x4096, {label}", "mode": 1, "B": 1, "H": 1, "W": 4096,
              "r": coeff * dt, "repeat_row": repeat_row(4096, d.cx[0], d.cx[1], d.cx[2], d.eps),
              "us": round(ms * 1e3, 2)})
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
