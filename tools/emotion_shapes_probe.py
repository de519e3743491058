#!/usr/bin/env python
"""Kernel times of emotion_recognition.PDELayer on planes above 64 x 64 (emotion_halo.cu), next to the existing
48 x 48 kernels, one JSON line per configuration.

    python tools/emotion_shapes_probe.py [--reps 20] [--out profiles/emotion_shapes_probe.jsonl]

Each pass is timed through the C ABI with CUDA events: three warm-up calls, then --reps timed windows of five
calls each, median per call.  The batch is chosen so that one input tensor is about 1 GB, far past the 126 MB L2.
Rates: Gcell-updates/s = B N^2 Nt / time.  Algorithmic bytes: forward 8 B per cell (read u0, write out), backward
12 B per cell (read u0 and gout, write grad_input); the share of peak is against the measured HBM copy rate
DESIGN section 4.4 uses (6551 GB/s on one B200).  The bytes the backward moves through its workspace (replay
writes, and per reversed step one read of u^k and lambda^{k+1} and one write of lambda^k) are reported separately,
counted from the algorithm, not measured.  The card name and power limit are read in the same run.
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

INPUT_BYTES = 1 << 30
HBM_COPY_GBS = 6551.0
DT = 0.001
CASES = [("existing 48x48 kernels", 48, 10), ("halo", 96, 10), ("halo", 128, 10), ("halo", 224, 10),
         ("halo", 512, 10)]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:   # noqa: BLE001 -- the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def time_case(P, N, Nt, reps):
    import numpy as np
    import torch
    L = P._cabi.lib()
    B = max(1, INPUT_BYTES // (N * N * 4))
    f = lambda v: float(np.float32(v))
    d = P._cabi.EmoDesc(B, N, Nt, f(0.5 * DT), f(DT), f((1.0 / N) ** 2), f((1.0 / N) ** 2), 0)
    nws = L.pde_emotion_backward_workspace_bytes(byref(d))
    if nws == 0:
        raise RuntimeError(f"unsupported configuration N={N} Nt={Nt}")
    gen = torch.Generator(device="cuda").manual_seed(1)
    u = torch.randn(B, 1, N, N, device="cuda", generator=gen)
    g = torch.randn(B, 1, N, N, device="cuda", generator=gen)
    out, gin = torch.empty_like(u), torch.empty_like(u)
    # stable coefficients: a_i, b_j ~ 0.1
    w = torch.tensor([0.2, 0.02, 0.02, 0.1, 0.01, 0.01], device="cuda") / (DT * N * N)
    xs = torch.linspace(0, 1, N).cuda()
    gw = torch.empty(6, device="cuda")
    ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def fwd():
        P._cabi.check(L.pde_emotion_forward(byref(d), u.data_ptr(), w.data_ptr(), xs.data_ptr(), xs.data_ptr(),
                                            out.data_ptr(), st), "forward")

    def bwd():
        P._cabi.check(L.pde_emotion_backward(byref(d), u.data_ptr(), g.data_ptr(), w.data_ptr(), xs.data_ptr(),
                                             xs.data_ptr(), gin.data_ptr(), gw.data_ptr(), ws.data_ptr(),
                                             ctypes.c_size_t(nws), st), "backward")

    res = {}
    for name, fn in (("fwd", fwd), ("bwd", bwd)):
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
    torch.cuda.synchronize()
    if not (torch.isfinite(out).all() and torch.isfinite(gin).all() and torch.isfinite(gw).all()):
        raise RuntimeError(f"non-finite results at N={N}")
    return B, nws, res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "emotion_shapes_probe.jsonl"))
    a = ap.parse_args()
    import torch
    import cnn_with_pde_b200 as P
    if not torch.cuda.is_available():
        raise SystemExit("emotion_shapes_probe needs a CUDA device")
    name, power = card()
    lines = []
    for label, N, Nt in CASES:
        B, nws, t = time_case(P, N, Nt, a.reps)
        cells = B * N * N
        row = {"case": label, "B": B, "N": N, "Nt": Nt, "gpu": name, "power_limit": power,
               "fwd_ms": round(t["fwd"], 4), "bwd_ms": round(t["bwd"], 4), "workspace_bytes": nws}
        for k, bpc in (("fwd", 8.0), ("bwd", 12.0)):
            sec = t[k] * 1e-3
            row[f"{k}_Gcell_updates_per_s"] = round(cells * Nt / sec / 1e9, 1)
            gbs = cells * bpc / sec / 1e9
            row[f"{k}_GBps"] = round(gbs, 1)
            row[f"{k}_of_hbm_copy_peak"] = round(gbs / HBM_COPY_GBS, 3)
        if N > 64:   # replay: Nt - 1 writes; step Nt - 1: 2 planes, steps Nt - 2 ... 1: 3 planes, step 0: 1 plane
            ws_bytes = cells * 4 * 4 * (Nt - 1)
            row["bwd_workspace_GB_moved"] = round(ws_bytes / 1e9, 2)
            row["bwd_GBps_incl_workspace"] = round((cells * 12 + ws_bytes) / (t["bwd"] * 1e-3) / 1e9, 1)
        print(json.dumps(row), flush=True)
        lines.append(json.dumps(row))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
