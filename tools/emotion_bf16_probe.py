#!/usr/bin/env python
"""Kernel times of emotion_recognition.PDELayer with fp32 planes against bf16 planes (pde_emotion_*_bf16), one JSON
line per (configuration, dtype).

    python tools/emotion_bf16_probe.py [--reps 20] [--rounds 3] [--out profiles/emotion_bf16_probe.jsonl]

Each pass is timed through the C ABI with CUDA events: three warm-up calls, then --reps timed windows of five calls
each; the two dtypes alternate --rounds times within the run, and the median window over all rounds is reported.
The batch is the one tools/emotion_shapes_probe.py uses: one fp32 input tensor of about 1 GB, far past the 126 MB L2
(116,508 planes at 48 x 48).  Rates: Gcell-updates/s = B N^2 Nt / time.  Algorithmic bytes per cell: forward 8 (fp32:
read u0, write out) or 4 (bf16), backward 12 (read u0 and gout, write grad_input) or 6; the share of peak is against
the HBM copy rate DESIGN section 4.4 measured (6551 GB/s on one B200).  The card name and power limit are read in the
same run.
"""
import argparse
import ctypes
import json
import os
import sys
from ctypes import byref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from emotion_shapes_probe import DT, HBM_COPY_GBS, INPUT_BYTES, card  # noqa: E402

CASES = [(48, 10), (96, 10), (224, 10), (512, 10)]


def setup(P, N, Nt):
    import numpy as np
    import torch
    L = P._cabi.lib()
    B = max(1, INPUT_BYTES // (N * N * 4))
    f = lambda v: float(np.float32(v))   # noqa: E731
    d = P._cabi.EmoDesc(B, N, Nt, f(0.5 * DT), f(DT), f((1.0 / N) ** 2), f((1.0 / N) ** 2), 0)
    gen = torch.Generator(device="cuda").manual_seed(1)
    u32 = torch.randn(B, 1, N, N, device="cuda", generator=gen)
    g32 = torch.randn(B, 1, N, N, device="cuda", generator=gen)
    w = torch.tensor([0.2, 0.02, 0.02, 0.1, 0.01, 0.01], device="cuda") / (DT * N * N)   # stable: a_i, b_j ~ 0.1
    xs = torch.linspace(0, 1, N).cuda()
    gw = torch.empty(6, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    passes = {}
    for name, dtype, fwd, bwd, query in (
            ("fp32", torch.float32, L.pde_emotion_forward, L.pde_emotion_backward, L.pde_emotion_backward_workspace_bytes),
            ("bf16", torch.bfloat16, L.pde_emotion_forward_bf16, L.pde_emotion_backward_bf16,
             L.pde_emotion_backward_workspace_bytes_bf16)):
        u, g = u32.to(dtype), g32.to(dtype)
        out, gin = torch.empty_like(u), torch.empty_like(u)
        nws = query(byref(d))
        if nws == 0:
            raise RuntimeError(f"unsupported configuration N={N} Nt={Nt}")
        ws = torch.empty(nws, dtype=torch.uint8, device="cuda")

        def f_fwd(fwd=fwd, u=u, out=out):
            P._cabi.check(fwd(byref(d), u.data_ptr(), w.data_ptr(), xs.data_ptr(), xs.data_ptr(), out.data_ptr(), st),
                          "forward")

        def f_bwd(bwd=bwd, u=u, g=g, gin=gin, ws=ws, nws=nws):
            P._cabi.check(bwd(byref(d), u.data_ptr(), g.data_ptr(), w.data_ptr(), xs.data_ptr(), xs.data_ptr(),
                              gin.data_ptr(), gw.data_ptr(), ws.data_ptr(), ctypes.c_size_t(nws), st), "backward")

        passes[name] = {"fwd": f_fwd, "bwd": f_bwd, "nws": nws, "out": out, "gin": gin}
    return B, passes


def time_windows(fn, reps):
    import torch
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
    return times


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "emotion_bf16_probe.jsonl"))
    a = ap.parse_args()
    import torch
    import cnn_with_pde_b200 as P
    if not torch.cuda.is_available():
        raise SystemExit("emotion_bf16_probe needs a CUDA device")
    name, power = card()
    lines = []
    for N, Nt in CASES:
        B, passes = setup(P, N, Nt)
        times = {(dt, k): [] for dt in passes for k in ("fwd", "bwd")}
        for _ in range(a.rounds):   # fp32 and bf16 alternate
            for dt, p in passes.items():
                for k in ("fwd", "bwd"):
                    times[(dt, k)] += time_windows(p[k], a.reps)
        torch.cuda.synchronize()
        for dt, p in passes.items():
            if not (torch.isfinite(p["out"]).all() and torch.isfinite(p["gin"]).all()):
                raise RuntimeError(f"non-finite results at N={N} {dt}")
        cells = B * N * N
        for dt in passes:
            row = {"N": N, "Nt": Nt, "B": B, "dtype": dt, "gpu": name, "power_limit": power,
                   "workspace_bytes": passes[dt]["nws"]}
            for k, bpc in (("fwd", 8.0), ("bwd", 12.0)):
                bpc = bpc / 2 if dt == "bf16" else bpc
                t = sorted(times[(dt, k)])[len(times[(dt, k)]) // 2]
                sec = t * 1e-3
                gbs = cells * bpc / sec / 1e9
                row[f"{k}_ms"] = round(t, 4)
                row[f"{k}_bytes_per_cell"] = bpc
                row[f"{k}_Gcell_updates_per_s"] = round(cells * Nt / sec / 1e9, 1)
                row[f"{k}_GBps"] = round(gbs, 1)
                row[f"{k}_of_hbm_copy_peak"] = round(gbs / HBM_COPY_GBS, 3)
            print(json.dumps(row), flush=True)
            lines.append(json.dumps(row))
        del passes
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
