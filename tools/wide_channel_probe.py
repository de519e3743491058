#!/usr/bin/env python
"""Kernel times of the implicit layers with 5 ... 64 channels (adi_wide.cu), one JSON line per configuration.

    python tools/wide_channel_probe.py [--reps 5] [--out FILE]

Each configuration is timed through the C ABI with CUDA events (two warm-up calls, then --reps calls, median):
forward (pde_adi_forward_train without checkpoints) and backward (pde_adi_backward, replay included).  The batch
is chosen so that the input alone is larger than the 126 MB L2.  Reported beside each: the same layer with no
channel op (the difference is the time spent in the O(C^2) channel op and its gradient), and as a reference
point the same cells as C / 3 independent three-channel layers on the existing kernels (a three-channel layer at
C / 3 times the batch, scaled to the same cell count).  Gcell/s counts cell updates: cells x sweeps / time.
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


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:   # noqa: BLE001 -- the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def time_layer(P, cfg, B, reps):
    """(forward ms, backward ms, workspace bytes) of one layer call on a batch of B."""
    import torch
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    C, N = cfg.C, cfg.N
    d = cfg.desc(B, 0)
    sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
    nt, nws = L.pde_adi_tables_bytes(byref(d)), L.pde_adi_backward_workspace_bytes(byref(d))
    if nt == 0 or nws == 0:
        raise RuntimeError(f"unsupported configuration {cfg}")
    gen = torch.Generator(device="cuda").manual_seed(1)
    u = torch.randn(B, C, N, N, device="cuda", generator=gen)
    g = torch.randn(B, C, N, N, device="cuda", generator=gen)
    out, gin = torch.empty_like(u), torch.empty_like(u)
    maps = [1.0 + 0.3 * torch.rand(C, N, N, device="cuda", generator=gen) for _ in range(2)] + \
           [0.01 * torch.randn(C, N, N, device="cuda", generator=gen) for _ in range(2)]
    chan = (torch.eye(C, device="cuda") + 0.1 / C ** 0.5 * torch.randn(C, C, device="cuda", generator=gen)) if cfg.chan_op else None
    skw = torch.tensor(0.3, device="cuda") if cfg.skip else None
    tables = torch.empty(nt, dtype=torch.uint8, device="cuda")
    ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
    gm = [torch.empty(C, N, N, device="cuda") for _ in range(4)]
    gchan = torch.empty(C, C, device="cuda") if cfg.chan_op else None
    gskip = torch.empty((), device="cuda") if cfg.skip else None
    st = torch.cuda.current_stream().cuda_stream
    p = lambda t: None if t is None else t.data_ptr()   # noqa: E731
    P._cabi.check(L.pde_adi_prepare(byref(d), byref(sched), *[p(m) for m in maps], p(tables), st), "prepare")

    def fwd():
        P._cabi.check(L.pde_adi_forward_train(byref(d), p(tables), p(u), p(chan), p(skw), p(out), None, st), "forward")

    def bwd():
        P._cabi.check(L.pde_adi_backward(byref(d), p(tables), p(u), p(g), p(chan), p(skw), p(gin), *[p(t) for t in gm],
                                         p(gchan), p(gskip), p(ws), nws, st), "backward")

    res = []
    for fn in (fwd, bwd):
        for _ in range(2):
            fn()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        res.append(ts[len(ts) // 2])
    del u, g, out, gin, ws, tables
    torch.cuda.empty_cache()
    return res[0], res[1], nws


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import cnn_with_pde_b200 as P
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    name, power = card()
    cifar = dict(dt=0.001, hx=1.0, hy=1.0, has_max=True, chan_op=1)
    svhn = dict(dt=0.01, hx=1.0, hy=1.0, smooth=True, chan_op=2, skip=True)
    todo = [("cifar10", 32, C, 5, cifar) for C in (8, 16, 32, 48)] + [("svhn", 32, 16, 10, svhn)] + \
           [("cifar10", 16, 64, 5, cifar), ("cifar10", 64, 12, 5, cifar)]
    lines = []
    for kind, N, C, steps, kw in todo:
        cfg = P.AdiConfig(N=N, C=C, steps=steps, **kw)
        B = -(-2 * L2_BYTES // (C * N * N * 4))   # input ~ 2x L2
        S = steps * (2 if cfg.lie else 3)
        f, b, ws = time_layer(P, cfg, B, args.reps)
        f0, b0, _ = time_layer(P, P.AdiConfig(N=N, C=C, steps=steps, **{**kw, "chan_op": 0}), B, args.reps)
        B3 = -(-B * C // 3)
        f3, b3, _ = time_layer(P, P.AdiConfig(N=N, C=3, steps=steps, **kw), B3, args.reps)
        scale = (B * C) / (B3 * 3)
        upd = B * C * N * N * S
        rec = {
            "config": f"{kind} N={N} C={C} steps={steps}", "batch": B, "input_bytes": B * C * N * N * 4,
            "fwd_ms": round(f, 4), "bwd_ms": round(b, 4),
            "fwd_gcell_s": round(upd / f / 1e6, 2), "bwd_gcell_s": round(upd / b / 1e6, 2),
            "workspace_bytes": ws,
            "fwd_ms_no_chan_op": round(f0, 4), "bwd_ms_no_chan_op": round(b0, 4),
            "chan_op_share_fwd": round(1 - f0 / f, 3), "chan_op_share_bwd": round(1 - b0 / b, 3),
            "ref_3ch_fwd_ms": round(f3 * scale, 4), "ref_3ch_bwd_ms": round(b3 * scale, 4),
            "gpu": name, "power_limit": power,
        }
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
