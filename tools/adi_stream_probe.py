#!/usr/bin/env python
"""Times of the implicit layers on the streaming kernels (adi_stream.cu), one JSON line per configuration.

    python tools/adi_stream_probe.py [--windows 20] [--calls 5] [--out FILE]

Each configuration is timed through the C ABI with CUDA events: after two warm-up calls, --windows windows of
--calls calls each, the median window divided by --calls.  Forward is pde_adi_stream_forward; backward is
pde_adi_stream_backward (its own replay of the trajectory included).  The batch is chosen so that the input is at
least twice the 126 MB L2.  Context rows time the shared-memory kernels on the same descriptor (prepare +
forward_train, backward_saved).  Beside each row: tests/adi_reference.py in fp32 on the GPU on the same batch --
the reference's own algorithm vectorised over lines, differentiated by autograd -- timed over 3 single calls (it
issues several kernels per cell position, so it is slow; "oom" / "skipped" where it does not run).

Gcell/s counts cell updates (cells x sweeps / time).  Algorithmic bytes: forward 8 B a cell and sweep (read and
write the state once) plus the map reads of the factor tables (8 B a cell and sweep, shared by the batch);
backward 3 x the forward's bytes (forward, replay, adjoint).  Shares are of the 6551 GB/s HBM copy peak (DESIGN 4.4).
"""
import argparse
import json
import os
import subprocess
import sys
import time
from ctypes import byref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 1024 * 1024
HBM_PEAK = 6551e9

# (label, kind, C, N, steps, lie, smooth, chan_op, skip): the scripts' step counts (mnist / cifar10 10, svhn 10)
ROWS = [
    ("mnist 1x224^2", 1, 224, 10, False, False, 0, False),
    ("cifar10 3x224^2", 3, 224, 10, False, False, 1, False),
    ("svhn 3x227^2", 3, 227, 10, False, True, 2, True),
    ("mnist 1x512^2", 1, 512, 10, False, False, 0, False),
    ("cifar10 3x512^2", 3, 512, 10, False, False, 1, False),
    ("mnist 1x2048^2 1 step", 1, 2048, 1, False, False, 0, False),
    ("cifar10 3x4096^2 1 step", 3, 4096, 1, False, False, 1, False),
    ("cifar10 16x64^2 chan_op 1", 16, 64, 5, False, False, 1, False),
    ("cifar10 64x56^2 chan_op 1", 64, 56, 5, False, False, 1, False),
]
CONTEXT = [
    ("context mnist 1x128^2", 1, 128, 10, False, False, 0, False),
    ("context cifar10 3x64^2", 3, 64, 10, False, False, 1, False),
]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:   # noqa: BLE001 -- the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def timed(fn, windows, calls):
    import torch
    fn()
    fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(windows)]
    for a, b in ev:
        a.record()
        for _ in range(calls):
            fn()
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) / calls for a, b in ev)
    return ts[len(ts) // 2]


def inputs(cfg, B):
    import torch
    C, N = cfg.C, cfg.N
    gen = torch.Generator(device="cuda").manual_seed(1)
    u = torch.randn(B, C, N, N, device="cuda", generator=gen)
    g = torch.randn(B, C, N, N, device="cuda", generator=gen)
    maps = [1.0 + 0.3 * torch.rand(C, N, N, device="cuda", generator=gen) for _ in range(2)] + \
           [0.01 * torch.randn(C, N, N, device="cuda", generator=gen) for _ in range(2)]
    chan = (torch.eye(C, device="cuda") + 0.1 / C ** 0.5 * torch.randn(C, C, device="cuda", generator=gen)) if cfg.chan_op else None
    skw = torch.full((1,), 0.3, device="cuda") if cfg.skip else None
    return u, g, maps, chan, skw


def p(t):
    return None if t is None else t.data_ptr()


def time_stream(P, cfg, B, windows, calls):
    import torch
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    C, N = cfg.C, cfg.N
    d = cfg.desc(B, 0)
    sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
    nf, nb = L.pde_adi_stream_forward_workspace_bytes(byref(d)), L.pde_adi_stream_backward_workspace_bytes(byref(d))
    u, g, maps, chan, skw = inputs(cfg, B)
    out, gin = torch.empty_like(u), torch.empty_like(u)
    wf, wb = torch.empty(nf, dtype=torch.uint8, device="cuda"), torch.empty(nb, dtype=torch.uint8, device="cuda")
    gm = [torch.empty(C, N, N, device="cuda") for _ in range(4)]
    gch = torch.empty(C, C, device="cuda") if cfg.chan_op else None
    gsk = torch.empty((), device="cuda") if cfg.skip else None
    st = torch.cuda.current_stream().cuda_stream
    mp = [m.data_ptr() for m in maps]
    fwd = lambda: P._cabi.check(L.pde_adi_stream_forward(byref(d), byref(sched), *mp, p(u), p(chan), p(skw), p(out), p(wf),   # noqa: E731
                                                         nf, st), "stream forward")
    bwd = lambda: P._cabi.check(L.pde_adi_stream_backward(byref(d), byref(sched), *mp, p(u), p(g), p(chan), p(skw), p(gin),   # noqa: E731
                                                          *[p(x) for x in gm], p(gch), p(gsk), p(wb), nb, st), "stream backward")
    return timed(fwd, windows, calls), timed(bwd, windows, calls), nf, nb


def time_tables(P, cfg, B, windows, calls):
    import torch
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    C, N = cfg.C, cfg.N
    d = cfg.desc(B, 0)
    sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
    nt, nck = L.pde_adi_tables_bytes(byref(d)), L.pde_adi_checkpoint_bytes(byref(d))
    nws = L.pde_adi_backward_saved_workspace_bytes(byref(d)) if nck else L.pde_adi_backward_workspace_bytes(byref(d))
    u, g, maps, chan, skw = inputs(cfg, B)
    out, gin = torch.empty_like(u), torch.empty_like(u)
    tables, ws = torch.empty(nt, dtype=torch.uint8, device="cuda"), torch.empty(nws, dtype=torch.uint8, device="cuda")
    ck = torch.empty(nck, dtype=torch.uint8, device="cuda") if nck else None
    gm = [torch.empty(C, N, N, device="cuda") for _ in range(4)]
    gch = torch.empty(C, C, device="cuda") if cfg.chan_op else None
    gsk = torch.empty((), device="cuda") if cfg.skip else None
    st = torch.cuda.current_stream().cuda_stream
    mp = [m.data_ptr() for m in maps]

    def fwd():
        P._cabi.check(L.pde_adi_prepare(byref(d), byref(sched), *mp, p(tables), st), "prepare")
        P._cabi.check(L.pde_adi_forward_train(byref(d), p(tables), p(u), p(chan), p(skw), p(out), p(ck), st), "forward")

    bwd = lambda: P._cabi.check(L.pde_adi_backward_saved(byref(d), p(tables), p(u), p(g), p(chan), p(skw), p(ck), p(gin),   # noqa: E731
                                                         *[p(x) for x in gm], p(gch), p(gsk), p(ws), nws, st), "backward")
    return timed(fwd, windows, calls), timed(bwd, windows, calls), nt + nws + nck


def time_reference(cfg, B):
    """tests/adi_reference.py in fp32 on the GPU: (forward ms, backward ms), median of 3 single calls."""
    import torch
    from tests import adi_reference as AR
    u, g, maps, chan, skw = inputs(cfg, B)
    maps = [m.requires_grad_(True) for m in maps]
    spec = type("Spec", (), dict(steps=cfg.steps, lie=cfg.lie, dt=cfg.dt, hx=cfg.hx, hy=cfg.hy, cmin=cfg.cmin, cmax=cfg.cmax,
                                 has_max=cfg.has_max, smooth=cfg.smooth, eps=cfg.eps, chan_op=cfg.chan_op, skip=cfg.skip))
    sk = skw.reshape(()) if skw is not None else None
    fw, bw = [], []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        y = AR.forward(spec, u, *maps, chan, sk)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        torch.autograd.grad(y, maps, grad_outputs=g)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        fw.append((t1 - t0) * 1e3)
        bw.append((t2 - t1) * 1e3)
        del y
    return sorted(fw)[1], sorted(bw)[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=20)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    import cnn_with_pde_b200 as P
    name, power = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with (open(args.out, "w") if args.out else open(os.devnull, "w")) as f:
        for label, C, N, steps, lie, smooth, chan_op, skip in ROWS + CONTEXT:
            cfg = P.AdiConfig(N=N, C=C, steps=steps, dt=0.01, hx=1.0, hy=1.0, lie=lie, smooth=smooth, chan_op=chan_op,
                              skip=skip)
            B = max(1, -(-2 * L2_BYTES // (C * N * N * 4)))
            S = steps * (2 if lie else 3)
            cells = B * C * N * N
            fwd_ms, bwd_ms, nf, nb = time_stream(P, cfg, B, args.windows, args.calls)
            fwd_bytes = 8.0 * cells * S + 8.0 * C * N * N * S
            row = {"config": label, "batch": B, "input_bytes": cells * 4, "sweeps": S,
                   "fwd_ms": round(fwd_ms, 4), "bwd_ms": round(bwd_ms, 4),
                   "fwd_gcell_s": round(cells * S / fwd_ms / 1e6, 2), "bwd_gcell_s": round(cells * S / bwd_ms / 1e6, 2),
                   "fwd_alg_gb_s": round(fwd_bytes / fwd_ms / 1e6, 1), "bwd_alg_gb_s": round(3 * fwd_bytes / bwd_ms / 1e6, 1),
                   "fwd_hbm_share": round(fwd_bytes / fwd_ms / 1e-3 / HBM_PEAK, 3),
                   "bwd_hbm_share": round(3 * fwd_bytes / bwd_ms / 1e-3 / HBM_PEAK, 3),
                   "fwd_workspace_bytes": nf, "bwd_workspace_bytes": nb}
            if label.startswith("context"):
                tf, tb, tbytes = time_tables(P, cfg, B, args.windows, args.calls)
                row.update({"tables_fwd_ms": round(tf, 4), "tables_bwd_ms": round(tb, 4), "tables_buffer_bytes": tbytes})
            try:
                rf, rb = time_reference(cfg, B)
                row.update({"torch_ref_fwd_ms": round(rf, 2), "torch_ref_bwd_ms": round(rb, 2),
                            "speedup_fwd": round(rf / fwd_ms, 1), "speedup_bwd": round(rb / bwd_ms, 1)})
            except torch.cuda.OutOfMemoryError:
                row.update({"torch_ref_fwd_ms": "oom", "torch_ref_bwd_ms": "oom"})
            torch.cuda.empty_cache()
            row.update({"gpu": name, "power_limit": power})
            print(json.dumps(row), flush=True)
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
