#!/usr/bin/env python
"""bench.py -- PDE-layer forward+backward throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--layer NAME] [--dump-outputs DIR]

One "step" = one forward + backward pass of the PDE layer over one batch of synthetic input
(u, g_out ~ N(0,1), seeded).  Headline workload: fashion_mnist.DiffusionLayer (BASELINE.json
configs[1]: 1x28x28, dt=0.3, 4 Strang steps) at a batch whose tensors exceed the L2 (126 MB),
because at the script's batch of 256 the whole tensor (0.8 MB) sits in L2 and a call is launch
latency; the config-batch latency is reported beside it.  Unit: cell-updates = B*C*H*W*num_steps
per step.  Under torchrun every rank runs its own batch (weak scaling; the only exchange is the
all-reduce of the coefficient gradients) and rank 0 prints ONE JSON line.

The timed region is the K steps back to back inside one CUDA-event bracket (--inner N makes every
step N passes; ms_per_step is the time of ONE pass).  At the headline batch a pass takes ~3.5 ms on a
B200 (1000 W limit), so a window of about a second, with enough NVML clock samples for `clocks` and
`issue_frac`, takes K ~ 300; with fewer samples `issue_frac` uses the maximum SM clock.
--dump-outputs DIR writes what the last timed step handed its caller -- the layer output, grad_input
and the coefficient gradients -- as DIR/<name>.npy (float32; a fixed, seeded sample of the batch where the full arrays would exceed
64 MB), so that two builds can be compared output for output on identical inputs.
Beside the default-init weights the same batch is timed with perturbed
weights that put cells outside both clamp edges (`clamped`: the masked / in-sweep smoothing-adjoint
path), and at N = 1 the CPU leg doubles as a parity self-check: the oracle runs on the very batch the
GPU was timed on and `parity_rel_err` holds the worst relative error per output.

--impl reference times the CPU restatement (oracle/, C + OpenMP on all host cores; the
reference itself is pure Python and does not travel to the GPU box) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "pde_layer_fwd_bwd_cell_updates_per_s"
UNIT = "Gcell-updates/s"

# layer -> (kind, ctor kwargs, roofline-size batch (one fp32 tensor ~0.8-1 GB), script batch)
LAYERS = {
    "fashion": ("fashion", dict(), 262144, 256),
    "mnist": ("mnist", dict(), 262144, 64),
    "cifar10_pde1": ("cifar10", dict(size=32, channels=3, dt=0.001, num_steps=5, dx=1.0, dy=1.0), 65536, 512),
    "cifar10_pde2": ("cifar10", dict(size=32, channels=3, dt=0.002, num_steps=8, dx=2.0, dy=2.0), 65536, 512),
    "cifar2_diffusion1": ("cifar2", dict(size=32, channels=3, dt=0.001, num_steps=8), 65536, 512),
    "svhn": ("svhn", dict(size=32, channels=3), 65536, 256),
    "emotion": ("emotion", dict(Nx=48, Ny=48), 98304, 64),
    "tiny": ("tiny", dict(size=64, channels=3, num_steps=1, use_implicit=False), 16384, 32),
    # plane sizes no script uses: the run-time-sized kernels (csrc/adi_generic.cu) -- reported under other_layers
    "mnist_48x48": ("mnist", dict(size=48), 32768, 64),
    "svhn_64x64": ("svhn", dict(size=64, channels=3), 4096, 256),
}


def _steps_of(kind, ctor):
    if kind == "emotion":
        return int(ctor.get("T", 0.01) / ctor.get("dt", 0.001))
    dflt = {"fashion": 4, "tiny": 1}.get(kind, 10)
    return ctor.get("num_steps", dflt)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _csrc_sha():
    """Hash of the kernel sources: ties the ncu-derived counters to the build being timed."""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(ROOT, "cnn-with-pde_b200", "csrc")
    for f in sorted(os.listdir(d)):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(f.encode())
            h.update(fh.read())
    return h.hexdigest()[:12]


def _profile_counters(layer):
    """Per-launch ncu counters of the layer's backward / forward kernels at the bench batch
    (profiles/kernel_counters.json, written by tools/ncu_counters.py from the round's `ncu --set full`
    capture): dram bytes and executed warp instructions.  `csrc_sha` says which sources they were
    captured from."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_counters.json")) as f:
            allc = json.load(f)
        c = dict(allc.get(layer) or {})
        c["csrc_sha"] = allc.get("_csrc_sha")
        return c
    except Exception:
        return {}


def _bind_to_gpu_numa(index):
    """Restrict this process to the CPUs NVML reports as local to GPU `index` (first-touch policy then
    places the pinned staging buffer on that NUMA node).  Best effort: returns what was done."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = [i for i in range(n) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [i for i in cpus if i in allowed]
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            return f"bound to {len(cpus)} of {len(allowed)} CPUs local to GPU {index}"
        return "no narrower CPU set reported for this GPU"
    except Exception as ex:   # NVML or affinity not available: keep going unbound
        return f"unbound ({type(ex).__name__})"


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, index=0, period=0.02):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.armed = False   # samples count only once the timed region has started (begin())
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None
            return self
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def _run(self):
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                if self.armed:
                    self.samples.append(mhz)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def begin(self):
        self.armed = True
        return self

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1.0)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


DUMP_BYTES = 64_000_000


def timed_inputs(B, shape, dev, rank=0):
    """The seeded batch of the timed path: input u and upstream gradient g, the same on every run with the same
    arguments, and the generator they came from (the script-batch section keeps drawing from it)."""
    import torch
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    u = torch.randn(B, *shape, device=dev, generator=gen)
    g = torch.randn(B, *shape, device=dev, generator=gen)
    return u, g, gen


def dump_rows(B, keep):
    """The batch rows --dump-outputs keeps when it cannot keep all B: a fixed, seeded sample, in batch order."""
    import numpy as np
    return np.sort(np.random.default_rng(0).choice(B, size=keep, replace=False))


def dump_outputs(out_dir, y, grad_input, layer):
    """Write the arrays one forward + backward hands its caller as out_dir/<name>.npy (float32):
    `out`, `grad_input` and `grad_<parameter>`.  The coefficient gradients are written whole; `out` and
    `grad_input` keep a fixed, seeded sample of the batch (same rows in both, in batch order) when the
    full arrays would take more than DUMP_BYTES in all."""
    import numpy as np
    import torch
    grads = {"grad_" + n: p.grad for n, p in layer.named_parameters() if p.grad is not None}
    batched = {"out": y, "grad_input": grad_input}
    batched = {k: v for k, v in batched.items() if v is not None}
    B = y.shape[0]
    row_bytes = sum(v[0].numel() * 4 for v in batched.values())
    room = DUMP_BYTES - sum(g.numel() * 4 + 1024 for g in grads.values()) - 1024 * len(batched)   # + .npy headers
    keep = min(B, max(1, room // row_bytes))
    if keep < B:
        idx = torch.from_numpy(dump_rows(B, keep)).to(y.device)
        batched = {k: v.detach().index_select(0, idx) for k, v in batched.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in {**batched, **grads}.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------ b200
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from tests import cases as K
    from tests import runners
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.parallel import allreduce_coefficient_grads

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    kind, ctor, big_b, script_b = LAYERS[args.layer]
    B = args.batch or big_b
    c = K.case("bench_" + args.layer, kind, B=B, perturb=False, **ctor)
    C, H, W = c.shape
    nsteps = _steps_of(kind, ctor)
    cells = B * C * H * W
    layer = runners.make_cuda_layer(c, device=dev)
    params = [p for p in layer.parameters()]
    nparam = sum(p.numel() for p in params if p.requires_grad)
    # same layer, weights perturbed so that cells sit outside both clamp edges (tests/cases.make_params)
    c_pert = K.case("bench_clamped_" + args.layer, kind, B=B, perturb=True, **ctor)
    layer_c = runners.make_cuda_layer(c_pert, device=dev)
    u, g, gen = timed_inputs(B, (C, H, W), dev, rank)
    info = P._cabi.device_info()

    def grads():
        return [p.grad for p in params if p.grad is not None]

    def step(x):
        for p in params:
            p.grad = None
        x.grad = None      # as a training loop's zero_grad(set_to_none=True): grad_input is handed over, not
        y = layer(x)       # added to last step's by a separate torch kernel (2.5 GB of traffic at this batch)
        y.backward(g)
        if world > 1:
            allreduce_coefficient_grads(params)   # the path's only exchange: one flat NCCL all-reduce
        return y

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- kernel-only (HBM-resident)
    x = u.clone().requires_grad_(True)
    # NVML is initialised and polling before the warm-up (its first calls take the driver's locks for
    # milliseconds); samples count from begin() on
    sampler = ClockSampler(index=local).start() if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step(x)
    inner = args.inner
    sync_all()
    # one more untimed pass: the host enqueues the first timed one while the device runs it, so the bracket
    # opens on a busy device instead of timing the host's way to the first launch
    step(x)
    if sampler:
        sampler.begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps * inner - 1):
        step(x)
    y_last = step(x)
    e1.record()
    sync_all()
    clocks = sampler.stop() if sampler else None
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / (args.steps * inner)
    value = world * cells * nsteps / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y_last, x.grad, layer)
    del y_last

    # ----------------------------------------- per-kernel timing through the C ABI (roofline)
    def time_phase(fn, n):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    n_k = max(20, min(args.steps * inner, 100))
    with torch.no_grad():
        fwd_eval_ms = time_phase(lambda: layer(u), n_k)      # inference forward (no checkpoints)
    fwd_ms = time_phase(lambda: layer(x), n_k)               # training forward: also writes the step checkpoints
    y = layer(x)
    bwd_ms = time_phase(lambda: torch.autograd.grad(y, [x] + [p for p in params if p.requires_grad], g,
                                                    retain_graph=True, allow_unused=True), n_k)
    xn = u.clone()  # no grad_input: what real training needs (the layer is the first op)
    yn = layer(xn)
    bwd_nogin_ms = time_phase(lambda: torch.autograd.grad(yn, [p for p in params if p.requires_grad], g,
                                                          retain_graph=True, allow_unused=True), n_k)
    # the clamped-cell variant of the same batch (masks read, smoothing adjoint inside every sweep)
    pc = [p for p in layer_c.parameters() if p.requires_grad]
    fwd_c_ms = time_phase(lambda: layer_c(x), n_k)
    yc = layer_c(x)
    bwd_c_ms = time_phase(lambda: torch.autograd.grad(yc, [x] + pc, g, retain_graph=True, allow_unused=True), n_k)
    del yc
    peak, peak_src = _peaks()
    bwd_bytes = 12 * cells + 4 * nparam       # read u, read g_out, write g_in, write coefficient grads
    fwd_bytes = 8 * cells + 4 * nparam        # read u, write out, read coefficient maps
    bwd_gbs = bwd_bytes / (bwd_ms * 1e-3) / 1e9
    fwd_gbs = fwd_bytes / (fwd_ms * 1e-3) / 1e9

    # ---------------------------------------------------------------- end to end (host buffers)
    # Per step: H2D of the step's input batch from pinned memory (chunked, copy stream overlaps
    # compute), forward + backward through the nn.Module, D2H of the coefficient gradients.
    # g_out stays on the device: in training it is produced there by the classifier's backward.
    nchunk = 8 if B >= 8 * 1024 else 1
    cb = (B + nchunk - 1) // nchunk
    # the staging buffer is first touched by this process: bind it to the CPUs next to this rank's GPU so
    # that with several ranks the pinned pages do not all land on NUMA node 0
    numa = _bind_to_gpu_numa(local) if world > 1 else None
    host_u = torch.empty((B, C, H, W), dtype=torch.float32).pin_memory()
    host_u.copy_(u)
    host_g = torch.empty(nparam, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    dev_bufs = [torch.empty((cb, C, H, W), device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def e2e_step():
        for p in params:
            p.grad = None
        main = torch.cuda.current_stream()
        for i in range(nchunk):
            lo, hi = i * cb, min(B, (i + 1) * cb)
            buf = dev_bufs[i % 2][: hi - lo]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % 2])
                buf.copy_(host_u[lo:hi], non_blocking=True)
                ready[i % 2].record(copy_stream)
            main.wait_event(ready[i % 2])
            yy = layer(buf)
            yy.backward(g[lo:hi])
            freed[i % 2].record(main)
        if world > 1:
            allreduce_coefficient_grads(params)
        flat = torch.cat([t.reshape(-1) for t in grads()])
        host_g.copy_(flat, non_blocking=True)

    for ev in freed:
        ev.record(torch.cuda.current_stream())
    for _ in range(2):
        e2e_step()
    sync_all()
    k_e2e = max(3, min(args.steps, 10))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(k_e2e):
        e2e_step()
    b.record()
    sync_all()
    t = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item()) / k_e2e
    e2e_value = world * cells * nsteps / (e2e_ms * 1e-3) / 1e9

    # ------------------------------- N > 1: sharded gradients + all-reduce against one GPU, on hardware
    # Every rank runs its shard and the coefficient gradients are all-reduced; rank 0 then runs the
    # concatenated global batch alone.  The two must agree to fp32 reduction-order noise.
    dp_parity = None
    if world > 1:
        bc = min(B, 4096)
        uc, gc = u[:bc].contiguous(), g[:bc].contiguous()
        for p in params:
            p.grad = None
        layer(uc.clone().requires_grad_(True)).backward(gc)
        allreduce_coefficient_grads(params)
        sharded = [p.grad.clone() for p in params if p.grad is not None]
        U = [torch.empty_like(uc) for _ in range(world)]
        G = [torch.empty_like(gc) for _ in range(world)]
        dist.all_gather(U, uc)
        dist.all_gather(G, gc)
        if rank == 0:
            for p in params:
                p.grad = None
            layer(torch.cat(U).requires_grad_(True)).backward(torch.cat(G))
            single = [p.grad for p in params if p.grad is not None]
            errs = [max(runners.rel_l2(a.cpu().numpy(), b.cpu().numpy()), runners.rel_max(a.cpu().numpy(), b.cpu().numpy()))
                    for a, b in zip(sharded, single)]
            dp_parity = {"worst": float(f"{max(errs):.3e}"), "global_batch": bc * world, "ranks": world, "tolerance": 1e-5,
                         "what": "all-reduced coefficient gradients of the sharded batch vs a single-GPU run of the same global batch"}
        del U, G

    # ------------------------------------------------------- latency at the script's own batch
    cs = K.case("bench_small", kind, B=script_b, perturb=False, **ctor)
    us = torch.randn(script_b, C, H, W, device=dev, generator=gen)
    gs = torch.randn(script_b, C, H, W, device=dev, generator=gen)
    xs = us.clone().requires_grad_(True)

    def small():
        for p in params:
            p.grad = None
        xs.grad = None
        layer(xs).backward(gs)

    torch.cuda.synchronize()
    torch.cuda.empty_cache()   # the big-batch buffers of the sections above go back to the driver first
    for _ in range(5):
        small()
    small_ms = time_phase(small, 200)
    # ------------------------------------------- whole-model training step (BASELINE metric, part ii)
    # cifar10.CIFAR10PDENoConv (BASELINE configs[2]: 3x32x32, batch 512 per GPU), three PDE layers +
    # the reference's dense head, AdamW recipe of cifar10.py:400-527, synthetic device-resident data,
    # one flat NCCL all-reduce of the gradients per step, step captured in CUDA graphs.
    train = None
    if args.train:
        from cnn_with_pde_b200 import train as T
        del x, y, yn, xn
        torch.cuda.empty_cache()
        try:
            kw = dict(steps=max(args.steps, 100), warmup=max(args.warmup, 10), graph=True, quiet=True)
            train = T.run(args.train_model, args.train_batch, **kw)
            if world == 1 and args.train_model == "cifar10":
                # the same step with the three PDE layers fused into one launch per pass (opt-in, see
                # classifiers.MultiScaleExtractor), then the default once more: the first run of a process also
                # pays for library initialisation effects, so the default is reported as the better of its two runs
                import cnn_with_pde_b200.classifiers as Cl
                Cl.MultiScaleExtractor.fused_branches = True
                try:
                    fused = T.run(args.train_model, args.train_batch, **kw)
                finally:
                    Cl.MultiScaleExtractor.fused_branches = False
                again = T.run(args.train_model, args.train_batch, **kw)
                first_ms = train["ms_per_step"]
                if again["ms_per_step"] < train["ms_per_step"]:
                    train = again
                train["runs_ms_per_step"] = {"default_first": first_ms, "fused_branches": fused["ms_per_step"],
                                             "default_again": again["ms_per_step"]}
                train["fused_branches"] = {"ms_per_step": fused["ms_per_step"], "img_per_s": fused["img_per_s"]}
        except Exception as ex:   # the headline line survives a failure of the side measurement
            train = {"error": f"{type(ex).__name__}: {ex}"}
        x = u.clone().requires_grad_(True)
        y = yn = xn = None

    # the same call replayed from a CUDA graph (how the launcher trains): the kernels without the host side
    small_graph_ms, small_graph_err = None, None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                small()
            side.synchronize()
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg, stream=side, capture_error_mode="thread_local"):
                small()
        torch.cuda.current_stream().wait_stream(side)
        small_graph_ms = time_phase(cg.replay, 200)
        del cg
    except Exception as ex:
        small_graph_err = f"{type(ex).__name__}: {ex}"


    out = None
    if rank == 0:
        # the CPU leg runs on rank 0 at N = 1 only (the other ranks would idle at the barrier)
        cpu, parity, parity_c = None, None, None
        if world == 1:
            x = y = yn = xn = None
            torch.cuda.empty_cache()
            cpu, parity = cpu_baseline_and_parity(args.layer, c, layer, u, g, args.cpu_seconds)
            _, parity_c = cpu_baseline_and_parity(args.layer, c_pert, layer_c, u, g, args.cpu_seconds)
        if train is not None and "error" not in train and world == 1:
            try:
                train["cpu_baseline"] = cpu_train_baseline(args.train_model)
            except Exception as ex:
                train["cpu_baseline"] = {"error": f"{type(ex).__name__}: {ex}"}
        others = {}
        if args.all_layers and world == 1:
            x = y = yn = xn = host_u = dev_bufs = None
            torch.cuda.empty_cache()
            for name in LAYERS:
                if name != args.layer:
                    try:
                        others[name] = _quick_layer(name, dev, peak)
                    except Exception as ex:  # keep the headline line even if a side measurement fails
                        others[name] = {"error": f"{type(ex).__name__}: {ex}"}
        ctr = _profile_counters(args.layer)
        sm_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
        sweeps = nsteps * (3 if kind in ("fashion", "mnist", "svhn", "cifar10") else (2 if kind == "cifar2" else 1))

        def issue(inst, ms):
            """warp instructions / (SMs x 4 schedulers x f x t): share of the issue slots a launch used"""
            if not inst:
                return None
            return round(inst / (info["sm_count"] * 4 * sm_mhz * 1e6 * ms * 1e-3), 4)

        def per_cell_sweep(inst):
            return round(inst * 32 / (cells * sweeps), 2) if inst else None

        out = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "timed_region_s": round(ms_total * 1e-3, 3),
            "config": {
                "inner_repeats": inner,
                "timing": f"{args.steps} steps x {inner} back-to-back passes inside one CUDA-event bracket; ms_per_step = one pass",
                "workload": f"{args.layer} PDE layer forward+backward (grad_input + coefficient grads), "
                            f"{C}x{H}x{W}, num_steps={nsteps}, batch {B} per GPU "
                            f"(script batch {script_b} scaled so every tensor ({cells * 4 / 1e6:.0f} MB) exceeds L2)",
                "layer": args.layer, "batch_per_gpu": B, "shape": [C, H, W], "num_steps": nsteps,
                "l2": f"inputs {cells * 4 / 1e6:.0f} MB each > L2 {info['l2_bytes'] / 1e6:.0f} MB; no flush needed",
                "parallelism": f"dp{world} (batch sharded, coefficient grads all-reduced)" if world > 1 else "single GPU",
            },
            "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": cells * 4,
                    "d2h_bytes_per_step": nparam * 4, "ms_per_step": round(e2e_ms, 4), "chunks": nchunk,
                    "note": "pinned host input -> H2D -> nn.Module forward+backward -> D2H coefficient grads; PCIe bound"},
            "gpu_launches": ((5 if kind not in ("emotion", "tiny") else 3) * args.steps * inner),
            "gpu_launches_per_step": {"prepare_kernel": 1, "flags_kernel": 1, "sfwd_kernel": 1, "sbwd_kernel": 1,
                                      "finish_kernel": 1} if kind not in ("emotion", "tiny") else
                                     {"fwd_kernel": 1, "bwd_kernel": 1, "finish_kernel": 1},
            "roofline": {"bound": "hbm", "kernel": "backward (adjoint + coefficient-gradient reduction)",
                         "achieved": round(bwd_gbs, 1), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": round(bwd_gbs / peak, 4), "traffic": ctr.get("bwd_dram_bytes"),
                         "algorithmic_bytes_per_launch": bwd_bytes, "ms_per_launch": round(bwd_ms, 4),
                         # the binding roof of the implicit kernels is instruction issue, not HBM (SURVEY 8d):
                         # executed warp instructions per launch (ncu smsp__inst_executed.sum of the capture in
                         # profiles/, sources `counters_csrc_sha`) over the issue slots of the live-timed launch
                         "issue_frac": issue(ctr.get("bwd_inst_executed"), bwd_ms),
                         "inst_executed_per_launch": ctr.get("bwd_inst_executed"),
                         "thread_inst_per_cell_sweep": per_cell_sweep(ctr.get("bwd_inst_executed")),
                         "issue_clock_mhz": sm_mhz,
                         "counters_csrc_sha": ctr.get("csrc_sha"), "csrc_sha": _csrc_sha(),
                         "counters_match_build": ctr.get("csrc_sha") == _csrc_sha(),
                         "traffic_note": ("ncu dram bytes of the backward kernel; for the implicit layers they include the step "
                                          "checkpoints (num_steps x 4 B/cell) the training forward wrote on purpose: HBM is the "
                                          "idle resource of these kernels, shared memory the busy one (DESIGN.md 4.0)")
                         if kind not in ("emotion", "tiny") else None},
            "roofline_fwd": {"bound": "hbm", "achieved": round(fwd_gbs, 1), "peak": peak, "unit": "GB/s",
                             "frac": round(fwd_gbs / peak, 4), "algorithmic_bytes_per_launch": fwd_bytes,
                             "ms_per_launch": round(fwd_ms, 4), "traffic": ctr.get("fwd_dram_bytes"),
                             "issue_frac": issue(ctr.get("fwd_inst_executed"), fwd_ms),
                             "thread_inst_per_cell_sweep": per_cell_sweep(ctr.get("fwd_inst_executed"))},
            # forward + backward against the HBM roof, on the step the driver's clock sees (ms_per_step)
            "fwd_bwd_hbm_frac": round((fwd_bytes + bwd_bytes) / (ms_per_step * 1e-3) / 1e9 / peak, 4),
            "clamped": {"note": "same batch, weights perturbed so that cells sit outside both clamp edges and the time "
                                "coefficients cross a clamp inside [0, T] (masked path, smoothing adjoint inside every sweep)",
                        "fwd_ms": round(fwd_c_ms, 4), "bwd_ms": round(bwd_c_ms, 4),
                        "fwd_bwd_gcell_updates_per_s": round(cells * nsteps / ((fwd_c_ms + bwd_c_ms) * 1e-3) / 1e9, 2),
                        "bwd_hbm_frac": round(bwd_bytes / (bwd_c_ms * 1e-3) / 1e9 / peak, 4)},
            "dp_parity_rel_err": dp_parity,
            "numa_binding": numa,
            "parity_rel_err": parity,
            "parity_rel_err_clamped": parity_c,
            "fwd_inference_ms": round(fwd_eval_ms, 4),
            "bwd_no_grad_input_ms": round(bwd_nogin_ms, 4),
            "script_batch_latency_us": round(small_ms * 1e3, 1),
            "script_batch_latency_note": f"forward+backward at the script's batch ({script_b}) through the nn.Module, eager: bound by the "
                                         "host (autograd engine + Python + launches; a trivial custom Function costs 55 us on this box)",
            "script_batch_graph_us": round(small_graph_ms * 1e3, 1) if small_graph_ms else small_graph_err,
            "cpu_baseline": cpu,
            "clocks": clocks,
            "device": info,
        }
        if train is not None:
            out["train"] = train
        if others:
            out["other_layers"] = others
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def _quick_layer(name, dev, peak):
    """fwd / bwd Gcell-updates/s and HBM fraction of another layer at its roofline batch."""
    import torch
    from tests import cases as K
    from tests import runners
    kind, ctor, big_b, _ = LAYERS[name]
    c = K.case("q_" + name, kind, B=big_b, perturb=False, **ctor)
    C, H, W = c.shape
    nsteps = _steps_of(kind, ctor)
    cells = big_b * C * H * W
    layer = runners.make_cuda_layer(c, device=dev)
    gen = torch.Generator(device=dev).manual_seed(99)
    u = torch.randn(big_b, C, H, W, device=dev, generator=gen)
    g = torch.randn(big_b, C, H, W, device=dev, generator=gen)
    params = [p for p in layer.parameters() if p.requires_grad]

    def t(fn, n=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    x = u.clone().requires_grad_(True)
    fwd = t(lambda: layer(x))     # training forward (the implicit layers also write their step checkpoints)
    y = layer(x)
    bwd = t(lambda: torch.autograd.grad(y, [x] + params, g, retain_graph=True, allow_unused=True))
    tot = fwd + bwd
    res = {"batch": big_b, "num_steps": nsteps, "fwd_ms": round(fwd, 3), "bwd_ms": round(bwd, 3),
           "fwd_bwd_gcell_updates_per_s": round(cells * nsteps / (tot * 1e-3) / 1e9, 2),
           "fwd_hbm_frac": round(8 * cells / (fwd * 1e-3) / 1e9 / peak, 4),
           "bwd_hbm_frac": round(12 * cells / (bwd * 1e-3) / 1e9 / peak, 4),
           "fwd_bwd_hbm_frac": round(20 * cells / (tot * 1e-3) / 1e9 / peak, 4)}
    if kind == "tiny":
        # the bf16-I/O variant of the one bandwidth-bound layer (pde_tiny_*_bf16): same arithmetic, half the bytes
        ub, gb = u.bfloat16(), g.bfloat16()
        xb = ub.clone().requires_grad_(True)
        fb = t(lambda: layer(xb))
        yb = layer(xb)
        bb = t(lambda: torch.autograd.grad(yb, [xb] + params, gb, retain_graph=True, allow_unused=True))
        res["bf16_io"] = {"fwd_ms": round(fb, 3), "bwd_ms": round(bb, 3),
                          "fwd_bwd_gcell_updates_per_s": round(cells * nsteps / ((fb + bb) * 1e-3) / 1e9, 2),
                          "fwd_bwd_hbm_frac": round(10 * cells / ((fb + bb) * 1e-3) / 1e9 / peak, 4)}
        del ub, gb, xb, yb
    del u, g, x, y
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------- CPU baseline
def _oracle_step(c, params, io, nthreads):
    from tests import runners
    import numpy as np
    return runners.run_oracle(c, params=params, io=io, dtype=np.float32, nthreads=nthreads)


def cpu_baseline(layer, budget_s=12.0, fixed_batch=None, reps=1):
    """The C oracle (a port: the reference is Python and is not on this box) on all host cores,
    forward + backward, on a bounded sample of the same workload."""
    from tests import cases as K
    kind, ctor, _, script_b = LAYERS[layer]
    cores = os.cpu_count() or 1
    nsteps = _steps_of(kind, ctor)
    b = max(script_b, cores * 8)
    c = K.case("cpu_" + layer, kind, B=b, perturb=False, **ctor)
    params, io = K.make_params(c), K.make_io(c)
    _oracle_step(c, params, io, cores)  # warm (library load, page faults)
    t0 = time.perf_counter()
    _oracle_step(c, params, io, cores)
    dt = time.perf_counter() - t0
    if fixed_batch is None:
        scale = max(1.0, min(budget_s / max(dt, 1e-4), 4096.0))
        b2 = int(b * scale) // cores * cores or b
    else:
        b2 = fixed_batch
    c2 = K.case("cpu_" + layer, kind, B=b2, perturb=False, **ctor)
    params, io = K.make_params(c2), K.make_io(c2)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        _oracle_step(c2, params, io, cores)
        times.append(time.perf_counter() - t0)
    dt2 = min(times)
    C, H, W = c2.shape
    val = b2 * C * H * W * nsteps / dt2 / 1e9
    return {"value": round(val, 4), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle/pde_oracle.c (fp32, OpenMP x{cores}) forward+backward of {layer}, batch {b2}, "
                      f"{dt2:.2f} s", "batch": b2, "seconds": round(dt2, 3)}


def cpu_baseline_and_parity(layer_name, c, layer, u, g, budget_s):
    """The CPU leg at N = 1, doubling as a parity self-check of what was just timed: the oracle (all
    host cores) runs forward + backward on the benched batch itself -- or, if that would take more
    than ~3x the budget, on its first samples -- and the GPU results for exactly those samples are
    compared with it (worst of rel-L2 and max-abs / max-ref per output, tests/runners.compare)."""
    import numpy as np
    import torch
    from tests import cases as K
    from tests import runners
    kind, ctor, _, _ = LAYERS[layer_name]
    cores = os.cpu_count() or 1
    nsteps = _steps_of(kind, ctor)
    C, H, W = c.shape
    probe = cpu_baseline(layer_name, budget_s=1.0)
    full_s = c.B * C * H * W * nsteps / 1e9 / max(probe["value"], 1e-9)
    b2 = c.B if full_s <= 3.0 * budget_s else max(cores * 8, int(c.B * budget_s / full_s))
    c2 = K.case(c.name + "_cpu", kind, B=b2, perturb=c.perturb, **ctor)
    params = K.make_params(c2)
    for p in layer.parameters():
        p.grad = None
    xs = u[:b2].clone().requires_grad_(True)
    ys = layer(xs)
    ys.backward(g[:b2])
    torch.cuda.synchronize()
    got = {"y": ys.detach().cpu().numpy(), "gin": xs.grad.cpu().numpy()}
    for k, p in layer.named_parameters():
        if p.grad is not None:
            got["g_" + k] = p.grad.detach().cpu().numpy()
    io = (u[:b2].cpu().numpy(), g[:b2].cpu().numpy())
    del xs, ys
    t0 = time.perf_counter()
    want = runners.run_oracle(c2, params=params, io=io, dtype=np.float32, nthreads=cores)
    dt = time.perf_counter() - t0
    errs = runners.compare(got, want)
    val = b2 * C * H * W * nsteps / dt / 1e9
    cpu = {"value": round(val, 4), "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"oracle/pde_oracle.c (fp32, OpenMP x{cores}) forward+backward of {layer_name} on "
                     f"{'the benched batch' if b2 == c.B else 'the first samples of the benched batch'} ({b2} samples), {dt:.2f} s",
           "batch": b2, "seconds": round(dt, 3)}
    parity = {"worst": float(f"{max(errs.values()):.3e}"), "batch": b2, "tolerance": 1e-5,
              "per_output": {k: float(f"{v:.3e}") for k, v in errs.items()},
              "against": "oracle fp32 on the same inputs and weights" + ("" if not c.perturb else " (perturbed, clamped cells)")}
    return cpu, parity


def cpu_train_baseline(model_name="cifar10", batch=64, steps=2):
    """Whole-model training step on the host CPU: the classifier of cnn_with_pde_b200.classifiers in
    stock CPU torch (all cores) with every PDE layer's forward/backward routed to the C oracle
    (OpenMP, all cores) -- a port: the reference's own Python layer is ~1000x slower than the C
    restatement (BASELINE.md section 2) and does not exist on this box.  Checker-side only."""
    import numpy as np
    import torch
    import oracle
    from cnn_with_pde_b200 import train as T
    from cnn_with_pde_b200.cifar10 import EnhancedDiffusionLayer
    if model_name != "cifar10":
        raise NotImplementedError("CPU training baseline is wired for cifar10 only")
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    r = T._recipes()[model_name]
    torch.manual_seed(1234)
    model = r.build()
    model.train()

    class OracleAdi(torch.autograd.Function):
        @staticmethod
        def forward(ctx, u, ab, bb, atc, btc, chan, spec):
            ctx.spec = spec
            ctx.save_for_backward(u, ab, bb, atc, btc, chan)
            out = oracle.adi_forward(spec, u.numpy(), ab.detach().numpy(), bb.detach().numpy(), atc.detach().numpy(),
                                     btc.detach().numpy(), chan=chan.detach().numpy(), nthreads=cores)
            return torch.from_numpy(out)

        @staticmethod
        def backward(ctx, gout):
            u, ab, bb, atc, btc, chan = ctx.saved_tensors
            g = oracle.adi_backward(ctx.spec, u.numpy(), gout.contiguous().numpy(), ab.detach().numpy(),
                                    bb.detach().numpy(), atc.detach().numpy(), btc.detach().numpy(),
                                    chan=chan.detach().numpy(), need_gin=False, nthreads=cores)
            f = lambda k: torch.from_numpy(np.asarray(g[k], np.float32))
            return (None, f("alpha_base"), f("beta_base"), f("alpha_time_coeff"), f("beta_time_coeff"), f("chan"), None)

    for m in model.modules():
        if isinstance(m, EnhancedDiffusionLayer):
            spec = oracle.spec_cifar10(m.size, m.channels, m.dt, m.dx, m.dy, m.num_steps)
            m.forward = (lambda u, m=m, spec=spec: OracleAdi.apply(u, m.alpha_base, m.beta_base, m.alpha_time_coeff,
                                                                   m.beta_time_coeff, m.channel_mixing, spec))
    opt = T.make_optimizer(model, r, capturable=False)
    crit = torch.nn.CrossEntropyLoss(label_smoothing=r.label_smoothing)
    gen = torch.Generator().manual_seed(7)
    xb = torch.randn(batch, *r.shape, generator=gen)
    yb = torch.randint(0, r.classes, (batch,), generator=gen)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = crit(model(xb), yb)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=1.0)
        opt.step()
        return float(loss.detach())

    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": round(batch / dt, 1), "unit": "img/s", "cores": cores, "kind": "port",
            "sample": f"{model_name} classifier in CPU torch + oracle/pde_oracle.c PDE layers (fp32, OpenMP x{cores}), "
                      f"batch {batch}, {steps} optimiser steps, {dt * 1e3:.1f} ms/step",
            "reference_python_img_per_s_build_container": 48.4}


def run_reference(args):
    """--impl reference: the CPU implementation of the path on the host cores, same metric."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from tests import cases as K
    kind, ctor, big_b, script_b = LAYERS[args.layer]
    cores = os.cpu_count() or 1
    nsteps = _steps_of(kind, ctor)
    probe = cpu_baseline(args.layer, budget_s=1.5)
    # one step ~1.5 s of CPU work so that steps + warmup stay within a few minutes
    b = probe["batch"]
    c = K.case("ref_" + args.layer, kind, B=b, perturb=False, **ctor)
    params, io = K.make_params(c), K.make_io(c)
    for _ in range(args.warmup):
        _oracle_step(c, params, io, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _oracle_step(c, params, io, cores)
    dt = (time.perf_counter() - t0) / args.steps
    C, H, W = c.shape
    val = b * C * H * W * nsteps / dt / 1e9
    sample = (f"oracle/pde_oracle.c (C port of the reference's CPU path, fp32, OpenMP x{cores}), "
              f"forward+backward of {args.layer}, batch {b} per step")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.layer} PDE layer forward+backward, {C}x{H}x{W}, num_steps={nsteps}, "
                               f"bounded sample: batch {b} per step on the host CPU", "layer": args.layer},
        "cpu_baseline": {"value": round(val, 4), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(val, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--layer", default="fashion", choices=sorted(LAYERS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: roofline-size batch of the layer)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--inner", type=int, default=1, help="back-to-back passes per timed step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (--impl b200)")
    ap.add_argument("--all-layers", type=int, default=1, help="also time the other layers (N=1 only)")
    ap.add_argument("--train", type=int, default=1, help="also time a whole-model training step (img/s)")
    ap.add_argument("--train-model", default="cifar10")
    ap.add_argument("--train-batch", type=int, default=512, help="per-GPU batch of the training step")
    args = ap.parse_args()
    if args.steps < 1 or args.inner < 1:
        ap.error("--steps and --inner must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path: it needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
