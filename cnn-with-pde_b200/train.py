"""Data-parallel training launcher for the reference's PDE classifiers on B200s.

One process per GPU (``torch.distributed``, NCCL over NVLink).  The only exchange is the sum of
the parameter gradients: every ``.grad`` is a view into one flat fp32 buffer, so gradient sync is a
single NCCL all-reduce per step (0.8 - 36 MB for these models; the PDE coefficient gradients,
<= 49 KB per layer, ride along) that also captures cleanly into a CUDA graph.  ``--sync ddp`` uses
``DistributedDataParallel`` (bucketed all-reduce overlapped with backward) instead.  Data is
synthetic and resident on the device (the reference's datasets need a network); each script's
optimiser recipe is reproduced (SURVEY.md section 2, row 14):

    model      reference loop                    optimiser                         loss              batch
    mnist      mnist_test.py:263-345             AdamW 1e-3, wd 1e-4               CE, smoothing .1  128
    fashion    fashion_mnist.py:256-331          AdamW 2e-3, wd 5e-4               CE, smoothing .1  128
    cifar10    cifar10.py:400-527                AdamW, alpha/beta group + rest    CE, smoothing .1   64
    svhn       SVHN.py:300-406                   AdamW 1e-2, wd 1e-4               CE                256
    emotion    emotion_recognition.py:265-415    AdamW 1e-3, wd 1e-4               CE                 64

every loop clips the gradient norm at 1.0.  Weak scaling: --batch is the per-GPU batch.  --image-size N trains
the tiny_imagenet ResNet on N x N images (it ends in a global average pool, so any size works; 224 is ImageNet's);
the other models' heads are sized for their images, so they refuse it.

    python train.py --model cifar10 --batch 512 --steps 50
    python train.py --model tiny --image-size 224 --batch 64 --steps 20 --graph
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29511 train.py --model cifar10 --batch 512 --steps 50

With --graph the step is captured in CUDA graphs: after the PDE kernels a step is a few dozen tiny
dense kernels and launch bound.  On several GPUs the flat all-reduce stays an eager NCCL call between
two graphs (forward + backward | clipping + AdamW): measured on two B200s the step costs 1.259 ms that
way against 1.236 ms on one GPU, so the exchange (1 MB) is ~2 % of the step.  --nccl-in-graph captures
the all-reduce inside ONE graph instead (thread-local capture mode, after a warm-up collective on the
capture stream); it takes the same optimiser steps (tests/test_gpu_multi.py) and the same time
(1.264 ms), but a 220-step run of it stopped making progress on the two-GPU box here, so it is opt-in.

--compile trains torch.compile(model, fullgraph=True) instead (the PDE layers are pde_b200:: custom ops in the
graph, ops.py); it excludes --graph and works with --amp and the flat all-reduce.

--amp reproduces the CIFAR scripts' mixed-precision recipe (cifar10.py:440,458-467): autocast,
GradScaler.scale(loss).backward(), unscale_, clip_grad_norm_, scaler.step, scaler.update -- the PDE
layers themselves stay fp32 (custom_fwd(cast_inputs=float32)).
"""
from __future__ import annotations

import argparse
import json
import os
import time
from dataclasses import dataclass
from typing import Callable, Tuple

import torch
import torch.distributed as dist
import torch.nn as nn


@dataclass(frozen=True)
class Recipe:
    build: Callable[[], nn.Module]
    shape: Tuple[int, int, int]
    classes: int
    batch: int                 # the reference script's batch size
    lr: float
    weight_decay: float
    label_smoothing: float
    split_groups: bool = False  # cifar10.py:423-434: alpha/beta parameters get their own group
    group_keys: Tuple[str, ...] = ("alpha", "beta")   # substrings that put a parameter in the coefficient group
    rest_lr_scale: float = 0.5                         # learning-rate factor of the other group


def _recipes():
    from . import SVHN, cifar10, cifar_2version, emotion_recognition, fashion_mnist, mnist_test, tiny_imagenet

    def tiny():
        # diff.beta_base takes no part in the forward pass (tiny_imagenet.py:21,26): its .grad stays None in
        # the reference, so AdamW never touches it; with one flat gradient buffer that means "frozen"
        m = tiny_imagenet.ImprovedTinyImageNetClassifier()
        m.diff.beta_base.requires_grad_(False)
        return m

    return {
        "tiny": Recipe(tiny, (3, 64, 64), 200, 32, 1e-3, 1e-4, 0.1),   # tiny_imagenet.py:543-556
        # cifar_2version.py:487-499: coefficient group (alpha, beta, channel_mixing, combination_weights)
        # lr 1e-3 / weight_decay 1e-6, the rest 0.8 x lr / 1e-4
        "cifar2": Recipe(cifar_2version.CIFAR10HybridPDEModel, (3, 32, 32), 10, 64, 1e-3, 1e-4, 0.1, split_groups=True,
                         group_keys=("alpha", "beta", "channel_mixing", "combination_weights"), rest_lr_scale=0.8),
        "mnist": Recipe(mnist_test.PDEClassifier, (1, 28, 28), 10, 128, 1e-3, 1e-4, 0.1),
        "fashion": Recipe(fashion_mnist.FashionPDEClassifier, (1, 28, 28), 10, 128, 2e-3, 5e-4, 0.1),
        "cifar10": Recipe(cifar10.CIFAR10PDENoConv, (3, 32, 32), 10, 64, 1e-3, 1e-4, 0.1, split_groups=True),
        "svhn": Recipe(SVHN.PDEClassifier, (3, 32, 32), 10, 256, 1e-2, 1e-4, 0.0),
        "emotion": Recipe(emotion_recognition.DiffusionClassifier, (1, 48, 48), 7, 64, 1e-3, 1e-4, 0.0),
    }


MODELS = ("mnist", "fashion", "cifar10", "cifar2", "svhn", "emotion", "tiny")
GRAPH_PRIMING_STEPS = 3   # eager steps on the capture stream before a CUDA graph is recorded


class FlatGradSync:
    """All parameter gradients as views of one flat buffer; sync = one all-reduce (mean, as DDP)."""

    def __init__(self, model: nn.Module, world: int):
        params = [p for p in model.parameters() if p.requires_grad]
        self.world = world
        self.flat = torch.zeros(sum(p.numel() for p in params), dtype=torch.float32, device=params[0].device)
        off = 0
        for p in params:
            n = p.numel()
            p.grad = self.flat[off:off + n].view_as(p)   # autograd accumulates into it in place
            off += n

    def zero(self):
        self.flat.zero_()

    def all_reduce(self):
        if self.world > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.flat.mul_(1.0 / self.world)


def make_optimizer(model: nn.Module, r: Recipe, capturable: bool):
    # the scripts' AdamW recipe; on CUDA the fused implementation (one kernel per parameter group
    # instead of ~30 multi-tensor launches per step; same update rule, capturable)
    on_cuda = all(p.is_cuda for p in model.parameters())
    extra = {"fused": True, "capturable": capturable} if on_cuda else {"capturable": capturable}
    if r.split_groups:
        in_coef = lambda n: any(k in n for k in r.group_keys)   # noqa: E731
        coef = [p for n, p in model.named_parameters() if in_coef(n)]
        rest = [p for n, p in model.named_parameters() if not in_coef(n)]
        groups = [{"params": coef, "lr": r.lr, "weight_decay": 1e-6},
                  {"params": rest, "lr": r.lr * r.rest_lr_scale, "weight_decay": r.weight_decay}]
        return torch.optim.AdamW(groups, **extra)
    return torch.optim.AdamW(model.parameters(), lr=r.lr, weight_decay=r.weight_decay, **extra)


def _dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


def run(model_name: str, batch: int, steps: int, warmup: int, graph: bool = False, amp: bool = False,
        seed: int = 1234, pool: int = 4, quiet: bool = False, sync: str = "flat", nccl_in_graph: bool = False,
        no_dropout: bool = False, keep_model: bool = False, image_size: int | None = None, compile: bool = False):
    """Train `steps` timed steps (after `warmup`) of `model_name` at per-GPU batch `batch` on the
    current rank's GPU; returns a dict with whole-job img/s (max-over-ranks device time).
    `image_size` (tiny only) trains on image_size x image_size images instead of the recipe's 64 x 64.
    `compile` trains torch.compile(model, fullgraph=True): the PDE layers enter the graph as pde_b200:: custom ops
    (ops.py), the stock layers are Inductor's; the first warm-up step compiles."""
    if compile and graph:
        raise ValueError("--compile and --graph are exclusive: --compile traces the model with torch.compile, "
                         "--graph captures the eager step in CUDA graphs")
    if compile and sync == "ddp":
        raise ValueError("--compile needs --sync flat")
    r = _recipes()[model_name]
    shape = r.shape
    if image_size is not None:
        if model_name != "tiny":
            raise ValueError(f"--image-size: only the tiny model takes other image sizes (its ResNet ends in a global "
                             f"average pool); {model_name}'s classifier head is sized for {r.shape[1]} x {r.shape[2]}")
        if image_size < 1:
            raise ValueError(f"--image-size must be positive, got {image_size}")
        shape = (r.shape[0], image_size, image_size)
    world, rank, local = _dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("train.py needs a CUDA device: the PDE layers have no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    own_pg = False
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
        own_pg = True
    torch.manual_seed(seed)            # identical initial weights on every rank
    model = r.build().to(dev)
    model.train()
    if no_dropout:   # a step without random masks: what the graph-vs-eager equality test compares
        for m in model.modules():
            if isinstance(m, nn.Dropout):
                m.p = 0.0
    criterion = nn.CrossEntropyLoss(label_smoothing=r.label_smoothing)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):      # DDP built on the capture stream, as whole-step capture requires
        use_ddp = world > 1 and sync == "ddp"
        net = nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True) \
            if use_ddp else model
        if compile:
            net = torch.compile(model, fullgraph=True)
        flat = None if use_ddp else FlatGradSync(model, world)
        opt = make_optimizer(model, r, capturable=graph)
    torch.cuda.current_stream().wait_stream(side)

    gen = torch.Generator(device=dev).manual_seed(seed + 1 + rank)   # a different shard per rank
    xs = [torch.randn(batch, *shape, device=dev, generator=gen) for _ in range(pool)]
    ys = [torch.randint(0, r.classes, (batch,), device=dev, generator=gen) for _ in range(pool)]
    x_in, y_in = xs[0].clone(), ys[0].clone()
    loss_out = torch.zeros((), device=dev)

    state = {"done": 0}   # optimiser steps taken so far: step k trains on batch k % pool, captured or not

    def feed(k):
        x_in.copy_(xs[k % pool], non_blocking=True)
        y_in.copy_(ys[k % pool], non_blocking=True)

    # cifar10.py:440: GradScaler on CUDA; a disabled scaler is the identity (scale = 1, plain step).
    # With the flat all-reduce the ranks exchange SCALED gradients; unscale_ runs after the exchange,
    # so an overflow on one rank is seen by all and the scalers stay in step.
    scaler = torch.amp.GradScaler("cuda", enabled=amp)

    def fwd_bwd():
        if flat is not None:
            flat.zero()
        else:
            opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", enabled=amp):
            loss = criterion(net(x_in), y_in)
        scaler.scale(loss).backward()
        loss_out.copy_(loss.detach())

    def update():
        scaler.unscale_(opt)
        nn.utils.clip_grad_norm_(model.parameters(), max_norm=1.0)
        scaler.step(opt)      # fused AdamW takes grad_scale / found_inf on the device: no host sync
        scaler.update()

    def step_body():
        fwd_bwd()
        if flat is not None:
            flat.all_reduce()
        update()

    # CUDA graphs: one graph for the whole step on one GPU.  With several ranks the flat all-reduce stays
    # an eager NCCL call between two graphs (forward + backward | clipping + AdamW) unless nccl_in_graph
    # asks for it inside ONE graph (thread-local capture mode: the NCCL watchdog thread polls events
    # concurrently, which a global-mode capture would treat as a violation; the priming steps below run
    # the collective on the capture stream first so that no communicator is created under capture).
    graphs = []
    if graph:
        if use_ddp:
            raise RuntimeError("--graph needs --sync flat (DDP's reducer is not captured)")
        with torch.cuda.stream(side):
            for _ in range(GRAPH_PRIMING_STEPS):   # real optimiser steps on the rotating batches, like every other
                feed(state["done"])
                step_body()
                state["done"] += 1
            side.synchronize()
            parts = [step_body] if (world == 1 or nccl_in_graph) else [fwd_bwd, update]
            pool_id = None
            for fn in parts:
                cg = torch.cuda.CUDAGraph()
                with torch.cuda.graph(cg, stream=side, pool=pool_id, capture_error_mode="thread_local"):
                    fn()
                pool_id = cg.pool()
                graphs.append(cg)
                if world > 1 and fn is fwd_bwd:
                    flat.all_reduce()          # keep the eager sequence of the step intact
        torch.cuda.current_stream().wait_stream(side)

    def one_step(_i):
        feed(state["done"])
        state["done"] += 1
        if not graphs:
            step_body()
        elif len(graphs) == 1:
            graphs[0].replay()
        else:
            graphs[0].replay()
            flat.all_reduce()
            graphs[1].replay()

    for i in range(warmup):
        one_step(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        one_step(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    out = {
        "model": model_name, "image_shape": list(shape), "n_gpus": world, "batch_per_gpu": batch, "global_batch": batch * world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms / max(steps, 1),
        "img_per_s": batch * world * steps / (ms * 1e-3) if ms > 0 else 0.0,
        "loss": float(loss_out.item()), "cuda_graph": bool(graphs), "compiled": compile, "autocast": amp, "optimizer_steps": state["done"],
        "grad_sync": "none" if world == 1 else ("ddp" if use_ddp else (
            "flat all-reduce inside the CUDA graph" if len(graphs) == 1 else "flat all-reduce")),
        "grad_scaler": bool(amp),
        "params": sum(p.numel() for p in model.parameters()), "data": "synthetic, device resident",
        "scaling": "weak",
    }
    if keep_model:
        out["_model"] = model
    if own_pg:
        dist.destroy_process_group()
    if rank == 0 and not quiet:
        print(json.dumps({k: v for k, v in out.items() if not k.startswith("_")}), flush=True)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--model", choices=MODELS, default="cifar10")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the reference script's)")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--graph", action="store_true", help="capture the whole step in a CUDA graph")
    ap.add_argument("--compile", action="store_true",
                    help="train torch.compile(model, fullgraph=True); not with --graph (compiled in the first warm-up step)")
    ap.add_argument("--amp", action="store_true", help="autocast as in cifar10.py:459 (the PDE layer stays fp32)")
    ap.add_argument("--sync", choices=("flat", "ddp"), default="flat", help="gradient sync for N > 1")
    ap.add_argument("--nccl-in-graph", action="store_true", help="capture the all-reduce inside the CUDA graph (opt-in)")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--image-size", type=int, default=None, help="tiny only: train on N x N images (e.g. 224)")
    a = ap.parse_args(argv)
    batch = a.batch or _recipes()[a.model].batch
    t0 = time.time()
    out = run(a.model, batch, a.steps, a.warmup, graph=a.graph, amp=a.amp, seed=a.seed, sync=a.sync,
              nccl_in_graph=a.nccl_in_graph, image_size=a.image_size, compile=a.compile)
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"# {out['img_per_s']:.0f} img/s on {out['n_gpus']} GPU(s), {out['ms_per_step']:.3f} ms/step, "
              f"wall {time.time() - t0:.1f} s", flush=True)


if __name__ == "__main__":
    main()
