"""The PDE passes as torch.library custom ops (namespace ``pde_b200``): what torch.compile, torch.export and
FakeTensor / meta-device shape inference see of the layers.

    adi_fwd / adi_bwd            implicit layers (both kernel families: the route is chosen inside the op)
    emotion_fwd / emotion_bwd    emotion_recognition.PDELayer (fp32 or bf16 planes, after the input)
    tiny_fwd / tiny_bwd          tiny_imagenet.ImprovedDiffusionLayer (fp32 or bf16 planes, after the input)
    tiny_split                   its dormant split methods (self-adjoint: the backward pass is the same op)

Each op's real implementation calls the same pass helper of functional.py as the eager autograd.Function, so a
traced call runs the same kernels with the same plans.  Schemas take the configuration as plain numbers.  What
goes from a forward op to its backward op is an op output or an op input kept by autograd; the kernel-variant
value (`functional.env_tuning`) is an argument of both.  Fake implementations size every output from the input
shapes and, where they need one, a host-only library size query at batch 1: no output size is a non-linear
function of the batch, so `torch.compile(..., dynamic=True)` compiles once for every batch.  That is why the
implicit layers' step checkpoints (`pde_adi_checkpoint_bytes`: rounded to whole sample groups, and it asks the
device) are not an output: under autograd the forward op runs the kernel that writes them, as the eager call does,
into a buffer it drops, and the backward op makes them again inside its own workspace with the same kernel, so
outputs and gradients equal the eager ones bit for bit.
"""
from __future__ import annotations

import functools
from ctypes import byref
from typing import Optional

import torch
from torch import Tensor

from . import _cabi
from . import functional as F


# ------------------------------------------------------------------------------ implicit ADI
@functools.lru_cache(maxsize=256)
def _adi_cfg(N, C, steps, dt, hx, hy, lie, smooth, has_max, chan_op, skip, cmin, cmax, eps) -> F.AdiConfig:
    return F.AdiConfig(N, C, steps, dt, hx, hy, lie, smooth, has_max, chan_op, skip, cmin, cmax, eps)


def _device_index(dev) -> int:
    return dev.index if dev.index is not None else torch.cuda.current_device()


@torch.library.custom_op("pde_b200::adi_fwd", mutates_args=())
def adi_fwd(u: Tensor, alpha_base: Tensor, beta_base: Tensor, alpha_time_coeff: Tensor, beta_time_coeff: Tensor,
            chan: Optional[Tensor], skip_weight: Optional[Tensor], N: int, C: int, steps: int, dt: float, hx: float,
            hy: float, lie: bool, smooth: bool, has_max: bool, chan_op: int, skip: bool, cmin: float, cmax: float,
            eps: float, tuning: int, training: bool) -> tuple[Tensor, Tensor]:
    """(out, coefficient tables): the tables are empty where the streaming kernels serve the configuration.
    `training` picks the forward kernel the eager call would pick (the one that also writes step checkpoints), so
    that the outputs are the eager ones bit for bit; the checkpoints themselves are not kept (module docstring)."""
    cfg = _adi_cfg(N, C, steps, dt, hx, hy, lie, smooth, has_max, chan_op, skip, cmin, cmax, eps)
    params = (alpha_base, beta_base, alpha_time_coeff, beta_time_coeff)
    if F.adi_route(cfg) == "stream":
        out = F._adi_stream_forward(u, params, chan, skip_weight, cfg)[0]
        return out, torch.empty(0, dtype=torch.uint8, device=u.device)
    out, tables = F._adi_tables_forward(u, params, chan, skip_weight, cfg, tuning, training, False)[:2]
    return out, tables


@adi_fwd.register_fake
def _(u, alpha_base, beta_base, alpha_time_coeff, beta_time_coeff, chan, skip_weight, N, C, steps, dt, hx, hy, lie,
      smooth, has_max, chan_op, skip, cmin, cmax, eps, tuning, training):
    cfg = _adi_cfg(N, C, steps, dt, hx, hy, lie, smooth, has_max, chan_op, skip, cmin, cmax, eps)
    # the table size does not depend on the batch (include/pde_b200.h: one set of tables per call)
    n = _cabi.lib().pde_adi_tables_bytes(byref(cfg.desc(1))) if F.adi_route(cfg) == "tables" else 0
    return u.new_empty(u.shape), u.new_empty((n,), dtype=torch.uint8)


@torch.library.custom_op("pde_b200::adi_bwd", mutates_args=())
def adi_bwd(gout: Tensor, u: Tensor, alpha_base: Tensor, beta_base: Tensor, alpha_time_coeff: Tensor,
            beta_time_coeff: Tensor, chan: Optional[Tensor], skip_weight: Optional[Tensor], tables: Tensor, N: int, C: int,
            steps: int, dt: float, hx: float, hy: float, lie: bool, smooth: bool, has_max: bool, chan_op: int, skip: bool,
            cmin: float, cmax: float, eps: float, tuning: int, training: bool,
            need_gin: bool) -> tuple[Tensor, Tensor, Tensor, Tensor]:
    """(grad_input, the four map gradients as one (4, ...) tensor, g_chan, g_skip); a gradient that is not wanted
    (need_gin false, no chan / skip_weight) is an empty tensor."""
    cfg = _adi_cfg(N, C, steps, dt, hx, hy, lie, smooth, has_max, chan_op, skip, cmin, cmax, eps)
    u = F._contig(u)
    chan = None if chan is None else F._contig(chan)
    skip_weight = None if skip_weight is None else F._contig(skip_weight)
    shape = alpha_base.shape
    with F._guard(u.device):
        if F.adi_route(cfg) == "stream":
            plan = F._adi_stream_plan(cfg, u.shape[0], _device_index(u.device))
            maps = [F._contig(p) for p in (alpha_base, beta_base, alpha_time_coeff, beta_time_coeff)]
            gin, gm, gchan, gskip = F._adi_stream_backward(plan, u, maps, chan, skip_weight, gout, shape, need_gin)
        else:
            plan = F._adi_plan(cfg, u.shape[0], tuning, _device_index(u.device))
            gin, gm, gchan, gskip = F._adi_tables_backward(plan, u, tables, chan, skip_weight, None, gout, shape, need_gin)
    none = lambda t: u.new_empty(0) if t is None else t   # noqa: E731  (one tensor per output: outputs may not alias)
    return none(gin), gm, none(gchan), none(gskip)


@adi_bwd.register_fake
def _(gout, u, alpha_base, beta_base, alpha_time_coeff, beta_time_coeff, chan, skip_weight, tables, N, C, steps, dt, hx,
      hy, lie, smooth, has_max, chan_op, skip, cmin, cmax, eps, tuning, training, need_gin):
    return (u.new_empty(u.shape if need_gin else (0,)), u.new_empty((4,) + tuple(alpha_base.shape)),
            u.new_empty((C, C) if chan is not None else (0,)), u.new_empty(() if skip_weight is not None else (0,)))


def _adi_setup(ctx, inputs, output):
    ctx.config = inputs[7:]
    ctx.save_for_backward(*inputs[:7], output[1])


def _adi_backward(ctx, gout, _gtables):
    F._no_double_backward("PDE layer")
    u, ab, bb, atc, btc, chan, skipw, tables = ctx.saved_tensors
    need_gin = ctx.needs_input_grad[0]
    gin, gm, gchan, gskip = torch.ops.pde_b200.adi_bwd(gout, u, ab, bb, atc, btc, chan, skipw, tables, *ctx.config,
                                                       need_gin)
    g = gm.unbind(0)
    return (gin if need_gin else None, g[0], g[1], g[2], g[3], gchan if chan is not None else None,
            gskip if skipw is not None else None) + (None,) * len(ctx.config)


adi_fwd.register_autograd(_adi_backward, setup_context=_adi_setup)


# ------------------------------------------------------------------- explicit, frozen ghost ring
@torch.library.custom_op("pde_b200::emotion_fwd", mutates_args=())
def emotion_fwd(u0: Tensor, w6: Tensor, xs: Tensor, ys: Tensor, N: int, Nt: int, dt: float, dx: float, dy: float,
                generic: bool) -> Tensor:
    return F._emotion_forward(u0, w6, xs, ys, F.EmoConfig(N=N, Nt=Nt, dt=dt, dx=dx, dy=dy), generic)[0]


@emotion_fwd.register_fake
def _(u0, w6, xs, ys, N, Nt, dt, dx, dy, generic):
    return u0.new_empty(u0.shape)


@torch.library.custom_op("pde_b200::emotion_bwd", mutates_args=())
def emotion_bwd(gout: Tensor, u0: Tensor, w6: Tensor, xs: Tensor, ys: Tensor, N: int, Nt: int, dt: float, dx: float,
                dy: float, generic: bool, need_gin: bool) -> tuple[Tensor, Tensor]:
    """(grad_input or an empty tensor, the gradient of the six weights); grad_input in u0's dtype, the weight
    gradient fp32."""
    plan = F._emo_plan(F.EmoConfig(N=N, Nt=Nt, dt=dt, dx=dx, dy=dy), u0.shape[0], generic, _device_index(u0.device),
                       u0.dtype == torch.bfloat16)
    gin, gw = F._emotion_backward(plan, F._contig(u0), F._fp32(w6), F._fp32(xs), F._fp32(ys), gout, need_gin)
    return (u0.new_empty(0) if gin is None else gin), gw


@emotion_bwd.register_fake
def _(gout, u0, w6, xs, ys, N, Nt, dt, dx, dy, generic, need_gin):
    return u0.new_empty(u0.shape if need_gin else (0,)), u0.new_empty((6,), dtype=torch.float32)


def _emotion_setup(ctx, inputs, output):
    ctx.config = inputs[4:]
    ctx.save_for_backward(*inputs[:4])


def _emotion_backward(ctx, gout):
    F._no_double_backward("PDELayer")
    u0, w6, xs, ys = ctx.saved_tensors
    need_gin = ctx.needs_input_grad[0]
    gin, gw = torch.ops.pde_b200.emotion_bwd(gout, u0, w6, xs, ys, *ctx.config, need_gin)
    return (gin if need_gin else None, gw, None, None) + (None,) * len(ctx.config)


emotion_fwd.register_autograd(_emotion_backward, setup_context=_emotion_setup)


# ----------------------------------------------------------------------- explicit, zero ghosts
@torch.library.custom_op("pde_b200::tiny_fwd", mutates_args=())
def tiny_fwd(u: Tensor, alpha_base: Tensor, channel_scaling: Tensor, steps: int, dt: float, cmin: float, cmax: float,
             blend: float) -> Tensor:
    return F._tiny_forward(u, alpha_base, channel_scaling, F.TinyConfig(steps, dt, cmin, cmax, blend))[0]


@tiny_fwd.register_fake
def _(u, alpha_base, channel_scaling, steps, dt, cmin, cmax, blend):
    return u.new_empty(u.shape)


@torch.library.custom_op("pde_b200::tiny_bwd", mutates_args=())
def tiny_bwd(gout: Tensor, u: Tensor, alpha_base: Tensor, channel_scaling: Tensor, steps: int, dt: float, cmin: float,
             cmax: float, blend: float, need_gin: bool) -> tuple[Tensor, Tensor, Tensor]:
    """(grad_input or an empty tensor, g_alpha_base, g_channel_scaling); the parameter gradients are fp32."""
    u = F._contig(u)
    al, sc = F._contig(alpha_base).float(), F._contig(channel_scaling).float()
    plan = F._tiny_plan(F.TinyConfig(steps, dt, cmin, cmax, blend), tuple(u.shape), _device_index(u.device))
    gin, ga, gs = F._tiny_backward(plan, u, al, sc, gout, need_gin)
    return (u.new_empty(0) if gin is None else gin), ga, gs


@tiny_bwd.register_fake
def _(gout, u, alpha_base, channel_scaling, steps, dt, cmin, cmax, blend, need_gin):
    C = u.shape[1]
    return (u.new_empty(u.shape if need_gin else (0,)), u.new_empty((C,), dtype=torch.float32),
            u.new_empty((C,), dtype=torch.float32))


def _tiny_setup(ctx, inputs, output):
    ctx.config = inputs[3:]
    ctx.save_for_backward(*inputs[:3])


def _tiny_backward(ctx, gout):
    F._no_double_backward("ImprovedDiffusionLayer")
    u, al, sc = ctx.saved_tensors
    need_gin = ctx.needs_input_grad[0]
    gin, ga, gs = torch.ops.pde_b200.tiny_bwd(gout, u, al, sc, *ctx.config, need_gin)
    return (gin if need_gin else None, ga, gs) + (None,) * len(ctx.config)


tiny_fwd.register_autograd(_tiny_backward, setup_context=_tiny_setup)


# --------------------------------------------- tiny_imagenet's dormant scalar-coefficient methods
@torch.library.custom_op("pde_b200::tiny_split", mutates_args=())
def tiny_split(u: Tensor, mode: int, coeff_x: float, coeff_y: float, dt: float, eps: float) -> Tensor:
    B, H, W = u.shape
    return F._tiny_split_run(F._tiny_split_desc(mode, B, H, W, coeff_x, coeff_y, dt, eps), u,
                             "ImprovedDiffusionLayer dormant-path input")


@tiny_split.register_fake
def _(u, mode, coeff_x, coeff_y, dt, eps):
    return u.new_empty(u.shape)


def _tiny_split_setup(ctx, inputs, output):
    ctx.config = inputs[1:]


def _tiny_split_backward(ctx, gout):
    F._no_double_backward("ImprovedDiffusionLayer dormant path")
    return (torch.ops.pde_b200.tiny_split(gout.float(), *ctx.config),) + (None,) * len(ctx.config)


tiny_split.register_autograd(_tiny_split_backward, setup_context=_tiny_split_setup)
