"""A second reference for tiny_imagenet.ImprovedDiffusionLayer's live path (tiny_imagenet.py:34-72), restated in
torch for any (B, C, H, W), with gradients from autograd.

Per step: alpha = clamp(alpha_base, cmin, cmax); v = s u; w = v + alpha dt conv2d(v, Laplacian, padding=1);
u <- u + blend (w - u).  It holds no hand-derived adjoint, so it checks the oracle's (oracle/pde_oracle.c) at
plane shapes the stored fixtures (16 x 16, 64 x 64) do not reach; tests/test_tiny_reference.py pins the two
together, and the GPU tests of the tiled kernels compare against the oracle.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

import oracle as O

LAPLACIAN = ((0.0, 1.0, 0.0), (1.0, -4.0, 1.0), (0.0, 1.0, 0.0))


def step(u, alpha_base, scaling, dt, cmin, cmax, blend):
    C = u.shape[1]
    alpha = torch.clamp(alpha_base, cmin, cmax)
    v = u * scaling.view(1, C, 1, 1)
    k = torch.tensor(LAPLACIAN, dtype=u.dtype).view(1, 1, 3, 3).repeat(C, 1, 1, 1)
    lap = F.conv2d(v, k, padding=1, groups=C)
    w = v + (alpha * dt).view(1, C, 1, 1) * lap
    return u + blend * (w - u)


def run(u, g, alpha_base, scaling, steps, dt=0.01, cmin=1e-6, cmax=0.15, blend=0.1, need_gin=True):
    """fp64 forward and gradients: {"y", "gin", "alpha_base", "channel_scaling"} as numpy arrays."""
    x = torch.tensor(np.asarray(u, np.float64), requires_grad=need_gin)
    a = torch.tensor(np.asarray(alpha_base, np.float64), requires_grad=True)
    s = torch.tensor(np.asarray(scaling, np.float64), requires_grad=True)
    y = x
    for _ in range(steps):
        y = step(y, a, s, dt, cmin, cmax, blend)
    wrt = [x, a, s] if need_gin else [a, s]
    if y.requires_grad:
        grads = torch.autograd.grad(y, wrt, torch.tensor(np.asarray(g, np.float64)), allow_unused=True)
    else:                                       # no steps and no grad_input: nothing depends on a parameter
        grads = [None] * len(wrt)
    out = {k: (np.zeros(t.shape) if d is None else d.numpy()) for k, t, d in
           zip(("gin", "alpha_base", "channel_scaling")[3 - len(wrt):], wrt, grads)}
    out["y"] = y.detach().numpy()
    out.setdefault("gin", None)
    return out


def oracle(u, g, alpha_base, scaling, steps, dt=0.01, cmin=1e-6, cmax=0.15, blend=0.1, need_gin=True,
           dtype=np.float64):
    """The C oracle on the same inputs, in the same layout."""
    C = np.asarray(u).shape[1]
    spec = O.TinySpec(channels=C, dt=dt, num_steps=steps, cmin=cmin, cmax=cmax, blend=blend)
    u, g = np.asarray(u, dtype), np.asarray(g, dtype)
    al, sc = np.asarray(alpha_base, dtype), np.asarray(scaling, dtype)
    y = O.tiny_forward(spec, u, al, sc)
    r = O.tiny_backward(spec, u, g, al, sc, need_gin=need_gin)
    return {"y": y, "gin": r["gin"], "alpha_base": r["alpha_base"], "channel_scaling": r["channel_scaling"]}


def make_inputs(B, C, H, W, seed, clamp=False):
    """Seeded planes and parameters; alpha_base inside (cmin, cmax), or straddling it when `clamp` is set."""
    rs = np.random.RandomState(seed)
    u = rs.randn(B, C, H, W).astype(np.float32)
    g = rs.randn(B, C, H, W).astype(np.float32)
    alpha = (0.05 + 0.08 * rs.rand(C) - 0.04).astype(np.float32)
    if clamp:
        alpha[::2] = np.float32(0.3)          # above cmax: clamped, gradient 0
        if C > 1:
            alpha[1] = np.float32(-0.1)       # below cmin
    scaling = (1.0 + 0.2 * rs.randn(C)).astype(np.float32)
    return u, g, alpha, scaling
