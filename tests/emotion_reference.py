"""A second reference for emotion_recognition.PDELayer (emotion_recognition.py:56-97), restated in torch for any
plane edge N, with gradients from autograd.

The input is reflect-padded once; the ghost ring keeps those values in every step.  Each step is a Jacobi update
of the interior slice: u <- u + a_i d2_row u + b_j d2_col u with a_i = 0.5 dt (w1 + w2 sin 2 pi y_i +
w3 sin 4 pi y_i) / dx^2 and b_j = dt (w4 + w5 cos 2 pi x_j + w6 cos 4 pi x_j) / dy^2.  It holds no hand-derived
adjoint, so it checks the oracle's (oracle/pde_oracle.c) above 64 x 64, where no stored fixture reaches;
tests/test_emotion_large_oracle.py pins the two together, and the GPU tests of the halo kernels compare against the
oracle.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

import oracle as O

DEFAULT_W = (0.1, 0.1, 0.1, 0.3, 0.2, 0.2)   # the reference's init values


def buffers(N, dtype=np.float32):
    """The registered buffers x, y: torch.linspace(0, 1, N) in fp32, as the module builds them."""
    t = torch.linspace(0, 1.0, N, dtype=torch.float32).numpy()
    return t.astype(dtype), t.astype(dtype)


def run(u, g, w, Nt, dt=0.001, need_gin=True):
    """fp64 forward and gradients of B x 1 x N x N planes: {"y", "gin", "w"} as numpy arrays."""
    N = np.asarray(u).shape[-1]
    dx = dy = 1.0 / N
    xs, ys = (torch.tensor(v, dtype=torch.float64) for v in buffers(N, np.float64))
    x = torch.tensor(np.asarray(u, np.float64), requires_grad=need_gin)
    wt = torch.tensor(np.asarray(w, np.float64), requires_grad=True)
    a = 0.5 * dt * (wt[0] + wt[1] * torch.sin(2 * np.pi * ys) + wt[2] * torch.sin(4 * np.pi * ys)) / dx ** 2
    b = dt * (wt[3] + wt[4] * torch.cos(2 * np.pi * xs) + wt[5] * torch.cos(4 * np.pi * xs)) / dy ** 2
    p = F.pad(x, (1, 1, 1, 1), mode="reflect")
    ring = p
    for _ in range(Nt):
        c = p[..., 1:-1, 1:-1]
        dr = p[..., 2:, 1:-1] - 2 * c + p[..., :-2, 1:-1]
        dc = p[..., 1:-1, 2:] - 2 * c + p[..., 1:-1, :-2]
        new = c + a.view(N, 1) * dr + b.view(1, N) * dc
        p = ring.clone()
        p[..., 1:-1, 1:-1] = new
    y = p[..., 1:-1, 1:-1]
    wrt = [x, wt] if need_gin else [wt]
    if Nt == 0:
        grads = [torch.tensor(np.asarray(g, np.float64)), torch.zeros(6, dtype=torch.float64)][2 - len(wrt):]
    else:
        grads = torch.autograd.grad(y, wrt, torch.tensor(np.asarray(g, np.float64)))
    out = {"y": y.detach().numpy(), "w": grads[-1].numpy(), "gin": grads[0].numpy() if need_gin else None}
    return out


def oracle(u, g, w, Nt, dt=0.001, need_gin=True, dtype=np.float64):
    """The C oracle on the same inputs, in the same layout."""
    N = np.asarray(u).shape[-1]
    spec = O.EmoSpec(Nx=N, Ny=N, T=dt * Nt, dt=dt)
    spec.Nt = Nt   # int(T / dt) can round down
    xs, ys = buffers(N, dtype)
    u, g, w = np.asarray(u, dtype), np.asarray(g, dtype), np.asarray(w, dtype)
    y = O.emotion_forward(spec, u, w, xs, ys)
    r = O.emotion_backward(spec, u, g, w, xs, ys, need_gin=need_gin)
    return {"y": y, "gin": r["gin"], "w": r["w"]}


def stable_weights(N, seed, dt=0.001):
    """Seeded weights with a_i, b_j > 0 and max_i a_i + max_j b_j <= 1/2: the explicit scheme does not amplify."""
    rs = np.random.RandomState(seed)
    r = np.clip(rs.randn(6), -1.5, 1.5)
    w = np.array([1 + abs(r[0]), 0.3 * r[1], 0.3 * r[2], 1 + abs(r[3]), 0.3 * r[4], 0.3 * r[5]])   # a, b > 0
    sa = abs(w[0]) + abs(w[1]) + abs(w[2])
    sb = abs(w[3]) + abs(w[4]) + abs(w[5])
    # a <= 0.5 dt sa N^2, b <= dt sb N^2
    scale = 0.45 / ((0.5 * sa + sb) * dt * N * N)
    return (w * scale).astype(np.float32)


def make_inputs(B, N, seed):
    rs = np.random.RandomState(seed)
    return rs.randn(B, 1, N, N).astype(np.float32), rs.randn(B, 1, N, N).astype(np.float32)
