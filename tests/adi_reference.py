"""A second reference for the channel-aware implicit layers: the oracle's arithmetic restated in torch, with
gradients from autograd, in fp32 or fp64, on any device and at any channel count.

The oracle's adjoint keeps its channel-matrix gradient in an 8 x 8 array, so it serves C <= 8 only.  This
module restates the oracle's forward (oracle/pde_oracle.c: build_schedule, build_tables, sweep_plane,
chan_apply, the skip blend) op for op, and lets autograd differentiate it, so it holds no hand-derived
adjoint of its own.  tests/test_adi_reference.py pins it to the oracle where both serve (forward at every C,
every gradient at C <= 8); tests/test_gpu_wide_channels.py uses it above eight channels.
"""
from __future__ import annotations

from typing import Dict

import numpy as np

from . import cases as K
from . import runners

MAP_KEYS = ("alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff")


def _schedule(spec):
    """(axis, t, dts, h) per sweep, current_time accumulated in double (oracle build_schedule)."""
    out, t = [], 0.0
    for _ in range(spec.steps):
        if not spec.lie:
            out.append((0, t, spec.dt / 2, spec.hx)); t += spec.dt / 2
            out.append((1, t, spec.dt, spec.hy)); t += spec.dt / 2
            out.append((0, t, spec.dt / 2, spec.hx))
        else:
            out.append((0, t, spec.dt / 2, spec.hx)); t += spec.dt / 2
            out.append((1, t, spec.dt / 2, spec.hy)); t += spec.dt / 2
    return out


def _tables(spec, base, tc, tt, dts, h2):
    """r and the Thomas pivots of one sweep, in line coordinates [c][line][i] (oracle build_tables)."""
    import torch
    R = base.dtype
    one, two, three = (torch.tensor(v, dtype=R, device=base.device) for v in (1.0, 2.0, 3.0))
    third = one / three
    raw = base + tc * tt
    k = torch.clamp(raw, min=spec.cmin, max=spec.cmax) if spec.has_max else torch.clamp(raw, min=spec.cmin)
    if spec.smooth:
        kp = torch.cat([k[..., :1], k[..., :-1]], -1)
        kn = torch.cat([k[..., 1:], k[..., -1:]], -1)
        k = (kp * third + k * third) + kn * third
    r = (k * dts) / h2
    N = r.shape[-1]
    eps = torch.tensor(spec.eps, dtype=R, device=base.device)
    dn, cst = [], []
    for i in range(N):
        ri = r[..., i]
        b = one + ri if i in (0, N - 1) else one + two * ri
        d = b + eps if i == 0 else (b - (-ri) * cst[i - 1]) + eps
        dn.append(d)
        cst.append((-ri) / d if i < N - 1 else torch.zeros_like(d))
    return r, dn, cst


def _sweep(x, r, dn, cst):
    """Thomas solve of every line of x [B][C][line][i] (oracle sweep_plane)."""
    import torch
    N = x.shape[-1]
    ds = [x[..., 0] / dn[0]]
    for i in range(1, N):
        ds.append((x[..., i] - (-r[..., i]) * ds[i - 1]) / dn[i])
    out = [None] * N
    out[N - 1] = ds[N - 1]
    for i in range(N - 2, -1, -1):
        out[i] = ds[i] - cst[i] * out[i + 1]
    return torch.stack(out, -1)


def _chan(M, u):
    """u[c] <- sum_d M[c][d] u[d], summed over d in order (oracle chan_apply)."""
    acc = None
    for d in range(M.shape[0]):
        pr = M[:, d, None, None] * u[:, d:d + 1]
        acc = pr if acc is None else acc + pr
    return acc


def forward(spec, u, ab, bb, atc, btc, chan=None, skipw=None):
    """The layer on torch tensors [B][C][N][N] (maps [C][N][N]); differentiable in every argument."""
    import torch
    R = u.dtype
    cur = u
    tabs = []
    for axis, t, dts, h in _schedule(spec):
        base, tc = (ab, atc) if axis == 0 else (bb, btc)
        if axis == 1:   # line coordinates: lines along H
            base, tc = base.transpose(-1, -2), tc.transpose(-1, -2)
        tabs.append((axis,) + _tables(spec, base, tc, torch.tensor(t, dtype=R, device=u.device),
                                      torch.tensor(dts, dtype=R, device=u.device),
                                      torch.tensor(h * h, dtype=R, device=u.device)))
    sps = 2 if spec.lie else 3
    for step in range(spec.steps):
        if spec.chan_op == 1:
            cur = _chan(chan, cur)
        for k in range(sps):
            axis, r, dn, cst = tabs[step * sps + k]
            if axis == 0:
                cur = _sweep(cur, r, dn, cst)
            else:
                cur = _sweep(cur.transpose(-1, -2), r, dn, cst).transpose(-1, -2)
        if spec.chan_op == 2:
            cur = _chan(chan, cur)
    if spec.skip:
        one = torch.tensor(1.0, dtype=R, device=u.device)
        sig = one / (one + torch.exp(-skipw))
        cur = sig * u + (one - sig) * cur
    return cur


def run(c: K.Case, params=None, io=None, dtype=np.float64, need_gin=True, device="cpu") -> Dict[str, np.ndarray]:
    """Output and gradients of sum(gout * y), keyed like runners.run_oracle (gradients as float64 arrays)."""
    import torch
    params = params if params is not None else K.make_params(c)
    u_np, g_np = io if io is not None else K.make_io(c)
    spec = runners.oracle_spec(c)
    t = lambda a: torch.tensor(np.asarray(a).astype(dtype), device=device)   # noqa: E731
    shp = (spec.C, spec.N, spec.N)
    P = {k: t(params[k]).reshape(shp).requires_grad_(True) for k in MAP_KEYS}
    ck = "channel_mixing" if "channel_mixing" in params else ("channel_coupling" if "channel_coupling" in params else None)
    chan = t(params[ck]).requires_grad_(True) if ck else None
    skipw = t(params["skip_weight"]).reshape(()).requires_grad_(True) if "skip_weight" in params else None
    u = t(u_np).requires_grad_(need_gin)
    g = t(g_np)
    y = forward(spec, u, P["alpha_base"], P["beta_base"], P["alpha_time_coeff"], P["beta_time_coeff"], chan, skipw)
    wrt = [P[k] for k in MAP_KEYS] + ([chan] if ck else []) + ([skipw] if skipw is not None else []) + ([u] if need_gin else [])
    # zero steps: the maps are unused (and without skip weight or grad_input, so is everything else)
    grads = torch.autograd.grad(y, wrt, grad_outputs=g, allow_unused=True) if y.requires_grad else [None] * len(wrt)
    grads = [torch.zeros_like(w) if gr is None else gr for w, gr in zip(wrt, grads)]
    out = {"y": y.detach().cpu().numpy().astype(dtype)}
    shp_param = np.asarray(params["alpha_base"]).shape
    for k, gr in zip(MAP_KEYS, grads):
        out["g_" + k] = gr.detach().cpu().numpy().astype(np.float64).reshape(shp_param)
    i = 4
    if ck:
        out["g_" + ck] = grads[i].detach().cpu().numpy().astype(np.float64)
        i += 1
    if skipw is not None:
        out["g_skip_weight"] = grads[i].detach().cpu().numpy().astype(np.float64).reshape(())
        i += 1
    out["gin"] = grads[i].detach().cpu().numpy().astype(dtype) if need_gin else None
    return out
