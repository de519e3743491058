"""The implicit layers with 5 ... 64 channels (adi_wide.cu), on the GPU.

There is no reference fixture with more than four channels, so these layers are tied to the reference two ways:
against the oracle (whose C <= 4 results are pinned to the reference fixtures), and against the already-validated
kernels: a layer whose channel matrix is block-diagonal is two independent narrower layers, and a layer without a
channel op is C single-channel layers.  The oracle's adjoint serves C <= 8; above that the expected values come
from tests/adi_reference.py (the oracle's forward restated in torch, differentiated by autograd, pinned to the
oracle by tests/test_adi_reference.py), and the outputs are also checked against the oracle's forward.

Bar: 1e-5 (max of rel-L2 and max-abs/max-ref) against the fp32 reference, and no further from the fp64 reference
than the fp32 one is, plus 1e-5.  The channel-matrix and skip-weight gradients are cancelling sums (DESIGN.md
section 2): where they miss the plain bar they are held to the ill-conditioned-scalar rule (within 3x the fp32
reference's own distance from fp64, plus 1e-5).
"""
import ctypes
from ctypes import byref

import numpy as np
import pytest

from . import adi_reference as AR
from . import cases as K
from . import runners
from .test_gpu_guards import Arena, _adi_case

pytestmark = pytest.mark.gpu
TOL = 1e-5
SCALARS = {"g_skip_weight", "g_channel_mixing", "g_channel_coupling"}
KINDS = ("cifar10", "cifar2", "svhn")   # Strang + pre-step mix, Lie + pre-step mix, smoothing + coupling + skip


def _case(kind, C, N, steps, B, seed=1234, **kw):
    return K.case(f"wide_{kind}_c{C}_n{N}_s{steps}_b{B}", kind, B=B, seed=seed, size=N, channels=C, num_steps=steps, **kw)


def _tame(c, params, gain=0.2):
    """Channel matrices I + gain / sqrt(C) * randn: long runs stay O(1) whatever C (make_params uses 0.2 randn)."""
    rs = np.random.RandomState(c.seed + 99)
    C = c.shape[0]
    for k in ("channel_mixing", "channel_coupling"):
        if k in params:
            params[k] = (np.eye(C) + gain / np.sqrt(C) * rs.randn(C, C)).astype(np.float32)
    return params


ORACLE_MAX_C = 8   # the oracle's adjoint holds the channel-matrix gradient in an 8 x 8 array


def _expected(c, params, io, need_gin, dtype, nthreads=0):
    if c.shape[0] <= ORACLE_MAX_C:
        return runners.run_oracle(c, params=params, io=io, dtype=dtype, need_gin=need_gin, nthreads=nthreads)
    want = AR.run(c, params=params, io=io, dtype=dtype, need_gin=need_gin, device="cuda")
    if dtype == np.float32:   # and the outputs against the oracle's forward, which takes any C
        y = runners.run_oracle(c, params=params, io=io, dtype=np.float32, forward_only=True)["y"]
        e = runners.compare({"y": want["y"]}, {"y": y})["y"]
        assert e <= TOL, (c.name, "reference vs oracle forward", e)
    return want


def _judge(got, c, params, io, need_gin, what, nthreads=0):
    """Returns the error of every key against the fp32 reference."""
    want32 = _expected(c, params, io, need_gin, np.float32, nthreads)
    want64 = _expected(c, params, io, need_gin, np.float64, nthreads)
    got = {k: v for k, v in got.items() if v is not None}
    want32 = {k: want32[k] for k in got}
    errs = runners.compare(got, want32)
    assert set(errs) == set(got), (what, sorted(errs), sorted(got))
    e64, r64 = runners.compare(got, want64), runners.compare(want32, want64)
    for k in errs:
        if errs[k] <= TOL:
            assert e64[k] <= r64[k] + TOL, (what, k, e64[k], r64[k])
        else:
            assert k in SCALARS, (what, k, errs[k])
            assert e64[k] <= 3.0 * r64[k] + TOL, (what, k, errs[k], e64[k], r64[k])
    return errs


def _check(c, params=None, need_gin=True):
    params = params if params is not None else _tame(c, K.make_params(c))
    io = K.make_io(c)
    got = runners.run_cuda(c, params=params, io=io, need_gin=need_gin)
    _judge(got, c, params, io, need_gin, c.name)


def _named_cases():
    """Every C in {5, 6, 8, 12, 16, 32, 48} with every edge in {8, 16, 28, 31, 32} (and 64 at C = 12); the
    variant, step count (0 ... 3), odd batch and grad_input cycle so that each appears with each C."""
    out, i = [], 0
    pairs = [(C, N) for C in (5, 6, 8, 12, 16, 32, 48) for N in (8, 16, 28, 31, 32)] + [(12, 64)]
    for C, N in pairs:
        out.append((_case(KINDS[i % 3], C, N, i % 4, (1, 3, 5, 7)[(i // 3) % 4], seed=500 + i), i % 5 != 4))
        i += 1
    return out


@pytest.mark.parametrize("c,need_gin", _named_cases(), ids=lambda v: v.name if hasattr(v, "name") else f"gin{int(v)}")
def test_wide_layers_match_the_references(c, need_gin):
    _check(c, need_gin=need_gin)


def test_seeded_random_sweep():
    rs = np.random.RandomState(20261020)
    for i in range(40):
        kind = KINDS[rs.randint(3)]
        N = int(rs.randint(2, 65))
        cmax = min(64, (200 * 1024) // (N * (N | 1) * 4))
        if cmax < 5:
            continue
        C = int(rs.randint(5, cmax + 1))
        steps = int(rs.randint(0, 5))
        B = int(rs.randint(1, 10))
        _check(_case(kind, C, N, steps, B, seed=9000 + i), need_gin=bool(rs.randint(2)))


# ------------------------------------------------------------------------------------------------------------
# against the already-validated kernels
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ("cifar10", "svhn"))
def test_block_diagonal_layer_is_two_three_channel_layers(kind):
    """C = 6 with M = blockdiag(M1, M2) at 32 x 32 against two C = 3 layers on the half-line kernels."""
    c6 = _case(kind, 6, 32, 3, 9, seed=77)
    p6 = K.make_params(c6)
    mk = "channel_mixing" if kind == "cifar10" else "channel_coupling"
    M = p6[mk].copy()
    M[:3, 3:] = 0.0
    M[3:, :3] = 0.0
    p6[mk] = M
    u, g = K.make_io(c6)
    got6 = runners.run_cuda(c6, params=p6, io=(u, g))
    c3 = _case(kind, 3, 32, 3, 9, seed=77)
    for h, sl in enumerate((slice(0, 3), slice(3, 6))):
        p3 = {k: (v[sl] if np.ndim(v) == 3 else v) for k, v in p6.items()}
        p3[mk] = M[sl, sl].copy()
        got3 = runners.run_cuda(c3, params=p3, io=(np.ascontiguousarray(u[:, sl]), np.ascontiguousarray(g[:, sl])))
        part = {"y": got6["y"][:, sl], "gin": got6["gin"][:, sl], "g_" + mk: got6["g_" + mk][sl, sl]}
        for k in ("alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff"):
            part["g_" + k] = got6["g_" + k][sl]
        errs = runners.compare(part, {k: got3[k] for k in part})
        assert max(errs.values()) <= TOL, (kind, h, errs)


def _abi_call(cfg, u, g, maps, chan=None, skw=None, need_gin=True, arena=None):
    """prepare + forward_train + backward through ctypes on buffers sized by the ABI's queries: torch allocations,
    or pieces of `arena` (test_gpu_guards.Arena: poisoned guard bands around every buffer)."""
    import torch
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    B, C, N = u.shape[0], cfg.C, cfg.N
    d = cfg.desc(B, 0)
    sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
    nt, nck = L.pde_adi_tables_bytes(byref(d)), L.pde_adi_checkpoint_bytes(byref(d))
    nws = L.pde_adi_backward_saved_workspace_bytes(byref(d)) if nck else L.pde_adi_backward_workspace_bytes(byref(d))
    assert nt > 0 and nws > 0
    if arena is None:
        take = lambda n, shape=None: torch.empty(max(int(n), 1), dtype=torch.uint8, device="cuda") if shape is None \
            else torch.empty(shape, device="cuda")   # noqa: E731
    else:
        take = lambda n, shape=None: arena.take(n) if shape is None else arena.take(n, torch.float32, shape)   # noqa: E731
    tables, ckpt, ws = take(nt), (take(nck) if nck else None), take(nws)
    out = take(4 * u.numel(), tuple(u.shape))
    gin = take(4 * u.numel(), tuple(u.shape)) if need_gin else None
    gm = [take(4 * C * N * N, (C, N, N)) for _ in range(4)]
    gchan = take(4 * C * C, (C, C)) if chan is not None else None
    gskip = take(4, ()) if skw is not None else None
    st = torch.cuda.current_stream().cuda_stream
    p = lambda t: None if t is None else t.data_ptr()   # noqa: E731
    P._cabi.check(L.pde_adi_prepare(byref(d), byref(sched), *[p(m) for m in maps], p(tables), st), "prepare")
    P._cabi.check(L.pde_adi_forward_train(byref(d), p(tables), p(u), p(chan), p(skw), p(out), p(ckpt), st), "forward")
    P._cabi.check(L.pde_adi_backward_saved(byref(d), p(tables), p(u), p(g), p(chan), p(skw), p(ckpt), p(gin), p(gm[0]),
                                           p(gm[1]), p(gm[2]), p(gm[3]), p(gchan), p(gskip), p(ws), nws, st), "backward")
    torch.cuda.synchronize()
    return out, gin, gm, gchan, gskip


def test_eight_channels_without_channel_op_are_eight_single_channel_layers():
    import torch
    import cnn_with_pde_b200 as P
    C, N, B = 8, 32, 6
    gen = torch.Generator(device="cuda").manual_seed(5)
    u = torch.randn(B, C, N, N, device="cuda", generator=gen)
    g = torch.randn(B, C, N, N, device="cuda", generator=gen)
    maps = [1.0 + 0.5 * torch.rand(C, N, N, device="cuda", generator=gen) for _ in range(2)] + \
           [0.3 * torch.randn(C, N, N, device="cuda", generator=gen) for _ in range(2)]
    cfg8 = P.AdiConfig(N=N, C=C, steps=4, dt=0.3, hx=1.0, hy=1.0, smooth=True)
    cfg1 = P.AdiConfig(N=N, C=1, steps=4, dt=0.3, hx=1.0, hy=1.0, smooth=True)
    out8, gin8, gm8, _, _ = _abi_call(cfg8, u, g, maps)
    for c in range(C):
        out1, gin1, gm1, _, _ = _abi_call(cfg1, u[:, c:c + 1].contiguous(), g[:, c:c + 1].contiguous(),
                                          [m[c:c + 1].contiguous() for m in maps])
        pairs = [(out8[:, c:c + 1], out1), (gin8[:, c:c + 1], gin1)] + [(a[c:c + 1], b) for a, b in zip(gm8, gm1)]
        for a, b in pairs:
            e = max(runners.rel_l2(a.cpu().numpy(), b.cpu().numpy()), runners.rel_max(a.cpu().numpy(), b.cpu().numpy()))
            assert e <= TOL, (c, e)


# ------------------------------------------------------------------------------------------------------------
# large batch, grid cap, guard bands
# ------------------------------------------------------------------------------------------------------------
def test_large_batch_every_gradient():
    """C = 16, N = 32, batch 2048: the input (128 MiB) is larger than L2."""
    _check(_case("cifar10", 16, 32, 2, 2048, seed=31))


def test_workspace_cap_shrinks_the_grid():
    """C = 48, N = 32, 64 Strang steps: the sweep history of a sample is 37 MiB, so the 1 GB cap leaves fewer
    slots than samples and blocks loop over samples."""
    import cnn_with_pde_b200 as P
    c = _case("cifar10", 48, 32, 64, 27, seed=41)
    L = P._cabi.lib()
    layer = runners.make_cuda_layer(c)
    d = layer._config().desc(c.B, 0)
    ws = L.pde_adi_backward_workspace_bytes(byref(d))
    per_slot = (4 + 3 * 64 + 64) * 48 * 32 * 32 * 4
    assert 0 < ws <= (1 << 30) + (1 << 20), ws
    assert ws < per_slot * c.B, "the grid was not capped"
    _check(c, params=_tame(c, K.make_params(c), gain=0.02))


def _guarded(c, need_gin):
    """Every buffer from one poisoned arena sized by the ABI's queries; guards intact, results as expected."""
    import torch
    params = _tame(c, K.make_params(c))
    u_np, g_np = K.make_io(c)
    layer = runners.make_cuda_layer(c, params)
    cfg = layer._config()
    C, N = cfg.C, cfg.N
    import cnn_with_pde_b200 as P
    L = P._cabi.lib()
    d = cfg.desc(c.B, 0)
    need = L.pde_adi_tables_bytes(byref(d)) + L.pde_adi_backward_workspace_bytes(byref(d)) + 3 * 4 * c.B * C * N * N + \
        4 * 4 * C * N * N + 4 * C * C + 64 * 1024 + 16 * 4096
    A = Arena(need)
    u, g = torch.from_numpy(u_np).cuda(), torch.from_numpy(g_np).cuda()
    maps = [t.detach().contiguous() for t in (layer.alpha_base, layer.beta_base, layer.alpha_time_coeff, layer.beta_time_coeff)]
    chan = getattr(layer, "channel_mixing", getattr(layer, "channel_coupling", None))
    skw = getattr(layer, "skip_weight", None)
    out, gin, gm, _, _ = _abi_call(cfg, u, g, maps, None if chan is None else chan.detach(),
                                   None if skw is None else skw.detach(), need_gin, arena=A)
    A.check(c.name)
    want = _expected(c, params, (u_np, g_np), need_gin, np.float32)
    got = {"y": out.cpu().numpy(), "gin": gin.cpu().numpy() if need_gin else None}
    for k, t in zip(AR.MAP_KEYS, gm):
        got["g_" + k] = t.cpu().numpy()
    errs = runners.compare(got, {k: want[k] for k in got})
    assert max(errs.values()) <= TOL, (c.name, errs)


def test_kernels_stay_inside_their_buffers():
    # oracle-checked through test_gpu_guards' own helper (C <= 8) ...
    for c, need_gin in ((_case("cifar10", 6, 31, 2, 5), True), (_case("cifar10", 5, 101, 1, 2), True)):
        _adi_case(c, 0, need_gin)
    # ... and the same arena above eight channels (odd planes, all three variants, 64 channels)
    for c, need_gin in ((_case("svhn", 12, 17, 2, 3), True), (_case("cifar2", 48, 32, 1, 3), False),
                        (_case("svhn", 64, 16, 1, 4), True), (_case("cifar10", 9, 7, 2, 5), True)):
        _guarded(c, need_gin)


# ------------------------------------------------------------------------------------------------------------
# module-level behaviour
# ------------------------------------------------------------------------------------------------------------
def _layer_io(c):
    import torch
    layer = runners.make_cuda_layer(c, _tame(c, K.make_params(c)))
    u, g = K.make_io(c)
    return layer, torch.from_numpy(u).cuda(), torch.from_numpy(g).cuda()


def _step(layer, u, g):
    import torch
    layer.zero_grad(set_to_none=True)
    x = u.clone().requires_grad_(True)
    y = layer(x)
    y.backward(g)
    torch.cuda.synchronize()
    return [y.detach().clone(), x.grad.clone()] + [p.grad.clone() for p in layer.parameters()]


def test_bit_reproducible():
    import torch
    for c in (_case("cifar10", 16, 32, 3, 37), _case("svhn", 40, 20, 2, 11)):
        layer, u, g = _layer_io(c)
        a, b = _step(layer, u, g), _step(layer, u, g)
        assert all(torch.equal(x, y) for x, y in zip(a, b)), c.name


def test_empty_batch_zeroes_the_gradients():
    """B = 0 (a rank without samples): the gradient outputs are overwritten with zeros; u / gout / gin may be NULL."""
    import torch
    import cnn_with_pde_b200 as P
    L = P._cabi.lib()
    C, N = 8, 24
    d = P.AdiConfig(N=N, C=C, steps=2, dt=0.01, hx=1.0, hy=1.0, smooth=True, chan_op=2, skip=True).desc(0, 0)
    gm = [torch.full((C, N, N), 7.0, device="cuda") for _ in range(4)]
    gchan, gskip = torch.full((C, C), 7.0, device="cuda"), torch.full((), 7.0, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    rc = L.pde_adi_backward(byref(d), None, None, None, None, None, None, *[t.data_ptr() for t in gm],
                            gchan.data_ptr(), gskip.data_ptr(), None, 0, st)
    assert rc == 0, rc
    torch.cuda.synchronize()
    for t in gm + [gchan, gskip]:
        assert torch.count_nonzero(t) == 0
    # and through the module
    layer, _, _ = _layer_io(_case("svhn", C, N, 2, 1))
    x = torch.zeros(0, C, N, N, device="cuda", requires_grad=True)
    layer(x).sum().backward()
    for p in layer.parameters():
        assert p.grad is None or torch.count_nonzero(p.grad) == 0


def test_multi_branch_entry_points_refuse_wide_layers():
    import cnn_with_pde_b200 as P
    L = P._cabi.lib()
    for B in (0, 4):
        cfgs = [P.AdiConfig(N=32, C=8, steps=s, dt=0.001, hx=1.0, hy=1.0, has_max=True, chan_op=1) for s in (2, 3)]
        descs = (P._cabi.AdiDesc * 2)(*[c.desc(B, 0) for c in cfgs])
        a = ctypes.addressof(descs)
        assert L.pde_adi_multi_prepare(2, a, None, None, None, None, None, None, None) == P._cabi.ERR_UNSUPPORTED, B
        assert L.pde_adi_multi_forward_train(2, a, None, None, None, None, None, None, None) == P._cabi.ERR_UNSUPPORTED, B
        assert L.pde_adi_multi_backward_saved(2, a, *([None] * 16)) == P._cabi.ERR_UNSUPPORTED, B


def test_multiscale_extractor_fused_equals_unfused():
    import torch
    from cnn_with_pde_b200.classifiers import MultiScaleExtractor
    torch.manual_seed(3)
    m = MultiScaleExtractor(input_size=16, channels=8).cuda()
    gen = torch.Generator(device="cuda").manual_seed(4)
    u = torch.randn(5, 8, 16, 16, device="cuda", generator=gen)
    res = []
    for fused in (False, True):
        m.fused_branches = fused
        m.zero_grad(set_to_none=True)
        x = u.clone().requires_grad_(True)
        ys = m(x)   # (combined, feature of each branch)
        sum(y.square().sum() for y in ys).backward()
        torch.cuda.synchronize()
        res.append([y.detach().clone() for y in ys] + [x.grad.clone()] + [p.grad.clone() for p in m.parameters()])
    # the wide layers cannot share a launch: the fused call falls back to one call per layer, so only the
    # gates' cuDNN weight gradients may differ, in summation order
    for a, b in zip(*res):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-7)
    for pde in (m.pde1, m.pde2, m.pde3):
        assert pde.channel_mixing.shape == (8, 8)


def test_graph_captured_step_equals_eager():
    import torch
    layer, u, g = _layer_io(_case("cifar10", 12, 28, 3, 9))
    x = torch.zeros_like(u, requires_grad=True)
    gs = torch.zeros_like(g)

    def step():
        y = layer(x)
        y.backward(gs)
        return y

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    x.grad = None
    layer.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_y = step()
    with torch.no_grad():
        x.copy_(u)
        gs.copy_(g)
    graph.replay()
    torch.cuda.synchronize()
    cap = [static_y.clone(), x.grad.clone()] + [p.grad.clone() for p in layer.parameters()]
    saved = [p.grad for p in layer.parameters()]
    eager = _step(layer, u, g)
    for a, b in zip(cap, eager):
        assert torch.equal(a, b)
    for p, s in zip(layer.parameters(), saved):
        p.grad = s
    del graph


def test_no_grad_and_autocast_match_fp32():
    import torch
    layer, u, g = _layer_io(_case("svhn", 16, 32, 3, 6))
    y = layer(u.clone().requires_grad_(True)).detach()
    with torch.no_grad():
        assert torch.equal(layer(u), y)
    x16 = u.half().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.float16):
        y16 = layer(x16)
    y16.float().backward(g)
    x32 = u.half().float().requires_grad_(True)
    y32 = layer(x32)
    y32.backward(g)
    assert y16.dtype == torch.float32 and torch.equal(y16.detach(), y32.detach())
    assert x16.grad.dtype == torch.float16 and torch.equal(x16.grad, x32.grad.half())
