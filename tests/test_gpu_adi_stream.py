"""The implicit layers on the streaming kernels (adi_stream.cu, pde_adi_stream_*), on the GPU.

These serve every plane up to 4096 x 4096 at 1 ... 64 channels.  References: the fp32 / fp64 oracle where C <= 8,
tests/adi_reference.py (fp64, autograd, on the GPU) above, with the bar and the cancelling-scalar rule of
test_gpu_wide_channels.py.  Where the shared-memory kernels also serve a descriptor, the two families are called on
it through the raw ABI: outputs must be equal bit for bit.
"""
import ctypes
import os
import subprocess
import sys
from ctypes import byref

import numpy as np
import pytest

from . import adi_reference as AR
from . import cases as K
from . import runners
from .test_gpu_guards import Arena
from .test_gpu_wide_channels import _judge, _tame

pytestmark = pytest.mark.gpu
TOL = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("mnist", "fashion", "svhn", "cifar10", "cifar2")
MAP_KEYS = ("alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff")


def _case(kind, C, N, steps, B, seed=1234, **kw):
    ctor = dict(size=N, num_steps=steps, **kw)
    if kind in ("svhn", "cifar10", "cifar2"):
        ctor["channels"] = C
    else:
        assert C == 1
    return K.case(f"stream_{kind}_c{C}_n{N}_s{steps}_b{B}", kind, B=B, seed=seed, **ctor)


def _route(c):
    from cnn_with_pde_b200 import functional as F
    return F.adi_route(runners.make_cuda_layer(c)._config())


def _check_module(c, need_gin=True):
    params = _tame(c, K.make_params(c))
    io = K.make_io(c)
    got = runners.run_cuda(c, params=params, io=io, need_gin=need_gin)
    _judge(got, c, params, io, need_gin, c.name)


# ------------------------------------------------------------------------------------------------------------
# raw ABI
# ------------------------------------------------------------------------------------------------------------
def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream_abi(cfg, u, g, maps, chan=None, skw=None, need_gin=True, take=None, ws_delta=0):
    """pde_adi_stream_forward + _backward on buffers sized by the queries; returns (rc_fwd, rc_bwd, out, gin, gm,
    gchan, gskip).  take(nbytes, shape=None) allocates (torch by default, an Arena for guard-band checks)."""
    import torch
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    B, C, N = u.shape[0], cfg.C, cfg.N
    d = cfg.desc(B, 0)
    sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
    nf = L.pde_adi_stream_forward_workspace_bytes(byref(d))
    nb = L.pde_adi_stream_backward_workspace_bytes(byref(d))
    assert nf > 0 and nb > 0
    if take is None:
        take = lambda n, shape=None: torch.empty(max(int(n), 1), dtype=torch.uint8, device="cuda") if shape is None \
            else torch.empty(shape, device="cuda")   # noqa: E731
    wf, wb = take(nf), take(nb)
    out = take(4 * u.numel(), tuple(u.shape))
    gin = take(4 * u.numel(), tuple(u.shape)) if need_gin else None
    gm = [take(4 * C * N * N, (C, N, N)) for _ in range(4)]
    gchan = take(4 * C * C, (C, C)) if chan is not None else None
    gskip = take(4, ()) if skw is not None else None
    st = torch.cuda.current_stream().cuda_stream
    rf = L.pde_adi_stream_forward(byref(d), byref(sched), *[_ptr(m) for m in maps], _ptr(u), _ptr(chan), _ptr(skw),
                                  _ptr(out), _ptr(wf), nf + ws_delta, st)
    rb = L.pde_adi_stream_backward(byref(d), byref(sched), *[_ptr(m) for m in maps], _ptr(u), _ptr(g), _ptr(chan),
                                   _ptr(skw), _ptr(gin), *[_ptr(m) for m in gm], _ptr(gchan), _ptr(gskip), _ptr(wb),
                                   nb + ws_delta, st)
    torch.cuda.synchronize()
    return rf, rb, out, gin, gm, gchan, gskip


def _tables_abi(cfg, u, g, maps, chan=None, skw=None, need_gin=True):
    from .test_gpu_wide_channels import _abi_call
    return _abi_call(cfg, u, g, maps, chan, skw, need_gin)


def _layer_inputs(c, params):
    """cfg and the parameter tensors of a case's module, for raw ABI calls."""
    import torch
    layer = runners.make_cuda_layer(c, params)
    cfg = layer._config()
    p = dict(layer.named_parameters())
    maps = [p[k].detach().contiguous() for k in MAP_KEYS]
    ck = "channel_mixing" if "channel_mixing" in p else ("channel_coupling" if "channel_coupling" in p else None)
    chan = p[ck].detach().contiguous() if ck else None
    skw = p["skip_weight"].detach().reshape(1).contiguous() if "skip_weight" in p else None
    u, g = (torch.from_numpy(a).cuda() for a in K.make_io(c))
    return cfg, maps, ck, chan, skw, u, g, layer


def _run_stream(c, params, need_gin):
    cfg, maps, ck, chan, skw, u, g, layer = _layer_inputs(c, params)
    rf, rb, out, gin, gm, gchan, gskip = _stream_abi(cfg, u, g, maps, chan, skw, need_gin)
    assert rf == 0 and rb == 0, (rf, rb)
    shp = tuple(layer.alpha_base.shape)
    got = {"y": out.cpu().numpy(), "gin": gin.cpu().numpy() if need_gin else None}
    for k, m in zip(MAP_KEYS, gm):
        got["g_" + k] = m.reshape(shp).cpu().numpy()
    if ck:
        got["g_" + ck] = gchan.cpu().numpy()
    if skw is not None:
        got["g_skip_weight"] = gskip.reshape(()).cpu().numpy()
    return got


# ------------------------------------------------------------------------------------------------------------
# both sides of every boundary of the shared-memory kernels, through the modules
# ------------------------------------------------------------------------------------------------------------
def _boundary_cases():
    pairs = [(1, 128), (1, 129), (3, 128), (3, 129), (4, 96), (4, 97), (4, 100), (4, 128), (12, 64), (13, 64),
             (5, 101), (5, 102), (48, 32), (49, 32), (63, 28), (64, 28)]
    out, i = [], 0
    for C, N in pairs:
        kinds = ("mnist", "fashion", "cifar10", "cifar2", "svhn") if C == 1 else ("cifar10", "cifar2", "svhn")
        for kind in kinds:
            if C == 1 and kind in ("cifar10", "cifar2", "svhn"):
                continue
            out.append((_case(kind, C, N, 2, 2, seed=700 + i), i % 2 == 0))
            i += 1
        if C == 1:   # the channel-aware layers at one channel too
            for kind in ("cifar10", "svhn"):
                out.append((_case(kind, 1, N, 2, 2, seed=700 + i), i % 2 == 1))
                i += 1
    return out


@pytest.mark.parametrize("c,need_gin", _boundary_cases(), ids=lambda v: v.name if hasattr(v, "name") else f"gin{int(v)}")
def test_boundaries_through_the_modules(c, need_gin):
    import cnn_with_pde_b200 as P
    L = P._cabi.lib()
    cfg = runners.make_cuda_layer(c)._config()
    served = L.pde_adi_tables_bytes(byref(cfg.desc(c.B))) > 0
    assert _route(c) == ("tables" if served else "stream")
    _check_module(c, need_gin)
    _check_module(c, not need_gin)


# ------------------------------------------------------------------------------------------------------------
# shared ground: both families on the same descriptor
# ------------------------------------------------------------------------------------------------------------
SHARED = [("mnist", 1, 7, 2), ("mnist", 1, 48, 1), ("cifar10", 3, 64, 1), ("cifar2", 3, 128, 1), ("svhn", 12, 64, 1),
          ("cifar10", 8, 32, 1), ("svhn", 3, 30, 3)]


@pytest.mark.parametrize("kind,C,N,B", SHARED, ids=[f"{k}_c{c}_n{n}_b{b}" for k, c, n, b in SHARED])
def test_outputs_equal_the_shared_memory_kernels_bit_for_bit(kind, C, N, B):
    import torch
    c = _case(kind, C, N, 3, B, seed=31 + C + N)
    params = _tame(c, K.make_params(c))
    cfg, maps, ck, chan, skw, u, g, _ = _layer_inputs(c, params)
    out_t, gin_t, gm_t, gch_t, gsk_t = _tables_abi(cfg, u, g, maps, chan, skw)
    rf, rb, out_s, gin_s, gm_s, gch_s, gsk_s = _stream_abi(cfg, u, g, maps, chan, skw)
    assert rf == 0 and rb == 0
    assert torch.equal(out_t, out_s), float((out_t - out_s).abs().max())
    pairs = [(gin_t, gin_s)] + list(zip(gm_t, gm_s))
    for a, b in pairs:
        a, b = a.cpu().numpy(), b.cpu().numpy()
        assert max(runners.rel_l2(b, a), runners.rel_max(b, a)) <= TOL
    print(f"{kind} C={C} N={N}: grad_input bit-identical: {bool(torch.equal(gin_t, gin_s))}")


# ------------------------------------------------------------------------------------------------------------
# large planes
# ------------------------------------------------------------------------------------------------------------
LARGE = [("mnist", 1, 224, 10, 1), ("cifar10", 3, 227, 10, 1), ("mnist", 1, 512, 1, 2), ("svhn", 3, 1000, 1, 1)]


@pytest.mark.parametrize("kind,C,N,steps,B", LARGE, ids=[f"{k}_c{c}_n{n}_s{s}" for k, c, n, s, _ in LARGE])
def test_large_planes_match_the_references(kind, C, N, steps, B):
    c = _case(kind, C, N, steps, B, seed=N)
    assert _route(c) == "stream"
    _check_module(c)


def _against_fp64_reference(c, need_gin=True):
    """Module vs tests/adi_reference.py in fp64 on the GPU (y, gin and the four maps at the 1e-5 bar)."""
    params = _tame(c, K.make_params(c))
    io = K.make_io(c)
    got = runners.run_cuda(c, params=params, io=io, need_gin=need_gin)
    want = AR.run(c, params=params, io=io, dtype=np.float64, need_gin=need_gin, device="cuda")
    keys = ["y"] + (["gin"] if need_gin else []) + ["g_" + k for k in MAP_KEYS]
    errs = runners.compare({k: got[k] for k in keys}, {k: want[k] for k in keys})
    assert max(errs.values()) <= TOL, (c.name, errs)


@pytest.mark.parametrize("C", (1, 3))
def test_4096_planes_forward_and_backward(C):
    c = _case("mnist" if C == 1 else "cifar10", C, 4096, 1, 1, seed=4096 + C)
    assert _route(c) == "stream"
    _against_fp64_reference(c)


@pytest.mark.parametrize("kind,C,N", [("cifar10", 64, 56), ("svhn", 64, 56), ("cifar10", 16, 112), ("svhn", 16, 112)])
def test_feature_maps_with_channel_ops(kind, C, N):
    c = _case(kind, C, N, 2, 2, seed=C * N)
    assert _route(c) == "stream"
    _check_module(c)


@pytest.mark.parametrize("kind,steps", [("mnist", 64), ("cifar2", 96)])
def test_full_schedules_above_128(kind, steps):
    import cnn_with_pde_b200 as P
    c = _case(kind, 1, 130, steps, 1, seed=steps, dt=0.0005)
    cfg = runners.make_cuda_layer(c)._config()
    assert cfg.steps * (2 if cfg.lie else 3) == P._cabi.MAX_SWEEPS
    _check_module(c)


def test_seeded_random_sweep():
    rs = np.random.RandomState(20261021)
    for i in range(30):
        N = int(rs.randint(2, 601))
        cmax = max(1, min(64, (1 << 19) // (N * N)))
        C = int(rs.randint(1, cmax + 1))
        kind = ("cifar10", "cifar2", "svhn")[rs.randint(3)]
        steps, B, need_gin = int(rs.randint(0, 6)), int(rs.randint(1, 5)), bool(rs.randint(2))
        c = _case(kind, C, N, steps, B, seed=9100 + i)
        params = _tame(c, K.make_params(c))
        got = _run_stream(c, params, need_gin)
        _judge(got, c, params, K.make_io(c), need_gin, c.name)


# ------------------------------------------------------------------------------------------------------------
# workspace and memory safety
# ------------------------------------------------------------------------------------------------------------
def _rand_layer(C, N, steps, B, seed, **kw):
    import torch
    import cnn_with_pde_b200 as P
    gen = torch.Generator(device="cuda").manual_seed(seed)
    cfg = P.AdiConfig(N=N, C=C, steps=steps, dt=0.2, hx=1.0, hy=1.0, **kw)
    u = torch.randn(B, C, N, N, device="cuda", generator=gen)
    g = torch.randn(B, C, N, N, device="cuda", generator=gen)
    maps = [1.0 + 0.5 * torch.rand(C, N, N, device="cuda", generator=gen) for _ in range(2)] + \
           [0.3 * torch.randn(C, N, N, device="cuda", generator=gen) for _ in range(2)]
    chan = torch.eye(C, device="cuda") + 0.1 * torch.randn(C, C, device="cuda", generator=gen) if cfg.chan_op else None
    skw = torch.full((1,), 0.3, device="cuda") if cfg.skip else None
    return cfg, u, g, maps, chan, skw


def test_batch_in_several_chunks_equals_single_sample_calls():
    """16 x 1024^2 at 10 steps: 940 MB a sample, so a batch of three runs one sample at a time."""
    import torch
    import cnn_with_pde_b200 as P
    cfg, u, g, maps, chan, skw = _rand_layer(16, 1024, 10, 3, 7, chan_op=1)
    d = cfg.desc(3)
    per = (10 + 3 + 1) * 16 * 1024 * 1024 * 4
    assert P._cabi.lib().pde_adi_stream_backward_workspace_bytes(byref(d)) == 512 * 256 + 16 * 16 * 1024 ** 2 + per
    rf, rb, out, gin, gm, gch, _ = _stream_abi(cfg, u, g, maps, chan)
    assert rf == 0 and rb == 0
    acc = [torch.zeros_like(m, dtype=torch.float64) for m in gm] + [torch.zeros_like(gch, dtype=torch.float64)]
    for b in range(3):
        r1 = _stream_abi(cfg, u[b:b + 1].contiguous(), g[b:b + 1].contiguous(), maps, chan)
        assert torch.equal(out[b:b + 1], r1[2]) and torch.equal(gin[b:b + 1], r1[3])
        for a, x in zip(acc, r1[4] + [r1[5]]):
            a += x.double()
    for a, x in zip(acc, gm + [gch]):
        assert max(runners.rel_l2(x.cpu().numpy(), a.cpu().numpy()), runners.rel_max(x.cpu().numpy(), a.cpu().numpy())) <= TOL


def test_workspace_exactly_as_queried():
    import cnn_with_pde_b200 as P
    cfg, u, g, maps, chan, skw = _rand_layer(5, 150, 2, 2, 8, chan_op=2, skip=True, smooth=True)
    assert _stream_abi(cfg, u, g, maps, chan, skw)[:2] == (0, 0)
    assert _stream_abi(cfg, u, g, maps, chan, skw, ws_delta=-1)[:2] == (P._cabi.ERR_WORKSPACE, P._cabi.ERR_WORKSPACE)


@pytest.mark.parametrize("C,N,kw", [(1, 131, dict(smooth=True)), (3, 200, dict(chan_op=1)), (7, 129, dict(chan_op=2, skip=True)),
                                    (4, 97, dict(lie=True, has_max=True))])
def test_guard_bands(C, N, kw):
    import torch
    cfg, u, g, maps, chan, skw = _rand_layer(C, N, 2, 3, 9, **kw)
    cnn = C * N * N
    arena = Arena(64 * cnn * 4 + 64 * (1 << 20) + 3 * 16 * cnn * 4 + 20 * cnn * 4 * 3)
    put = lambda t: (lambda a: (a.copy_(t), a)[1])(arena.take(t.numel() * 4, torch.float32, tuple(t.shape)))   # noqa: E731
    ua, ga = put(u), put(g)
    mapsa = [put(m) for m in maps]
    chana = put(chan) if chan is not None else None
    skwa = put(skw) if skw is not None else None
    rf, rb, out, gin, gm, gch, gsk = _stream_abi(cfg, ua, ga, mapsa, chana, skwa, take=lambda n, shape=None:
                                                 arena.take(n) if shape is None else arena.take(n, torch.float32, shape))
    assert rf == 0 and rb == 0
    arena.check(f"stream C={C} N={N} {kw}")
    ref = _stream_abi(cfg, u, g, maps, chan, skw)
    assert torch.equal(out, ref[2]) and torch.equal(gin, ref[3])
    assert all(torch.equal(a, b) for a, b in zip(gm, ref[4]))


def test_unaligned_batch_views():
    """x[1:] of odd planes is 4-byte aligned only; the results equal those of a contiguous copy bit for bit."""
    import torch
    import cnn_with_pde_b200 as P
    for kind, C, N in (("mnist", 1, 131), ("svhn", 3, 129)):
        c = _case(kind, C, N, 2, 3)
        layer = runners.make_cuda_layer(c)
        x = torch.from_numpy(K.make_io(c)[0]).cuda()
        v = x[1:]
        assert v.data_ptr() % 16 != 0
        assert torch.equal(layer(v), layer(v.contiguous()))


def test_forward_beyond_2_31_cells_equals_single_sample_calls():
    import torch
    cfg, _, _, maps, _, _ = _rand_layer(33, 4096, 1, 1, 10)
    B = 4
    assert B * 33 * 4096 * 4096 > 2 ** 31
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    gen = torch.Generator(device="cuda").manual_seed(11)
    u = torch.randn(B, 33, 4096, 4096, device="cuda", generator=gen)
    sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
    st = torch.cuda.current_stream().cuda_stream

    def fwd(x):
        d = cfg.desc(x.shape[0])
        n = L.pde_adi_stream_forward_workspace_bytes(byref(d))
        ws = torch.empty(n, dtype=torch.uint8, device="cuda")
        out = torch.empty_like(x)
        P._cabi.check(L.pde_adi_stream_forward(byref(d), byref(sched), *[m.data_ptr() for m in maps], x.data_ptr(), None,
                                               None, out.data_ptr(), ws.data_ptr(), n, st), "stream forward")
        return out

    out = fwd(u)
    for b in range(B):
        assert torch.equal(out[b:b + 1], fwd(u[b:b + 1])), b


# ------------------------------------------------------------------------------------------------------------
# behaviour under the modules
# ------------------------------------------------------------------------------------------------------------
def test_gradients_are_reproducible_and_independent_of_grad_input():
    import torch
    c = _case("svhn", 6, 150, 3, 3, seed=5)
    layer = runners.make_cuda_layer(c)
    u = torch.from_numpy(K.make_io(c)[0]).cuda()
    grads = []
    for need_gin in (True, True, False):
        layer.zero_grad()
        x = u.clone().requires_grad_(need_gin)
        layer(x).square().sum().backward()
        grads.append([p.grad.clone() for p in layer.parameters()])
    for other in grads[1:]:
        assert all(torch.equal(a, b) for a, b in zip(grads[0], other))


def test_empty_batch_zeroes_the_gradients():
    import torch
    c = _case("svhn", 3, 200, 2, 1)
    layer = runners.make_cuda_layer(c)
    x = torch.zeros(0, 3, 200, 200, device="cuda", requires_grad=True)
    y = layer(x)
    assert y.shape == x.shape
    y.sum().backward()
    for p in layer.parameters():
        assert p.grad is not None and int(torch.count_nonzero(p.grad)) == 0


def _five_modules(N):
    import cnn_with_pde_b200 as P
    return [P.mnist_test.DiffusionLayer(size=N), P.fashion_mnist.DiffusionLayer(size=N),
            P.SVHN.DiffusionLayer(size=N, channels=3), P.cifar10.EnhancedDiffusionLayer(size=N, channels=4),
            P.cifar_2version.LearnableDiffusionLayer(size=N, channels=3)]


def test_drop_in_modules_on_side_streams_no_grad_and_autocast():
    import torch
    for layer in _five_modules(224):
        layer = layer.cuda()
        C = layer.alpha_base.shape[0] if layer.alpha_base.dim() == 3 else 1
        x = torch.randn(2, C, 224, 224, device="cuda", requires_grad=True)
        y = layer(x)
        y.square().sum().backward()
        g = [p.grad.clone() for p in layer.parameters()] + [x.grad.clone()]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            layer.zero_grad()
            x2 = x.detach().clone().requires_grad_(True)
            y2 = layer(x2)
            y2.square().sum().backward()
        torch.cuda.current_stream().wait_stream(s)
        assert torch.equal(y, y2)
        assert all(torch.equal(a, b) for a, b in zip(g, [p.grad for p in layer.parameters()] + [x2.grad]))
        with torch.no_grad():
            assert torch.equal(layer(x), y)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            assert torch.equal(layer(x.detach()), y.detach())


def test_multiscale_extractor_at_224_fused_and_streams():
    import torch
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.classifiers import MultiScaleExtractor
    torch.manual_seed(0)
    m = MultiScaleExtractor(input_size=224).cuda()
    x = torch.randn(2, 3, 224, 224, device="cuda", requires_grad=True)
    res = []
    for fused in (False, True):
        m.fused_branches = fused
        m.zero_grad()
        x.grad = None
        ys = m(x)   # (combined, feature of each branch)
        ys[0].square().sum().backward()
        torch.cuda.synchronize()
        res.append([y.detach() for y in ys] + [p.grad.clone() for p in m.parameters() if p.grad is not None] +
                   [x.grad.clone()])
    # the PDE outputs come from the same kernels either way; the gradients are sums over the three branches whose
    # order follows the streams' schedule, so they agree to the fp32 summation order
    assert len(res[0]) == len(res[1])
    n_out = 4
    assert all(torch.equal(a, b) for a, b in zip(res[0][:n_out], res[1][:n_out]))
    for a, b in zip(res[0][n_out:], res[1][n_out:]):
        a, b = a.cpu().double().numpy(), b.cpu().double().numpy()
        assert max(runners.rel_l2(b, a), runners.rel_max(b, a)) <= TOL


def test_cuda_graph_training_step_equals_eager():
    import torch
    c = _case("cifar10", 3, 160, 2, 2, seed=3)
    layer = runners.make_cuda_layer(c)
    x = torch.from_numpy(K.make_io(c)[0]).cuda()

    def step():
        layer.zero_grad(set_to_none=False)
        y = layer(x)
        y.square().sum().backward()
        return y

    y_eager = step().detach().clone()
    g_eager = [p.grad.clone() for p in layer.parameters()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y_g = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_g, y_eager)
    assert all(torch.equal(a, p.grad) for a, p in zip(g_eager, layer.parameters()))


def test_debug_prints_the_stream_plans():
    code = ("import torch, cnn_with_pde_b200 as P\n"
            "m = P.mnist_test.DiffusionLayer(size=200).cuda()\n"
            "x = torch.randn(2, 1, 200, 200, device='cuda', requires_grad=True)\n"
            "m(x).sum().backward(); torch.cuda.synchronize()\n")
    env = dict(os.environ, PDE_B200_DEBUG="1")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "stream fwd plan" in r.stderr and "stream bwd plan" in r.stderr, r.stderr
    assert "ssweep<rows>(regs=" in r.stderr and "sadj<cols>(regs=" in r.stderr
