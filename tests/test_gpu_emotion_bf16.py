"""emotion_recognition.PDELayer on bfloat16 planes (pde_emotion_*_bf16), and a converted module's weights and buffers
read as fp32.

The bf16 contract: planes are widened on load, all arithmetic, weights and weight gradients stay fp32, and every
result is rounded once, to nearest even, on its final store; a descriptor takes the same kernels, grid and chunking in
both dtypes.  So the bf16 layer equals, bit for bit, the fp32 layer on the widened input, rounded to bf16 -- the
output and grad_input -- and its weight gradient equals the fp32 one.  The one exception is the weight gradient of
the whole-plane generic kernels (N <= 64 outside 16 / 32 / 48, and PDE_B200_EMO_TILED=0): they sum it with float
atomics, so two fp32 calls already agree on it only up to the summation order.
"""
import ctypes
from ctypes import byref

import numpy as np
import pytest
import torch

from . import emotion_reference as ER
from . import runners
from .test_gpu_emotion_shapes import _Guarded, _desc

pytestmark = pytest.mark.gpu
DT = 0.001
NAMES = ("alpha_w1", "alpha_w2", "alpha_w3", "beta_w1", "beta_w2", "beta_w3")
TILED = (16, 32, 48)


def _layer(N, Nt, w, dtype=torch.float32):
    from cnn_with_pde_b200.emotion_recognition import PDELayer
    m = PDELayer(Nx=N, Ny=N, dt=DT).cuda()
    m.Nt = Nt
    with torch.no_grad():
        for k, v in zip(NAMES, w):
            getattr(m, k).fill_(float(v))
    return m.to(dtype)


def _pass(m, x, g, need_gin):
    m.zero_grad(set_to_none=True)
    x = x.detach().clone().requires_grad_(need_gin)
    y = m(x)
    y.backward(g)
    torch.cuda.synchronize()
    return y.detach(), (x.grad if need_gin else None), torch.stack([getattr(m, k).grad for k in NAMES])


def _generic(N, env_generic):
    """Whether the whole-plane generic kernels (float atomics in the weight gradient) serve N."""
    return N <= 64 and (env_generic or N not in TILED)


def _check_bits(N, Nt, B, need_gin, seed, env_generic=False, oracle=False):
    """bf16 layer == fp32 layer on the widened input, rounded; the weight gradient equal (generic kernels: up to the
    atomics' summation order)."""
    u, g = ER.make_inputs(B, N, seed=seed)
    w = ER.stable_weights(N, seed)
    m = _layer(N, Nt, w)
    x16 = torch.from_numpy(u).cuda().bfloat16()
    g16 = torch.from_numpy(g).cuda().bfloat16()
    y16, gi16, gw16 = _pass(m, x16, g16, need_gin)
    y32, gi32, gw32 = _pass(m, x16.float(), g16.float(), need_gin)
    what = f"N={N} Nt={Nt} B={B} need_gin={need_gin} generic_env={env_generic}"
    assert y16.dtype == torch.bfloat16 and torch.equal(y16, y32.bfloat16()), what
    if need_gin:
        assert gi16.dtype == torch.bfloat16 and torch.equal(gi16, gi32.bfloat16()), what
    assert gw16.dtype == torch.float32
    if _generic(N, env_generic):
        torch.testing.assert_close(gw16, gw32, rtol=1e-5, atol=1e-6 * float(gw32.abs().max()), msg=what)
    else:
        assert torch.equal(gw16, gw32), (what, (gw16 - gw32).abs().max().item())
    if oracle:   # against the fp32 C oracle on the widened planes
        want = ER.oracle(x16.float().cpu().numpy(), g16.float().cpu().numpy(), w, Nt, need_gin=True, dtype=np.float32)
        err = max(runners.rel_l2(gw16.cpu().numpy(), want["w"]), runners.rel_max(gw16.cpu().numpy(), want["w"]))
        assert err <= 1e-5, (what, "g_w6 vs oracle", err)
        for got, k in ((y16, "y"), (gi16, "gin")):
            if got is None:
                continue
            ref = torch.from_numpy(want[k]).reshape(got.shape)
            # the bf16 value is the oracle's within its rounding: half a bf16 unit plus the fp32 path's own 1e-5
            bound = ref.abs() * (2.0 ** -8 + 1e-5) + 1e-5 * float(ref.abs().max())
            assert bool(((got.float().cpu() - ref).abs() <= bound).all()), (what, k)


# ------------------------------------------------------------------------------ bit identity per route
ROUTE_N = [3, 16, 17, 32, 47, 48, 63, 64, 65, 66, 97, 300]
STEPS = [0, 1, 2, 10, 16]


@pytest.mark.parametrize("N", ROUTE_N)
def test_bits_equal_the_widened_fp32_layer(N):
    from cnn_with_pde_b200._cabi import PdeB200Error
    for i, Nt in enumerate(STEPS):
        B = (3, 5, 7, 1, 6)[(N + i) % 5]
        if N in (63, 64) and Nt == 16:   # fp32 serves the forward and refuses the backward: so does bf16
            m = _layer(N, Nt, ER.stable_weights(N, 1))
            x = torch.randn(B, 1, N, N, device="cuda").bfloat16().requires_grad_()
            y = m(x)
            assert torch.equal(y, m(x.detach().float()).bfloat16())
            with pytest.raises(PdeB200Error, match="unsupported emotion PDELayer"):
                y.backward(torch.ones_like(y))
            continue
        for need_gin in (True, False):
            _check_bits(N, Nt, B, need_gin, seed=N * 100 + Nt, oracle=need_gin and Nt == 10 and N in (3, 48, 97))


@pytest.mark.parametrize("N", [16, 32, 48])
def test_bits_on_the_generic_kernels(N, monkeypatch):
    monkeypatch.setenv("PDE_B200_EMO_TILED", "0")
    for i, Nt in enumerate(STEPS):
        _check_bits(N, Nt, (3, 5, 7, 9, 11)[i], i % 2 == 0, seed=N + Nt, env_generic=True, oracle=Nt == 10)


def test_plane_4096():
    _check_bits(4096, 16, 1, True, seed=4096)


def test_batch_past_the_workspace_cap():
    """B = 130 at 512 x 512, 16 steps: three chunks."""
    _check_bits(512, 16, 130, True, seed=512)


# ------------------------------------------------------------------------------------------- C ABI
def _abi():
    import cnn_with_pde_b200._cabi as cabi
    return cabi, cabi.lib(), torch.cuda.current_stream().cuda_stream


def test_refusals_match_fp32():
    cabi, L, stream = _abi()
    x = torch.zeros(1, 1, 66, 66, device="cuda")
    w = torch.ones(6, device="cuda")
    xs = torch.linspace(0, 1, 66, device="cuda")
    ptr = x.data_ptr()
    for N, Nt in ((4097, 1), (65, 17), (4096, 17), (63, 16), (64, 16), (2, 1)):
        d = _desc(1, N, Nt)
        ws16 = L.pde_emotion_backward_workspace_bytes_bf16(byref(d))
        assert ws16 == L.pde_emotion_backward_workspace_bytes(byref(d)) and (ws16 > 0) == (N in (63, 64)), (N, Nt)
        f32 = L.pde_emotion_forward(byref(d), ptr, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), ptr, stream)
        f16 = L.pde_emotion_forward_bf16(byref(d), ptr, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), ptr, stream)
        b32 = L.pde_emotion_backward(byref(d), ptr, ptr, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), ptr, w.data_ptr(),
                                     ptr, ctypes.c_size_t(1 << 20), stream)
        b16 = L.pde_emotion_backward_bf16(byref(d), ptr, ptr, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), ptr,
                                          w.data_ptr(), ptr, ctypes.c_size_t(1 << 20), stream)
        assert (f16, b16) == (f32, b32), (N, Nt)
        assert b16 == (cabi.ERR_INVALID if N == 2 else cabi.ERR_UNSUPPORTED), (N, Nt)
        assert f16 == (0 if N in (63, 64) else b16), (N, Nt)
    torch.cuda.synchronize()


def test_empty_batch():
    _, L, stream = _abi()
    w = torch.ones(6, device="cuda")
    for N in (17, 48, 65, 224, 4096):
        d = _desc(0, N, 10)
        xs = torch.linspace(0, 1, N, device="cuda")
        assert L.pde_emotion_forward_bf16(byref(d), None, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), None, stream) == 0
        gw = torch.full((6,), 7.0, device="cuda")
        assert L.pde_emotion_backward_bf16(byref(d), None, None, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), None,
                                           gw.data_ptr(), None, ctypes.c_size_t(0), stream) == 0
        assert float(gw.abs().sum()) == 0.0


def _bf16_view(buf):
    return buf.raw[buf.start:buf.start + buf.n].view(torch.bfloat16)


@pytest.mark.parametrize("B,N,Nt", [(2, 65, 1), (3, 100, 10), (1, 227, 16), (2, 130, 0), (3, 48, 10), (5, 40, 3)])
def test_abi_guard_bands_and_workspace(B, N, Nt):
    """bf16 planes 2 bytes past a 256-byte boundary (an odd element offset) inside guard bands; the workspace exactly
    as the bf16 query answers, one byte less refused; the same bits as the module; a plane at an odd byte address
    refused."""
    cabi, L, stream = _abi()
    d = _desc(B, N, Nt)
    ws_bytes = L.pde_emotion_backward_workspace_bytes_bf16(byref(d))
    assert ws_bytes >= L.pde_emotion_backward_workspace_bytes(byref(d)) > 0
    n = B * N * N
    u, g = ER.make_inputs(B, N, seed=n)
    w = ER.stable_weights(N, n)
    u16, g16 = torch.from_numpy(u).cuda().bfloat16(), torch.from_numpy(g).cuda().bfloat16()
    bufs = {k: _Guarded(n * 2, 2) for k in ("u", "g", "out", "gin")}
    _bf16_view(bufs["u"]).copy_(u16.ravel())
    _bf16_view(bufs["g"]).copy_(g16.ravel())
    wt = torch.from_numpy(w).cuda()
    xs = torch.linspace(0, 1, N).cuda()
    assert L.pde_emotion_forward_bf16(byref(d), bufs["u"].ptr, wt.data_ptr(), xs.data_ptr(), xs.data_ptr(),
                                      bufs["out"].ptr, stream) == 0
    ws = _Guarded(ws_bytes, 0)
    gw = _Guarded(6 * 4, 4)
    assert L.pde_emotion_backward_bf16(byref(d), bufs["u"].ptr, bufs["g"].ptr, wt.data_ptr(), xs.data_ptr(),
                                       xs.data_ptr(), bufs["gin"].ptr, gw.ptr, ws.ptr, ctypes.c_size_t(ws_bytes),
                                       stream) == 0
    torch.cuda.synchronize()
    assert ws.guards_intact() and gw.guards_intact() and all(b.guards_intact() for b in bufs.values())
    m = _layer(N, Nt, w)
    y, gi, gwm = _pass(m, u16, g16, True)
    assert torch.equal(_bf16_view(bufs["out"]), y.ravel())
    assert torch.equal(_bf16_view(bufs["gin"]), gi.ravel())
    got_w = gw.view()
    if _generic(N, False):
        torch.testing.assert_close(got_w, gwm, rtol=1e-5, atol=1e-6 * float(gwm.abs().max()))
    else:
        assert torch.equal(got_w, gwm)
    # above 64 the answer is the halo kernels' exact need; up to 64 it is, as in fp32, what the whole-plane kernels
    # need at their largest grid (and with PDE_EMO_TUNE_GENERIC), so those routes are checked at 0 bytes
    short = ws_bytes - 1 if N > 64 else 0
    assert L.pde_emotion_backward_bf16(byref(d), bufs["u"].ptr, bufs["g"].ptr, wt.data_ptr(), xs.data_ptr(),
                                       xs.data_ptr(), bufs["gin"].ptr, gw.ptr, ws.ptr, ctypes.c_size_t(short),
                                       stream) == cabi.ERR_WORKSPACE
    odd = bufs["u"].ptr + 1
    assert L.pde_emotion_forward_bf16(byref(d), odd, wt.data_ptr(), xs.data_ptr(), xs.data_ptr(), bufs["out"].ptr,
                                      stream) == cabi.ERR_INVALID
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ modules
@pytest.mark.parametrize("N", [48, 96])
def test_bf16_module_grads_are_the_fp32_ones_rounded(N):
    torch.manual_seed(N)
    w = ER.stable_weights(N, 3)
    m16 = _layer(N, 10, w, torch.bfloat16)
    # the fp32 twin holds the bf16 module's weights and buffers widened
    m32 = _layer(N, 10, w)
    with torch.no_grad():
        for (_, p32), (_, p16) in zip(m32.named_parameters(), m16.named_parameters()):
            p32.copy_(p16.float())
        m32.x.copy_(m16.x.float())
        m32.y.copy_(m16.y.float())
    x = torch.randn(5, 1, N, N, device="cuda").bfloat16()
    g = torch.randn(5, 1, N, N, device="cuda").bfloat16()
    y16, gi16, _ = _pass(m16, x, g, True)
    y32, gi32, _ = _pass(m32, x.float(), g.float(), True)
    assert y16.dtype == torch.bfloat16
    assert torch.equal(y16, y32.bfloat16()) and torch.equal(gi16, gi32.bfloat16())
    for (k, p16), (_, p32) in zip(m16.named_parameters(), m32.named_parameters()):
        assert p16.grad.dtype == torch.bfloat16 and torch.equal(p16.grad, p32.grad.bfloat16()), k


def test_fp32_module_on_bf16_input():
    w = ER.stable_weights(48, 4)
    m = _layer(48, 10, w)
    x = torch.randn(3, 1, 48, 48, device="cuda").bfloat16()
    y, gi, gw = _pass(m, x, torch.ones(3, 1, 48, 48, device="cuda", dtype=torch.bfloat16), True)
    assert y.dtype == gi.dtype == torch.bfloat16
    assert all(p.grad.dtype == torch.float32 for p in m.parameters())
    # autocast: the input is cast up and the output is fp32, as before
    with torch.autocast("cuda", dtype=torch.bfloat16):
        ya = m(x)
    assert ya.dtype == torch.float32 and torch.equal(ya, m(x.float()))


def test_half_and_double_planes_refused():
    m = _layer(48, 10, ER.stable_weights(48, 4))
    for dtype in (torch.float16, torch.float64):
        with pytest.raises(RuntimeError, match="float32 or bfloat16"):
            m(torch.zeros(2, 1, 48, 48, device="cuda", dtype=dtype))


@pytest.mark.parametrize("img_size", [48, 96])
def test_bf16_classifier_trains_a_step(img_size):
    from cnn_with_pde_b200.emotion_recognition import DiffusionClassifier
    torch.manual_seed(img_size)
    model = DiffusionClassifier(img_size=img_size).cuda().bfloat16()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    x = torch.rand(8, 1, img_size, img_size, device="cuda").bfloat16()
    labels = torch.randint(0, 7, (8,), device="cuda")
    loss = torch.nn.functional.cross_entropy(model(x).float(), labels)
    loss.backward()
    assert torch.isfinite(loss)
    for name, p in model.named_parameters():
        assert p.grad is not None and p.grad.dtype == torch.bfloat16 and torch.isfinite(p.grad).all(), name
    opt.step()
    assert all(torch.isfinite(p).all() for p in model.parameters())


# ------------------------------------------------------------------------------------------ the defect
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64])
@pytest.mark.parametrize("N", [48, 40, 96])
def test_converted_module_reads_fp32_weights(dtype, N):
    """A module converted with .half() / .bfloat16() / .double() on an fp32 input equals an fp32 module holding the
    converted weights and x / y buffers widened to fp32, plainly and under autocast."""
    w = ER.stable_weights(N, 5)
    conv = _layer(N, 10, w, dtype)
    ref = _layer(N, 10, w)
    with torch.no_grad():
        for (_, pr), (_, pc) in zip(ref.named_parameters(), conv.named_parameters()):
            pr.copy_(pc.float())
        ref.x.copy_(conv.x.float())
        ref.y.copy_(conv.y.float())
    x = torch.randn(3, 1, N, N, device="cuda")
    g = torch.randn(3, 1, N, N, device="cuda")
    for autocast in (False, True):
        with torch.autocast("cuda", enabled=autocast):
            yc, gic, _ = _pass(conv, x, g, True)
            yr, gir, _ = _pass(ref, x, g, True)
        assert yc.dtype == torch.float32 and torch.equal(yc, yr), (dtype, autocast)
        assert torch.equal(gic, gir), (dtype, autocast)
        for (k, pc), (_, pr) in zip(conv.named_parameters(), ref.named_parameters()):
            assert pc.grad.dtype == dtype, k
            if not _generic(N, False):
                assert torch.equal(pc.grad, pr.grad.to(dtype)), (dtype, autocast, k)
            else:   # float atomics: the fp32 sums agree to ~1e-6, which may move the rounded value by one unit
                ulp = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7, torch.float64: 1e-5}[dtype]
                torch.testing.assert_close(pc.grad.double(), pr.grad.to(dtype).double(), rtol=ulp, atol=0)


# -------------------------------------------------------------------------------- compile / export / graphs
@pytest.mark.parametrize("N", [48, 96])
def test_compiled_and_exported_bf16_layer_match_eager_bitwise(N):
    m = _layer(N, 10, ER.stable_weights(N, 6), torch.bfloat16)
    x = torch.randn(4, 1, N, N, device="cuda").bfloat16()
    g = torch.randn(4, 1, N, N, device="cuda").bfloat16()

    def run(fn):
        m.zero_grad(set_to_none=True)
        xx = x.clone().requires_grad_()
        y = fn(xx)
        y.backward(g)
        return [y.detach(), xx.grad] + [p.grad for p in m.parameters()]

    want = run(m)
    torch._dynamo.reset()
    for got in (run(torch.compile(m, fullgraph=True)), run(torch.export.export(m, (x,)).module())):
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert a.dtype == b.dtype and torch.equal(a, b)


def test_compiled_and_exported_bf16_classifier():
    """The classifier's PDE layer compiled equals eager bit for bit; the whole bf16 classifier, compiled with
    fullgraph=True and exported, matches eager (its convolutions and matmuls are not this project's kernels and
    may round differently once compiled)."""
    from cnn_with_pde_b200.emotion_recognition import DiffusionClassifier, PDELayer
    torch.manual_seed(0)
    model = DiffusionClassifier().cuda().bfloat16().eval()
    x = torch.randn(8, 1, 48, 48, device="cuda").bfloat16()
    layers = [mod for mod in model.modules() if isinstance(mod, PDELayer)]
    assert layers
    for mod in layers:
        torch._dynamo.reset()
        assert torch.equal(torch.compile(mod, fullgraph=True)(x), mod(x))
    with torch.no_grad():
        want = model(x)
        torch._dynamo.reset()
        got_c = torch.compile(model, fullgraph=True)(x)
        got_e = torch.export.export(model, (x,)).module()(x)
    for got in (got_c, got_e):
        assert got.dtype == torch.bfloat16
        assert runners.rel_l2(got.float().cpu().numpy(), want.float().cpu().numpy()) <= 3e-2


def test_opcheck_bf16():
    for N in (48, 96):
        u = torch.randn(3, 1, N, N, device="cuda").bfloat16().requires_grad_()
        w6 = torch.tensor([0.1, 0.1, 0.1, 0.3, 0.2, 0.2], device="cuda") / (DT * N * N)
        w6.requires_grad_()
        xs = torch.linspace(0, 1, N, device="cuda")
        args = (u, w6, xs, xs.clone(), N, 10, DT, 1 / N, 1 / N, False)
        torch.library.opcheck(torch.ops.pde_b200.emotion_fwd, args,
                              test_utils=("test_schema", "test_autograd_registration", "test_faketensor",
                                          "test_aot_dispatch_dynamic"))
        with torch.no_grad():
            out = torch.ops.pde_b200.emotion_fwd(*args)
            torch.library.opcheck(torch.ops.pde_b200.emotion_bwd,
                                  (torch.randn_like(out), *[a.detach() for a in args[:4]], *args[4:], True))


@pytest.mark.parametrize("N", [48, 96])
def test_cuda_graph_bf16_training_step_equals_eager(N):
    layer = _layer(N, 10, ER.stable_weights(N, 8), torch.bfloat16)
    base = torch.randn(4, 1, N, N, device="cuda").bfloat16()
    xs = torch.zeros_like(base, requires_grad=True)
    gs = torch.zeros_like(base)

    def step():
        yy = layer(xs)
        yy.backward(gs)
        return yy

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    xs.grad = None
    layer.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_y = step()
    with torch.no_grad():
        xs.copy_(base)
        gs.copy_(base * 0.5 + 1.0)
    graph.replay()
    torch.cuda.synchronize()
    cap = [static_y.clone(), xs.grad.clone()] + [p.grad.clone() for p in layer.parameters()]
    layer.zero_grad(set_to_none=True)
    xe = base.clone().requires_grad_(True)
    ye = layer(xe)
    ye.backward(gs)
    eager = [ye.detach(), xe.grad] + [p.grad for p in layer.parameters()]
    assert len(cap) == len(eager) == 8
    for a, b in zip(cap, eager):
        assert a.dtype == b.dtype and torch.equal(a, b)
    del graph
