"""emotion_recognition.PDELayer on planes above 64 x 64 (emotion_halo.cu), and both sides of the dispatch boundary.

Every plane edge from 65 up was refused before the halo kernels existed, and the dispatch is exclusive (N <= 64
keeps the whole-plane kernels, 65 ... 4096 with Nt <= 16 takes the halo ones), so a case passing above 64 is also
the proof that the halo kernels ran.

Bar (tests/test_gpu_parity.py): 1e-5 against the fp32 oracle for the output, grad_input and the six weight
gradients, measured as rel-L2 and as max-abs / max-ref; the fp64 oracle's distance is reported beside it.
Coefficients: a stable set (tests/emotion_reference.stable_weights: a + b <= 1/2) and the reference's default
init, which amplifies.
"""
import ctypes
import os
import subprocess
import sys
from ctypes import byref

import numpy as np
import pytest

from . import emotion_reference as ER
from . import runners

pytestmark = pytest.mark.gpu
TOL = 1e-5
DT = 0.001
NAMES = ("alpha_w1", "alpha_w2", "alpha_w3", "beta_w1", "beta_w2", "beta_w3")
DOMAIN = "65 ... 4096 with Nt <= 16"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _err(a, b):
    return max(runners.rel_l2(a, b), runners.rel_max(a, b))


def _layer(N, Nt, w):
    import torch
    from cnn_with_pde_b200.emotion_recognition import PDELayer
    m = PDELayer(Nx=N, Ny=N, dt=DT).cuda()
    m.Nt = Nt
    with torch.no_grad():
        for k, v in zip(NAMES, w):
            getattr(m, k).fill_(float(v))
    return m


def _run(u, g, w, Nt, need_gin=True):
    import torch
    m = _layer(u.shape[-1], Nt, w)
    x = torch.from_numpy(u).cuda().requires_grad_(need_gin)
    y = m(x)
    y.backward(torch.from_numpy(g).cuda())
    torch.cuda.synchronize()
    return {"y": y.detach().cpu().numpy(), "gin": x.grad.cpu().numpy() if need_gin else None,
            "w": np.array([getattr(m, k).grad.item() for k in NAMES])}


def _check(u, g, w, Nt, need_gin=True, what=""):
    got = _run(u, g, w, Nt, need_gin)
    if not need_gin:
        assert got["gin"] is None
    want32 = ER.oracle(u, g, w, Nt, need_gin=need_gin, dtype=np.float32)
    want64 = ER.oracle(u, g, w, Nt, need_gin=need_gin, dtype=np.float64)
    for k in ("y", "gin", "w") if need_gin else ("y", "w"):
        assert np.all(np.isfinite(got[k])), (what, k)
        e32, e64, eref = _err(got[k], want32[k]), _err(got[k], want64[k]), _err(want32[k], want64[k])
        assert e32 <= TOL, (what, k, "vs fp32 oracle", e32, "vs fp64", e64, "fp32 oracle vs fp64", eref)
    return got


def _weights(N, seed, default):
    return np.array(ER.DEFAULT_W, np.float32) if default else ER.stable_weights(N, seed)


# ------------------------------------------------------------------------------------------ shapes
@pytest.mark.parametrize("N", [63, 64, 65, 66])
@pytest.mark.parametrize("Nt", [0, 1, 10, 16])
def test_both_sides_of_the_dispatch_boundary(N, Nt):
    """63 / 64 keep the whole-plane kernels, 65 / 66 take the halo kernels.  At 16 steps the whole-plane backward
    does not hold 63 x 63 or 64 x 64 (the step states exceed a block's shared memory): the forward is served and
    the backward refused, as before the halo kernels existed."""
    import torch
    import cnn_with_pde_b200._cabi as cabi
    for default in (False, True):
        u, g = ER.make_inputs(3, N, seed=N * 10 + Nt)
        w = _weights(N, N + Nt, default)
        what = f"N={N} Nt={Nt} default={default}"
        if N <= 64 and Nt == 16:
            m = _layer(N, Nt, w)
            x = torch.from_numpy(u).cuda().requires_grad_(True)
            y = m(x)
            assert _err(y.detach().cpu().numpy(), ER.oracle(u, g, w, Nt, dtype=np.float32)["y"]) <= TOL, what
            with pytest.raises(cabi.PdeB200Error):
                y.backward(torch.from_numpy(g).cuda())
            continue
        _check(u, g, w, Nt, need_gin=not default or Nt != 10, what=what)


def test_sixteen_steps_served_and_seventeen_refused():
    import torch
    import cnn_with_pde_b200._cabi as cabi
    u, g = ER.make_inputs(2, 65, seed=65)
    _check(u, g, ER.stable_weights(65, 1), 16, what="N=65 Nt=16")
    L = cabi.lib()
    stream = torch.cuda.current_stream().cuda_stream
    x = torch.zeros(1, 1, 65, 65, device="cuda")
    w = torch.ones(6, device="cuda")
    xs = torch.linspace(0, 1, 65, device="cuda")
    for N, Nt in ((65, 17), (4096, 17), (4097, 1), (5000, 0)):
        d = cabi.EmoDesc(1, N, Nt, 0.0005, 0.001, 1.0 / N ** 2, 1.0 / N ** 2, 0)
        assert L.pde_emotion_backward_workspace_bytes(byref(d)) == 0
        ptr = x.data_ptr()
        assert L.pde_emotion_forward(byref(d), ptr, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), ptr, stream) == \
            cabi.ERR_UNSUPPORTED
        assert L.pde_emotion_backward(byref(d), ptr, ptr, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), ptr, w.data_ptr(),
                                      ptr, ctypes.c_size_t(1 << 20), stream) == cabi.ERR_UNSUPPORTED
    m = _layer(65, 17, ER.stable_weights(65, 1))
    with pytest.raises(cabi.PdeB200Error, match=DOMAIN):
        m(torch.from_numpy(u).cuda())
    from cnn_with_pde_b200.emotion_recognition import PDELayer
    with pytest.raises(cabi.PdeB200Error, match=DOMAIN):
        PDELayer(Nx=4097, Ny=4097).cuda()(torch.zeros(1, 1, 4097, 4097, device="cuda"))


@pytest.mark.parametrize("N", [96, 97, 100, 112, 127, 128, 129, 224, 255, 256, 1000])
def test_tile_seams(N):
    """Plane edges on and off the 32 x 64 tile grid, cycling steps, batch and grad_input."""
    i = N % 7
    Nt = (1, 2, 5, 10, 16, 3, 7)[i]
    B = (1, 2, 3)[N % 3] if N <= 256 else 1
    u, g = ER.make_inputs(B, N, seed=N)
    _check(u, g, ER.stable_weights(N, N), Nt, need_gin=N % 4 != 1, what=f"N={N} Nt={Nt} B={B}")


def test_plane_4096():
    u, g = ER.make_inputs(1, 4096, seed=4096)
    _check(u, g, ER.stable_weights(4096, 7), 16, what="4096^2 Nt=16")


def test_random_configurations():
    """30 seeded draws: B 1 ... 4, N 65 ... 300, Nt 0 ... 16, stable or default coefficients, grad_input or not."""
    rs = np.random.RandomState(20261021)
    for n in range(30):
        N, Nt, B = int(rs.randint(65, 301)), int(rs.randint(0, 17)), int(rs.randint(1, 5))
        default = N <= 128 and Nt <= 10 and rs.randint(3) == 0   # beyond that the default init overflows fp32
        need_gin = bool(rs.randint(4))
        u, g = ER.make_inputs(B, N, seed=int(rs.randint(1 << 20)))
        _check(u, g, _weights(N, n, default), Nt, need_gin, what=f"draw {n}: B={B} N={N} Nt={Nt} default={default}")


@pytest.mark.parametrize("N", [65, 80, 96, 111, 128])
def test_default_init_stays_finite(N):
    """The reference's init amplifies (a + b up to ~20 at 128 x 128); ten steps stay finite and match."""
    u, g = ER.make_inputs(2, N, seed=N + 1)
    _check(u, g, np.array(ER.DEFAULT_W, np.float32), 10, what=f"default N={N}")


def test_adjoint_identity():
    """<J v, g> = <v, J^T g>: the layer is linear in its input (the ghost ring is a reflection of it)."""
    u, g = ER.make_inputs(2, 224, seed=5)
    w = ER.stable_weights(224, 5)
    for Nt in (1, 10, 16):
        got = _run(u, g, w, Nt)
        lhs = float(np.dot(got["y"].astype(np.float64).ravel(), g.astype(np.float64).ravel()))
        rhs = float(np.dot(u.astype(np.float64).ravel(), got["gin"].astype(np.float64).ravel()))
        scale = float(np.linalg.norm(got["y"]) * np.linalg.norm(g))
        assert abs(lhs - rhs) <= 1e-6 * scale, (Nt, lhs, rhs, scale)


def test_batch_past_the_workspace_cap():
    """512 x 512 at 16 steps keeps 16 planes per sample: 130 samples run in three chunks under 1 GiB."""
    import cnn_with_pde_b200._cabi as cabi
    d = cabi.EmoDesc(130, 512, 16, 0.0005, 0.001, 1.0 / 512 ** 2, 1.0 / 512 ** 2, 0)
    assert cabi.lib().pde_emotion_backward_workspace_bytes(byref(d)) <= (1 << 30) + (1 << 20)
    u, g = ER.make_inputs(130, 512, seed=512)
    _check(u, g, ER.stable_weights(512, 9), 16, what="B=130 N=512 Nt=16")


def test_forward_past_two_to_the_31_cells():
    """129 planes of 4096 x 4096: B N^2 > 2^31."""
    import torch
    B, N = 129, 4096
    assert B * N * N > 2 ** 31
    w = ER.stable_weights(N, 3)
    m = _layer(N, 2, w)
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(B, 1, N, N, device="cuda", generator=gen)
    with torch.no_grad():
        y = m(x)
    for b in (0, 64, B - 1):
        want = ER.oracle(x[b:b + 1].cpu().numpy(), x[b:b + 1].cpu().numpy(), w, 2, dtype=np.float32)["y"]
        assert _err(y[b:b + 1].cpu().numpy(), want) <= TOL, b
    del x, y


# --------------------------------------------------------------------------------------------- ABI
class _Guarded:
    """A device buffer `nbytes` long at `offset` bytes past a 256-byte boundary, with 4 KB guard bands of 0xA5."""
    GUARD = 4096

    def __init__(self, nbytes, offset):
        import torch
        self.raw = torch.full((nbytes + 2 * self.GUARD + 256,), 0xA5, dtype=torch.uint8, device="cuda")
        base = self.raw.data_ptr()
        self.start = self.GUARD + (-(base + self.GUARD)) % 256 + offset
        self.n = nbytes
        self.ptr = base + self.start

    def view(self):
        import torch
        return self.raw[self.start:self.start + self.n].view(torch.float32)

    def guards_intact(self):
        r = self.raw.cpu().numpy()
        return bool(np.all(r[:self.start] == 0xA5) and np.all(r[self.start + self.n:] == 0xA5))


def _desc(B, N, Nt):
    import cnn_with_pde_b200._cabi as cabi
    f = lambda v: float(np.float32(v))
    return cabi.EmoDesc(B, N, Nt, f(0.5 * DT), f(DT), f((1.0 / N) ** 2), f((1.0 / N) ** 2), 0)


@pytest.mark.parametrize("B,N,Nt", [(2, 65, 1), (3, 100, 10), (1, 227, 16), (2, 130, 0)])
def test_abi_guard_bands_workspace_and_reproducibility(B, N, Nt):
    """Unaligned (4-byte) planes with guard bands; the workspace exactly as queried, and one byte less refused;
    g_w6 bit-identical from call to call and with gin = NULL; the same values as the module."""
    import torch
    import cnn_with_pde_b200._cabi as cabi
    L = cabi.lib()
    d = _desc(B, N, Nt)
    ws_bytes = L.pde_emotion_backward_workspace_bytes(byref(d))
    assert ws_bytes > 0
    n = B * N * N
    u, g = ER.make_inputs(B, N, seed=n)
    w = ER.stable_weights(N, n)
    bufs = {k: _Guarded(n * 4, 4) for k in ("u", "g", "out", "gin")}
    bufs["u"].view().copy_(torch.from_numpy(u.ravel()))
    bufs["g"].view().copy_(torch.from_numpy(g.ravel()))
    wt = torch.from_numpy(w).cuda()
    xs = torch.linspace(0, 1, N).cuda()   # the module's buffer: built on the CPU
    stream = torch.cuda.current_stream().cuda_stream
    assert L.pde_emotion_forward(byref(d), bufs["u"].ptr, wt.data_ptr(), xs.data_ptr(), xs.data_ptr(), bufs["out"].ptr,
                                 stream) == 0
    results = []
    for gin in (bufs["gin"].ptr, bufs["gin"].ptr, None):
        ws = _Guarded(ws_bytes, 0)
        gw = _Guarded(6 * 4, 4)
        rc = L.pde_emotion_backward(byref(d), bufs["u"].ptr, bufs["g"].ptr, wt.data_ptr(), xs.data_ptr(), xs.data_ptr(),
                                    gin, gw.ptr, ws.ptr, ctypes.c_size_t(ws_bytes), stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert ws.guards_intact() and gw.guards_intact()
        results.append((gw.view().cpu().numpy(), bufs["gin"].view().cpu().numpy()))
    assert np.array_equal(results[0][0], results[1][0]) and np.array_equal(results[0][1], results[1][1])
    assert np.array_equal(results[0][0], results[2][0])
    assert all(b.guards_intact() for b in bufs.values())
    ref = _run(u, g, w, Nt)
    assert np.array_equal(bufs["out"].view().cpu().numpy(), ref["y"].ravel())
    assert np.array_equal(results[0][1], ref["gin"].ravel())
    assert np.array_equal(results[0][0], ref["w"].astype(np.float32))
    ws = _Guarded(ws_bytes, 0)
    rc = L.pde_emotion_backward(byref(d), bufs["u"].ptr, bufs["g"].ptr, wt.data_ptr(), xs.data_ptr(), xs.data_ptr(),
                                bufs["gin"].ptr, gw.ptr, ws.ptr, ctypes.c_size_t(ws_bytes - 1), stream)
    assert rc == cabi.ERR_WORKSPACE


def test_abi_empty_batch():
    import torch
    import cnn_with_pde_b200._cabi as cabi
    L = cabi.lib()
    stream = torch.cuda.current_stream().cuda_stream
    w = torch.ones(6, device="cuda")
    for N in (65, 224, 4096):
        d = _desc(0, N, 10)
        xs = torch.linspace(0, 1, N, device="cuda")
        assert L.pde_emotion_forward(byref(d), None, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), None, stream) == 0
        gw = torch.full((6,), 7.0, device="cuda")
        assert L.pde_emotion_backward(byref(d), None, None, w.data_ptr(), xs.data_ptr(), xs.data_ptr(), None,
                                      gw.data_ptr(), None, ctypes.c_size_t(0), stream) == 0
        assert float(gw.abs().sum()) == 0.0


def test_debug_plan_names_the_halo_kernels():
    code = ("import torch, cnn_with_pde_b200 as P\n"
            "from cnn_with_pde_b200.emotion_recognition import PDELayer\n"
            "for n in (48, 96):\n"
            "    m = PDELayer(Nx=n, Ny=n).cuda()\n"
            "    x = torch.randn(2, 1, n, n, device='cuda', requires_grad=True)\n"
            "    m(x).sum().backward()\n"
            "torch.cuda.synchronize()\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, PDE_B200_DEBUG="1"), timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stderr.splitlines() if "emotion halo" in ln]
    assert len(lines) == 2, r.stderr
    assert "emotion halo fwd plan" in lines[0] and "N=96 Nt=10" in lines[0] and "regs=" in lines[0], r.stderr
    assert "emotion halo bwd plan" in lines[1] and "chunk=2" in lines[1] and "workspace=" in lines[1], r.stderr


# ------------------------------------------------------------------------------------------ module
def test_module_semantics_at_100():
    import torch
    from cnn_with_pde_b200.emotion_recognition import PDELayer
    torch.manual_seed(0)
    N = 100
    w = ER.stable_weights(N, 11)
    m = _layer(N, 10, w)
    base = torch.randn(4, 1, N, N, device="cuda")
    # autograd on a batch slice: x[1:] starts 4 bytes past a 16-byte boundary
    x = base.clone().requires_grad_(True)
    y = m(x[1:])
    g = torch.randn_like(y)
    y.backward(g)
    want = ER.oracle(base[1:].cpu().numpy(), g.cpu().numpy(), w, 10, dtype=np.float32)
    assert _err(y.detach().cpu().numpy(), want["y"]) <= TOL
    assert _err(x.grad[1:].cpu().numpy(), want["gin"]) <= TOL and not x.grad[0].any()
    with torch.no_grad():
        y0 = m(base)
    assert not y0.requires_grad and torch.equal(y0[1:], y.detach())
    with torch.autocast("cuda", dtype=torch.float16):
        yh = m(base.half())
    assert yh.dtype == torch.float32
    assert runners.rel_l2(yh.detach().cpu().numpy(), y0.cpu().numpy()) <= 2e-3
    # CUDA-graph capture equals eager
    layer = _layer(N, 10, w)
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
        assert torch.equal(a, b)
    del graph


@pytest.mark.parametrize("img_size", [96, 224])
def test_classifier_trains_at_larger_images(img_size):
    """DiffusionClassifier(img_size=N): one forward + backward + AdamW step at the reference's default init."""
    import torch
    from cnn_with_pde_b200.emotion_recognition import DiffusionClassifier
    torch.manual_seed(img_size)
    model = DiffusionClassifier(img_size=img_size).cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    x = torch.rand(8, 1, img_size, img_size, device="cuda")
    labels = torch.randint(0, 7, (8,), device="cuda")
    loss = torch.nn.functional.cross_entropy(model(x), labels)
    loss.backward()
    assert torch.isfinite(loss)
    for name, p in model.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    opt.step()
    assert all(torch.isfinite(p).all() for p in model.parameters())
