"""tiny_imagenet.ImprovedDiffusionLayer at plane shapes the whole-plane ring kernels cannot hold (tiny_tiled.cu).

Every new shape here was refused before the tiled kernels existed, and the dispatch is exclusive: a
configuration the ring kernels serve keeps them, anything else in the domain (H, W <= 4096, steps <= 16,
C <= 1024) takes the tiled ones.  So a case passing at a new shape is also the proof that the tiled kernels ran.

Bar (tests/test_gpu_parity.py): 1e-5 against the fp32 oracle and no further from the fp64 oracle than the fp32
oracle plus 1e-5; the two parameter gradients are cancelling sums, held to "three times the fp32 oracle's own
distance from fp64, plus 1e-5" where they miss the plain bar.  Where a parameter gradient cancels to ~1e-4 of its
terms, the fp32 oracle (unfused multiply and add) can land far closer to fp64 than the kernels' arithmetic (fused,
op for op that of the whole-plane kernels) does: at 3 x 1 x 2 x 299 with 3 steps the kernels' per-cell arithmetic,
replayed in numpy with the sum in double, is 3e-4 from fp64 and the fp32 oracle 4e-5.  Such a gradient is held to
the size the sum would have without cancellation instead: an absolute error of at most 1e-6 of
steps x blend x |u| |gout| x max |s| / sqrt(cells) (times dt x 6 for alpha), which one cell counted twice or
missed still exceeds many times over.  bf16 I/O: the output and grad_input are the oracle's fp32 results on the
bf16-rounded inputs, rounded to bf16, to within one bf16 unit and almost always exact.
"""
import ctypes
import os
import subprocess
import sys
from ctypes import byref

import numpy as np
import pytest

from . import runners
from . import tiny_reference as TR

pytestmark = pytest.mark.gpu
TOL = 1e-5
DT = 0.01
PARAMS = ("alpha_base", "channel_scaling")
EDGES = (1, 2, 3, 7, 30, 63, 64, 65, 127, 129, 224, 227, 255, 257, 299, 512)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _err(a, b):
    return max(runners.rel_l2(a, b), runners.rel_max(a, b))


def _layer(C, steps, al, sc):
    import torch
    from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer
    m = ImprovedDiffusionLayer(channels=C, dt=DT, num_steps=steps).cuda()
    with torch.no_grad():
        m.alpha_base.copy_(torch.from_numpy(al))
        m.channel_scaling.copy_(torch.from_numpy(sc))
    return m


def _run(u, g, al, sc, steps, need_gin=True, bf16=False):
    import torch
    m = _layer(u.shape[1], steps, al, sc)
    x = torch.from_numpy(u).cuda()
    gg = torch.from_numpy(g).cuda()
    if bf16:
        x, gg = x.bfloat16(), gg.bfloat16()
    x.requires_grad_(need_gin)
    y = m(x)
    assert y.dtype == x.dtype
    y.backward(gg)
    torch.cuda.synchronize()
    out = {"y": y.detach().float().cpu().numpy(), "gin": x.grad.float().cpu().numpy() if need_gin else None}
    for k in PARAMS:
        out[k] = getattr(m, k).grad.cpu().numpy()
    return out


def _param_ok(k, got, want32, want64, u, g, sc, steps):
    """plain bar, the three-times rule, or the rounding bound of a sum that cancels (module docstring)"""
    e32, e64, eref = _err(got, want32), _err(got, want64), _err(want32, want64)
    if e32 <= TOL or e64 <= 3.0 * eref + TOL:
        return True
    scale = steps * 0.1 * float(np.linalg.norm(u)) * float(np.linalg.norm(g)) * float(np.max(np.abs(sc))) / np.sqrt(u.size)
    if k == "alpha_base":
        scale *= DT * 6.0
    return float(np.max(np.abs(np.asarray(got, np.float64) - want64))) <= 1e-6 * scale


def _check(u, g, al, sc, steps, need_gin=True, what=""):
    """fp32 planes through the module against the oracle."""
    got = _run(u, g, al, sc, steps, need_gin)
    if not need_gin:
        assert got["gin"] is None
    want32 = TR.oracle(u, g, al, sc, steps, need_gin=need_gin, dtype=np.float32)
    want64 = TR.oracle(u, g, al, sc, steps, need_gin=need_gin, dtype=np.float64)
    keys = ("y", "gin") + PARAMS if need_gin else ("y",) + PARAMS
    for k in keys:
        e32, e64, eref = _err(got[k], want32[k]), _err(got[k], want64[k]), _err(want32[k], want64[k])
        if k in PARAMS:
            assert _param_ok(k, got[k], want32[k], want64[k], u, g, sc, steps), (what, k, e32, e64, eref)
        else:
            assert e32 <= TOL and e64 <= eref + TOL, (what, k, e32, e64, eref)
    clamped = (al < 1e-6) | (al > 0.15)
    assert np.all(got["alpha_base"][clamped] == 0.0), what
    return got


def _check_bf16(u, g, al, sc, steps, what=""):
    import torch
    got = _run(u, g, al, sc, steps, bf16=True)
    ub = torch.from_numpy(u).bfloat16().float().numpy()
    gb = torch.from_numpy(g).bfloat16().float().numpy()
    want = TR.oracle(ub, gb, al, sc, steps, dtype=np.float32)
    for k in ("y", "gin"):
        ref_b = torch.from_numpy(want[k]).bfloat16().float().numpy()
        assert np.all(np.abs(got[k] - ref_b) <= 2.0 ** -7 * np.abs(ref_b) + 1e-30), (what, k)   # at most one bf16 unit
        assert np.mean(got[k] != ref_b) <= 0.01, (what, k)                                       # and almost always none
    want64 = TR.oracle(ub, gb, al, sc, steps, dtype=np.float64)
    for k in PARAMS:
        assert _param_ok(k, got[k], want[k], want64[k], ub, gb, sc, steps), (what, k)


# ------------------------------------------------------------------------------------------ shapes
@pytest.mark.parametrize("H", EDGES)
def test_every_plane_shape(H):
    """H x W for every W of the list (squares and rectangles), cycling channels, steps, batch and grad_input."""
    i = EDGES.index(H)
    for j, W in enumerate(EDGES):
        cells = H * W
        C = (1, 3, 17)[(i + j) % 3] if cells <= 70000 else (1, 3)[(i + j) % 2]
        steps = (0, 1, 2, 3, 7, 16)[(7 * i + j) % 6]
        B = 1 + (i + 2 * j) % 3 if cells <= 100000 else 1
        need_gin = (i + j) % 4 != 3
        u, g, al, sc = TR.make_inputs(B, C, H, W, seed=100 * i + j, clamp=(i + j) % 5 == 0)
        _check(u, g, al, sc, steps, need_gin, what=f"{B}x{C}x{H}x{W} K={steps} gin={need_gin}")


@pytest.mark.parametrize("H,W,steps", [(170, 170, 1), (171, 171, 1), (240, 240, 1), (241, 241, 1), (64, 64, 11),
                                       (64, 64, 12), (128, 128, 1), (128, 128, 2)])
def test_both_sides_of_the_ring_kernels_limits(H, W, steps):
    """170 / 171 (fp32 backward), 240 / 241 (fp32 forward), 64 x 64 at 11 / 12 steps, 128 x 128 at 1 / 2 steps."""
    u, g, al, sc = TR.make_inputs(3, 3, H, W, seed=H + steps)
    _check(u, g, al, sc, steps, what=f"{H}x{W} K={steps}")


@pytest.mark.parametrize("H,W,steps", [(3, 4, 1), (5, 12, 2), (64, 64, 1), (299, 299, 1), (224, 224, 2), (31, 45, 3),
                                       (7, 229, 1)])
def test_bf16_io(H, W, steps):
    """bf16 planes: H * W % 8 != 0 next to a plane the ring kernels serve, odd widths, 224^2 at two steps, 299^2."""
    u, g, al, sc = TR.make_inputs(2, 3, H, W, seed=7 * H + W)
    _check_bf16(u, g, al, sc, steps, what=f"bf16 {H}x{W} K={steps}")


def test_random_configurations():
    """40 seeded draws: H, W 1 ... 300, C 1 ... 5, steps 0 ... 16, batch, grad_input and I/O type."""
    rs = np.random.RandomState(20261020)
    for n in range(40):
        H, W = int(rs.randint(1, 301)), int(rs.randint(1, 301))
        C, steps, B = int(rs.randint(1, 6)), int(rs.randint(0, 17)), int(rs.choice([1, 2, 3, 5]))
        need_gin, bf16 = bool(rs.randint(2)), rs.randint(4) == 0
        u, g, al, sc = TR.make_inputs(B, C, H, W, seed=int(rs.randint(1 << 20)), clamp=bool(rs.randint(2)))
        what = f"draw {n}: {B}x{C}x{H}x{W} K={steps} gin={need_gin} bf16={bf16}"
        if bf16:
            _check_bf16(u, g, al, sc, steps, what)
        else:
            _check(u, g, al, sc, steps, need_gin, what)


# ------------------------------------------------------------------------------------ size and seams
def test_imagenet_batch_larger_than_l2():
    """3 x 224 x 224 at batch 1024 (616 MB a tensor): every output and gradient against the oracle."""
    u, g, al, sc = TR.make_inputs(1024, 3, 224, 224, seed=224)
    got = _run(u, g, al, sc, 1)
    want = TR.oracle(u, g, al, sc, 1, dtype=np.float32)
    for k in ("y", "gin"):
        assert _err(got[k], want[k]) <= TOL, k
    want64 = TR.oracle(u, g, al, sc, 1, dtype=np.float64)
    for k in PARAMS:
        assert _param_ok(k, got[k], want[k], want64[k], u, g, sc, 1), k


@pytest.mark.parametrize("B,C,H,W,steps", [(1, 1, 4096, 4096, 2), (2, 3, 1000, 1003, 1), (1, 2, 1000, 1003, 16)])
def test_large_planes_every_tile_seam(B, C, H, W, steps):
    u, g, al, sc = TR.make_inputs(B, C, H, W, seed=H + W)
    _check(u, g, al, sc, steps, what=f"{B}x{C}x{H}x{W} K={steps}")


def test_adjoint_identity():
    """<J v, w> = <v, J^T w> at 3 x 512 x 512 (the step is linear in u for fixed alpha and s)."""
    u, g, al, sc = TR.make_inputs(2, 3, 512, 512, seed=5)
    for steps in (1, 4, 16):
        got = _run(u, g, al, sc, steps)
        lhs = float(np.dot(got["y"].astype(np.float64).ravel(), g.astype(np.float64).ravel()))
        rhs = float(np.dot(u.astype(np.float64).ravel(), got["gin"].astype(np.float64).ravel()))
        scale = float(np.linalg.norm(got["y"]) * np.linalg.norm(g))
        assert abs(lhs - rhs) <= 1e-6 * scale, (steps, lhs, rhs, scale)


# --------------------------------------------------------------------------------------------- ABI
def _abi():
    import cnn_with_pde_b200._cabi as cabi
    return cabi, cabi.lib()


def _desc(B, C, H, W, steps):
    cabi, _ = _abi()
    return cabi.TinyDesc(B, C, H, W, steps, DT, 1e-6, 0.15, 0.1)


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

    def view(self, dtype):
        return self.raw[self.start:self.start + self.n].view(dtype)

    def guards_intact(self):
        r = self.raw.cpu().numpy()
        return bool(np.all(r[:self.start] == 0xA5) and np.all(r[self.start + self.n:] == 0xA5))


@pytest.mark.parametrize("bf16", [False, True], ids=["fp32", "bf16"])
@pytest.mark.parametrize("B,C,H,W,steps", [(2, 3, 227, 227, 1), (3, 2, 33, 71, 5), (1, 1, 7, 9, 16)])
def test_abi_guard_bands_workspace_and_reproducibility(bf16, B, C, H, W, steps):
    import torch
    cabi, L = _abi()
    d = _desc(B, C, H, W, steps)
    ws_bytes = L.pde_tiny_backward_workspace_bytes(byref(d))
    assert ws_bytes > 0
    es = 2 if bf16 else 4
    tdt = torch.bfloat16 if bf16 else torch.float32
    n = B * C * H * W
    u, g, al, sc = TR.make_inputs(B, C, H, W, seed=n)
    bufs = {k: _Guarded(n * es, es) for k in ("u", "g", "out", "gin")}   # element aligned, not 16-byte aligned
    bufs["u"].view(tdt).copy_(torch.from_numpy(u.ravel()).to(tdt))
    bufs["g"].view(tdt).copy_(torch.from_numpy(g.ravel()).to(tdt))
    a, s = torch.from_numpy(al).cuda(), torch.from_numpy(sc).cuda()
    fwd = L.pde_tiny_forward_bf16 if bf16 else L.pde_tiny_forward
    bwd = L.pde_tiny_backward_bf16 if bf16 else L.pde_tiny_backward
    stream = torch.cuda.current_stream().cuda_stream
    assert fwd(byref(d), bufs["u"].ptr, a.data_ptr(), s.data_ptr(), bufs["out"].ptr, stream) == 0
    results = []
    for _ in range(3):
        ws = _Guarded(ws_bytes, 0)
        ga, gs = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        rc = bwd(byref(d), bufs["u"].ptr, bufs["g"].ptr, a.data_ptr(), s.data_ptr(), bufs["gin"].ptr, ga.data_ptr(),
                 gs.data_ptr(), ws.ptr, ctypes.c_size_t(ws_bytes), stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert ws.guards_intact()
        results.append((ga.cpu().numpy(), gs.cpu().numpy(), bufs["gin"].view(tdt).float().cpu().numpy()))
    for r in results[1:]:   # bit-identical run to run
        for x, y in zip(r, results[0]):
            assert np.array_equal(x, y)
    assert all(b.guards_intact() for b in bufs.values())
    # the same values as the module on ordinary tensors
    ref = _run(u, g, al, sc, steps, bf16=bf16)
    assert np.array_equal(bufs["out"].view(tdt).float().cpu().numpy(), ref["y"].ravel())
    assert np.array_equal(results[0][2], ref["gin"].ravel())
    # one byte less than the query
    ws = _Guarded(ws_bytes, 0)
    ga, gs = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    rc = bwd(byref(d), bufs["u"].ptr, bufs["g"].ptr, a.data_ptr(), s.data_ptr(), bufs["gin"].ptr, ga.data_ptr(),
             gs.data_ptr(), ws.ptr, ctypes.c_size_t(ws_bytes - 1), stream)
    assert rc == cabi.ERR_WORKSPACE


def test_abi_empty_batch_identity_and_refusals():
    import torch
    cabi, L = _abi()
    stream = torch.cuda.current_stream().cuda_stream
    one = torch.ones(3, device="cuda")
    # B = 0 at odd widths and beyond the ring kernels: a no-op, gradients zeroed
    for H, W in ((7, 7), (227, 227), (4096, 4095)):
        d = _desc(0, 3, H, W, 2)
        assert L.pde_tiny_forward(byref(d), None, one.data_ptr(), one.data_ptr(), None, stream) == 0
        ga, gs = torch.full((3,), 7.0, device="cuda"), torch.full((3,), 7.0, device="cuda")
        assert L.pde_tiny_backward_bf16(byref(d), None, None, one.data_ptr(), one.data_ptr(), None, ga.data_ptr(),
                                        gs.data_ptr(), None, ctypes.c_size_t(0), stream) == 0
        assert float(ga.abs().sum() + gs.abs().sum()) == 0.0
    # outside the domain: refused by the library, with the supported domain from Python
    for B, C, H, W, steps in ((1, 3, 256, 256, 17), (1, 1, 8, 4097, 1), (1, 1, 4097, 9, 1), (1, 1025, 8, 8, 1)):
        d = _desc(B, C, H, W, steps)
        assert L.pde_tiny_backward_workspace_bytes(byref(d)) == 0
        x = torch.zeros(B, C, H, W, device="cuda")
        assert L.pde_tiny_forward(byref(d), x.data_ptr(), one.data_ptr(), one.data_ptr(), x.data_ptr(), stream) == \
            cabi.ERR_UNSUPPORTED
        if C <= 3:
            with pytest.raises(cabi.PdeB200Error, match="supported: any H, W 1 ... 4096 with at most 16 steps"):
                _layer(C, steps, np.full(C, 0.05, np.float32), np.ones(C, np.float32))(x)
    # small planes beyond 16 steps stay served by the ring kernels
    u, g, al, sc = TR.make_inputs(2, 2, 16, 16, seed=20)
    _check(u, g, al, sc, 20, what="16x16 K=20")
    # zero steps: the identity, zero parameter gradients
    u, g, al, sc = TR.make_inputs(2, 3, 31, 33, seed=0)
    got = _run(u, g, al, sc, 0)
    assert np.array_equal(got["y"], u) and np.array_equal(got["gin"], g)
    assert not got["alpha_base"].any() and not got["channel_scaling"].any()


def test_forward_only_configurations_stay_served():
    """64 x 64 at 20 steps: the whole-plane forward holds the plane and its two work planes, no backward pass holds
    the step states.  The forward runs, with and without autograd; the backward raises the domain message."""
    import torch
    import cnn_with_pde_b200._cabi as cabi
    u, g, al, sc = TR.make_inputs(2, 3, 64, 64, seed=64)
    m = _layer(3, 20, al, sc)
    x = torch.from_numpy(u).cuda()
    want = TR.oracle(u, g, al, sc, 20, dtype=np.float32)["y"]
    with torch.no_grad():
        y0 = m(x)
    assert _err(y0.cpu().numpy(), want) <= TOL
    xr = x.clone().requires_grad_(True)
    y = m(xr)
    assert torch.equal(y.detach(), y0)
    with pytest.raises(cabi.PdeB200Error, match="supported: any H, W 1 ... 4096 with at most 16 steps"):
        y.backward(torch.from_numpy(g).cuda())


def test_workspace_query_covers_both_io_types():
    """fp32 224^2 takes the tiled backward and bf16 224^2 the ring one: the query serves both, and where both
    passes take the ring kernels it is the number it always was."""
    import torch
    cabi, L = _abi()
    stream = torch.cuda.current_stream().cuda_stream
    for B, C, H, W, steps in ((2, 3, 224, 224, 1), (2, 3, 64, 64, 12), (2, 3, 36, 36, 2)):
        d = _desc(B, C, H, W, steps)
        q = L.pde_tiny_backward_workspace_bytes(byref(d))
        u, g, al, sc = TR.make_inputs(B, C, H, W, seed=1)
        a, s = torch.from_numpy(al).cuda(), torch.from_numpy(sc).cuda()
        for dt, bwd in ((torch.float32, L.pde_tiny_backward), (torch.bfloat16, L.pde_tiny_backward_bf16)):
            x, gg = torch.from_numpy(u).cuda().to(dt), torch.from_numpy(g).cuda().to(dt)
            gin = torch.empty_like(x)
            ws = torch.empty(q, dtype=torch.uint8, device="cuda")
            ga, gs = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
            assert bwd(byref(d), x.data_ptr(), gg.data_ptr(), a.data_ptr(), s.data_ptr(), gin.data_ptr(), ga.data_ptr(),
                       gs.data_ptr(), ws.data_ptr(), ctypes.c_size_t(q), stream) == 0, (H, W, steps, dt)
    props = cabi.device_info()
    d = _desc(2, 3, 36, 36, 2)   # both passes on the ring kernels: (sm_count * 8 + C) partial pairs + 256
    assert L.pde_tiny_backward_workspace_bytes(byref(d)) == (props["sm_count"] * 8 + 3) * 8 + 256


def test_debug_plan_names_the_tiled_kernels():
    code = ("import torch, cnn_with_pde_b200 as P\n"
            "from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer\n"
            "m = ImprovedDiffusionLayer().cuda()\n"
            "for n in (64, 224):\n"
            "    x = torch.randn(2, 3, n, n, device='cuda', requires_grad=True)\n"
            "    m(x).sum().backward()\n"
            "torch.cuda.synchronize()\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, PDE_B200_DEBUG="1"), timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stderr.splitlines() if "tiny tiled" in ln]
    # 224^2 fp32 at one step: the ring forward (one stage), the tiled backward; nothing tiled at 64^2
    assert len(lines) == 1 and "tiny tiled bwd plan" in lines[0] and "H=224 W=224" in lines[0], r.stderr


# ------------------------------------------------------------------------------------------ module
def test_module_semantics_at_227():
    import torch
    from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer
    torch.manual_seed(0)
    m = ImprovedDiffusionLayer(channels=3, num_steps=1).cuda()
    base = torch.randn(4, 3, 227, 227, device="cuda")
    # autograd on a batch slice: x[1:] starts 12 bytes past a 16-byte boundary
    x = base.clone().requires_grad_(True)
    y = m(x[1:])
    g = torch.randn_like(y)
    y.backward(g)
    al, sc = m.alpha_base.detach().cpu().numpy(), m.channel_scaling.detach().cpu().numpy()
    want = TR.oracle(base[1:].cpu().numpy(), g.cpu().numpy(), al, sc, 1, dtype=np.float32)
    assert _err(y.detach().cpu().numpy(), want["y"]) <= TOL
    assert _err(x.grad[1:].cpu().numpy(), want["gin"]) <= TOL and not x.grad[0].any()
    # no_grad
    with torch.no_grad():
        y0 = m(base)
    assert not y0.requires_grad and torch.equal(y0[1:], y.detach())
    # autocast with fp16 input: the layer runs in fp32
    with torch.autocast("cuda", dtype=torch.float16):
        yh = m(base.half())
    assert yh.dtype == torch.float32
    assert runners.rel_l2(yh.detach().cpu().numpy(), y0.cpu().numpy()) <= 2e-3
    # a bf16 module on bf16 input
    mb = ImprovedDiffusionLayer(channels=3, num_steps=1).cuda().bfloat16()
    xb = base.bfloat16().requires_grad_(True)
    yb = mb(xb)
    yb.float().sum().backward()
    assert yb.dtype == torch.bfloat16 and xb.grad.dtype == torch.bfloat16
    assert runners.rel_l2(yb.detach().float().cpu().numpy(), m(base.bfloat16().float()).detach().cpu().numpy()) <= 1e-2
    # CUDA-graph capture equals eager
    layer = ImprovedDiffusionLayer(channels=3, num_steps=2).cuda()
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
        gs.copy_(g.new_ones(base.shape) + base)
    graph.replay()
    torch.cuda.synchronize()
    cap = [static_y.clone(), xs.grad.clone()] + [p.grad.clone() for p in layer.parameters() if p.grad is not None]
    layer.zero_grad(set_to_none=True)
    xe = base.clone().requires_grad_(True)
    ye = layer(xe)
    ye.backward(gs)
    eager = [ye.detach(), xe.grad] + [p.grad for p in layer.parameters() if p.grad is not None]
    assert len(cap) == len(eager) == 4
    for a, b in zip(cap, eager):
        assert torch.equal(a, b)
    del graph


def test_train_tiny_at_imagenet_resolution():
    import cnn_with_pde_b200.train as train
    out = train.run("tiny", 8, 3, 2, graph=True, quiet=True, image_size=224)
    assert out["image_shape"] == [3, 224, 224] and np.isfinite(out["loss"]) and out["cuda_graph"]
