"""tiny_imagenet's dormant methods (tiny_imagenet.py:88-233) on planes beyond 64 x 64 (tiny_split_tiled.cu).

Every shape here with H or W above 64 was refused before the line-streaming kernels existed, and the dispatch is
exclusive (H <= 64 and W <= 64 keeps tiny_split_kernel), so a case passing at such a shape is also the proof that
the new kernels ran.  Bar (tests/test_tiny_split.py): rel-L2 and rel-max <= 1e-5 against the fp32 oracle, 1e-4
where pivots clamp.  The new kernels run tiny_split_kernel's recurrences op for op, so across the dispatch boundary
the two agree bit for bit on every line both compute.
"""
import os
import subprocess
import sys
from ctypes import byref

import numpy as np
import pytest

from . import runners

pytestmark = pytest.mark.gpu
TOL = 1e-5
METHODS = ("implicit_diffusion_step", "solve_implicit_x", "solve_implicit_y", "diffuse_x_explicit",
           "diffuse_y_explicit")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [
    (3, 64, 65), (3, 65, 64), (2, 65, 65), (3, 1, 65), (3, 65, 1),        # both sides of 64 in each dimension
    (2, 1, 4096), (2, 4096, 1), (2, 2, 4096), (2, 4096, 2),               # long thin planes
    (2, 97, 101), (2, 224, 224), (2, 227, 227), (1, 299, 299), (1, 1000, 1003),
    (1, 4096, 4096),
]


def _err(a, b):
    return max(runners.rel_l2(a, b), runners.rel_max(a, b))


def _kw(method, cx, cy, dt):
    return dict(coeff_x=cx, coeff_y=cy, dt=dt)


def _call(method, x, cx, cy, dt, eps=1e-6):
    from cnn_with_pde_b200.functional import tiny_split
    return tiny_split(method, x, cx, cy, dt, eps)


def _oracle(method, u, cx, cy, dt):
    import oracle as O
    return O.tiny_split(method, u, **_kw(method, cx, cy, dt))


def _check(method, u, cx, cy, dt, tol=TOL, what=""):
    import torch
    y = _call(method, torch.from_numpy(u).cuda(), cx, cy, dt).cpu().numpy()
    want = _oracle(method, u, cx, cy, dt)
    assert np.all(np.isfinite(y)), what
    err = _err(y, want)
    assert err <= tol, (what, method, err)
    return y


# ------------------------------------------------------------------------------------------ shapes
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_every_mode_against_oracle(shape):
    u = np.random.RandomState(sum(shape)).randn(*shape).astype(np.float32)
    for method in METHODS:
        _check(method, u, 0.7, 1.9, 0.3, what=shape)


def test_random_configurations():
    """30 seeded draws: H, W 1 ... 1100 with at least one above 64, every mode, coefficients and dt."""
    rs = np.random.RandomState(20261021)
    for n in range(30):
        H, W = int(rs.randint(1, 1101)), int(rs.randint(1, 1101))
        if max(H, W) <= 64:
            H = int(rs.randint(65, 1101))
        B = int(rs.choice([1, 2, 3, 5]))
        method = METHODS[rs.randint(len(METHODS))]
        cx, cy = float(rs.uniform(0, 5)), float(rs.uniform(0, 5))
        dt = float(rs.choice([0.01, 0.1, 0.3, 1.0]))
        u = rs.randn(B, H, W).astype(np.float32)
        _check(method, u, cx, cy, dt, what=f"draw {n}: {B}x{H}x{W} {cx:.3f} {cy:.3f} {dt}")


# --------------------------------------------------------------------------- across the dispatch boundary
@pytest.mark.parametrize("shape", [(3, 64, 100), (2, 33, 4096)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("method", ["solve_implicit_y", "diffuse_y_explicit"])
def test_columns_bit_identical_to_on_chip_kernel(method, shape):
    """Columns are independent in the y modes: the first 64 equal tiny_split_kernel on those 64 alone."""
    import torch
    x = torch.randn(*shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(shape[2]))
    big = _call(method, x, 0.7, 1.9, 0.3)
    small = _call(method, x[:, :, :64].contiguous(), 0.7, 1.9, 0.3)
    assert torch.equal(big[:, :, :64], small)


@pytest.mark.parametrize("shape", [(3, 100, 64), (2, 4096, 33)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("method", ["solve_implicit_x", "diffuse_x_explicit"])
def test_rows_bit_identical_to_on_chip_kernel(method, shape):
    import torch
    x = torch.randn(*shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(shape[1]))
    big = _call(method, x, 0.7, 1.9, 0.3)
    small = _call(method, x[:, :64, :].contiguous(), 0.7, 1.9, 0.3)
    assert torch.equal(big[:, :64, :], small)


@pytest.mark.parametrize("method,shape", [("solve_implicit_y", (2, 6, 4096)), ("solve_implicit_x", (2, 4096, 6))])
def test_clamped_pivots(method, shape):
    """r = -0.3 (the clamped fixture's coefficient): the pivots hit stability_eps on short solved lines."""
    u = np.random.RandomState(6).randn(*shape).astype(np.float32)
    y = _check(method, u, -0.3, -0.3, 1.0, tol=1e-4, what="clamped")
    assert np.max(np.abs(y)) > 1e12   # the clamp acted: every clamped row multiplies by 1 / eps


# ------------------------------------------------------------------------------------------ autograd
@pytest.mark.parametrize("method", METHODS)
def test_gradient_is_the_same_map(method):
    import torch
    gen = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(2, 224, 227, device="cuda", generator=gen).requires_grad_(True)
    g = torch.randn(2, 224, 227, device="cuda", generator=gen)
    _call(method, x, 0.7, 1.9, 0.3).backward(g)
    assert torch.equal(x.grad, _call(method, g, 0.7, 1.9, 0.3))


@pytest.mark.parametrize("shape", [(2, 224, 224), (1, 1000, 1003)], ids=lambda s: "x".join(map(str, s)))
def test_adjoint_identity(shape):
    import torch
    gen = torch.Generator(device="cuda").manual_seed(3)
    v = torch.randn(*shape, device="cuda", generator=gen)
    w = torch.randn(*shape, device="cuda", generator=gen)
    for method in METHODS:
        jv, jw = _call(method, v, 0.7, 1.9, 0.3).double(), _call(method, w, 0.7, 1.9, 0.3).double()
        lhs, rhs = float((jv * w.double()).sum()), float((v.double() * jw).sum())
        scale = float(jv.norm() * w.double().norm())
        assert abs(lhs - rhs) <= 1e-6 * scale, (method, lhs, rhs, scale)


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


def _abi():
    import cnn_with_pde_b200._cabi as cabi
    import cnn_with_pde_b200.functional as F
    return cabi, cabi.lib(), F


@pytest.mark.parametrize("offset", [4, 12])
@pytest.mark.parametrize("shape", [(2, 97, 101), (1, 65, 1), (3, 1, 227), (1, 300, 1001)],
                         ids=lambda s: "x".join(map(str, s)))
def test_abi_guard_bands_unaligned_and_in_place(shape, offset):
    import torch
    cabi, L, F = _abi()
    B, H, W = shape
    stream = torch.cuda.current_stream().cuda_stream
    x = torch.randn(*shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(B * H * W))
    for mode, method in enumerate(METHODS):
        d = F._tiny_split_desc(mode, B, H, W, 0.7, 1.9, 0.3, 1e-6)
        u, out = _Guarded(x.numel() * 4, offset), _Guarded(x.numel() * 4, offset)
        u.view().copy_(x.ravel())
        assert L.pde_tiny_split(byref(d), u.ptr, out.ptr, stream) == 0
        torch.cuda.synchronize()
        assert u.guards_intact() and out.guards_intact(), (mode, shape)
        assert torch.equal(u.view(), x.ravel())
        want = _call(method, x, 0.7, 1.9, 0.3).ravel()
        assert torch.equal(out.view(), want), (mode, shape)
        if mode <= 2:   # the implicit modes may run in place
            assert L.pde_tiny_split(byref(d), u.ptr, u.ptr, stream) == 0
            torch.cuda.synchronize()
            assert u.guards_intact() and torch.equal(u.view(), want), (mode, shape)


def test_indices_past_two_to_the_31():
    """130 planes of 4096^2 (2.18e9 cells, 8.7 GB a tensor) in one call: the last planes against the oracle."""
    import torch
    B, N = 130, 4096
    assert B * N * N > 2 ** 31
    x = torch.empty(B, N, N, device="cuda")
    x[-2:].normal_(generator=torch.Generator(device="cuda").manual_seed(130))
    x[:-2].copy_(x[-2:].repeat(64, 1, 1))
    for method in ("implicit_diffusion_step", "diffuse_y_explicit"):
        y = _call(method, x, 0.7, 1.9, 0.3)
        last = y[-2:].cpu().numpy()
        assert _err(last, _oracle(method, x[-2:].cpu().numpy(), 0.7, 1.9, 0.3)) <= TOL, method
        assert torch.equal(y[:2], y[-2:]), method
        del y
    del x
    torch.cuda.empty_cache()


def test_empty_batch_and_refusals():
    import torch
    cabi, L, F = _abi()
    stream = torch.cuda.current_stream().cuda_stream
    for mode, method in enumerate(METHODS):
        for H, W in ((224, 224), (4096, 4096), (1, 4096)):
            d = F._tiny_split_desc(mode, 0, H, W, 0.7, 1.9, 0.3, 1e-6)
            assert L.pde_tiny_split(byref(d), None, None, stream) == 0
            assert _call(method, torch.empty(0, H, W, device="cuda"), 0.7, 1.9, 0.3).shape == (0, H, W)
        for H, W in ((4097, 8), (8, 4097), (4097, 4097)):
            d = F._tiny_split_desc(mode, 1, H, W, 0.7, 1.9, 0.3, 1e-6)
            x = torch.zeros(1, H, W, device="cuda")
            assert L.pde_tiny_split(byref(d), x.data_ptr(), x.data_ptr(), stream) == cabi.ERR_UNSUPPORTED
            with pytest.raises(cabi.PdeB200Error, match="planes up to 4096 x 4096"):
                _call(method, x, 0.7, 1.9, 0.3)


def test_cuda_graph_capture_of_the_adi_step():
    import torch
    from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer
    layer = ImprovedDiffusionLayer(size=224, use_implicit=True).cuda()
    base = torch.randn(3, 224, 224, device="cuda")
    xs = torch.zeros_like(base)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            layer.implicit_diffusion_step(xs, 0.7, 1.9)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_y = layer.implicit_diffusion_step(xs, 0.7, 1.9)
    xs.copy_(base)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_y, layer.implicit_diffusion_step(base, 0.7, 1.9))
    del graph


def test_autocast_half_input_runs_in_fp32():
    import torch
    from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer
    layer = ImprovedDiffusionLayer(size=227, use_implicit=True).cuda()
    x = torch.randn(2, 227, 227, device="cuda")
    with torch.autocast("cuda", dtype=torch.float16):
        yh = layer.implicit_diffusion_step(x.half(), 0.7, 1.9)
    assert yh.dtype == torch.float32
    assert torch.equal(yh, layer.implicit_diffusion_step(x.half().float(), 0.7, 1.9))


def test_debug_plan_line():
    code = ("import torch\n"
            "from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer\n"
            "m = ImprovedDiffusionLayer(use_implicit=True).cuda()\n"
            "m.implicit_diffusion_step(torch.randn(2, 64, 64, device='cuda'), 0.7, 1.9)\n"
            "m.implicit_diffusion_step(torch.randn(2, 224, 227, device='cuda'), 0.7, 1.9)\n"
            "m.diffuse_y_explicit(torch.randn(2, 300, 20, device='cuda'), 0.3)\n"
            "torch.cuda.synchronize()\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, PDE_B200_DEBUG="1"), timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stderr.splitlines() if "tiny split tiled plan" in ln]
    # nothing for the 64^2 plane, which tiny_split_kernel holds
    assert len(lines) == 2, r.stderr
    assert "mode=0 B=2 H=224 W=227" in lines[0] and "x: grid=" in lines[0] and "y: grid=" in lines[0], lines[0]
    assert "regs=" in lines[0] and "smem=" in lines[0], lines[0]
    assert "mode=4 B=2 H=300 W=20 explicit_y" in lines[1], lines[1]


# ------------------------------------------------------------------------------------------ module
def test_module_methods_at_224():
    import torch
    from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer
    layer = ImprovedDiffusionLayer(size=224, channels=3, dt=0.01, use_implicit=True).cuda()
    u = np.random.RandomState(224).randn(4, 224, 224).astype(np.float32)
    x = torch.from_numpy(u).cuda()
    calls = {
        "implicit_diffusion_step": ((0.7, 1.9), dict(coeff_x=0.7, coeff_y=1.9, dt=0.01)),
        "solve_implicit_x": ((0.9, 0.3), dict(coeff_x=0.9, dt=0.3)),
        "solve_implicit_y": ((2.5, 0.1), dict(coeff_y=2.5, dt=0.1)),
        "diffuse_x_explicit": ((0.11,), dict(coeff_x=0.11, dt=0.01)),
        "diffuse_y_explicit": ((0.13,), dict(coeff_y=0.13, dt=0.01)),
    }
    import oracle as O
    for method, (args, kw) in calls.items():
        y = getattr(layer, method)(x, *args)
        assert y.shape == x.shape and y.dtype == torch.float32
        assert _err(y.cpu().numpy(), O.tiny_split(method, u, **kw)) <= TOL, method
    # forward() still ignores use_implicit, as the reference does (tiny_imagenet.py:21,34-51)
    u4 = torch.randn(2, 3, 224, 224, device="cuda")
    plain = ImprovedDiffusionLayer(size=224, channels=3, dt=0.01, use_implicit=False).cuda()
    assert torch.equal(layer(u4), plain(u4))
