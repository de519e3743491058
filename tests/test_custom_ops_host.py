"""The pde_b200:: custom ops without a GPU: their fake implementations (output dtype, shape and device from the
library's host-only size queries), and tracing of every layer and classifier -- FakeTensor mode, the meta device,
Dynamo with fullgraph=True, torch.export -- without ever entering a compute entry point of the library."""
import ctypes

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import cnn_with_pde_b200 as P
from cnn_with_pde_b200 import classifiers as Cl

OPS = ("adi_fwd", "adi_bwd", "emotion_fwd", "emotion_bwd", "tiny_fwd", "tiny_bwd", "tiny_split")

# (name, class, input shape without the batch, classes)
CLASSIFIERS = [
    ("mnist", Cl.MnistPDEClassifier, (1, 28, 28), 10),
    ("fashion", Cl.FashionPDEClassifier, (1, 28, 28), 10),
    ("svhn", Cl.SvhnPDEClassifier, (3, 32, 32), 10),
    ("emotion", Cl.DiffusionClassifier, (1, 48, 48), 7),
    ("cifar10", Cl.CIFAR10PDENoConv, (3, 32, 32), 10),
    ("cifar2", Cl.CIFAR10HybridPDEModel, (3, 32, 32), 10),
    ("tiny", Cl.ImprovedTinyImageNetClassifier, (3, 64, 64), 200),
]

LAYERS = [
    ("mnist", lambda: P.mnist_test.DiffusionLayer(), (1, 28, 28)),
    ("fashion", lambda: P.fashion_mnist.DiffusionLayer(), (1, 28, 28)),
    ("svhn", lambda: P.SVHN.DiffusionLayer(), (3, 32, 32)),
    ("cifar10", lambda: P.cifar10.EnhancedDiffusionLayer(), (3, 32, 32)),
    ("cifar10_stream", lambda: P.cifar10.EnhancedDiffusionLayer(size=224, channels=1, num_steps=2), (1, 224, 224)),
    ("cifar2", lambda: P.cifar_2version.LearnableDiffusionLayer(), (3, 32, 32)),
    ("emotion", lambda: P.emotion_recognition.PDELayer(), (1, 48, 48)),
    ("emotion_96", lambda: P.emotion_recognition.PDELayer(Nx=96, Ny=96), (1, 96, 96)),
    ("tiny", lambda: P.tiny_imagenet.ImprovedDiffusionLayer(), (3, 64, 64)),
]


@pytest.fixture
def no_passes(monkeypatch):
    """Every compute entry point of the library raises; the size queries (host-only, pure) stay."""
    L = P._cabi.lib()

    def entered(*_):
        raise AssertionError("a pde_b200 compute entry point was called while tracing")

    for name in P._cabi.EXPORTS:
        if name.startswith(("pde_adi", "pde_emotion", "pde_tiny")) and not name.endswith("_bytes"):
            monkeypatch.setattr(L, name, entered)
    return L


def _fake_cuda():
    return FakeTensorMode(allow_non_fake_inputs=False)


def test_every_op_is_registered():
    for name in OPS:
        assert hasattr(torch.ops.pde_b200, name), name
        assert torch._C._dispatch_has_kernel_for_dispatch_key(f"pde_b200::{name}", "Meta"), name


# ---------------------------------------------------------------------------- fake implementations
ADI_CASES = [   # (B, C, N, chan_op, skip, route)
    (4, 1, 28, 0, False, "tables"),
    (4, 3, 32, 1, False, "tables"),
    (4, 1, 48, 0, False, "tables"),
    (3, 12, 64, 1, False, "tables"),
    (1, 1, 224, 0, False, "stream"),
    (2, 64, 56, 2, True, "stream"),
]


@pytest.mark.parametrize("B,C,N,chan_op,skip,route", ADI_CASES)
def test_adi_fake_outputs(no_passes, B, C, N, chan_op, skip, route):
    cfg = P.AdiConfig(N=N, C=C, steps=3, dt=0.01, hx=1.0, hy=1.0, chan_op=chan_op, skip=skip)
    assert P.functional.adi_route(cfg) == route
    L = no_passes
    want_tables = L.pde_adi_tables_bytes(ctypes.byref(cfg.desc(B))) if route == "tables" else 0
    if route == "tables":   # one set of tables per call, whatever the batch
        assert all(L.pde_adi_tables_bytes(ctypes.byref(cfg.desc(b))) == want_tables for b in (1, 2, 7, 64, 1000))
    args = (cfg.N, cfg.C, cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie, cfg.smooth, cfg.has_max, cfg.chan_op, cfg.skip,
            cfg.cmin, cfg.cmax, cfg.eps, 0, True)
    pshape = (C, N, N) if C > 1 else (N, N)
    with _fake_cuda():
        u = torch.empty(B, C, N, N, device="cuda")
        maps = [torch.empty(pshape, device="cuda") for _ in range(4)]
        chan = torch.empty(C, C, device="cuda") if chan_op else None
        skipw = torch.empty((), device="cuda") if skip else None
        out, tables = torch.ops.pde_b200.adi_fwd(u, *maps, chan, skipw, *args)
        assert (out.shape, out.dtype, out.device.type) == (u.shape, torch.float32, "cuda")
        assert (tables.shape, tables.dtype) == ((want_tables,), torch.uint8)
        for need_gin in (True, False):
            gin, gm, gchan, gskip = torch.ops.pde_b200.adi_bwd(out, u, *maps, chan, skipw, tables, *args, need_gin)
            assert gin.shape == (u.shape if need_gin else (0,))
            assert gm.shape == (4,) + pshape and gm.dtype == torch.float32
            assert gchan.shape == ((C, C) if chan_op else (0,))
            assert gskip.shape == (() if skip else (0,))


@pytest.mark.parametrize("N", [48, 96])
def test_emotion_fake_outputs(no_passes, N):
    with _fake_cuda():
        u = torch.empty(5, 1, N, N, device="cuda")
        w6, xs, ys = (torch.empty(6, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, device="cuda"))
        args = (N, 10, 0.001, 1.0 / N, 1.0 / N, False)
        out = torch.ops.pde_b200.emotion_fwd(u, w6, xs, ys, *args)
        assert (out.shape, out.dtype, out.device.type) == (u.shape, torch.float32, "cuda")
        gin, gw = torch.ops.pde_b200.emotion_bwd(out, u, w6, xs, ys, *args, True)
        assert gin.shape == u.shape and gw.shape == (6,)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("size", [64, 224])
def test_tiny_fake_outputs(no_passes, size, dtype):
    with _fake_cuda():
        u = torch.empty(4, 3, size, size, device="cuda", dtype=dtype)
        al, sc = torch.empty(3, device="cuda"), torch.empty(3, device="cuda")
        args = (1, 0.01, 1e-6, 0.15, 0.1)
        out = torch.ops.pde_b200.tiny_fwd(u, al, sc, *args)
        assert (out.shape, out.dtype, out.device.type) == (u.shape, dtype, "cuda")
        gin, ga, gs = torch.ops.pde_b200.tiny_bwd(out, u, al, sc, *args, True)
        assert (gin.shape, gin.dtype) == (u.shape, dtype)
        assert ga.shape == gs.shape == (3,) and ga.dtype == gs.dtype == torch.float32


@pytest.mark.parametrize("method", sorted(P.functional.TINY_SPLIT_MODES))
def test_tiny_split_fake_outputs(no_passes, method):
    layer = P.tiny_imagenet.ImprovedDiffusionLayer()
    with _fake_cuda():
        u = torch.empty(3, 70, 200, device="cuda")
        if method == "implicit_diffusion_step":
            out = layer.implicit_diffusion_step(u, 0.7, 1.9)
        elif method.startswith("solve"):
            out = getattr(layer, method)(u, 0.7, 0.01)
        else:
            out = getattr(layer, method)(u, 0.7)
        assert (out.shape, out.dtype, out.device.type) == (u.shape, torch.float32, "cuda")


# ------------------------------------------------------------------------------------- tracing
@pytest.mark.parametrize("name,cls,shape,classes", CLASSIFIERS, ids=[c[0] for c in CLASSIFIERS])
def test_classifiers_trace_without_the_library(no_passes, name, cls, shape, classes):
    with _fake_cuda(), torch.device("cuda"):
        m = cls()
        assert m(torch.randn(4, *shape)).shape == (4, classes)
    with torch.device("meta"):
        m = cls()
        x = torch.randn(3, *shape)
    y = m(x)
    assert y.shape == (3, classes) and y.is_meta
    y.sum().backward()   # the backward ops' fake implementations
    torch._dynamo.reset()
    y = torch.compile(m, backend="eager", fullgraph=True)(x)
    assert y.shape == (3, classes)


@pytest.mark.parametrize("name,make,shape", LAYERS, ids=[c[0] for c in LAYERS])
def test_layers_export(no_passes, name, make, shape):
    with _fake_cuda(), torch.device("cuda"):
        m = make()
        x = torch.randn(2, *shape)
    ep = torch.export.export(m, (x,), dynamic_shapes=({0: torch.export.Dim("batch")},))
    targets = {str(n.target) for n in ep.graph.nodes if n.op == "call_function"}
    assert any(t.startswith("pde_b200.") for t in targets), targets


@pytest.mark.parametrize("name,cls,shape,classes", CLASSIFIERS, ids=[c[0] for c in CLASSIFIERS])
def test_classifiers_export(no_passes, name, cls, shape, classes):
    with _fake_cuda(), torch.device("cuda"):
        m = cls()
        x = torch.randn(4, *shape)
    ep = torch.export.export(m, (x,))
    out = [n for n in ep.graph.nodes if n.op == "output"][0].args[0][0]
    assert tuple(out.meta["val"].shape) == (4, classes)


def test_real_cpu_tensors_still_refused():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.mnist_test.DiffusionLayer()(torch.randn(2, 1, 28, 28))
