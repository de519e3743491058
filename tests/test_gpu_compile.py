"""The PDE layers under torch.compile(fullgraph=True) and torch.export: the pde_b200:: custom ops pass
torch.library.opcheck, and a traced layer runs the same kernels with the same plans as the eager autograd.Function,
so its outputs and gradients are bit-identical to eager."""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn as nn

import cnn_with_pde_b200 as P
from cnn_with_pde_b200 import classifiers as Cl

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LAYERS = [   # (id, constructor, input shape without the batch)
    ("mnist", lambda: P.mnist_test.DiffusionLayer(), (1, 28, 28)),
    ("fashion", lambda: P.fashion_mnist.DiffusionLayer(), (1, 28, 28)),
    ("svhn", lambda: P.SVHN.DiffusionLayer(), (3, 32, 32)),
    ("cifar10", lambda: P.cifar10.EnhancedDiffusionLayer(num_steps=5), (3, 32, 32)),
    ("cifar10_generic48", lambda: P.cifar10.EnhancedDiffusionLayer(size=48, num_steps=3), (3, 48, 48)),
    ("cifar10_wide", lambda: P.cifar10.EnhancedDiffusionLayer(size=64, channels=12, num_steps=2), (12, 64, 64)),
    ("cifar10_stream", lambda: P.cifar10.EnhancedDiffusionLayer(size=224, channels=1, num_steps=2), (1, 224, 224)),
    ("svhn_stream", lambda: P.SVHN.DiffusionLayer(size=56, channels=64, num_steps=2), (64, 56, 56)),
    ("cifar2", lambda: P.cifar_2version.LearnableDiffusionLayer(num_steps=5), (3, 32, 32)),
    ("emotion", lambda: P.emotion_recognition.PDELayer(), (1, 48, 48)),
    ("emotion_96", lambda: P.emotion_recognition.PDELayer(Nx=96, Ny=96), (1, 96, 96)),
    ("tiny", lambda: P.tiny_imagenet.ImprovedDiffusionLayer(), (3, 64, 64)),
    ("tiny_224", lambda: P.tiny_imagenet.ImprovedDiffusionLayer(size=224), (3, 224, 224)),
]


def _perturb(m, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(0.05 * torch.randn(p.shape, device="cuda", generator=g))
    return m


def _run(fn, m, x, seed=1):
    """Output, grad_input and every parameter gradient of one forward + backward."""
    m.zero_grad(set_to_none=True)
    x = x.detach().clone().requires_grad_(True)
    y = fn(x)
    g = torch.randn(y.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    y.backward(g)
    return [y.detach(), x.grad] + [p.grad for _, p in m.named_parameters() if p.grad is not None]


def _same(a, b):
    assert len(a) == len(b)
    for i, (s, t) in enumerate(zip(a, b)):
        assert s.dtype == t.dtype and s.shape == t.shape, i
        assert torch.equal(s, t), (i, (s - t).abs().max().item())


# ------------------------------------------------------------------------------------ opcheck
def _opcheck_cases():
    B = 3
    cases = []
    for C, N, chan_op, skip in ((1, 28, 0, False), (3, 32, 1, False), (1, 48, 0, False), (12, 64, 1, False),
                                (1, 224, 0, False), (64, 56, 2, True)):
        cfg = P.AdiConfig(N=N, C=C, steps=2, dt=0.01, hx=1.0, hy=1.0, smooth=True, chan_op=chan_op, skip=skip)
        pshape = (C, N, N) if C > 1 else (N, N)
        maps = [(1.0 + 0.1 * torch.rand(pshape, device="cuda")).requires_grad_() for _ in range(4)]
        chan = (torch.eye(C, device="cuda") + 0.01).requires_grad_() if chan_op else None
        skipw = torch.tensor(0.9, device="cuda", requires_grad=True) if skip else None
        u = torch.randn(1 if N == 224 else B, C, N, N, device="cuda", requires_grad=True)
        args = (cfg.N, cfg.C, cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie, cfg.smooth, cfg.has_max, cfg.chan_op, cfg.skip,
                cfg.cmin, cfg.cmax, cfg.eps, 0, True)
        cases.append((f"adi_{C}x{N}", torch.ops.pde_b200.adi_fwd, (u, *maps, chan, skipw, *args)))
    for N in (48, 96):
        u = torch.randn(B, 1, N, N, device="cuda", requires_grad=True)
        w6 = torch.tensor([0.1, 0.1, 0.1, 0.3, 0.2, 0.2], device="cuda", requires_grad=True)
        xs = torch.linspace(0, 1, N, device="cuda")
        cases.append((f"emotion_{N}", torch.ops.pde_b200.emotion_fwd, (u, w6, xs, xs.clone(), N, 10, 0.001, 1 / N, 1 / N, False)))
    for N in (64, 224):
        for dt in (torch.float32, torch.bfloat16):
            u = torch.randn(B, 3, N, N, device="cuda").to(dt).requires_grad_()
            al = torch.full((3,), 0.05, device="cuda", requires_grad=True)
            sc = torch.ones(3, device="cuda", requires_grad=True)
            cases.append((f"tiny_{N}_{dt}", torch.ops.pde_b200.tiny_fwd, (u, al, sc, 1, 0.01, 1e-6, 0.15, 0.1)))
    for mode in range(5):
        u = torch.randn(B, 70, 200, device="cuda", requires_grad=True)
        cases.append((f"tiny_split_{mode}", torch.ops.pde_b200.tiny_split, (u, mode, 0.7, 1.9, 0.01, 1e-6)))
    return cases


def test_opcheck_every_op():
    for name, op, args in _opcheck_cases():
        torch.library.opcheck(op, args, test_utils=("test_schema", "test_autograd_registration", "test_faketensor",
                                                    "test_aot_dispatch_dynamic"))
    # the backward ops, on what the forward ops hand them
    with torch.no_grad():
        _opcheck_backward_ops()


def _opcheck_backward_ops():
    for name, op, args in _opcheck_cases()[:1] + _opcheck_cases()[6:7] + _opcheck_cases()[8:9]:
        out = op(*args)
        gout = torch.randn_like(out[0] if isinstance(out, tuple) else out)
        if op is torch.ops.pde_b200.adi_fwd:
            bargs = (gout, *[a.detach() if isinstance(a, torch.Tensor) else a for a in args[:7]], out[1].detach(),
                     *args[7:], True)
            torch.library.opcheck(torch.ops.pde_b200.adi_bwd, bargs)
        elif op is torch.ops.pde_b200.emotion_fwd:
            torch.library.opcheck(torch.ops.pde_b200.emotion_bwd,
                                  (gout, *[a.detach() for a in args[:4]], *args[4:], True))
        else:
            torch.library.opcheck(torch.ops.pde_b200.tiny_bwd, (gout, *[a.detach() for a in args[:3]], *args[3:], True))


# ------------------------------------------------------------------------- bit-identical to eager
@pytest.mark.parametrize("name,make,shape", LAYERS, ids=[c[0] for c in LAYERS])
def test_compiled_and_exported_layers_match_eager_bitwise(name, make, shape):
    torch.manual_seed(0)
    m = _perturb(make().cuda())
    x = torch.randn(4 if shape[-1] < 200 else 2, *shape, device="cuda")
    want = _run(m, m, x)
    torch._dynamo.reset()
    _same(_run(torch.compile(m, fullgraph=True), m, x), want)
    ep = torch.export.export(m, (x,))
    _same(_run(ep.module(), m, x), want)


def test_compiled_whole_line_variant_matches_eager_bitwise(monkeypatch):
    """The whole-line implicit kernels: the switch reaches the traced call too."""
    monkeypatch.setenv("PDE_B200_ADI_LEGACY", "1")
    torch.manual_seed(0)
    m = _perturb(P.fashion_mnist.DiffusionLayer().cuda())
    x = torch.randn(8, 1, 28, 28, device="cuda")
    want = _run(m, m, x)
    torch._dynamo.reset()
    _same(_run(torch.compile(m, fullgraph=True), m, x), want)


def test_compiled_generic_emotion_variant_matches_eager(monkeypatch):
    """The generic emotion kernels: output and grad_input bit for bit.  They sum the six weight gradients with float
    atomics, so those agree up to the summation order only (as between two eager calls)."""
    monkeypatch.setenv("PDE_B200_EMO_TILED", "0")
    torch.manual_seed(0)
    m = _perturb(P.emotion_recognition.PDELayer().cuda())
    x = torch.randn(8, 1, 48, 48, device="cuda")
    want = _run(m, m, x)
    torch._dynamo.reset()
    got = _run(torch.compile(m, fullgraph=True), m, x)
    _same(got[:2], want[:2])
    for g, w in zip(got[2:], want[2:]):
        torch.testing.assert_close(g, w, rtol=1e-6, atol=0)


def test_tiny_split_compiled_matches_eager_bitwise():
    layer = P.tiny_imagenet.ImprovedDiffusionLayer().cuda()
    u = torch.randn(3, 70, 200, device="cuda")
    for method, args in (("implicit_diffusion_step", (0.7, 1.9)), ("solve_implicit_x", (0.7, 0.01)),
                         ("solve_implicit_y", (0.7, 0.01)), ("diffuse_x_explicit", (0.7,)), ("diffuse_y_explicit", (0.7,))):
        fn = lambda v: getattr(layer, method)(v, *args)   # noqa: E731
        want = _run(fn, layer, u)
        torch._dynamo.reset()
        _same(_run(torch.compile(fn, fullgraph=True), layer, u), want)


# ---------------------------------------------------------------------------------- dynamic batch
@pytest.mark.parametrize("name", ["fashion", "svhn", "cifar10_stream", "emotion", "tiny"])
def test_dynamic_batch_compiles_once(name, monkeypatch):
    make, shape = {c[0]: (c[1], c[2]) for c in LAYERS}[name]
    torch.manual_seed(0)
    m = _perturb(make().cuda())
    torch._dynamo.reset()
    monkeypatch.setattr(torch._dynamo.config, "error_on_recompile", True)
    fn = torch.compile(m, fullgraph=True)
    x0 = torch.randn(2, *shape, device="cuda").requires_grad_()
    torch._dynamo.mark_dynamic(x0, 0)
    fn(x0).sum().backward()
    for B in (3, 5, 64):
        x = torch.randn(B, *shape, device="cuda")
        _same(_run(fn, m, x), _run(m, m, x))


# ------------------------------------------------------------------------------------ classifiers
CLASSIFIERS = [("mnist", Cl.MnistPDEClassifier, (1, 28, 28), 10), ("fashion", Cl.FashionPDEClassifier, (1, 28, 28), 10),
               ("svhn", Cl.SvhnPDEClassifier, (3, 32, 32), 10), ("emotion", Cl.DiffusionClassifier, (1, 48, 48), 7),
               ("cifar10", Cl.CIFAR10PDENoConv, (3, 32, 32), 10), ("cifar2", Cl.CIFAR10HybridPDEModel, (3, 32, 32), 10),
               ("tiny", Cl.ImprovedTinyImageNetClassifier, (3, 64, 64), 200)]

PDE_TYPES = (P.mnist_test.DiffusionLayer, P.fashion_mnist.DiffusionLayer, P.SVHN.DiffusionLayer,
             P.cifar10.EnhancedDiffusionLayer, P.emotion_recognition.PDELayer, P.tiny_imagenet.ImprovedDiffusionLayer)


def _train_step(model, fn, x, y):
    """One training step (forward, loss, backward, AdamW): the loss and the gradients."""
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    opt.zero_grad(set_to_none=True)
    loss = nn.functional.cross_entropy(fn(x), y)
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    opt.step()
    return loss.detach(), grads


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("name,cls,shape,classes", CLASSIFIERS, ids=[c[0] for c in CLASSIFIERS])
def test_classifiers_compile_fullgraph(name, cls, shape, classes, monkeypatch):
    import copy
    # fp32 throughout: with TF32 the eager (cuDNN) and Inductor convolutions and matmuls round differently
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    torch.manual_seed(0)
    model = cls().cuda()
    for mod in model.modules():
        if isinstance(mod, nn.Dropout):
            mod.p = 0.0
    twin = copy.deepcopy(model)
    x = torch.randn(16, *shape, device="cuda")
    y = torch.randint(0, classes, (16,), device="cuda")
    # every PDE layer of these classifiers reads the network input: compiled, its output is the eager one bit for bit
    layers = [(n, mod) for n, mod in model.named_modules() if isinstance(mod, PDE_TYPES)]
    assert layers
    for n, mod in layers:
        torch._dynamo.reset()
        assert torch.equal(torch.compile(mod, fullgraph=True)(x), mod(x)), n
    loss_e, grads_e = _train_step(model, model, x, y)
    torch._dynamo.reset()
    loss_c, grads_c = _train_step(twin, torch.compile(twin, fullgraph=True), x, y)
    assert _rel(loss_c, loss_e) <= 1e-4
    assert grads_c.keys() == grads_e.keys()
    # relative to each gradient, with a floor at 1e-4 of the largest one: the bias of a linear layer that a batch
    # norm follows has a gradient that is zero up to rounding, whose relative error says nothing
    floor = 1e-4 * max(g.double().norm().item() for g in grads_e.values())
    for k in grads_e:
        diff = (grads_c[k].double() - grads_e[k].double()).norm().item()
        assert diff <= 1e-4 * grads_e[k].double().norm().item() + floor, k


def test_reduce_overhead_matches_default_mode():
    torch.manual_seed(0)
    model = Cl.CIFAR10PDENoConv().cuda().eval()
    x = torch.randn(64, 3, 32, 32, device="cuda")
    torch._dynamo.reset()
    want = torch.compile(model, fullgraph=True)(x).clone()
    torch._dynamo.reset()
    fn = torch.compile(model, fullgraph=True, mode="reduce-overhead")
    for _ in range(3):
        got = fn(x).clone()
    assert torch.equal(got, want)


# ----------------------------------------------------------------------------------- behaviour kept
def test_compiled_autocast_and_once_differentiable():
    torch.manual_seed(0)
    m = P.cifar10.EnhancedDiffusionLayer().cuda()
    fn = torch.compile(m, fullgraph=True)
    x = torch.randn(4, 3, 32, 32, device="cuda", dtype=torch.float16, requires_grad=True)
    with torch.autocast("cuda", dtype=torch.float16):
        y = fn(x)
    assert y.dtype == torch.float32
    y.sum().backward()
    assert x.grad.dtype == torch.float16
    # a second derivative is never taken silently: eager and exported modules refuse create_graph=True in the
    # layer's own backward; a torch.compile'd graph's backward is refused by torch itself, either at
    # create_graph=True or when the second derivative is asked for
    x2 = torch.randn(4, 3, 32, 32, device="cuda", requires_grad=True)
    with pytest.raises(RuntimeError, match="once differentiable"):
        torch.autograd.grad(m(x2).sum(), x2, create_graph=True)
    ep = torch.export.export(m, (x2,)).module()
    with pytest.raises(RuntimeError, match="once differentiable"):
        torch.autograd.grad(ep(x2).sum(), x2, create_graph=True)
    with pytest.raises(RuntimeError):
        g, = torch.autograd.grad(fn(x2).sum(), x2, create_graph=True)
        torch.autograd.grad(g.sum(), x2)


@pytest.mark.parametrize("model", ["mnist", "fashion", "cifar10", "cifar2", "svhn", "emotion", "tiny"])
def test_train_compile_runs(model):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "train.py"), "--model", model, "--compile", "--steps", "5",
                        "--warmup", "1", "--batch", "32"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert '"compiled": true' in r.stdout


def test_train_compile_rejects_graph():
    from cnn_with_pde_b200.train import run
    with pytest.raises(ValueError, match="exclusive"):
        run("fashion", 8, 1, 0, graph=True, compile=True)
