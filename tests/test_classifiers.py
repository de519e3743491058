"""The classifiers around the PDE layers (cnn_with_pde_b200.classifiers) against the reference's.

CPU: same state_dict keys / order / shapes / dtypes as the state_dicts stored from the reference
classifiers, which load unchanged; the launcher's optimiser groups follow cifar10.py:423-434.
GPU: logits, loss and every PDE-parameter gradient of a whole model against fixtures generated
from the unmodified reference (tests/golden/make_golden_models.py), tolerance 1e-5 (north_star).
"""
import os

import numpy as np
import pytest
import torch

from .golden.make_golden_models import MODELS, is_pde_param

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OURS = {
    "mnist": ("mnist_test", "PDEClassifier"),
    "fashion": ("fashion_mnist", "FashionPDEClassifier"),
    "cifar10": ("cifar10", "CIFAR10PDENoConv"),
    "cifar2": ("cifar_2version", "CIFAR10HybridPDEModel"),
    "svhn": ("SVHN", "PDEClassifier"),
    "emotion": ("emotion_recognition", "DiffusionClassifier"),
    "tiny": ("tiny_imagenet", "ImprovedTinyImageNetClassifier"),
}


def ours(name):
    import importlib
    import cnn_with_pde_b200  # noqa: F401
    mod, cls = OURS[name]
    return getattr(importlib.import_module("cnn_with_pde_b200." + mod), cls)()


@pytest.mark.parametrize("name", sorted(MODELS))
def test_state_dict_layout_matches_reference_fixture(name):
    """The whole state_dicts stored from the reference classifiers (tests/golden/model_*.npz): same keys in
    the same order, same shapes and dtypes, and they load into ours unchanged."""
    z = np.load(os.path.join(GOLDEN_DIR, f"model_{name}.npz"))
    rsd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd_")}
    mine = ours(name)
    msd = mine.state_dict()
    assert list(rsd.keys()) == list(msd.keys())
    assert [(tuple(v.shape), v.dtype) for v in rsd.values()] == [(tuple(v.shape), v.dtype) for v in msd.values()]
    mine.load_state_dict(rsd)
    for k, v in mine.state_dict().items():
        assert torch.equal(v, rsd[k]), k


def test_cifar2_optimizer_groups_follow_the_script():
    from cnn_with_pde_b200 import train
    r = train._recipes()["cifar2"]
    model = r.build()
    opt = train.make_optimizer(model, r, capturable=False)
    coef, rest = opt.param_groups
    keys = ("alpha", "beta", "channel_mixing", "combination_weights")
    n_coef = sum(p.numel() for n, p in model.named_parameters() if any(k in n for k in keys))
    assert sum(p.numel() for p in coef["params"]) == n_coef == 2 * (4 * 3 * 32 * 32 + 9) + 4
    assert coef["lr"] == 1e-3 and coef["weight_decay"] == 1e-6
    assert abs(rest["lr"] - 8e-4) < 1e-12 and rest["weight_decay"] == 1e-4


def test_cifar10_optimizer_groups_follow_the_script():
    from cnn_with_pde_b200 import train
    r = train._recipes()["cifar10"]
    model = r.build()
    opt = train.make_optimizer(model, r, capturable=False)
    coef, rest = opt.param_groups
    n_coef = sum(p.numel() for n, p in model.named_parameters() if "alpha" in n or "beta" in n)
    assert sum(p.numel() for p in coef["params"]) == n_coef == 3 * 4 * 3 * 32 * 32
    assert coef["lr"] == 1e-3 and coef["weight_decay"] == 1e-6
    assert rest["lr"] == 5e-4 and rest["weight_decay"] == 1e-4
    assert sum(p.numel() for g in opt.param_groups for p in g["params"]) == sum(p.numel() for p in model.parameters())


def test_launcher_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from cnn_with_pde_b200 import train
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        train.run("mnist", 4, 1, 0, quiet=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS) + ["cifar10/fused"])
def test_whole_model_matches_reference_fixture(name, monkeypatch):
    if name.endswith("/fused"):
        # the three PDE layers of MultiScaleExtractor through one launch per pass (pde_adi_multi_*)
        import cnn_with_pde_b200.classifiers as C
        monkeypatch.setattr(C.MultiScaleExtractor, "fused_branches", True)
        name = name.split("/")[0]
    z = np.load(os.path.join(GOLDEN_DIR, f"model_{name}.npz"))
    model = ours(name)
    model.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd_")})
    model = model.cuda().eval()
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    logits = model(x)
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    tol = 1e-5

    def rel(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))

    assert rel(logits.detach().cpu().numpy(), z["logits"]) <= tol
    assert abs(loss.item() - float(z["loss"])) <= tol * abs(float(z["loss"]))
    checked = 0
    for n, p in model.named_parameters():
        if is_pde_param(n) and ("g_" + n) in z.files:
            assert p.grad is not None, n
            assert rel(p.grad.cpu().numpy(), z["g_" + n]) <= tol, n
            checked += 1
    assert checked >= 4


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_launcher_trains_one_gpu(graph):
    from cnn_with_pde_b200 import train
    out = train.run("fashion", 32, 4, 2, graph=graph, quiet=True)
    assert out["img_per_s"] > 0 and np.isfinite(out["loss"]) and out["cuda_graph"] == graph


@pytest.mark.gpu
@pytest.mark.parametrize("name,batch", [("fashion", 64), ("cifar10", 48)])
def test_graph_captured_step_equals_eager_step(name, batch):
    """The CUDA-graph-captured optimiser step (forward, loss, backward, clipping, fused AdamW) against
    the same step run eagerly: same seed, same synthetic batches, dropout off (its masks come from
    different Philox offsets under capture).  After six steps the loss and every parameter agree to
    the noise of the atomics in stock torch's pooling / embedding backward kernels."""
    from cnn_with_pde_b200 import train
    # the captured run takes GRAPH_PRIMING_STEPS eager steps before it records the graph: same total
    runs = [train.run(name, batch, 4, 2 + (0 if g else train.GRAPH_PRIMING_STEPS), graph=g, quiet=True, no_dropout=True,
                      keep_model=True) for g in (False, True)]
    assert runs[0]["cuda_graph"] is False and runs[1]["cuda_graph"] is True
    assert runs[0]["optimizer_steps"] == runs[1]["optimizer_steps"] == 6 + train.GRAPH_PRIMING_STEPS
    assert abs(runs[0]["loss"] - runs[1]["loss"]) <= 1e-5 * abs(runs[0]["loss"]), (runs[0]["loss"], runs[1]["loss"])
    sd_e, sd_g = runs[0]["_model"].state_dict(), runs[1]["_model"].state_dict()
    worst = 0.0
    for k in sd_e:
        a, b = sd_e[k].double(), sd_g[k].double()
        if a.numel() and a.dtype.is_floating_point:
            worst = max(worst, float((a - b).norm() / a.norm().clamp_min(1e-30)))
    assert worst <= 1e-5, worst
    # the PDE coefficients really moved (the step is not a no-op) and moved identically
    moved = [k for k in sd_e if is_pde_param(k)]
    assert moved
    fresh = train._recipes()[name].build().state_dict()
    assert any(not torch.equal(sd_g[k].cpu(), fresh[k]) for k in moved)


@pytest.mark.gpu
def test_models_survive_deepcopy_and_pickle_after_running():
    """EMA / checkpointing code copies models that have already run: the layers' cached launch plans and the
    extractors' side streams must not get in the way."""
    import copy
    import io
    for name in ("cifar10", "fashion"):
        torch.manual_seed(0)
        model = ours(name).cuda().eval()
        shape = (3, 32, 32) if name == "cifar10" else (1, 28, 28)
        x = torch.randn(4, *shape, device="cuda")
        y = model(x)
        y.sum().backward()
        twin = copy.deepcopy(model)
        buf = io.BytesIO()
        torch.save(model, buf)
        buf.seek(0)
        loaded = torch.load(buf, weights_only=False)
        with torch.no_grad():
            assert torch.allclose(twin(x), y, rtol=1e-5, atol=1e-6) and torch.allclose(loaded(x), y, rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_amp_recipe_scales_unscales_and_steps():
    """--amp is the CIFAR scripts' recipe (cifar10.py:440,458-467): autocast forward, GradScaler.scale(loss)
    .backward(), unscale_, clip_grad_norm_, scaler.step, scaler.update.  The PDE layers stay fp32 inside; the
    run must train (finite loss, parameters move) eagerly and under a CUDA graph."""
    from cnn_with_pde_b200 import train
    for graph in (False, True):
        out = train.run("cifar10", 32, 4, 2, graph=graph, amp=True, quiet=True, keep_model=True)
        assert out["grad_scaler"] is True and out["autocast"] is True and np.isfinite(out["loss"])
        fresh = train._recipes()["cifar10"].build().state_dict()
        sd = out["_model"].state_dict()
        assert any(not torch.equal(sd[k].cpu(), fresh[k]) for k in sd if "alpha_base" in k)


@pytest.mark.gpu
def test_cifar2_hybrid_model_trains_and_branch_order_does_not_matter(monkeypatch):
    """cifar_2version's hybrid model on the B200 diffusion layers: serial and concurrent branches
    give the same logits and PDE gradients; the launcher trains it under a CUDA graph."""
    from cnn_with_pde_b200 import train
    from cnn_with_pde_b200.cifar_2version import CIFAR10HybridPDEModel
    torch.manual_seed(0)
    model = CIFAR10HybridPDEModel().cuda().eval()
    x = torch.randn(6, 3, 32, 32, device="cuda")
    y = torch.randint(0, 10, (6,), device="cuda")
    outs = []
    for serial in ("1", ""):
        if serial:
            monkeypatch.setenv("PDE_B200_SERIAL_BRANCHES", "1")
        else:
            monkeypatch.delenv("PDE_B200_SERIAL_BRANCHES", raising=False)
        model.zero_grad(set_to_none=True)
        logits = model(x)
        torch.nn.functional.cross_entropy(logits, y).backward()
        torch.cuda.synchronize()
        outs.append((logits.detach().clone(), model.feature_extractor.diffusion2.alpha_base.grad.clone(),
                     model.feature_extractor.diffusion1.channel_mixing.grad.clone()))
    for a, b in zip(*outs):
        assert torch.isfinite(a).all() and torch.allclose(a, b, rtol=1e-5, atol=1e-7)
    out = train.run("cifar2", 32, 3, 2, graph=True, quiet=True)
    assert out["img_per_s"] > 0 and np.isfinite(out["loss"])
    out = train.run("tiny", 16, 3, 2, graph=True, quiet=True)     # tiny_imagenet's ResNet behind the explicit layer
    assert out["img_per_s"] > 0 and np.isfinite(out["loss"])
