"""Layer calls on input and gradient tensors that are views at 4- and 8-byte offsets of their storage.

The half-line ADI kernels move whole planes by 16-byte bulk copies; the module copies such a view to
an aligned buffer before the call, and the results must still be the oracle's.  Two pairs per group
(small batch) and four (forced), plus a layer with a channel mix and a skip connection.
"""
import numpy as np
import pytest

from . import cases as K
from . import runners

pytestmark = pytest.mark.gpu


def _offset_view(a: np.ndarray, offset_floats: int):
    """A cuda tensor holding `a`, starting `offset_floats` floats into a fresh allocation."""
    import torch
    base = torch.zeros(a.size + 4, dtype=torch.float32, device="cuda")
    v = base[offset_floats:offset_floats + a.size].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.data_ptr() % 16 == 4 * offset_floats
    return v


def _run_offset(c, offset_floats):
    import torch
    params, (u, g) = K.make_params(c), K.make_io(c)
    layer = runners.make_cuda_layer(c, params)
    x = _offset_view(u, offset_floats).requires_grad_(True)
    y = layer(x)
    y.backward(_offset_view(g, offset_floats))
    torch.cuda.synchronize()
    got = {"y": y.detach().cpu().numpy(), "gin": x.grad.detach().cpu().numpy()}
    for k, p in layer.named_parameters():
        if p.grad is not None:
            got["g_" + k] = p.grad.detach().cpu().numpy()
    want = runners.run_oracle(c, params=params, io=(u, g), dtype=np.float32)
    return runners.compare(got, want)


@pytest.mark.parametrize("offset_floats", [1, 2])
@pytest.mark.parametrize("pairs", [None, "4"])
def test_fashion_offset_views(offset_floats, pairs, monkeypatch):
    if pairs:
        monkeypatch.setenv("PDE_B200_SPLIT_P", pairs)
    errs = _run_offset(K.case("align_fashion", "fashion", B=13), offset_floats)
    assert max(errs.values()) <= 1e-5, errs


@pytest.mark.parametrize("offset_floats", [1, 2])
def test_cifar10_offset_views(offset_floats):
    c = K.case("align_cifar10", "cifar10", B=5, **K.SCRIPT_INSTANCES["cifar10_pde3"])
    errs = _run_offset(c, offset_floats)
    assert max(errs.values()) <= 1e-5, errs
