"""The emotion layer's bf16 planes without a GPU: the custom ops' fake implementations (bf16 grad_input, fp32 weight
gradient), tracing of a bf16 module, and the bf16 backward workspace query of the halo kernels (host-only)."""
import ctypes

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import cnn_with_pde_b200 as P

from .test_custom_ops_host import no_passes  # noqa: F401  (fixture)


@pytest.mark.parametrize("N", [48, 96])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_emotion_fake_outputs_follow_the_planes(no_passes, N, dtype):  # noqa: F811
    with FakeTensorMode(allow_non_fake_inputs=False):
        u = torch.empty(5, 1, N, N, device="cuda", dtype=dtype)
        w6, xs, ys = (torch.empty(6, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, device="cuda"))
        args = (N, 10, 0.001, 1.0 / N, 1.0 / N, False)
        out = torch.ops.pde_b200.emotion_fwd(u, w6, xs, ys, *args)
        assert (out.shape, out.dtype) == (u.shape, dtype)
        for need_gin in (True, False):
            gin, gw = torch.ops.pde_b200.emotion_bwd(out, u, w6, xs, ys, *args, need_gin)
            assert (gin.shape, gin.dtype) == ((u.shape if need_gin else (0,)), dtype)
            assert (gw.shape, gw.dtype) == ((6,), torch.float32)


@pytest.mark.parametrize("convert", ["bfloat16", "half", "double"])
def test_converted_module_traces_with_fp32_weights(no_passes, convert):  # noqa: F811
    """A converted module's weights reach the op widened to fp32; its output follows the input (bf16 or fp32)."""
    with torch.device("meta"):
        m = getattr(P.emotion_recognition.PDELayer(), convert)()
        for dtype in (torch.float32, torch.bfloat16):
            x = torch.randn(3, 1, 48, 48, dtype=dtype)
            y = m(x)
            assert y.dtype == dtype and y.shape == x.shape
            y.float().sum().backward()
            assert all(p.grad.dtype == p.dtype for p in m.parameters())
            m.zero_grad(set_to_none=True)


def test_bf16_classifier_exports(no_passes):  # noqa: F811
    m = P.emotion_recognition.DiffusionClassifier().bfloat16()   # (export fakes the CPU tensors itself)
    x = torch.randn(4, 1, 48, 48, dtype=torch.bfloat16)
    ep = torch.export.export(m, (x,))
    out = [n for n in ep.graph.nodes if n.op == "output"][0].args[0][0]
    assert tuple(out.meta["val"].shape) == (4, 7) and out.meta["val"].dtype == torch.bfloat16


@pytest.mark.parametrize("B,N,Nt", [(2, 65, 0), (2, 65, 1), (3, 100, 10), (130, 512, 16), (1, 4096, 16)])
def test_halo_bf16_workspace(B, N, Nt):
    """Above 64 the bf16 backward needs the fp32 workspace plus one fp32 [slot][4][N] side buffer (chunk slots: the
    fp32 chunking, min(B, 512) where the planes are small)."""
    L = P._cabi.lib()
    d = P._cabi.EmoDesc(B, N, Nt, 0.0005, 0.001, 1.0 / N ** 2, 1.0 / N ** 2, 0)
    ws32 = L.pde_emotion_backward_workspace_bytes(ctypes.byref(d))
    ws16 = L.pde_emotion_backward_workspace_bytes_bf16(ctypes.byref(d))
    assert ws32 > 0 and ws16 > ws32
    extra = ws16 - ws32
    assert extra % (4 * N * 4) == 0
    chunk = extra // (4 * N * 4)
    assert 1 <= chunk <= min(B, 512)
    if Nt <= 1 and N < 1000:
        assert chunk == min(B, 512)


def test_refused_descriptors_have_no_bf16_workspace():
    L = P._cabi.lib()
    for N, Nt in ((65, 17), (4096, 17), (4097, 1), (2, 1)):
        d = P._cabi.EmoDesc(1, N, Nt, 0.0005, 0.001, 1.0 / N ** 2, 1.0 / N ** 2, 0)
        assert L.pde_emotion_backward_workspace_bytes_bf16(ctypes.byref(d)) == 0

