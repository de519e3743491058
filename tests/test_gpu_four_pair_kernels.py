"""The four-pair half-line kernels (adi_split.cu: sfwd_kernel<N, 4, Q>, sbwd_kernel<N, 4>) in the modes the kernel
ledger's rows do not reach: exact mode, the checkpoint-free backward, a compiled training step, and the claim that a
sample's result does not depend on how many pairs share a group (P) or groups share a block (Q).

Single-channel layers without a channel op take four pairs per group once (B + 7) // 8 >= 2 * SMs, so every batch
here is derived from the device's SM count and leaves a ragged last group (B % 8 != 0).  Bar: 1e-5 against the fp32
oracle for the output, grad_input and every coefficient gradient, and no further from the fp64 oracle than the fp32
oracle is, plus 1e-5 (test_gpu_large_batch._check).
"""
import os

import numpy as np
import pytest

from . import cases as K
from . import runners
from .test_gpu_kernel_ledger import profiled, sm_count

pytestmark = pytest.mark.gpu


def _first_p4_batch(extra=2):
    """A batch just past the first one with four pairs per group (16 * SMs - 7), ragged: B % 8 == 1 + extra."""
    return 16 * sm_count() - 7 + extra


def _case(kind, N, B, exact=False, perturb=True):
    ctor = dict(size=N)
    if exact:   # fashion's init with dt = 5: the reconstruction bound (DESIGN.md section 4.3) asks for exact mode
        ctor["dt"], perturb = 5.0, False
    return K.case(f"{kind}{N}{'_exact' if exact else ''}_b{B}", kind, B=B, perturb=perturb, **ctor)


def _oracle_check(c, params, io, got):
    from .test_gpu_large_batch import _check
    nt = os.cpu_count() or 1
    o32 = runners.run_oracle(c, params=params, io=io, dtype=np.float32, nthreads=nt)
    o64 = runners.run_oracle(c, params=params, io=io, dtype=np.float64, nthreads=nt)
    return _check(c, got, o32, o64)


def _four_pair_run(c, params, io, N):
    """runners.run_cuda, asserting that the four-pair forward and backward kernels served it."""
    got, launched, exc = profiled(lambda: runners.run_cuda(c, params=params, io=io))
    if exc is not None:
        raise exc
    assert any(k.startswith(f"adi::split::sfwd_kernel<{N}, 4,") for k in launched), sorted(launched)
    assert f"adi::split::sbwd_kernel<{N}, 4, false>" in launched, sorted(launched)
    return got


@pytest.mark.parametrize("N", [28, 32])
def test_exact_mode_with_four_pairs(N):
    """Exact mode (per-sweep checkpoints; step 0 takes the layer input by bulk copy, zero_tail for the ragged
    group) exists only for four pairs per group.  The checkpoint header proves the mode."""
    from .test_gpu_multi_branch import _single_flags
    B = _first_p4_batch()
    c = _case("fashion", N, B, exact=True)
    params, io = K.make_params(c), K.make_io(c)
    assert _single_flags(c, params, B)[0] == 1, "expected mode_exact in the checkpoint header"
    got = _four_pair_run(c, params, io, N)
    errs = _oracle_check(c, params, io, got)
    print(f"{c.name}: worst rel-err {max(errs.values()):.2e}")


@pytest.mark.parametrize("kind,N,exact", [("fashion", 28, False), ("mnist", 32, False), ("fashion", 28, True),
                                          ("fashion", 32, True)], ids=["fashion28", "mnist32", "fashion28_exact",
                                                                       "fashion32_exact"])
def test_checkpoint_free_backward_with_four_pairs(kind, N, exact, monkeypatch):
    """PDE_B200_NO_CKPT=1: the backward rebuilds the checkpoints in its workspace (pde_adi_backward).  The same
    half-line kernels replay the same trajectory, so grad_input and every gradient equal the saved-checkpoint
    call's bit for bit.  The output does not: a forward with no checkpoints to write is the inference forward
    (whole-line kernels), which rounds differently; it equals the no_grad call's output bit for bit."""
    import torch
    B = _first_p4_batch(extra=4)
    c = _case(kind, N, B, exact=exact)
    params, io = K.make_params(c), K.make_io(c)
    saved = _four_pair_run(c, params, io, N)
    monkeypatch.setenv("PDE_B200_NO_CKPT", "1")
    rebuilt = _four_pair_run(c, params, io, N)
    assert set(saved) == set(rebuilt)
    for k in saved:
        if k != "y":
            assert np.array_equal(saved[k], rebuilt[k]), (c.name, k)
    with torch.no_grad():
        y = runners.make_cuda_layer(c, params)(torch.from_numpy(io[0]).cuda())
    assert np.array_equal(y.cpu().numpy(), rebuilt["y"]), c.name
    _oracle_check(c, params, io, saved)
    _oracle_check(c, params, io, rebuilt)


@pytest.mark.parametrize("kind,N", [("fashion", 28), ("mnist", 32)])
def test_compiled_training_step_with_four_pairs_equals_eager(kind, N):
    """torch.compile(fullgraph=True): the traced backward rebuilds the checkpoints in its own workspace, which is the
    checkpoint-free backward of every compiled mnist / fashion training step at these batches."""
    import torch
    from .test_gpu_compile import _run, _same
    c = _case(kind, N, _first_p4_batch(extra=6))
    m = runners.make_cuda_layer(c, K.make_params(c))
    x = torch.from_numpy(K.make_io(c)[0]).cuda()
    eager = _run(m, m, x)
    compiled = torch.compile(m, fullgraph=True)
    got, launched, exc = profiled(lambda: _run(compiled, m, x))
    if exc is not None:
        raise exc
    assert f"adi::split::sbwd_kernel<{N}, 4, false>" in launched, sorted(launched)
    _same(got, eager)


# tuning -> the forward kernel it selects at _first_p4_batch(): pairs per group and groups per block
_LAYOUTS = [({}, 4, 1), ({"PDE_B200_SPLIT_QF": "2"}, 4, 2), ({"PDE_B200_SPLIT_QF": "4"}, 4, 4),
            ({"PDE_B200_SPLIT_P": "2", "PDE_B200_SPLIT_QF": "1"}, 2, 1), ({"PDE_B200_SPLIT_P": "2", "PDE_B200_SPLIT_QF": "2"}, 2, 2)]


@pytest.mark.parametrize("kind,N", [("fashion", 28), ("mnist", 32)])
def test_pairs_and_groups_per_block_do_not_change_a_sample(kind, N, monkeypatch):
    """The per-sample arithmetic does not depend on P or Q: the output and grad_input of every layout are
    bit-identical.  (The coefficient gradients are sums over the batch in a layout-dependent order.)"""
    c = _case(kind, N, _first_p4_batch(extra=0))
    params, io = K.make_params(c), K.make_io(c)
    ref = None
    for env, P, Q in _LAYOUTS:
        for k in ("PDE_B200_SPLIT_P", "PDE_B200_SPLIT_QF"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        got, launched, exc = profiled(lambda: runners.run_cuda(c, params=params, io=io))
        if exc is not None:
            raise exc
        assert f"adi::split::sfwd_kernel<{N}, {P}, {Q}, false>" in launched, (env, sorted(launched))
        if ref is None:
            ref = got
            _oracle_check(c, params, io, got)
            continue
        for k in ("y", "gin"):
            d = np.abs(got[k].astype(np.float64) - ref[k])
            assert np.array_equal(got[k], ref[k]), (env, k, float(d.max()), int(np.count_nonzero(d)))
