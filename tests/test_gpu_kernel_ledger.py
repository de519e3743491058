"""Every kernel of the library, launched by a case that compares its results with the oracle (tests/kernel_ledger.py).

Each row runs under torch.profiler; the test asserts that the row's kernels are among the `pde::` kernels of the
trace, then holds the results to the bar of the suite for that layer:

- implicit layers (module rows): 1e-5 against the fp32 oracle (rel-L2 and max-abs / max-ref) for the output,
  grad_input and every parameter gradient, and no further from the fp64 oracle than the fp32 oracle is, plus 1e-5;
  above eight channels tests/adi_reference.py takes the oracle's place.  The channel-matrix and skip-weight
  gradients, cancelling sums, are held to the ill-conditioned-scalar rule where they miss the plain bar
  (test_gpu_wide_channels._judge);
- multi-branch rows: test_gpu_multi_branch.check_fused;
- emotion and tiny_imagenet rows: the fp32 layer against the oracle, and the bf16 layer bit for bit against the fp32
  layer on the widened input (and against the oracle within a bf16 unit);
- tiny_imagenet's dormant methods against the oracle.

The last test asserts that the rows together launched every kernel of the library and prints one line per row
(run with -s to see it).
"""
import os

import numpy as np
import pytest

from . import cases as K
from . import kernel_ledger as KL
from . import runners

pytestmark = pytest.mark.gpu

_LAUNCHED = {}   # row name -> normalised pde:: kernels its case launched
_SUMMARY = {}    # row name -> summary line
_RAW = set()     # a few kernel names as the profiler spells them


def sm_count():
    import cnn_with_pde_b200 as P
    return P._cabi.device_info()["sm_count"]


def profiled(fn):
    """(fn()'s result, the normalised names of the pde:: kernels it launched, the exception it raised or None)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    res, exc = None, None
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            res = fn()
            torch.cuda.synchronize()
        except Exception as e:   # the kernels it launched are still reported
            exc = e
    raw = {e.name for e in prof.events() if KL.normalise(e.name)}
    for n in sorted(raw):
        if "<" in n and len(_RAW) < 4:
            _RAW.add(n)
    return res, {KL.normalise(n) for n in raw}, exc


# ------------------------------------------------------------------------------------------------ runners
def _module(spec, name):
    """One implicit layer through its module; returns the worst error against the fp32 reference."""
    import torch
    from .test_gpu_wide_channels import _judge, _tame
    c = K.case(name, spec["kind"], B=KL.batch(spec["B"], sm_count()), perturb=spec["perturb"], seed=spec["seed"],
               **spec["ctor"])
    params = K.make_params(c)
    if c.shape[0] > 4:   # long runs of wide channel matrices stay O(1)
        params = _tame(c, params)
    io = K.make_io(c)
    if spec["no_grad"]:
        layer = runners.make_cuda_layer(c, params)
        with torch.no_grad():
            got = {"y": layer(torch.from_numpy(io[0]).cuda()).cpu().numpy()}
    else:
        got = runners.run_cuda(c, params=params, io=io, need_gin=spec["need_gin"])
        want = {"y"} | ({"gin"} if spec["need_gin"] else set()) | {"g_" + k for k in K.grad_names(c)}
        assert {k for k, v in got.items() if v is not None} == want, (name, sorted(got))
    errs = _judge(got, c, params, io, spec["need_gin"] and not spec["no_grad"], name, nthreads=os.cpu_count() or 1)
    return max(errs.values())


def _multi(spec, name, monkeypatch):
    from . import test_gpu_multi_branch as MB
    brs, B, env = MB.NAMED[spec["name"]]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    MB.check_fused(brs, B, what=name, open_keys=MB.OPEN_BAR.get(spec["name"], ()))


def _emotion(spec, name):
    from . import emotion_reference as ER
    from .test_gpu_emotion_bf16 import _check_bits
    from .test_gpu_emotion_shapes import _check
    N, Nt, B = spec["N"], spec["Nt"], spec["B"]
    u, g = ER.make_inputs(B, N, seed=N + Nt)
    _check(u, g, ER.stable_weights(N, N + Nt), Nt, what=name)
    _check_bits(N, Nt, B, True, seed=N + Nt, oracle=True)


def _tiny(spec, name):
    import torch
    from . import tiny_reference as TR
    from .test_gpu_tiny_shapes import _check, _check_bf16, _run
    u, g, al, sc = TR.make_inputs(spec["B"], spec["C"], spec["H"], spec["W"], seed=spec["H"] + spec["steps"], clamp=True)
    if not spec.get("bf16"):
        _check(u, g, al, sc, spec["steps"], what=name)
        return
    _check_bf16(u, g, al, sc, spec["steps"], what=name)
    ub = torch.from_numpy(u).bfloat16().float().numpy()
    gb = torch.from_numpy(g).bfloat16().float().numpy()
    got16 = _run(u, g, al, sc, spec["steps"], bf16=True)
    got32 = _run(ub, gb, al, sc, spec["steps"])
    for k in ("y", "gin"):   # the fp32 arithmetic on the widened planes, rounded once
        want = torch.from_numpy(got32[k]).bfloat16().float().numpy()
        assert np.array_equal(got16[k], want), (name, k, float(np.mean(got16[k] != want)))


def _tiny_split(spec, name):
    from .test_gpu_tiny_split_shapes import METHODS, _check
    u = np.random.RandomState(sum(spec["shape"])).randn(*spec["shape"]).astype(np.float32)
    for method in METHODS:
        _check(method, u, 0.7, 1.9, 0.3, what=name)


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("row", KL.ROWS, ids=lambda r: r.name)
def test_row_launches_its_kernels_and_matches_the_oracle(row, monkeypatch):
    import cnn_with_pde_b200.functional as F
    for k, v in row.env.items():
        monkeypatch.setenv(k, v)
    if not row.env:
        assert F.env_tuning() == 0, "a PDE_B200_* tuning switch is set: the rows without one must run the default dispatch"
    run = {"module": lambda: _module(row.spec, row.name), "multi": lambda: _multi(row.spec, row.name, monkeypatch),
           "emotion": lambda: _emotion(row.spec, row.name), "tiny": lambda: _tiny(row.spec, row.name),
           "tiny_split": lambda: _tiny_split(row.spec, row.name)}[row.run]
    worst, launched, exc = profiled(run)
    _LAUNCHED[row.name] = launched
    missing = sorted(set(row.kernels) - launched)
    assert not missing, f"{row.name}: not launched {missing}; launched {sorted(launched)}; comparison raised {exc!r}"
    if exc is not None:
        raise exc
    err = "within the bar" if worst is None else f"worst rel-err {worst:.2e}"
    _SUMMARY[row.name] = f"{row.name}: {err}; {', '.join(row.kernels)}"


def test_rows_together_launch_every_kernel_of_the_library():
    """Runs after the rows (same module): the union of what they launched is the library's kernel set."""
    from .test_kernel_ledger_host import library_kernels
    if set(_LAUNCHED) != {r.name for r in KL.ROWS}:
        pytest.skip("only a subset of the rows ran")
    launched = set().union(*_LAUNCHED.values())
    have = library_kernels()
    for r in KL.ROWS:
        print("ledger", _SUMMARY.get(r.name, f"{r.name}: FAILED"))
    print(f"ledger: {len(launched & have)} of {len(have)} kernels launched; profiler spelling: {sorted(_RAW)[:4]}")
    assert not sorted(have - launched), f"never launched: {sorted(have - launched)}"
    assert len(_SUMMARY) == len(KL.ROWS), f"rows that failed: {sorted({r.name for r in KL.ROWS} - set(_SUMMARY))}"
