"""The torch restatement of the channel-aware implicit layers (tests/adi_reference.py) against the oracle (CPU).

Where both serve, they must agree: the forward at every channel count (the oracle's forward takes any C), and
every gradient at C <= 8 (the oracle's adjoint keeps an 8 x 8 channel-gradient array).  The restatement's
gradients come from autograd over the same code for every C, so agreement at C <= 8 carries to the wide layers;
a finite-difference check at 12 channels covers the channel-matrix and skip-weight gradients there directly.
"""
import numpy as np
import pytest

from . import adi_reference as AR
from . import cases as K
from . import runners

KINDS = ("cifar10", "cifar2", "svhn")


def _err(a, b):
    return max(runners.rel_l2(a, b), runners.rel_max(a, b))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("C", (1, 3, 5, 8))
def test_gradients_match_the_oracle_up_to_eight_channels(kind, C):
    c = K.case(f"ref_{kind}_{C}", kind, B=3, size=9 if C < 8 else 7, channels=C, num_steps=3, seed=60 + C)
    want = runners.run_oracle(c, dtype=np.float64, nthreads=1)
    got = AR.run(c, dtype=np.float64)
    assert set(got) == set(want), (sorted(got), sorted(want))
    for k in want:
        e = _err(got[k], want[k])
        assert e <= 1e-10, (k, e)
    # fp32: the same operations in the same order
    want32 = runners.run_oracle(c, dtype=np.float32, nthreads=1, forward_only=True)
    got32 = AR.run(c, dtype=np.float32)
    assert _err(got32["y"], want32["y"]) <= 1e-6


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("C,N", ((12, 8), (33, 5), (64, 3)))
def test_forward_matches_the_oracle_at_any_channel_count(kind, C, N):
    c = K.case(f"ref_fwd_{kind}_{C}", kind, B=2, size=N, channels=C, num_steps=2, seed=70 + C)
    params = K.make_params(c)
    for k in ("channel_mixing", "channel_coupling"):
        if k in params:
            params[k] = (np.eye(C) + 0.2 / np.sqrt(C) * np.random.RandomState(C).randn(C, C)).astype(np.float32)
    io = K.make_io(c)
    for dtype, tol in ((np.float64, 1e-12), (np.float32, 1e-6)):
        want = runners.run_oracle(c, params=params, io=io, dtype=dtype, nthreads=1, forward_only=True)
        got = AR.run(c, params=params, io=io, dtype=dtype, need_gin=False)
        assert _err(got["y"], want["y"]) <= tol, dtype


@pytest.mark.parametrize("kind", ("cifar10", "svhn"))
def test_finite_differences_at_twelve_channels(kind):
    """fp64 central differences of sum(gout * y) for every channel-matrix entry, the skip weight, sampled map
    entries and grad_input."""
    C, N = 12, 6
    c = K.case(f"ref_fd_{kind}", kind, B=2, size=N, channels=C, num_steps=2, dt=0.02)
    rs = np.random.RandomState(7)
    base = 1.0 if kind == "cifar10" else 0.1      # maps well inside the clamp interval: a smooth loss
    p = {k: np.asarray(v, np.float64) for k, v in K.default_params(c).items()}
    for k in ("alpha_base", "beta_base"):
        p[k] = base * (1.0 + 0.2 * rs.rand(C, N, N))
    for k in ("alpha_time_coeff", "beta_time_coeff"):
        p[k] = 0.05 * base * rs.randn(C, N, N)
    mk = "channel_mixing" if kind == "cifar10" else "channel_coupling"
    p[mk] = np.eye(C) + 0.3 / np.sqrt(C) * rs.randn(C, C)
    if "skip_weight" in p:
        p["skip_weight"] = np.array(0.4)
    u, g = rs.randn(2, C, N, N), rs.randn(2, C, N, N)
    r = AR.run(c, params=p, io=(u, g), dtype=np.float64)

    def loss(pp, uu):
        y = runners.run_oracle(c, params=pp, io=(uu, g), dtype=np.float64, forward_only=True, nthreads=1)["y"]
        return float(np.sum(y * g))

    h = 1e-5
    checks = [(mk, q) for q in range(C * C)] + [(k, int(q)) for k in AR.MAP_KEYS for q in rs.choice(C * N * N, 4, replace=False)]
    if "skip_weight" in p:
        checks.append(("skip_weight", 0))
    for key, q in checks:
        vals = []
        for sgn in (1, -1):
            pp = {k: np.array(v, np.float64) for k, v in p.items()}
            pp[key].reshape(-1)[q] += sgn * h
            vals.append(loss(pp, u))
        want = (vals[0] - vals[1]) / (2 * h)
        got = float(np.asarray(r["g_" + key]).reshape(-1)[q])
        assert abs(got - want) <= 1e-6 * max(1.0, float(np.max(np.abs(r["g_" + key])))), (key, q, got, want)
    for q in rs.choice(u.size, 6, replace=False):   # linear in u
        uu = u.copy().reshape(-1)
        uu[q] += 1.0
        want = loss(p, uu.reshape(u.shape)) - loss(p, u)
        assert abs(float(r["gin"].reshape(-1)[q]) - want) <= 1e-9 * max(1.0, abs(want)), q


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("need_gin", (True, False))
def test_zero_steps(kind, need_gin):
    c = K.case(f"ref_zero_{kind}", kind, B=2, size=5, channels=6, num_steps=0)
    want = runners.run_oracle(c, dtype=np.float64, nthreads=1, need_gin=need_gin)
    got = AR.run(c, dtype=np.float64, need_gin=need_gin)
    for k in want:
        if want[k] is not None:
            assert _err(got[k], want[k]) <= 1e-12, k
