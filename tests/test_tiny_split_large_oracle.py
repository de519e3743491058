"""The oracle of tiny_imagenet's dormant methods (tiny_imagenet.py:88-233) on planes beyond 64 x 64.

The stored fixtures pin the oracle to the reference up to 64 x 64 only, so its larger planes are pinned to
independent solvers here.  For r >= 0 every pivot is at least 1 + r >= 1 (denom_i = 1 + 2r - r^2 / denom_{i-1} >
1 + r once denom_{i-1} >= 1 + r), so the clamp at stability_eps never acts and the implicit modes are exact
tridiagonal solves: the fp64 oracle is compared with scipy.linalg.solve_banded.  The explicit modes are restated
in numpy with the oracle's operation order, bit-exact in fp32 and fp64.  Clamped pivots stay covered by the
fixtures of tests/test_tiny_split.py.
"""
import numpy as np
import pytest

from . import runners

SHAPES = [(2, 1, 4096), (2, 4096, 1), (1, 2, 4096), (1, 224, 227), (1, 1000, 1003)]
IMPLICIT = ("implicit_diffusion_step", "solve_implicit_x", "solve_implicit_y")
EXPLICIT = ("diffuse_x_explicit", "diffuse_y_explicit")
# (coeff_x, coeff_y, dt): the model's init values, moderate r, and r = 100 (pivots far from 1 + 2r)
COEFFS = [(0.05, 0.05, 0.01), (0.7, 1.9, 0.3), (50.0, 200.0, 1.0)]


def _solve_lines(u, bands):
    """Solve the tridiagonal system of `bands` = (a, b_mid, b_end) along the last axis of u (fp64)."""
    from scipy.linalg import solve_banded
    n = u.shape[-1]
    a, bmid, bend = (float(v) for v in bands)
    ab = np.zeros((3, n))
    ab[0, 1:] = a
    ab[1, :] = bmid
    ab[1, 0] = ab[1, -1] = bend
    ab[2, :-1] = a
    rhs = u.reshape(-1, n).T
    return solve_banded((1, 1), ab, rhs).T.reshape(u.shape)


def _explicit_lines(u, k):
    """explicit_line along the last axis, in the oracle's order: u + k (u[i-1] - 2 u[i] + u[i+1]), one-sided ends."""
    out = u.copy()
    n = u.shape[-1]
    if n < 2:
        return out
    t = u.dtype.type
    k = t(k)
    out[..., 1:-1] = u[..., 1:-1] + k * ((u[..., :-2] - t(2) * u[..., 1:-1]) + u[..., 2:])
    out[..., 0] = u[..., 0] + k * (u[..., 1] - u[..., 0])
    out[..., -1] = u[..., -1] + k * (u[..., -2] - u[..., -1])
    return out


def _kw(method, cx, cy, dt):
    return dict(coeff_x=cx, coeff_y=cy, dt=dt)


@pytest.mark.parametrize("coeffs", COEFFS, ids=lambda c: f"cx{c[0]}_cy{c[1]}_dt{c[2]}")
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("method", IMPLICIT)
def test_implicit_modes_are_exact_tridiagonal_solves(method, shape, coeffs):
    import oracle as O
    cx, cy, dt = coeffs
    u = np.random.RandomState(sum(shape) + int(10 * cx)).randn(*shape)
    got = O.tiny_split(method, u, **_kw(method, cx, cy, dt))
    bx, by = O.tiny_split_coefficients(O.TINY_SPLIT_MODES[method], cx, cy, dt, np.float64)
    want = u
    if method != "solve_implicit_y":
        want = _solve_lines(want, bx)
    if method != "solve_implicit_x":
        want = np.swapaxes(_solve_lines(np.swapaxes(want, 1, 2), by), 1, 2)
    assert max(runners.rel_l2(got, want), runners.rel_max(got, want)) <= 1e-12


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("method", EXPLICIT)
def test_explicit_modes_match_numpy_restatement(method, shape, dtype):
    import oracle as O
    u = np.random.RandomState(sum(shape)).randn(*shape).astype(dtype)
    coeff, dt = 0.37, 0.3
    got = O.tiny_split(method, u, coeff_x=coeff, coeff_y=coeff, dt=dt)
    k = O.tiny_split_coefficients(O.TINY_SPLIT_MODES[method], coeff, coeff, dt, dtype)[0][0]
    if method == "diffuse_x_explicit":
        want = _explicit_lines(u, k)
    else:
        want = np.swapaxes(_explicit_lines(np.swapaxes(u, 1, 2), k), 1, 2)
    np.testing.assert_array_equal(got, want)
