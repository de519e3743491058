"""The torch restatement of tiny_imagenet's diffusion layer (tests/tiny_reference.py) against the C oracle (CPU).

The oracle's hand-derived adjoint was tied to the reference only by the stored fixtures at 16 x 16 and 64 x 64.
The GPU tests of the tiled kernels compare against the oracle at odd, rectangular and one-cell planes, so here
the oracle's forward and every gradient are pinned, in fp64, to autograd over the reference step at those shapes.
"""
import numpy as np
import pytest

from . import tiny_reference as TR

SHAPES = ((1, 1), (1, 9), (9, 1), (7, 7), (13, 31), (64, 64), (227, 227))
STEPS = (0, 1, 2, 5, 16)


def _err(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    den = max(np.max(np.abs(b)) if b.size else 0.0, 1e-300)
    return float(np.max(np.abs(a - b)) / den) if b.any() else float(np.max(np.abs(a), initial=0.0))


@pytest.mark.parametrize("H,W", SHAPES, ids=lambda v: str(v))
@pytest.mark.parametrize("steps", STEPS)
def test_oracle_matches_the_torch_reference(H, W, steps):
    for C, clamp in ((1, False), (2, True), (3, False)) if H * W < 50000 else ((3, True),):
        B = 2 if H * W < 50000 else 1
        u, g, al, sc = TR.make_inputs(B, C, H, W, seed=H * 1000 + W * 10 + steps + C, clamp=clamp)
        for need_gin in (True, False):
            want = TR.run(u, g, al, sc, steps, need_gin=need_gin)
            got = TR.oracle(u, g, al, sc, steps, need_gin=need_gin)
            for k in ("y", "gin", "alpha_base", "channel_scaling"):
                if not need_gin and k == "gin":
                    assert got[k] is None
                    continue
                assert _err(got[k], want[k]) <= 1e-12, (H, W, steps, C, need_gin, k, _err(got[k], want[k]))
            if clamp:
                assert got["alpha_base"][0] == 0.0 and want["alpha_base"][0] == 0.0


def test_clamped_and_unclamped_channels_differ_only_in_the_alpha_gradient():
    u, g, al, sc = TR.make_inputs(2, 2, 5, 11, seed=3)
    r = TR.run(u, g, al, sc, 3)
    assert np.all(r["alpha_base"] != 0.0)
    al2 = al.copy()
    al2[0] = np.float32(0.3)
    r2 = TR.oracle(u, g, al2, sc, 3)
    assert r2["alpha_base"][0] == 0.0 and r2["alpha_base"][1] != 0.0

