"""The torch restatement of emotion_recognition.PDELayer (tests/emotion_reference.py) against the C oracle (CPU).

The stored fixtures tie the oracle to the reference at 48 x 48 only.  The GPU tests of the halo kernels
(emotion_halo.cu) compare against the oracle from 65 x 65 up, so here the oracle's forward and every gradient
are pinned, in fp64, to autograd over the reference step at those plane sizes: a stable coefficient set
(a + b <= 1/2) and the reference's default init, which amplifies.
"""
import numpy as np
import pytest

from . import emotion_reference as ER

SIZES = (65, 96, 100, 127, 224)
STEPS = (0, 1, 10, 16)


def _err(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    den = np.max(np.abs(b)) if b.size else 0.0
    return float(np.max(np.abs(a - b)) / den) if den > 0 else float(np.max(np.abs(a), initial=0.0))


@pytest.mark.parametrize("N", SIZES)
@pytest.mark.parametrize("Nt", STEPS)
def test_oracle_matches_the_torch_reference(N, Nt):
    for name, w in (("stable", ER.stable_weights(N, seed=N + Nt)), ("default", np.array(ER.DEFAULT_W, np.float32))):
        u, g = ER.make_inputs(2, N, seed=N * 100 + Nt)
        for need_gin in (True, False):
            want = ER.run(u, g, w, Nt, need_gin=need_gin)
            got = ER.oracle(u, g, w, Nt, need_gin=need_gin)
            for k in ("y", "gin", "w"):
                if not need_gin and k == "gin":
                    assert got[k] is None
                    continue
                e = _err(got[k], want[k])
                assert e <= 1e-12, (N, Nt, name, need_gin, k, e)


def test_stable_weights_do_not_amplify():
    N = 127
    w = ER.stable_weights(N, seed=3).astype(np.float64)
    xs, ys = ER.buffers(N, np.float64)
    a = 0.5 * 0.001 * (w[0] + w[1] * np.sin(2 * np.pi * ys) + w[2] * np.sin(4 * np.pi * ys)) * N * N
    b = 0.001 * (w[3] + w[4] * np.cos(2 * np.pi * xs) + w[5] * np.cos(4 * np.pi * xs)) * N * N
    assert np.max(np.abs(a)) + np.max(np.abs(b)) <= 0.5
    u, g = ER.make_inputs(1, N, seed=4)
    y = ER.run(u, g, w, 16)["y"]
    assert np.max(np.abs(y)) <= np.max(np.abs(u)) * 1.0001
