"""Size queries of the implicit layers with 5 ... 64 channels (CPU: no device needed).

Domain: 5 <= C <= PDE_ADI_MAX_CHANNELS (64), 2 <= N <= 128, one sample's planes in one block's shared memory:
C * N * (N | 1) * 4 bytes <= 200 KB.  These layers use the run-time-sized table layout (header + one float4 per
cell and sweep) and keep no checkpoints (the backward pass replays the trajectory).
"""
import ctypes

import pytest


def _lib():
    import cnn_with_pde_b200 as P
    return P, P._cabi.lib()


def _desc(P, N, C, steps=2, lie=False, chan_op=1):
    return P.AdiConfig(N=N, C=C, steps=steps, dt=0.01, hx=1.0, hy=1.0, lie=lie, has_max=True, chan_op=chan_op).desc(3)


def _served(N, C):
    return 5 <= C <= 64 and 2 <= N <= 128 and C * N * (N | 1) * 4 <= 200 * 1024


def test_constants():
    P, _ = _lib()
    assert P._cabi.ADI_MAX_CHANNELS == 64 and P._cabi.MAX_CHANNELS == 4


def test_tables_bytes_is_nonzero_exactly_on_the_domain():
    P, L = _lib()
    for N in range(1, 131):
        for C in range(5, 70):
            d = _desc(P, N, C)
            S = 2 * 3
            want = 4096 + 16 * S * C * N * N if _served(N, C) else 0
            assert L.pde_adi_tables_bytes(ctypes.byref(d)) == want, (N, C)


@pytest.mark.parametrize("N,c_ok", [(32, 48), (64, 12), (16, 64), (101, 5), (28, 63), (48, 21)])
def test_boundaries(N, c_ok):
    P, L = _lib()
    assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, N, c_ok))) > 0, (N, c_ok)
    assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, N, c_ok + 1))) == 0, (N, c_ok + 1)


def test_five_channels_stop_at_101():
    P, L = _lib()
    assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, 101, 5))) > 0
    assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, 102, 5))) == 0


@pytest.mark.parametrize("lie,chan_op,steps", [(False, 1, 5), (True, 1, 96), (False, 2, 64), (False, 0, 1), (False, 1, 0)])
def test_every_variant_and_no_checkpoints(lie, chan_op, steps):
    P, L = _lib()
    for N, C in ((32, 16), (31, 6), (64, 12), (16, 64), (2, 64), (8, 5)):
        d = _desc(P, N, C, steps=steps, lie=lie, chan_op=chan_op)
        S = steps * (2 if lie else 3)
        assert L.pde_adi_tables_bytes(ctypes.byref(d)) == 4096 + 16 * S * C * N * N
        assert L.pde_adi_checkpoint_bytes(ctypes.byref(d)) == 0


def test_sweep_limit_still_applies():
    P, L = _lib()
    assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, 32, 8, steps=65))) == 0        # 195 Strang sweeps
    assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, 32, 8, steps=97, lie=True))) == 0


def test_narrow_channel_rules_are_unchanged():
    """C <= 4 keeps its own limits (C * N <= 384 on the run-time-sized path)."""
    P, L = _lib()
    for N, C in ((100, 4), (128, 4), (200, 1)):
        assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, N, C))) == 0, (N, C)
    for N, C in ((96, 4), (128, 3), (30, 3)):
        assert L.pde_adi_tables_bytes(ctypes.byref(_desc(P, N, C))) == 4096 + 16 * 6 * C * N * N, (N, C)


def test_unsupported_message_names_the_channel_bound():
    P, _ = _lib()
    from cnn_with_pde_b200 import functional as F
    cfg = P.AdiConfig(N=32, C=49, steps=2, dt=0.01, hx=1.0, hy=1.0, has_max=True, chan_op=1)
    with pytest.raises(P._cabi.PdeB200Error, match="channels <= 64"):
        F._AdiPlan(cfg, 2, 0)
