"""Host-side logic of the streaming implicit kernels (pde_adi_stream_*): their domain, the documented workspace
formulas and the Python routing between them and the shared-memory kernels.  No GPU needed: the queries are pure
functions of the descriptor."""
import ctypes

import pytest

MiB = 1 << 20


def _lib():
    import cnn_with_pde_b200 as P
    return P, P._cabi.lib()


def _desc(P, N, C, steps=2, lie=False, B=2, chan_op=0, skip=False):
    return P.AdiConfig(N=N, C=C, steps=steps, dt=0.01, hx=1.0, hy=1.0, lie=lie, chan_op=chan_op, skip=skip).desc(B, 0)


def _formula(d):
    """include/pde_b200.h: the two workspace sizes of the stream group."""
    P = 2 if d.lie else 3
    cnn = d.C * d.N * d.N
    per = (d.steps + P + 1) * cnn * 4
    K = min(max(d.B, 1), max(1, (1 << 30) // per))
    fwd = 16 * cnn
    bwd = 512 * d.C * d.C * (d.chan_op != 0) + 2048 * int(d.skip) + 16 * cnn + K * per
    return fwd, bwd


def _queries(L, d):
    return (L.pde_adi_stream_forward_workspace_bytes(ctypes.byref(d)),
            L.pde_adi_stream_backward_workspace_bytes(ctypes.byref(d)))


def test_queries_are_nonzero_exactly_on_the_domain():
    P, L = _lib()
    Ns = sorted(set(range(1, 40)) | set(range(120, 140)) | {255, 256, 257, 1000, 2047, 2048, 4095, 4096, 4097, 4100})
    for C in list(range(1, 9)) + [12, 16, 31, 48, 63, 64, 65, 66, 70]:
        for N in Ns:
            d = _desc(P, N, C, steps=1)
            inside = 2 <= N <= 4096 and C <= 64
            f, b = _queries(L, d)
            assert (f > 0) == inside and (b > 0) == inside, (N, C, f, b)
    for steps, lie, inside in ((64, False, True), (65, False, False), (96, True, True), (97, True, False)):
        f, b = _queries(L, _desc(P, 200, 3, steps=steps, lie=lie))
        assert (f > 0) == inside and (b > 0) == inside, (steps, lie)


def test_queries_match_the_documented_formulas():
    P, L = _lib()
    for N, C, steps, lie, B, chan_op, skip in ((2, 1, 0, False, 0, 0, False), (7, 2, 3, True, 5, 1, False),
                                               (224, 1, 10, False, 64, 0, False), (227, 3, 10, False, 8, 2, True),
                                               (56, 64, 2, False, 32, 1, False), (4096, 3, 1, False, 3, 0, False),
                                               (4096, 64, 1, True, 2, 2, True), (512, 1, 64, False, 1000, 0, False)):
        d = _desc(P, N, C, steps=steps, lie=lie, B=B, chan_op=chan_op, skip=skip)
        assert _queries(L, d) == _formula(d), (N, C, steps, lie, B)


def test_large_samples_run_one_at_a_time():
    """3 x 4096^2 at one Strang step: 1 GiB a sample, so one sample in flight whatever the batch."""
    P, L = _lib()
    d = _desc(P, 4096, 3, steps=1, B=16)
    _, b = _queries(L, d)
    assert b == 16 * 3 * 4096 ** 2 + 5 * 3 * 4096 ** 2 * 4


@pytest.mark.parametrize("N,C", [(200, 1), (128, 4), (100, 4), (64, 16), (56, 64)])
def test_routing_picks_the_stream_kernels_beyond_shared_memory(N, C):
    P, L = _lib()
    from cnn_with_pde_b200 import functional as F
    cfg = P.AdiConfig(N=N, C=C, steps=3, dt=0.01, hx=1.0, hy=1.0, chan_op=1 if C > 1 else 0)
    assert L.pde_adi_tables_bytes(ctypes.byref(cfg.desc(2))) == 0
    assert F.adi_route(cfg) == "stream"


@pytest.mark.parametrize("N,C", [(28, 1), (32, 3), (128, 3), (64, 12)])
def test_routing_keeps_the_shared_memory_kernels_where_they_serve(N, C):
    P, _ = _lib()
    from cnn_with_pde_b200 import functional as F
    cfg = P.AdiConfig(N=N, C=C, steps=3, dt=0.01, hx=1.0, hy=1.0, chan_op=1 if C > 1 else 0)
    assert F.adi_route(cfg) == "tables"


@pytest.mark.parametrize("N,C,steps,lie", [(4097, 1, 1, False), (64, 65, 1, False), (300, 3, 65, False),
                                           (300, 3, 97, True), (1, 1, 1, False)])
def test_refusal_names_the_new_domain(N, C, steps, lie):
    P, _ = _lib()
    from cnn_with_pde_b200 import functional as F
    cfg = P.AdiConfig(N=N, C=C, steps=steps, dt=0.01, hx=1.0, hy=1.0, lie=lie)
    with pytest.raises(P._cabi.PdeB200Error, match=r"size 2 \.\.\. 4096, channels <= 64, at most 64 Strang / 96 Lie steps"):
        F.adi_route(cfg)
