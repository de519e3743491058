"""Several implicit layers on one input, one launch per pass (`pde_adi_multi_*`, DESIGN.md section 4.7).

include/pde_b200.h promises that the multi-branch entry points serve any 2 ... 4 layers that agree in B, C, N,
chan_op, skip and tuning, whatever their steps, dt, spacing and splitting; that every gin[i] may be NULL; that
buffers sized by the single-layer queries suffice; and that outputs and grad_input are bit-identical to
single-layer calls.  This file checks each of those against the fp32 oracle and against single-layer calls on
the same module objects.  Every case meant to be fused asserts that the library accepted it
(`functional._adi_multi_plan(...).ok`) and that autograd recorded the multi-branch function, so none of them
can pass by quietly running the layers one by one.

The library builds twelve multi-branch kernels; the named cases reach each of them:

    sfwd_multi_kernel<32, 2, 1, MIX1=1>   cifar2_pair (B 3, 512), mixed_strang_lie, one_step_beside_24
    sfwd_multi_kernel<32, 2, 2, MIX1=1>   cifar2_pair_q2 (PDE_B200_SPLIT_QF=2), big_cifar2_pair (B 3000, Q=2 by default)
    sfwd_multi_kernel<32, 2, 1, MIX1=0>   svhn32_n2, mnist32
    sfwd_multi_kernel<32, 2, 2, MIX1=0>   svhn32_n4_q2, mnist32_q2 (PDE_B200_SPLIT_P=2, _QF=2)
    sfwd_multi_kernel<28, 2, 1, MIX1=1>   cifar10_28_c1, cifar10_28_c2
    sfwd_multi_kernel<28, 2, 2, MIX1=1>   cifar10_28_c2_q2
    sfwd_multi_kernel<28, 2, 1, MIX1=0>   svhn28_n2, mnist_fashion_28
    sfwd_multi_kernel<28, 2, 2, MIX1=0>   svhn28_n4_q2, mnist_fashion_28_q2
    sbwd_multi_kernel<32, 2, CHAN=1>      every 32 x 32 cifar / SVHN case
    sbwd_multi_kernel<32, 2, CHAN=0>      mnist32, mnist32_q2
    sbwd_multi_kernel<28, 2, CHAN=1>      cifar10_28_*, svhn28_*
    sbwd_multi_kernel<28, 2, CHAN=0>      mnist_fashion_28*, the single-channel batch edges

Tolerances: each branch against the fp32 oracle on its own (u, g_i) at 1e-5 (rel-L2 and max-abs / max-ref),
the fused grad_input against the sum of the oracle grad_inputs at 1e-5; against single-layer calls outputs
bit-identical, summed grad_input <= 1e-6 and coefficient gradients <= 2e-6 (rel-L2: the branches share the
resident blocks, so each block sums a different subset of the batch).  The skip-weight gradient and a 1 x 1
channel-matrix gradient (one channel with a channel op) are the ill-conditioned scalars of DESIGN.md section 2
and are judged by the rule of `test_gpu_parity._assert_close_or_as_good_as_fp32`: within three times the fp32
oracle's own distance from the fp64 oracle, plus 1e-5.
"""
import ctypes

import numpy as np
import pytest

from . import cases as K
from . import runners
from .test_gpu_guards import GUARD, Arena

pytestmark = pytest.mark.gpu
TOL = 1e-5
SINGLE_GIN_TOL = 1e-6
SINGLE_GRAD_TOL = 2e-6
MAPS = ("alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff")
SCALARS = ("g_channel_mixing", "g_channel_coupling", "g_skip_weight")


# ------------------------------------------------------------------------------------------------ helpers
def _br(kind, seed, exact=False, perturb=True, **ctor):
    """One branch: (case, parameters).  exact=True sets alpha_base = beta_base = 6 everywhere: with dt = 1,
    unit spacing and Strang splitting the reconstruction bound of DESIGN.md section 4.3 is
    (1 + 4 * 6) * (1 + 4 * 3) = 325 > 256 (per-sweep checkpoints), while 6 +- the perturbed time terms stays
    inside the clamp interval."""
    c = K.case(f"{kind}_{seed}", kind, B=1, perturb=perturb, seed=seed, **ctor)
    p = K.make_params(c)
    if exact:
        for k in ("alpha_base", "beta_base"):
            p[k] = np.full_like(p[k], 6.0)
    return c, p


def _cifar(key, seed, **kw):
    kind = "cifar2" if key.startswith("cifar2") else "cifar10"
    return _br(kind, seed, **dict(K.SCRIPT_INSTANCES[key], **kw))


def _branch(layer):
    chan = getattr(layer, "channel_mixing", None)
    if chan is None:
        chan = getattr(layer, "channel_coupling", None)
    return (layer.alpha_base, layer.beta_base, layer.alpha_time_coeff, layer.beta_time_coeff, chan,
            getattr(layer, "skip_weight", None), layer._config())


def _plan_ok(layers, B):
    import torch
    from cnn_with_pde_b200 import functional as F
    return F._adi_multi_plan(tuple(l._config() for l in layers), B, F.env_tuning(), torch.cuda.current_device()).ok


def _inputs(c, B, n, seed):
    import torch
    gen = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.randn(B, *c.shape, device="cuda", generator=gen)
    return u, [torch.randn(B, *c.shape, device="cuda", generator=gen) for _ in range(n)]


def _distinct(layers):
    out = {}
    for l in layers:
        out.setdefault(id(l), l)
    return list(out.values())


def _run(layers, u, gs, need_gin, fused):
    """Forward + backward of the layers on u, fused (adi_multi_layer) or one call per layer."""
    import torch
    from cnn_with_pde_b200 import functional as F
    for l in _distinct(layers):
        for p in l.parameters():
            p.grad = None
    x = u.clone().requires_grad_(need_gin)
    if fused:
        ys = F.adi_multi_layer(x, [_branch(l) for l in layers])
    else:
        ys = [l(x) for l in layers]
    torch.autograd.backward(list(ys), list(gs))
    torch.cuda.synchronize()
    grads = {id(l): {"g_" + k: p.grad.clone() for k, p in l.named_parameters()} for l in _distinct(layers)}
    return {"ys": [y.detach().clone() for y in ys], "gin": x.grad.clone() if need_gin else None, "grads": grads,
            "fn": type(ys[0].grad_fn).__name__}


def _scalar_keys(c):
    """Gradients that are one number left over from ~1e4 cancelling products: the skip weight always, the
    channel matrix when it is 1 x 1."""
    return set(SCALARS) if c.shape[0] == 1 else {"g_skip_weight"}


def _judge(got, want32, c, o64, what, open_keys=()):
    """<= 1e-5, or for the ill-conditioned scalars of `c` (and `open_keys`, see OPEN_BAR) within 3x the fp32
    oracle's own distance from fp64 plus 1e-5.  o64: callable returning the fp64 oracle values of the same keys."""
    errs = runners.compare(got, want32)
    assert set(errs) == set(got), (sorted(errs), sorted(got))
    bad = {k: e for k, e in errs.items() if not e <= TOL}
    assert set(bad) <= _scalar_keys(c) | set(open_keys), f"{what}: {bad}"
    if bad:
        want64 = o64()
        e_cuda, e_ref = runners.compare(got, want64), runners.compare(want32, want64)
        worse = {k: (e_cuda[k], e_ref[k]) for k in bad if not e_cuda[k] <= 3.0 * e_ref[k] + TOL}
        assert not worse, f"{what}: {worse}"


def _oracle_sum(cs, ps, owners, u_np, g_nps, need_gin, dtype, nthreads=0):
    """Per-branch outputs, the summed grad_input and the parameter gradients summed per owning layer."""
    ys, gin, grads = [], None, {}
    for c, p, o, g in zip(cs, ps, owners, g_nps):
        r = runners.run_oracle(c, params=p, io=(u_np, g), dtype=dtype, need_gin=need_gin, nthreads=nthreads)
        ys.append(r["y"])
        if need_gin:
            gin = r["gin"].astype(np.float64) if gin is None else gin + r["gin"]
        acc = grads.setdefault(o, {})
        for k, v in r.items():
            if k.startswith("g_"):
                acc[k] = np.asarray(v, np.float64) + acc.get(k, 0.0)
    return ys, gin, grads


def check_fused(brs, B, *, need_gin=True, fused=True, alias=None, oracle="full", seed=0, what="", open_keys=()):
    """brs: [(case, params)] per branch; alias {i: j}: branch i runs the layer object of branch j.
    oracle: "full" (whole batch), "ends" (first and last three samples; coefficient gradients against the
    single-layer calls only) or None.  open_keys: gradients known to miss the plain 1e-5 against the oracle
    (OPEN_BAR), held to the ill-conditioned-scalar rule here and to 1e-5 by a strict expected failure."""
    n = len(brs)
    alias = alias or {}
    brs = [brs[alias.get(i, i)] for i in range(n)]
    cs, ps = [b[0] for b in brs], [b[1] for b in brs]
    own = [runners.make_cuda_layer(c, p) for c, p in zip(cs, ps)]
    layers = [own[alias.get(i, i)] for i in range(n)]
    owners = [id(l) for l in layers]
    what = what or "+".join(c.name for c in cs)
    what = f"{what} B={B} gin={need_gin}"
    assert _plan_ok(layers, B) is fused, what
    u, gs = _inputs(cs[0], B, n, seed)
    a = _run(layers, u, gs, need_gin, fused=True)
    assert (a["fn"] == "_AdiMultiFunctionBackward") is fused, (what, a["fn"])
    b = _run(layers, u, gs, need_gin, fused=False)
    # against n single-layer calls on the same module objects
    for i, (ya, yb) in enumerate(zip(a["ys"], b["ys"])):
        assert torch_equal(ya, yb), f"{what}: output {i} differs from the single-layer call"
    if need_gin:
        assert runners.rel_l2(a["gin"].cpu().numpy(), b["gin"].cpu().numpy()) <= SINGLE_GIN_TOL, what
    else:
        assert a["gin"] is None and b["gin"] is None
    u_np, g_nps = u.cpu().numpy(), [g.cpu().numpy() for g in gs]
    o64_cache = {}

    def o64():   # the fp64 oracle on the whole batch, computed at most once
        if "v" not in o64_cache:
            o64_cache["v"] = _oracle_sum(cs, ps, owners, u_np, g_nps, need_gin, np.float64)
        return o64_cache["v"]

    c_of = {o: cs[i] for i, o in reversed(list(enumerate(owners)))}
    for o, ga in a["grads"].items():
        for k, t in ga.items():
            e = runners.rel_l2(t.cpu().numpy(), b["grads"][o][k].cpu().numpy())
            if e <= SINGLE_GRAD_TOL:
                continue
            assert k in _scalar_keys(c_of[o]), f"{what}: {k} {e:.2e} from the single-layer calls"
            w32, w64 = _oracle_sum(cs, ps, owners, u_np, g_nps, need_gin, np.float32)[2][o][k], o64()[2][o][k]
            e_ref = runners.rel_l2(w32, w64)
            assert e <= 3.0 * e_ref + TOL, f"{what}: {k} {e:.2e} from the single-layer calls, fp32 oracle {e_ref:.2e}"
    if oracle == "full":
        ys, gin, grads = _oracle_sum(cs, ps, owners, u_np, g_nps, need_gin, np.float32)
        for i, (y, c) in enumerate(zip(ys, cs)):
            e = runners.compare({"y": a["ys"][i].cpu().numpy()}, {"y": y})["y"]
            assert e <= TOL, f"{what}: output {i} {e:.2e} from the oracle"
        if need_gin:
            e = runners.compare({"gin": a["gin"].cpu().numpy()}, {"gin": gin})["gin"]
            assert e <= TOL, f"{what}: summed grad_input {e:.2e} from the oracle"
        for o, ga in a["grads"].items():
            got = {k: t.cpu().numpy() for k, t in ga.items()}
            _judge(got, grads[o], c_of[o], lambda o=o: o64()[2][o], f"{what} gradients of {c_of[o].name}", open_keys)
    elif oracle == "ends":
        for sl in (slice(0, 3), slice(B - 3, B)):
            ys, gin, _ = _oracle_sum(cs, ps, owners, u_np[sl], [g[sl] for g in g_nps], need_gin, np.float32)
            for i, y in enumerate(ys):
                assert runners.rel_l2(a["ys"][i][sl].cpu().numpy(), y) <= TOL, (what, i, sl)
            if need_gin:
                assert runners.rel_l2(a["gin"][sl].cpu().numpy(), gin) <= TOL, (what, sl)
    return a


def torch_equal(a, b):
    import torch
    return torch.equal(a, b)


# ------------------------------------------------------------------------------- 1. autograd path, named cases
def _named_cases():
    """name -> (branches, batch, environment).  Comments: the multi-branch kernels a case reaches."""
    Q1, P2Q2 = {"PDE_B200_SPLIT_QF": "1"}, {"PDE_B200_SPLIT_P": "2", "PDE_B200_SPLIT_QF": "2"}
    pair = lambda: [_cifar("cifar2_diffusion1", 11), _cifar("cifar2_diffusion2", 12)]   # noqa: E731
    svhn = lambda N, n: [_br("svhn", 20 + i, size=N, channels=3, num_steps=2 + i, dt=[0.01, 0.05, 0.02, 0.1][i])  # noqa: E731
                         for i in range(n)]
    mf28 = lambda: [_br("mnist", 31, num_steps=10), _br("fashion", 32, num_steps=4)]   # noqa: E731
    mn32 = lambda: [_br("mnist", 41, size=32, num_steps=3, dt=0.05), _br("mnist", 42, size=32, num_steps=2, dt=0.3)]  # noqa: E731
    c28 = lambda C, n=2: [_br("cifar10", 50 + i, size=28, channels=C, dt=[0.002, 0.01, 0.005][i], num_steps=2 + i,  # noqa: E731
                              dx=[1.0, 1.5, 2.0][i], dy=1.0) for i in range(n)]
    return {
        # sfwd<32,2,1,1>, sbwd<32,2,1>: cifar_2version's HybridPDEExtractor pair (Lie), its training batch too
        "cifar2_pair_B3": (pair(), 3, {}),
        "cifar2_pair_B512": (pair(), 512, {}),
        # sfwd<32,2,2,1>
        "cifar2_pair_q2": (pair(), 9, {"PDE_B200_SPLIT_QF": "2"}),
        # Strang beside Lie in one launch
        "mixed_strang_lie": ([_cifar("cifar10_pde2", 13), _cifar("cifar2_diffusion1", 14)], 5, {}),
        # sfwd<32,2,1,0> / sfwd<32,2,2,0>, sbwd<32,2,1>: post-step coupling + skip
        "svhn32_n2": (svhn(32, 2), 5, Q1),
        "svhn32_n4_q2": (svhn(32, 4), 17, {"PDE_B200_SPLIT_QF": "2"}),
        # sfwd<28,2,1,0> / sfwd<28,2,2,0>, sbwd<28,2,1>
        "svhn28_n2": (svhn(28, 2), 5, Q1),
        "svhn28_n4_q2": (svhn(28, 4), 6, {"PDE_B200_SPLIT_QF": "2"}),
        # sfwd<28,2,1,0> / sfwd<28,2,2,0>, sbwd<28,2,0>: single channel, smoothing, 10 and 4 steps
        "mnist_fashion_28": (mf28(), 9, Q1),
        "mnist_fashion_28_q2": (mf28(), 9, P2Q2),
        # sfwd<32,2,1,0> / sfwd<32,2,2,0>, sbwd<32,2,0>: the 32 x 32 kernels without a channel op
        "mnist32": (mn32(), 5, {}),
        "mnist32_q2": (mn32(), 7, P2Q2),
        # sfwd<28,2,1,1> / sfwd<28,2,2,1>, sbwd<28,2,1>: 1 x 1 (ill-conditioned) and 2 x 2 channel mixing
        "cifar10_28_c1": (c28(1), 5, Q1),
        "cifar10_28_c2": (c28(2, 3), 3, {}),
        "cifar10_28_c2_q2": (c28(2, 3), 7, {"PDE_B200_SPLIT_QF": "2"}),
        # deal_blocks with very unequal work: 3 sweeps per item beside 72 (beside 90 for the single-channel pair)
        "one_step_beside_24": ([_br("cifar10", 61, dt=0.002, num_steps=1), _br("cifar10", 62, dt=0.0005, num_steps=24)], 7, {}),
        "one_step_beside_30_c1": ([_br("mnist", 63, num_steps=1, dt=0.05), _br("fashion", 64, num_steps=30, dt=0.05)], 5, {}),
        # per-branch call-wide flags (test_per_branch_flags_differ reads them): exact + unclamped beside
        # rebuilt + clamped
        "exact_c1": ([_br("fashion", 71, perturb=False, dt=5.0), _br("mnist", 72)], 6, {}),
        "exact_c3": ([_br("cifar10", 73, exact=True, dt=1.0, num_steps=2), _cifar("cifar10_pde1", 74)], 4, {}),
        "exact_svhn": ([_br("svhn", 75, exact=True, dt=1.0, num_steps=2), _br("svhn", 76, num_steps=3)], 5, {}),
    }


NAMED = _named_cases()


# Open finding, not a fusion defect (the fused gradients equal the single-layer call's to 2e-6): the 3 x 3
# channel-matrix gradient of this case's 24-step layer misses the plain 1e-5 against the fp32 oracle.  It is a
# cancelling sum like the scalars (DESIGN.md section 2: the fp32 oracle itself is up to 1.2e-5 from fp64 on other
# inputs), so here it is held to the ill-conditioned-scalar rule; the plain bar is a strict expected failure of its
# own (test_open_bar_channel_matrix_gradient_after_24_steps), so every other check of the case stays a hard one.
OPEN_BAR = {"one_step_beside_24": ("g_channel_mixing",)}


@pytest.mark.parametrize("name", sorted(NAMED))
def test_fused_branches_match_single_layer_calls_and_oracle(name, monkeypatch):
    brs, B, env = NAMED[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    check_fused(brs, B, what=name, open_keys=OPEN_BAR.get(name, ()))


@pytest.mark.xfail(strict=True, reason="half-line backward: 3 x 3 channel-matrix gradient after 24 Strang steps is "
                                       "1.0e-5 from the fp32 oracle, a cancelling sum (DESIGN.md section 2)")
def test_open_bar_channel_matrix_gradient_after_24_steps():
    """The one comparison OPEN_BAR takes out of one_step_beside_24, at the plain 1e-5: the 24-step branch called
    alone on the same input and upstream gradient (the fused call equals it to 2e-6)."""
    brs, B, _ = NAMED["one_step_beside_24"]
    c, p = brs[1]
    u, gs = _inputs(c, B, len(brs), 0)
    io = (u.cpu().numpy(), gs[1].cpu().numpy())
    got = runners.run_cuda(c, params=p, io=io)
    want = runners.run_oracle(c, params=p, io=io, dtype=np.float32)
    e = runners.compare({"g_channel_mixing": got["g_channel_mixing"]}, want)["g_channel_mixing"]
    assert e <= TOL, e


@pytest.mark.parametrize("B", [1, 2, 3, 5, 17])
def test_fused_branches_at_ragged_batches(B):
    """One sample, pairs and groups cut short in every position of the last item."""
    check_fused([_cifar("cifar2_diffusion1", 81), _cifar("cifar2_diffusion2", 82)], B, what="cifar2_pair")
    check_fused([_br("mnist", 83), _br("fashion", 84), _br("mnist", 85, num_steps=3, dt=0.05)], B, what="c1_triple")


def test_three_channel_exact_mode_single_layer():
    """The half-line kernels in exact mode (per-sweep checkpoints) with three channels, pre-step channel mix or
    post-step coupling + skip: one layer, no fusion.  The checkpoint header proves the mode."""
    c, p = _br("cifar10", 73, exact=True, dt=1.0, num_steps=2)
    assert _single_flags(c, p, 6) == (1, 0)
    c = K.case("cifar10_exact", "cifar10", B=6, seed=73, **c.ctor)
    io = K.make_io(c)
    got = runners.run_cuda(c, params=p, io=io)
    want = runners.run_oracle(c, params=p, io=io, dtype=np.float32)
    errs = runners.compare(got, want)
    assert max(errs.values()) <= TOL, errs
    cs, ps = _br("svhn", 75, exact=True, dt=1.0, num_steps=2)
    assert _single_flags(cs, ps, 5) == (1, 0)
    cs = K.case("svhn_exact", "svhn", B=5, seed=75, **cs.ctor)
    io = K.make_io(cs)
    got = runners.run_cuda(cs, params=ps, io=io)
    want = runners.run_oracle(cs, params=ps, io=io, dtype=np.float32)
    errs = runners.compare(got, want)
    assert max(errs.values()) <= TOL, errs


def test_fused_branches_many_items_per_block():
    """A few thousand samples of a three-channel pair (Q = 2 by default): every branch's blocks walk many
    items.  First and last samples against the oracle, everything against the single-layer calls."""
    check_fused([_cifar("cifar2_diffusion1", 91), _cifar("cifar2_diffusion2", 92)], 3000, oracle="ends", what="big_cifar2_pair")
    check_fused([_br("svhn", 93, num_steps=3), _br("svhn", 94, num_steps=1, dt=0.05)], 2049, oracle="ends", what="big_svhn_pair")


def test_single_channel_fusion_ends_where_four_pairs_per_group_begin():
    """Single-channel layers take four sample pairs per group once (B + 7) // 8 >= 2 * SMs, and the
    multi-branch kernels are built for two: the largest batch below that fuses, the next one falls back.
    Both must match the single-layer calls."""
    import cnn_with_pde_b200 as P
    sms = P._cabi.device_info()["sm_count"]
    first_p4 = 8 * 2 * sms - 7
    assert (first_p4 + 7) // 8 >= 2 * sms > (first_p4 - 1 + 7) // 8
    brs = [_br("mnist", 101, num_steps=3, dt=0.05), _br("fashion", 102)]
    check_fused(brs, first_p4 - 1, oracle="ends", what="c1_last_fused")
    check_fused(brs, first_p4, fused=False, oracle="ends", what="c1_first_p4")


def test_fused_branches_without_grad_input():
    """The models' case: the layers are the first op, the input does not require grad."""
    check_fused([_cifar("cifar2_diffusion1", 111), _cifar("cifar2_diffusion2", 112)], 5, need_gin=False)
    check_fused([_br("svhn", 113), _br("svhn", 114, num_steps=2), _br("svhn", 115, num_steps=1)], 3, need_gin=False)
    check_fused([_br("mnist", 116), _br("fashion", 117)], 4, need_gin=False)


def test_same_layer_twice_sums_its_gradients():
    check_fused([_cifar("cifar10_pde3", 121), _cifar("cifar10_pde3", 121)], 5, alias={1: 0}, what="cifar10_twice")
    check_fused([_br("fashion", 122), _br("mnist", 123), _br("fashion", 122)], 3, alias={2: 0}, what="fashion_twice")


def test_fallbacks_run_the_layers_one_by_one(monkeypatch):
    """n = 1, n = 5, different channels or plane sizes, whole-line tuning: the library refuses the shared
    launch and adi_multi_layer calls the layers one by one, with the same results."""
    check_fused([_cifar("cifar10_pde1", 131)], 3, fused=False, what="n1")
    check_fused([_br("mnist", 132 + i, num_steps=1 + i) for i in range(5)], 3, fused=False, what="n5")
    c3, c2 = _cifar("cifar10_pde1", 137), _br("cifar10", 138, channels=2, dt=0.002, num_steps=2)
    c3d = runners.make_cuda_layer(*c3)
    assert not _plan_ok([c3d, runners.make_cuda_layer(*c2)], 3)   # (no input fits both: the plan alone is asked)
    n28 = _br("cifar10", 139, size=28, dt=0.002, num_steps=2)
    assert not _plan_ok([c3d, runners.make_cuda_layer(*n28)], 3)
    monkeypatch.setenv("PDE_B200_ADI_LEGACY", "1")
    check_fused([_cifar("cifar2_diffusion1", 140), _cifar("cifar2_diffusion2", 141)], 3, fused=False, what="whole_line")


def test_fused_branches_random_configurations(monkeypatch):
    """Seeded sweep: kernel family (cifar Strang / Lie mix, SVHN, single channel), plane edge 28 / 32, channels
    1 ... 3, two to four branches with 1 ... 8 steps and different dt and spacing, ragged batches, Q forced to
    1 or 2 or left automatic, grad_input on / off, occasionally one layer object twice."""
    rs = np.random.RandomState(4711)
    for draw in range(30):
        n, N, B = int(rs.randint(2, 5)), int(rs.choice([28, 32])), int(rs.choice([1, 2, 3, 5, 9, 17, 33]))
        fam = ["cifar", "svhn", "single"][rs.randint(3)]
        C = 1 if fam == "single" else int(rs.randint(1, 4))
        brs = []
        for i in range(n):
            seed, steps = int(rs.randint(1 << 20)), int(rs.randint(1, 9))
            if fam == "cifar":
                kind = ["cifar10", "cifar2"][rs.randint(2)]
                brs.append(_br(kind, seed, size=N, channels=C, num_steps=steps, dt=float(rs.choice([0.001, 0.005, 0.02])),
                               dx=float(rs.choice([1.0, 1.5, 2.0])), dy=float(rs.choice([1.0, 2.0]))))
            elif fam == "svhn":
                brs.append(_br("svhn", seed, size=N, channels=C, num_steps=steps, dt=float(rs.choice([0.01, 0.05])),
                               dx=float(rs.choice([1.0, 1.5]))))
            else:
                kind = ["mnist", "fashion"][rs.randint(2)]
                extra = dict(dy=float(rs.choice([1.0, 1.3]))) if kind == "mnist" else {}
                brs.append(_br(kind, seed, size=N, num_steps=steps, dt=float(rs.choice([0.001, 0.05, 0.3])),
                               dx=float(rs.choice([0.7, 1.0])), **extra))
        qf = int(rs.choice([0, 1, 2]))
        for k in ("PDE_B200_SPLIT_P", "PDE_B200_SPLIT_QF"):
            monkeypatch.delenv(k, raising=False)
        if qf:
            monkeypatch.setenv("PDE_B200_SPLIT_QF", str(qf))
            if fam == "single":
                monkeypatch.setenv("PDE_B200_SPLIT_P", "2")
        alias = {n - 1: 0} if rs.randint(6) == 0 else None
        need_gin = bool(rs.randint(3))
        check_fused(brs, B, need_gin=need_gin, alias=alias, seed=draw,
                    what=f"draw {draw} {fam} N={N} C={C} n={n} qf={qf} alias={alias}")


# ------------------------------------------------------------------------------------- 2. the C ABI, ctypes
def _ptrs(ts):
    arr = (ctypes.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])
    return arr, ctypes.addressof(arr)


def _single_abi(L, d, sched, maps, chan, skw, u, g, P):
    """One layer through pde_adi_prepare / _forward_train / _backward_saved, buffers from torch."""
    import torch
    from cnn_with_pde_b200 import functional as F
    dev = u.device
    nt, nck, nws = L.pde_adi_tables_bytes(ctypes.byref(d)), L.pde_adi_checkpoint_bytes(ctypes.byref(d)), \
        L.pde_adi_backward_saved_workspace_bytes(ctypes.byref(d))
    tables, ckpt, ws = F._bytes(nt, dev), F._bytes(nck, dev), F._bytes(nws, dev)
    out, gin = torch.empty_like(u), torch.empty_like(u)
    gm = [torch.empty_like(m) for m in maps]
    gchan = torch.empty_like(chan) if chan is not None else None
    gskip = torch.empty_like(skw) if skw is not None else None
    st = torch.cuda.current_stream().cuda_stream
    p = lambda t: None if t is None else t.data_ptr()   # noqa: E731
    P._cabi.check(L.pde_adi_prepare(ctypes.byref(d), ctypes.byref(sched), *[p(m) for m in maps], p(tables), st), "prepare")
    P._cabi.check(L.pde_adi_forward_train(ctypes.byref(d), p(tables), p(u), p(chan), p(skw), p(out), p(ckpt), st), "forward")
    P._cabi.check(L.pde_adi_backward_saved(ctypes.byref(d), p(tables), p(u), p(g), p(chan), p(skw), p(ckpt), p(gin),
                                           *[p(t) for t in gm], p(gchan), p(gskip), p(ws), nws, st), "backward")
    return out, gin, gm, gchan, gskip, ckpt


def _ck_flags(ckpt):
    """CkFlags {mode_exact, any_clamped}: the first two int32 of a checkpoint buffer (DESIGN.md section 3)."""
    import torch
    return tuple(int(v) for v in ckpt[:8].view(torch.int32).cpu())


def _single_flags(c, p, B):
    """CkFlags of one single-layer training call of the layer (c, p) through the C ABI."""
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.schedule import adi_schedule
    layer = runners.make_cuda_layer(c, p)
    cfg = layer._config()
    br = [None if t is None else t.detach().contiguous() for t in _branch(layer)[:6]]
    u, gs = _inputs(c, B, 1, 0)
    res = _single_abi(P._cabi.lib(), cfg.desc(B), adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie), br[:4], br[4],
                      br[5], u, gs[0], P)
    return _ck_flags(res[5])


def _abi_case(brs, B, gin_mask, tuning=0, seed=0):
    """The three multi entry points on buffers carved out of one poisoned arena, each sized exactly by the
    single-layer queries.  Checks the guard bands, the results against the oracle and the single-layer
    calls, the workspace / checkpoint refusals; returns each branch's CkFlags {mode_exact, any_clamped}."""
    import torch
    import cnn_with_pde_b200 as P
    from cnn_with_pde_b200.schedule import adi_schedule
    L = P._cabi.lib()
    n = len(brs)
    layers = [runners.make_cuda_layer(c, p) for c, p in brs]
    cfgs = [l._config() for l in layers]
    descs = (P._cabi.AdiDesc * n)(*[cfg.desc(B, tuning) for cfg in cfgs])
    scheds = (P._cabi.AdiSchedule * n)(*[adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie) for cfg in cfgs])
    C, N = cfgs[0].C, cfgs[0].N
    cells = B * C * N * N
    nt = [L.pde_adi_tables_bytes(ctypes.byref(descs[i])) for i in range(n)]
    nck = [L.pde_adi_checkpoint_bytes(ctypes.byref(descs[i])) for i in range(n)]
    nws = [L.pde_adi_backward_saved_workspace_bytes(ctypes.byref(descs[i])) for i in range(n)]
    assert all(nck) and all(nws), (nck, nws)
    A = Arena(sum(nt) + sum(nck) + sum(nws) + n * (8 * cells + 16 * C * N * N + 4 * C * C + 4) + 24 * n * GUARD + 64 * 1024)
    f32 = torch.float32
    tables = [A.take(b) for b in nt]
    ckpt = [A.take(b) for b in nck]
    ws = [A.take(b) for b in nws]
    out = [A.take(4 * cells, f32, (B, C, N, N)) for _ in range(n)]
    gin = [A.take(4 * cells, f32, (B, C, N, N)) if m else None for m in gin_mask]
    gm = [[A.take(4 * C * N * N, f32, tuple(l.alpha_base.shape)) for _ in range(4)] for l in layers]
    chans = [_branch(l)[4] for l in layers]
    skws = [_branch(l)[5] for l in layers]
    chans = [None if t is None else t.detach().contiguous() for t in chans]
    skws = [None if t is None else t.detach().contiguous() for t in skws]
    gch = [A.take(4 * C * C, f32, (C, C)) if t is not None else None for t in chans]
    gsk = [A.take(4, f32, ()) if t is not None else None for t in skws]
    maps = [[getattr(l, k).detach().contiguous() for k in MAPS] for l in layers]
    u, gs = _inputs(brs[0][0], B, n, seed)
    st = torch.cuda.current_stream().cuda_stream
    keep = []

    def arr(ts):
        a, addr = _ptrs(ts)
        keep.append(a)
        return addr

    D, S = ctypes.addressof(descs), ctypes.addressof(scheds)
    ck = lambda: arr(ckpt)   # noqa: E731
    P._cabi.check(L.pde_adi_multi_prepare(n, D, S, *[arr([m[k] for m in maps]) for k in range(4)], arr(tables), st),
                  "pde_adi_multi_prepare")
    P._cabi.check(L.pde_adi_multi_forward_train(n, D, arr(tables), u.data_ptr(), arr(chans), arr(skws), arr(out), ck(), st),
                  "pde_adi_multi_forward_train")
    gin_arr = arr(gin) if any(gin_mask) else None
    gp = [arr([g[k] for g in gm]) for k in range(4)]
    wsb = (ctypes.c_size_t * n)(*nws)

    def backward(wsizes, ckarr):
        return L.pde_adi_multi_backward_saved(n, D, arr(tables), u.data_ptr(), arr(gs), arr(chans), arr(skws), ckarr, gin_arr,
                                              *gp, arr(gch), arr(gsk), arr(ws), ctypes.addressof(wsizes), st)

    # refusals first (nothing is launched): one branch's workspace one byte short of its query, a NULL checkpoint
    short = (ctypes.c_size_t * n)(*nws)
    short[n - 1] -= 1
    assert backward(short, ck()) == P._cabi.ERR_WORKSPACE
    assert backward(wsb, arr(ckpt[:-1] + [None])) == P._cabi.ERR_WORKSPACE
    P._cabi.check(backward(wsb, ck()), "pde_adi_multi_backward_saved")
    torch.cuda.synchronize()
    A.check("multi " + "+".join(c.name for c, _ in brs) + f" B={B}")
    flags = [_ck_flags(c) for c in ckpt]
    # against single-layer calls through the same ABI
    for i in range(n):
        so, sg, sgm, sgc, sgs, _ = _single_abi(L, descs[i], scheds[i], maps[i], chans[i], skws[i], u, gs[i], P)
        assert torch.equal(out[i], so), i
        if gin[i] is not None:
            assert torch.equal(gin[i], sg), i
        c = brs[i][0]
        for k, a, b in zip(MAPS, gm[i], sgm):
            assert runners.rel_l2(a.cpu().numpy(), b.cpu().numpy()) <= SINGLE_GRAD_TOL, (c.name, k)
        for k, a, b in (("g_channel", gch[i], sgc), ("g_skip_weight", gsk[i], sgs)):
            if a is not None and (k == "g_skip_weight" or c.shape[0] > 1):
                assert runners.rel_l2(a.cpu().numpy(), b.cpu().numpy()) <= SINGLE_GRAD_TOL, (c.name, k)
    # against the oracle, branch by branch
    u_np = u.cpu().numpy()
    for i, (c, p) in enumerate(brs):
        g_np = gs[i].cpu().numpy()
        want = runners.run_oracle(c, params=p, io=(u_np, g_np), dtype=np.float32, need_gin=gin[i] is not None)
        got = {"y": out[i].cpu().numpy()}
        if gin[i] is not None:
            got["gin"] = gin[i].cpu().numpy()
        for k, t in zip(MAPS, gm[i]):
            got["g_" + k] = t.cpu().numpy()
        chan_key = "g_channel_mixing" if "channel_mixing" in p else "g_channel_coupling"
        if gch[i] is not None:
            got[chan_key] = gch[i].cpu().numpy()
        if gsk[i] is not None:
            got["g_skip_weight"] = gsk[i].cpu().numpy()
        _judge(got, {k: want[k] for k in got}, c,
               lambda c=c, p=p, g_np=g_np, need=gin[i] is not None: runners.run_oracle(
                   c, params=p, io=(u_np, g_np), dtype=np.float64, need_gin=need), f"abi {c.name} B={B}")
    return flags


def test_multi_abi_stays_inside_single_layer_sized_buffers():
    # cifar_2version's pair, grad_input for the first branch only
    _abi_case([_cifar("cifar2_diffusion1", 201), _cifar("cifar2_diffusion2", 202)], 9, [True, False])
    # four SVHN layers, one of them in exact mode, gin == NULL
    flags = _abi_case([_br("svhn", 203, num_steps=3), _br("svhn", 204, exact=True, dt=1.0, num_steps=2),
                       _br("svhn", 205, num_steps=1, dt=0.05), _br("svhn", 206, num_steps=2)], 6, [False] * 4)
    assert [f[0] for f in flags] == [0, 1, 0, 0], flags
    # three single-channel layers, gin = [buf, NULL, buf]
    _abi_case([_br("mnist", 207), _br("fashion", 208), _br("mnist", 209, num_steps=2, dt=0.05)], 19, [True, False, True])


@pytest.mark.parametrize("name", ["exact_c1", "exact_c3", "exact_svhn"])
def test_per_branch_flags_differ(name):
    """The call-wide flags of the backward pass live in each branch's checkpoint header (DESIGN.md section 3):
    one branch in exact mode (per-sweep checkpoints) and unclamped -- smoothing deferred where the layer
    smooths -- beside one that rebuilds its sweep inputs and has clamped cells, in one launch."""
    brs, B, _ = NAMED[name]
    flags = _abi_case(brs, B, [True, True])
    assert flags[0] == (1, 0) and flags[1] == (0, 1), flags


def _descs(cfgs, B, tuning=0):
    import cnn_with_pde_b200 as P
    return (P._cabi.AdiDesc * len(cfgs))(*[c.desc(B, tuning) for c in cfgs])


def test_multi_abi_error_contract():
    import dataclasses
    import torch
    import cnn_with_pde_b200 as P
    L = P._cabi.lib()
    T = P._cabi.adi_tuning
    cif = [runners.make_cuda_layer(*_cifar(k, 300 + i))._config() for i, k in enumerate(("cifar10_pde1", "cifar10_pde2"))]
    c1 = [runners.make_cuda_layer(*_br(k, 310 + i))._config() for i, k in enumerate(("mnist", "fashion"))]

    def prep(n, ds):
        return L.pde_adi_multi_prepare(n, ctypes.addressof(ds), None, None, None, None, None, None, None)

    assert prep(2, _descs(cif, 8)) == P._cabi.ERR_INVALID        # compatible: only the buffers are missing
    assert prep(4, _descs(cif * 2, 8)) == P._cabi.ERR_INVALID
    assert prep(2, _descs(c1, 8)) == P._cabi.ERR_INVALID
    U = P._cabi.ERR_UNSUPPORTED
    for field, value in (("B", 9), ("C", 2), ("N", 28), ("chan_op", 0), ("skip", 1), ("tuning", T(qf=1))):
        ds = _descs(cif, 8)
        setattr(ds[1], field, value)
        assert prep(2, ds) == U, field
    assert prep(2, _descs(cif, 8, T(impl=P._cabi.TUNE_IMPL_WHOLE_LINE))) == U
    edge30 = [dataclasses.replace(c, N=30) for c in cif]
    assert prep(2, _descs(edge30, 8)) == U                        # run-time-sized kernels: single calls only
    assert prep(2, _descs(c1, 8, T(pairs=4))) == U                # four pairs per group: no multi kernel
    assert prep(1, _descs(cif[:1], 8)) == U
    assert prep(0, _descs(cif, 8)) < 0
    assert prep(5, _descs((cif * 3)[:5], 8)) < 0
    # B = 0: every branch's gradients are zeroed, poison first
    n = 3
    cfg3 = cif + cif[:1]
    ds = _descs(cfg3, 0)
    C, N = 3, 32
    g = [[torch.full((C, N, N), float("nan"), device="cuda") for _ in range(4)] for _ in range(n)]
    gch = [torch.full((C, C), float("nan"), device="cuda") for _ in range(n)]
    keep = []

    def arr(ts):
        a, addr = _ptrs(ts)
        keep.append(a)
        return addr

    st = torch.cuda.current_stream().cuda_stream
    assert L.pde_adi_multi_forward_train(n, ctypes.addressof(ds), None, None, None, None, None, None, st) == 0
    rc = L.pde_adi_multi_backward_saved(n, ctypes.addressof(ds), None, None, None, None, None, None, None,
                                        *[arr([g[i][k] for i in range(n)]) for k in range(4)], arr(gch), None, None, None, st)
    assert rc == 0
    torch.cuda.synchronize()
    for t in [t for row in g for t in row] + gch:
        assert torch.count_nonzero(t).item() == 0 and not torch.isnan(t).any()


# ----------------------------------------------------------------------------- 3. graph capture, the models
def _graph_vs_eager(brs, B, seed):
    import torch
    from cnn_with_pde_b200 import functional as F
    layers = [runners.make_cuda_layer(c, p) for c, p in brs]
    assert _plan_ok(layers, B)
    params = [p for l in layers for p in l.parameters()]
    branches = [_branch(l) for l in layers]
    x = torch.zeros(B, *brs[0][0].shape, device="cuda", requires_grad=True)
    gs = [torch.zeros_like(x) for _ in layers]

    def step():
        ys = F.adi_multi_layer(x, branches)
        torch.autograd.backward(list(ys), gs)
        return ys

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    x.grad = None
    for p in params:
        p.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_ys = step()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(2):   # two replays on new data: the second must not see the first
        u = torch.randn(x.shape, device="cuda", generator=gen)
        g_new = [torch.randn(x.shape, device="cuda", generator=gen) for _ in layers]
        with torch.no_grad():
            x.copy_(u)
            for a, b in zip(gs, g_new):
                a.copy_(b)
        graph.replay()
        torch.cuda.synchronize()
        cap = ([y.clone() for y in static_ys], x.grad.clone(), [p.grad.clone() for p in params])
        xe = u.clone().requires_grad_(True)
        saved = [p.grad for p in params]
        for p in params:
            p.grad = None
        ys = F.adi_multi_layer(xe, branches)
        assert type(ys[0].grad_fn).__name__ == "_AdiMultiFunctionBackward"
        torch.autograd.backward(list(ys), g_new)
        for a, b in zip(cap[0], ys):
            assert torch.equal(a, b.detach())
        assert torch.equal(cap[1], xe.grad)
        for a, p in zip(cap[2], params):
            assert torch.equal(a, p.grad)
        for p, s in zip(params, saved):   # the graph's gradient buffers stay the ones it writes
            p.grad = s
    del graph


def test_graph_captured_fused_step_equals_eager_fused_step():
    """What bench.py times (train.fused_branches): the fused forward + backward captured in a CUDA graph,
    replayed on new data, against an eager fused call -- bit for bit (fixed-order sums, no atomics)."""
    _graph_vs_eager([_cifar(k, 400 + i) for i, k in enumerate(("cifar10_pde1", "cifar10_pde2", "cifar10_pde3"))], 512, 1)
    _graph_vs_eager([_cifar("cifar2_diffusion1", 410), _cifar("cifar2_diffusion2", 411)], 512, 2)


def test_cifar10_training_step_with_fused_branches_graph_equals_eager(monkeypatch):
    import torch
    import cnn_with_pde_b200.classifiers as C
    from cnn_with_pde_b200 import train
    from .golden.make_golden_models import is_pde_param
    monkeypatch.setattr(C.MultiScaleExtractor, "fused_branches", True)
    runs = [train.run("cifar10", 48, 4, 2 + (0 if g else train.GRAPH_PRIMING_STEPS), graph=g, quiet=True, no_dropout=True,
                      keep_model=True) for g in (False, True)]
    assert runs[1]["cuda_graph"] is True
    ext = [m for m in runs[1]["_model"].modules() if isinstance(m, C.MultiScaleExtractor)]
    assert ext and _plan_ok([ext[0].pde1, ext[0].pde2, ext[0].pde3], 48)
    assert abs(runs[0]["loss"] - runs[1]["loss"]) <= 1e-5 * abs(runs[0]["loss"])
    sd_e, sd_g = runs[0]["_model"].state_dict(), runs[1]["_model"].state_dict()
    worst = 0.0
    for k in sd_e:
        a, b = sd_e[k].double(), sd_g[k].double()
        if a.numel() and a.dtype.is_floating_point:
            worst = max(worst, float((a - b).norm() / a.norm().clamp_min(1e-30)))
    assert worst <= 1e-5, worst
    fresh = train._recipes()["cifar10"].build().state_dict()
    assert any(not torch.equal(sd_g[k].cpu(), fresh[k]) for k in sd_e if is_pde_param(k))


def test_cifar2_hybrid_model_fused_branches_on_and_off(monkeypatch):
    import torch
    import cnn_with_pde_b200.classifiers as C
    from cnn_with_pde_b200.cifar_2version import CIFAR10HybridPDEModel
    torch.manual_seed(0)
    model = CIFAR10HybridPDEModel().cuda().eval()
    fe = model.feature_extractor
    B = 6
    x = torch.randn(B, 3, 32, 32, device="cuda")
    y = torch.randint(0, 10, (B,), device="cuda")
    assert _plan_ok([fe.diffusion1, fe.diffusion2], B)
    seen = {}
    fe.register_forward_hook(lambda m, i, o: seen.__setitem__("d", (o[1].detach().clone(), o[2].detach().clone())))
    outs = []
    for fused in (True, False):
        monkeypatch.setattr(C.HybridPDEExtractor, "fused_branches", fused)
        model.zero_grad(set_to_none=True)
        logits = model(x)
        torch.nn.functional.cross_entropy(logits, y).backward()
        torch.cuda.synchronize()
        grads = {n: p.grad.clone() for n, p in model.named_parameters() if ".diffusion" in n}
        outs.append((logits.detach().clone(), seen["d"], grads))
    (la, da, ga), (lb, db, gb) = outs
    assert torch.equal(da[0], db[0]) and torch.equal(da[1], db[1])
    assert runners.rel_l2(la.cpu().numpy(), lb.cpu().numpy()) <= TOL
    assert len(ga) == 10
    for n in ga:
        assert runners.rel_l2(ga[n].cpu().numpy(), gb[n].cpu().numpy()) <= SINGLE_GRAD_TOL, n
