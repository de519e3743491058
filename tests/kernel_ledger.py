"""The kernel ledger: every `__global__` instantiation the library builds, and a small case that launches it.

A row is one case plus the set of kernels that case must launch.  `tests/test_kernel_ledger_host.py` checks, without
a GPU, that the union of the rows equals the set of kernels in the built library (so a kernel added without a row, or
a row left behind by a deleted kernel, fails there); `tests/test_gpu_kernel_ledger.py` runs every row under
torch.profiler, asserts that the row's kernels were launched, and compares the row's results with the oracle or the
reference the rest of the suite uses for that layer.

Kernel names are kept in one normalised spelling (`normalise`): the `pde::` namespace, `void`, the parameter list and
the integer casts `cu++filt` prints are dropped, and `(bool)0` / `(bool)1` become `false` / `true`.

Adding a kernel: add its name to the row whose case launches it, or add a row.  A row's `run` names the runner in
tests/test_gpu_kernel_ledger.py that executes `spec`:

    module       one layer through its nn.Module (tests/runners.py), forward + backward (or no_grad), against the
                 fp32 and fp64 oracle; above eight channels against tests/adi_reference.py
    multi        several layers on one input through the multi-branch launch (test_gpu_multi_branch.check_fused),
                 spec["name"] is one of its named cases
    emotion      the emotion layer in fp32 against the oracle, and in bf16 bit for bit against the fp32 layer on
                 the widened input
    tiny         the tiny_imagenet layer against the oracle (fp32, or bf16 within one bf16 unit and bit for bit
                 against the fp32 layer on the widened input)
    tiny_split   tiny_imagenet's dormant methods against the oracle

A batch written as "sm * a + b" is derived from the device's SM count, because the library chooses several kernels
from the batch per SM.
"""
from __future__ import annotations

import re
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple

_CAST = re.compile(r"\((?:unsigned |signed )?(?:int|long|long long|short|char)\)")


def normalise(name: str) -> Optional[str]:
    """One spelling for a kernel name from cu++filt or from the profiler; None for a name outside namespace pde.

    >>> normalise("pde::adi::split::sfwd_kernel<(int)28, (int)4, (int)1, (bool)0>(pde::adi::split::Args)")
    'adi::split::sfwd_kernel<28, 4, 1, false>'
    >>> normalise("void pde::adi::split::sfwd_kernel<28, 4, 1, false>(pde::adi::split::Args)")
    'adi::split::sfwd_kernel<28, 4, 1, false>'
    """
    s = name.strip()
    if s.startswith("void "):
        s = s[5:]
    s = s.replace("(bool)0", "false").replace("(bool)1", "true")
    s = _CAST.sub("", s)
    depth = 0
    for i, ch in enumerate(s):   # the parameter list: the first '(' outside the template arguments
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            s = s[:i]
            break
    s = re.sub(r"\s*,\s*", ", ", s.strip())
    if not s.startswith("pde::"):
        return None
    return s[len("pde::"):]


@dataclass(frozen=True)
class Row:
    name: str
    kernels: Tuple[str, ...]
    run: str
    spec: Dict = field(default_factory=dict)
    env: Dict = field(default_factory=dict)


def _m(name, kernels, kind, B, ctor=None, env=None, perturb=True, seed=1234, need_gin=True, no_grad=False):
    spec = dict(kind=kind, B=B, ctor=dict(ctor or {}), perturb=perturb, seed=seed, need_gin=need_gin, no_grad=no_grad)
    return Row(name, tuple(kernels), "module", spec, dict(env or {}))


def _whole(N, chan=False, np2=False):
    return (f"adi::prepare_kernel<{N}>", f"adi::fwd_kernel<{N}, {2 if np2 else 1}>",
            f"adi::bwd_kernel<{N}, {'true' if chan else 'false'}>", "adi::finish_kernel")


def _split(N, P, Q, mix1=False, chan=False):
    return (f"adi::prepare_kernel<{N}>", f"adi::split::sfwd_kernel<{N}, {P}, {Q}, {'true' if mix1 else 'false'}>",
            f"adi::split::sbwd_kernel<{N}, {P}, {'true' if chan else 'false'}>", "adi::finish_kernel")


def _multi(N, Q, mix1, chan):
    b = lambda v: "true" if v else "false"   # noqa: E731
    return (f"adi::prepare_multi_kernel<{N}>", f"adi::split::sfwd_multi_kernel<{N}, 2, {Q}, {b(mix1)}>",
            f"adi::split::sbwd_multi_kernel<{N}, 2, {b(chan)}>", "adi::finish_multi_kernel")


_GENERIC = ("adi::generic::gprepare_kernel", "adi::generic::gfwd_kernel", "adi::generic::gfinish_kernel")
_WIDE = ("adi::generic::gprepare_kernel", "adi::wide::wfinish_kernel")
_STREAM = ("adi::stream::sprep_kernel", "adi::stream::ssweep_kernel<true>", "adi::stream::ssweep_kernel<false>",
           "adi::stream::sadj_kernel<true>", "adi::stream::sadj_kernel<false>", "adi::stream::sred_kernel",
           "adi::stream::sinit_kernel", "adi::stream::sgin_kernel")
_SMIX = lambda CB: (f"adi::stream::smix_kernel<{CB}, false>", f"adi::stream::smix_kernel<{CB}, true>")   # noqa: E731
_P4_FIRST = "sm * 16 - 7"      # the first batch with four pairs per group: (B + 7) // 8 >= 2 * SMs; B % 8 == 1
_P4_Q2 = "sm * 32 - 13"        # ceil(groups / 2) >= 2 * SMs; B % 8 == 3
_P4_Q4 = "sm * 64 - 29"        # ceil(groups / 4) >= 2 * SMs (28 x 28 only: four 32 x 32 slots do not fit); B % 8 == 3
_P2_Q2 = "sm * 16 - 5"         # two pairs per group (channel op or C > 1): ceil(groups / 2) >= 2 * SMs; B % 4 == 3
_NP2 = "sm * 64 - 3"           # whole-line forward, one channel: (B + 3) // 4 >= 16 * SMs; B % 4 == 1

_CIFAR = dict(dt=0.002, num_steps=3, dx=1.0, dy=1.5)

ROWS = [
    # ------------------------------------------------------------ whole-line kernels (adi.cu), edges 8 ... 24
    *[_m(f"whole_n{N}_mnist", _whole(N), "mnist", 5, dict(size=N, num_steps=3, dt=0.05, dx=0.7, dy=1.3)) for N in (8, 12, 16, 20, 24)],
    *[_m(f"whole_n{N}_cifar10_c3", _whole(N, chan=True), "cifar10", 3, dict(size=N, channels=3, **_CIFAR)) for N in (8, 12, 16, 20, 24)],
    # two sample pairs per warp: the single-channel training forward at large batch
    *[_m(f"whole_np2_n{N}_mnist", _whole(N, np2=True), "mnist", _NP2, dict(size=N, num_steps=2, dt=0.05)) for N in (8, 12, 20, 24)],
    _m("whole_np2_n16_cifar10_c1", _whole(16, chan=True, np2=True), "cifar10", _NP2, dict(size=16, channels=1, **_CIFAR)),
    # 28 / 32 x 32: the whole-line forward serves inference; four channels leave the half-line kernels' domain
    _m("whole_np2_n28_fashion_no_grad", ("adi::prepare_kernel<28>", "adi::fwd_kernel<28, 2>"), "fashion", _NP2, no_grad=True),
    _m("whole_np2_n32_mnist_no_grad", ("adi::prepare_kernel<32>", "adi::fwd_kernel<32, 2>"), "mnist", _NP2,
       dict(size=32), no_grad=True),
    _m("whole_n28_cifar10_c4", _whole(28, chan=True), "cifar10", 3, dict(size=28, channels=4, **_CIFAR)),
    _m("whole_n32_cifar10_c4", _whole(32, chan=True), "cifar10", 3, dict(size=32, channels=4, **_CIFAR)),
    # the whole-line backward without a channel op at 28 / 32: only on request (every such layer has one channel)
    _m("whole_n28_fashion_legacy", _whole(28), "fashion", 9, env={"PDE_B200_ADI_LEGACY": "1"}),
    _m("whole_n32_mnist_legacy", _whole(32), "mnist", 9, dict(size=32, num_steps=3, dt=0.05), env={"PDE_B200_ADI_LEGACY": "1"}),
    # ------------------------------------------------------------ half-line kernels (adi_split.cu), 28 and 32
    _m("split_n28_p2_q1_fashion", _split(28, 2, 1), "fashion", 9),
    _m("split_n32_p2_q1_mnist", _split(32, 2, 1), "mnist", 5, dict(size=32, num_steps=3, dt=0.05)),
    _m("split_n28_p2_q1_cifar10_mix", _split(28, 2, 1, mix1=True, chan=True), "cifar10", 3, dict(size=28, channels=3, **_CIFAR)),
    _m("split_n32_p2_q1_cifar10_mix", _split(32, 2, 1, mix1=True, chan=True), "cifar10", 3, dict(size=32, channels=3, **_CIFAR)),
    _m("split_n28_p2_q2_svhn", _split(28, 2, 2, chan=True), "svhn", _P2_Q2, dict(size=28, channels=3, num_steps=2)),
    _m("split_n32_p2_q2_svhn", _split(32, 2, 2, chan=True), "svhn", _P2_Q2, dict(size=32, channels=3, num_steps=2)),
    _m("split_n28_p2_q2_cifar10_mix", _split(28, 2, 2, mix1=True, chan=True), "cifar10", _P2_Q2, dict(size=28, channels=2, **_CIFAR)),
    _m("split_n32_p2_q2_cifar10_mix", _split(32, 2, 2, mix1=True, chan=True), "cifar10", _P2_Q2, dict(size=32, channels=3, **_CIFAR)),
    # four pairs per group: single-channel layers without a channel op at large batch
    _m("split_n28_p4_q1_fashion", _split(28, 4, 1), "fashion", _P4_FIRST),
    _m("split_n28_p4_q2_fashion_init_no_gin", _split(28, 4, 2), "fashion", _P4_Q2, perturb=False, need_gin=False),
    _m("split_n28_p4_q4_fashion", _split(28, 4, 4), "fashion", _P4_Q4),
    _m("split_n32_p4_q1_mnist", _split(32, 4, 1), "mnist", _P4_FIRST, dict(size=32)),
    _m("split_n32_p4_q1_fashion_init_no_gin", _split(32, 4, 1), "fashion", _P4_FIRST, dict(size=32), perturb=False, need_gin=False),
    _m("split_n32_p4_q2_mnist_no_gin", _split(32, 4, 2), "mnist", _P4_Q2, dict(size=32), need_gin=False),
    _m("split_n32_p4_q2_fashion_init", _split(32, 4, 2), "fashion", _P4_Q2, dict(size=32), perturb=False),
    # four 32 x 32 slots exceed the tile budget: only the tuning switch reaches Q = 4 (a candidate for removal)
    _m("split_n32_p4_q4_mnist_forced", _split(32, 4, 4), "mnist", _P4_FIRST, dict(size=32), env={"PDE_B200_SPLIT_QF": "4"}),
    # ------------------------------------------------------------ multi-branch launch (pde_adi_multi_*)
    *[Row(f"multi_{n}", _multi(*k), "multi", dict(name=n)) for n, k in (
        ("cifar2_pair_B3", (32, 1, True, True)), ("cifar2_pair_q2", (32, 2, True, True)),
        ("mnist32", (32, 1, False, False)), ("mnist32_q2", (32, 2, False, False)),
        ("svhn32_n2", (32, 1, False, True)), ("svhn28_n4_q2", (28, 2, False, True)),
        ("cifar10_28_c1", (28, 1, True, True)), ("cifar10_28_c2_q2", (28, 2, True, True)),
        ("mnist_fashion_28", (28, 1, False, False)), ("mnist_fashion_28_q2", (28, 2, False, False)))],
    # ------------------------------------------------------------ run-time-sized edges (adi_generic.cu), 1 ... 4 channels
    _m("generic_n36_mnist_c1", _GENERIC + ("adi::generic::gbwd_kernel<1>",), "mnist", 5, dict(size=36, num_steps=3, dt=0.05)),
    _m("generic_n30_cifar2_c2", _GENERIC + ("adi::generic::gbwd_kernel<2>",), "cifar2", 7, dict(size=30, channels=2, dt=0.02, num_steps=3)),
    _m("generic_n37_svhn_c3", _GENERIC + ("adi::generic::gbwd_kernel<3>",), "svhn", 3, dict(size=37, channels=3, num_steps=2)),
    _m("generic_n30_cifar10_c4", _GENERIC + ("adi::generic::gbwd_kernel<4>",), "cifar10", 3, dict(size=30, channels=4, **_CIFAR)),
    # ------------------------------------------------------------ 5 ... 64 channels (adi_wide.cu)
    _m("wide_c6_cifar10", _WIDE + ("adi::wide::wfwd_kernel<8>", "adi::wide::wbwd_kernel<8>"), "cifar10", 3,
       dict(size=16, channels=6, **_CIFAR)),
    _m("wide_c12_svhn", _WIDE + ("adi::wide::wfwd_kernel<16>", "adi::wide::wbwd_kernel<16>"), "svhn", 3,
       dict(size=12, channels=12, num_steps=2)),
    _m("wide_c24_cifar2", _WIDE + ("adi::wide::wfwd_kernel<32>", "adi::wide::wbwd_kernel<32>"), "cifar2", 2,
       dict(size=9, channels=24, dt=0.02, num_steps=2)),
    _m("wide_c48_cifar10", _WIDE + ("adi::wide::wfwd_kernel<64>", "adi::wide::wbwd_kernel<64>"), "cifar10", 2,
       dict(size=8, channels=48, **_CIFAR)),
    # ------------------------------------------------------------ planes beyond one block (adi_stream.cu)
    _m("stream_n130_svhn_c3", _STREAM + ("adi::stream::sout_kernel", "adi::stream::sdot_kernel", "adi::stream::sfin_kernel")
       + _SMIX(4), "svhn", 2, dict(size=130, channels=3, num_steps=2)),
    _m("stream_n130_mnist_c1", _STREAM, "mnist", 2, dict(size=130, num_steps=2, dt=0.05)),
    _m("stream_n130_cifar10_c8", _SMIX(8) + ("adi::stream::sdot_kernel", "adi::stream::sfin_kernel"), "cifar10", 1,
       dict(size=130, channels=8, num_steps=1, dt=0.002)),
    _m("stream_n130_cifar10_c16", _SMIX(16), "cifar10", 1, dict(size=130, channels=16, num_steps=1, dt=0.002)),
    _m("stream_n130_cifar2_c32", _SMIX(32), "cifar2", 1, dict(size=130, channels=32, num_steps=1, dt=0.002)),
    _m("stream_n130_cifar10_c64", _SMIX(64), "cifar10", 1, dict(size=130, channels=64, num_steps=1, dt=0.002)),
    # ------------------------------------------------------------ emotion layer (explicit.cu, emotion_halo.cu)
    *[Row(f"emotion_tiled_n{N}", (f"expl::emo_fwd_tiled<{N}, float>", f"expl::emo_fwd_tiled<{N}, __nv_bfloat16>",
                                  f"expl::emo_bwd_tiled<{N}, float>", f"expl::emo_bwd_tiled<{N}, __nv_bfloat16>",
                                  "expl::emo_finish_tiled"), "emotion", dict(N=N, Nt=3, B=3)) for N in (16, 32, 48)],
    Row("emotion_generic_n40", ("expl::emo_fwd_kernel<float>", "expl::emo_fwd_kernel<__nv_bfloat16>",
                                "expl::emo_bwd_kernel<float>", "expl::emo_bwd_kernel<__nv_bfloat16>",
                                "expl::emo_finish_kernel"), "emotion", dict(N=40, Nt=3, B=3)),
    Row("emotion_halo_n70_3_steps", ("halo::emo_halo_fwd_kernel<false, float>", "halo::emo_halo_fwd_kernel<false, __nv_bfloat16>",
                                     "halo::emo_halo_fwd_kernel<true, float>", "halo::emo_halo_fwd_kernel<true, __nv_bfloat16>",
                                     "halo::emo_halo_adj_kernel<float, false, false>",
                                     "halo::emo_halo_adj_kernel<__nv_bfloat16, true, false>",
                                     "halo::emo_halo_adj_kernel<__nv_bfloat16, false, false>",
                                     "halo::emo_halo_adj_kernel<__nv_bfloat16, false, true>",
                                     "halo::emo_halo_fold_kernel<float>", "halo::emo_halo_fold_kernel<__nv_bfloat16>",
                                     "halo::emo_halo_sum_kernel", "halo::emo_halo_finish_kernel"),
        "emotion", dict(N=70, Nt=3, B=3)),
    Row("emotion_halo_n67_1_step", ("halo::emo_halo_adj_kernel<__nv_bfloat16, true, true>",), "emotion", dict(N=67, Nt=1, B=2)),
    # ------------------------------------------------------------ tiny_imagenet layer (explicit.cu, tiny_tiled.cu)
    Row("tiny_ring_64", ("expl::tiny_fwd_kernel<float>", "expl::tiny_bwd_kernel<float>", "expl::tiny_finish_kernel"),
        "tiny", dict(B=3, C=3, H=64, W=64, steps=1)),
    Row("tiny_ring_64_bf16", ("expl::tiny_fwd_kernel<__nv_bfloat16>", "expl::tiny_bwd_kernel<__nv_bfloat16>"),
        "tiny", dict(B=3, C=3, H=64, W=64, steps=1, bf16=True)),
    Row("tiny_tiled_227_1_step", ("tiled::tiny_tiled_fwd_kernel<float, 1>", "tiled::tiny_tiled_bwd_kernel<float, 1>",
                                  "tiled::tiny_tiled_finish_kernel"), "tiny", dict(B=2, C=3, H=227, W=227, steps=1)),
    Row("tiny_tiled_227_2_steps", ("tiled::tiny_tiled_fwd_kernel<float, 16>", "tiled::tiny_tiled_bwd_kernel<float, 16>"),
        "tiny", dict(B=2, C=3, H=227, W=227, steps=2)),
    Row("tiny_tiled_227_1_step_bf16", ("tiled::tiny_tiled_fwd_kernel<__nv_bfloat16, 1>", "tiled::tiny_tiled_bwd_kernel<__nv_bfloat16, 1>"),
        "tiny", dict(B=2, C=3, H=227, W=227, steps=1, bf16=True)),
    Row("tiny_tiled_227_2_steps_bf16", ("tiled::tiny_tiled_fwd_kernel<__nv_bfloat16, 16>",
                                        "tiled::tiny_tiled_bwd_kernel<__nv_bfloat16, 16>"),
        "tiny", dict(B=2, C=3, H=227, W=227, steps=2, bf16=True)),
    # ------------------------------------------------------------ tiny_imagenet's dormant methods (tiny_split*.cu)
    Row("tiny_split_on_chip_64", ("tsplit::tiny_split_kernel",), "tiny_split", dict(shape=(3, 64, 64))),
    Row("tiny_split_lines_65x97", ("tsplit_tiled::tiny_split_solve_kernel<true>", "tsplit_tiled::tiny_split_solve_kernel<false>",
                                   "tsplit_tiled::tiny_split_explicit_kernel<true>", "tsplit_tiled::tiny_split_explicit_kernel<false>"),
        "tiny_split", dict(shape=(2, 65, 97))),
]


def batch(B, sm_count: int) -> int:
    """A row's batch: an int, or "sm * a + b" / "sm * a - b" evaluated at the device's SM count."""
    if isinstance(B, int):
        return B
    m = re.fullmatch(r"sm \* (\d+) ([+-]) (\d+)", B)
    assert m, B
    a, sign, b = int(m.group(1)), m.group(2), int(m.group(3))
    return sm_count * a + (b if sign == "+" else -b)


def ledger_kernels():
    """The union of the rows' kernels."""
    out = set()
    for r in ROWS:
        out.update(r.kernels)
    return out
