"""The kernel ledger (tests/kernel_ledger.py) names every kernel the built library contains, and nothing else.

The library's kernels are the `.text.<mangled name>` sections `cuobjdump -elf` lists for its sm_100a code,
demangled by `cu++filt`.  No GPU is needed.
"""
import os
import re
import shutil
import subprocess
import sys

import pytest

from . import kernel_ledger as KL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")


def _tool(name):
    path = shutil.which(name) or os.path.join(CUDA_BIN, name)
    if not os.path.exists(path):
        pytest.fail(f"{name} not found (CUDA toolkit at {CUDA_BIN}): it lists the library's kernels")
    return path


def _library():
    sys.path.insert(0, os.path.join(ROOT, "cnn-with-pde_b200"))
    try:
        import build   # rebuilds only when a source is newer than the library
    finally:
        sys.path.pop(0)
    return build.build()


def library_kernels():
    """Normalised names of every kernel in the built library."""
    elf = subprocess.run([_tool("cuobjdump"), "-elf", _library()], check=True, capture_output=True, text=True).stdout
    mangled = sorted(set(re.findall(r"\.text\.(_Z\S+)", elf)))
    assert mangled, "cuobjdump listed no kernel sections"
    names = subprocess.run([_tool("cu++filt")], input="\n".join(mangled) + "\n", check=True, capture_output=True,
                           text=True).stdout.splitlines()
    assert len(names) == len(mangled)
    out = {KL.normalise(n) for n in names}
    assert None not in out, [n for n in names if KL.normalise(n) is None]
    return out


def test_normalise_both_spellings():
    """cu++filt's spelling and the profiler's of the same kernels.  The profiler's, as a B200 run of
    test_gpu_kernel_ledger printed it, has `void ` before a template instantiation and none before a plain kernel."""
    pairs = [
        ("pde::adi::split::sfwd_kernel<(int)28, (int)4, (int)1, (bool)0>(pde::adi::split::Args)",
         "void pde::adi::split::sfwd_kernel<28, 4, 1, false>(pde::adi::split::Args)"),
        ("pde::adi::fwd_kernel<(int)16, (int)2>(pde::adi::Args)", "void pde::adi::fwd_kernel<16, 2>(pde::adi::Args)"),
        ("pde::halo::emo_halo_adj_kernel<__nv_bfloat16, (bool)1, (bool)0>(pde::halo::AdjArgs)",
         "void pde::halo::emo_halo_adj_kernel<__nv_bfloat16, true, false>(pde::halo::AdjArgs)"),
        ("pde::halo::emo_halo_fold_kernel<float>(int, long long, const float *, const float *, T1 *)",
         "void pde::halo::emo_halo_fold_kernel<float>(int, long long, float const*, float const*, float*)"),
        ("pde::adi::stream::sred_kernel(pde_adi_desc, int, int, float, float, const float *, const float *, "
         "const float *, float *, float *)",
         "pde::adi::stream::sred_kernel(pde_adi_desc, int, int, float, float, float const*, float const*, "
         "float const*, float*, float*)"),
        ("pde::adi::bwd_kernel<(int)12, (bool)0>", "void pde::adi::bwd_kernel<12, false>(pde::adi::Args)"),
        ("pde::adi::finish_multi_kernel(pde::adi::FinishMulti)", "pde::adi::finish_multi_kernel(pde::adi::FinishMulti)"),
    ]
    want = ["adi::split::sfwd_kernel<28, 4, 1, false>", "adi::fwd_kernel<16, 2>",
            "halo::emo_halo_adj_kernel<__nv_bfloat16, true, false>", "halo::emo_halo_fold_kernel<float>",
            "adi::stream::sred_kernel", "adi::bwd_kernel<12, false>", "adi::finish_multi_kernel"]
    for (a, b), w in zip(pairs, want):
        assert KL.normalise(a) == w and KL.normalise(b) == w, (a, b, w)
    assert KL.normalise("void at::native::vectorized_elementwise_kernel<4, float>(int, float)") is None


def test_rows_are_well_formed():
    names = [r.name for r in KL.ROWS]
    assert len(names) == len(set(names)), "row names repeat"
    for r in KL.ROWS:
        assert r.kernels and r.run in ("module", "multi", "emotion", "tiny", "tiny_split"), r.name
        for k in r.kernels:
            assert KL.normalise("pde::" + k) == k, (r.name, k, "not in normalised spelling")
        if r.run == "module":
            assert KL.batch(r.spec["B"], 148) >= 1


def test_ledger_names_every_kernel_of_the_library():
    have = library_kernels()
    rows = KL.ledger_kernels()
    missing, stale = sorted(have - rows), sorted(rows - have)
    assert not missing, f"kernels without a ledger row (tests/kernel_ledger.py): {missing}"
    assert not stale, f"ledger rows name kernels the library does not contain: {stale}"
