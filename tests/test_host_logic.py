"""CPU-only tests: C-ABI surface, drop-in contract of the modules, schedule, sharding."""
import os
import re

import numpy as np
import pytest
import torch

from . import cases as K
from . import runners

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_exports_every_declared_symbol():
    import cnn_with_pde_b200 as P
    hdr = open(os.path.join(ROOT, "include", "pde_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(pde_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(P._cabi.EXPORTS), declared ^ set(P._cabi.EXPORTS)
    lib = P._cabi.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pde_b200_abi_version() == 3
    assert b"unsupported" in lib.pde_b200_error_string(-2).lower() or b"not supported" in lib.pde_b200_error_string(-2)


def test_cabi_host_only_queries():
    import ctypes
    import cnn_with_pde_b200 as P
    lib = P._cabi.lib()
    cfg = P.AdiConfig(N=28, C=1, steps=4, dt=0.3, hx=1.0, hy=1.0, smooth=True)
    d = cfg.desc(256)
    n = lib.pde_adi_tables_bytes(ctypes.byref(d))
    # header + the tables of both implementations (28 cells / line; 2 halves x 16 padded cells / line)
    assert n == 4096 + 4 * (12 * 1 * 28 * 28) * 4 + 4 * (12 * 1 * 28 * 32) * 4
    if not torch.cuda.is_available():
        # without a device the half-line kernels cannot be planned: no checkpoints are asked for and
        # the size queries answer 0 instead of guessing
        assert lib.pde_adi_checkpoint_bytes(ctypes.byref(d)) == 0
        big = cfg.desc(1 << 16)
        assert lib.pde_adi_checkpoint_bytes(ctypes.byref(big)) == 0
    # plane edges without kernels of their own go to the run-time-sized path (one table set, no checkpoints)
    gen = P.AdiConfig(N=30, C=3, steps=4, dt=0.3, hx=1.0, hy=1.0).desc(5)
    assert lib.pde_adi_tables_bytes(ctypes.byref(gen)) == 4096 + 4 * (12 * 3 * 30 * 30) * 4
    assert lib.pde_adi_checkpoint_bytes(ctypes.byref(gen)) == 0
    for N, C in ((128, 3), (96, 4), (127, 2), (2, 1)):
        ok = P.AdiConfig(N=N, C=C, steps=2, dt=0.3, hx=1.0, hy=1.0).desc(1)
        assert lib.pde_adi_tables_bytes(ctypes.byref(ok)) == 4096 + 4 * (6 * C * N * N) * 4, (N, C)
    for N, C in ((200, 1), (128, 4), (100, 4), (1, 1)):     # shared memory / threads of a block exceeded; not a plane
        bad = P.AdiConfig(N=N, C=C, steps=4, dt=0.3, hx=1.0, hy=1.0).desc(1)
        assert lib.pde_adi_tables_bytes(ctypes.byref(bad)) == 0, (N, C)
    # struct layouts must match the header
    assert ctypes.sizeof(P._cabi.AdiDesc) == 9 * 4 + 3 * 4 + 4      # ... + tuning
    assert ctypes.sizeof(P._cabi.AdiSchedule) == 3 * 192 * 4
    assert ctypes.sizeof(P._cabi.EmoDesc) == 3 * 4 + 4 * 4 + 4     # ... + tuning
    assert ctypes.sizeof(P._cabi.TinyDesc) == 5 * 4 + 4 * 4


def test_product_does_not_touch_the_oracle():
    """The oracle is a checker: nothing under cnn-with-pde_b200/ may import or link it."""
    pkg = os.path.join(ROOT, "cnn-with-pde_b200")
    for dirpath, _, files in os.walk(pkg):
        if os.path.basename(dirpath) in ("build", "__pycache__"):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle-free", ""), os.path.join(dirpath, f)


def test_schedule_matches_python_double_accumulation():
    from cnn_with_pde_b200.schedule import adi_schedule, adi_schedule_lists
    t, dts, h = adi_schedule_lists(3, 0.3, 1.0, 2.0, lie=False)
    cur = 0.0
    want = []
    for _ in range(3):
        want.append(cur); cur += 0.3 / 2
        want.append(cur); cur += 0.3 / 2
        want.append(cur)
    assert t == want
    assert dts == [0.15, 0.3, 0.15] * 3 and h == [1.0, 2.0, 1.0] * 3
    t, dts, h = adi_schedule_lists(2, 0.002, 1.0, 1.0, lie=True)
    assert t == [0.0, 0.001, 0.002, 0.003] and dts == [0.001] * 4
    s = adi_schedule(10, 0.001, 1.0, 1.0, False)
    assert s.t[29] == float(np.float32(sum([0.0005] * 20))) or abs(s.t[29] - 0.01) < 1e-8
    with pytest.raises(ValueError):
        adi_schedule(65, 0.1, 1.0, 1.0, False)


EXPECTED_KEYS = {
    "mnist": ["alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff"],
    "fashion": ["alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff"],
    "svhn": ["alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff", "channel_coupling", "skip_weight"],
    "cifar10": ["alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff", "channel_mixing"],
    "cifar2": ["alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff", "channel_mixing"],
    "emotion": ["alpha_w1", "alpha_w2", "alpha_w3", "beta_w1", "beta_w2", "beta_w3", "x", "y"],
    "tiny": ["alpha_base", "beta_base", "channel_scaling"],
}


def _ours(kind):
    import importlib
    mod, cls = runners.OUR_CLASS[kind]
    return getattr(importlib.import_module("cnn_with_pde_b200." + mod), cls)


@pytest.mark.parametrize("kind", sorted(EXPECTED_KEYS))
def test_state_dict_layout(kind):
    layer = _ours(kind)()
    assert list(layer.state_dict().keys()) == EXPECTED_KEYS[kind]
    assert all(v.dtype == torch.float32 for v in layer.state_dict().values())


def test_modules_reject_cpu_input_loudly():
    for kind in ("mnist", "cifar10", "emotion", "tiny"):
        layer = _ours(kind)()
        c = K.case("x", kind)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            layer(torch.zeros(1, *c.shape))


def test_shard_bounds_cover_ragged_batches():
    from cnn_with_pde_b200.parallel import shard_bounds
    for n in (0, 1, 7, 8, 513):
        for world in (1, 2, 3, 8):
            spans = [shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
