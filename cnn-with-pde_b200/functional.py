"""torch.autograd.Function wrappers over the C ABI (the only callers of _cabi).

Each Function saves its inputs and, for the implicit family, the factorised coefficient tables of
the call plus -- when the half-line kernels serve it -- the state at the end of every step
(`pde_adi_forward_train`); everything else of the forward trajectory is rebuilt on-chip by the
backward kernels.

Host-side cost matters at the reference's own batch sizes (a call is a few tens of microseconds of
GPU time): everything that depends only on (configuration, batch, device) -- descriptor, sweep
schedule, buffer sizes -- is computed once and cached (`_adi_plan`), the gradient outputs share one
allocation, and under `torch.no_grad()` the coefficient tables are reused while the parameters'
version counters have not moved.
"""
from __future__ import annotations

import contextlib
import ctypes
import functools
import os
import weakref

from ctypes import byref
from dataclasses import dataclass

import torch
from torch._subclasses.fake_tensor import FakeTensor

from . import _cabi
from .schedule import adi_schedule


def _traced(t) -> bool:
    """Whether a layer call is traced rather than run: under torch.compile, or on FakeTensor / meta-device inputs
    (torch.export, shape inference).  Such calls go through the custom ops of ops.py, which Dynamo and FakeTensor
    mode can see through; a call on real tensors keeps the autograd.Functions below (less host time per call)."""
    return torch.compiler.is_compiling() or isinstance(t, FakeTensor) or (isinstance(t, torch.Tensor) and t.is_meta)


def _require_cuda(x: torch.Tensor, what: str):
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise RuntimeError(
            f"{what}: expected a CUDA tensor -- the B200 PDE layers have no CPU fallback "
            f"(got {'a ' + str(x.device) + ' tensor' if isinstance(x, torch.Tensor) else type(x)})")
    if x.dtype != torch.float32:
        raise RuntimeError(f"{what}: expected float32, got {x.dtype}")


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(device=None):
    """cudaStream_t of torch's current stream (the raw query: torch.cuda.current_stream() builds a
    Python Stream object, ~10 us, every call)."""
    idx = torch.cuda.current_device() if device is None or device.index is None else device.index
    return torch._C._cuda_getCurrentRawStream(idx)


def _no_double_backward(what: str):
    # the backward passes call raw-pointer kernels: autograd cannot differentiate them again, and
    # returning their results under create_graph=True would silently treat them as constants
    if torch.is_grad_enabled():
        raise RuntimeError(f"{what}: the B200 PDE layers are once differentiable (no create_graph=True / double backward)")


def _autocast_to_fp32(t):
    """What custom_fwd(cast_inputs=torch.float32) does for the input, at a fraction of its host cost:
    under CUDA autocast a half-precision input is cast up (tracked by autograd, so its gradient comes
    back in its own dtype); the layers themselves always compute in fp32 and call no op that autocast
    would touch."""
    if t.dtype != torch.float32 and t.is_floating_point() and torch.is_autocast_enabled("cuda"):
        return t.float()
    return t


def _guard(device):
    """Device guard only when the tensor does not live on the current device."""
    if device.index is None or device.index == torch.cuda.current_device():
        return contextlib.nullcontext()
    return torch.cuda.device(device)


def _bytes(n: int, device) -> torch.Tensor:
    # caching-allocator blocks are 512-byte aligned, which covers the 256-byte requirement
    return torch.empty(max(int(n), 1), dtype=torch.uint8, device=device)


def _contig(t):
    """Contiguous and 16-byte aligned: the half-line ADI kernels move whole planes by bulk copies,
    which need 16-byte-aligned addresses.  A view at an odd offset of its storage is copied."""
    if t.is_contiguous() and t.data_ptr() % 16 == 0:
        return t
    return t.clone(memory_format=torch.contiguous_format)


def env_tuning() -> int:
    """The kernel-variant switches of the test suite and of A/B timing runs, as a
    `pde_adi_desc.tuning` value.  This is the only place they are read: the value travels inside the
    descriptor, is saved with the autograd context, and so cannot differ between forward and backward.

        PDE_B200_ADI_LEGACY=1   whole-line kernels (adi.cu) everywhere
        PDE_B200_ADI_SPLIT=1    half-line kernels (adi_split.cu) also for small batches
        PDE_B200_SPLIT_P=2|4    sample pairs per half-line group
        PDE_B200_SPLIT_QF=1|2|4 groups per half-line forward block
        PDE_B200_FWD_NP=1|2     sample pairs per whole-line forward warp
    """
    raw = getattr(os.environ, "_data", None)   # bytes-keyed dict behind os.environ: membership costs ~50 ns
    if raw is not None and not (_TUNING_KEYS_B & raw.keys()):
        return 0
    env = os.environ
    impl = _cabi.TUNE_IMPL_WHOLE_LINE if env.get("PDE_B200_ADI_LEGACY") else (
        _cabi.TUNE_IMPL_HALF_LINE if env.get("PDE_B200_ADI_SPLIT") else 0)
    num = lambda k: int(env.get(k) or 0)   # noqa: E731
    return _cabi.adi_tuning(impl, num("PDE_B200_SPLIT_P"), num("PDE_B200_SPLIT_QF"), num("PDE_B200_FWD_NP"))


@torch.compiler.assume_constant_result
def _traced_tuning() -> int:
    """env_tuning() for a traced call: Dynamo takes the value as a constant of the graph."""
    return env_tuning()


_TUNING_KEYS = ("PDE_B200_ADI_LEGACY", "PDE_B200_ADI_SPLIT", "PDE_B200_SPLIT_P", "PDE_B200_SPLIT_QF", "PDE_B200_FWD_NP")
_TUNING_KEYS_B = frozenset(k.encode() for k in _TUNING_KEYS)


# ------------------------------------------------------------------------------ implicit ADI
@dataclass(frozen=True)
class AdiConfig:
    N: int
    C: int
    steps: int
    dt: float
    hx: float
    hy: float
    lie: bool = False
    smooth: bool = False
    has_max: bool = False
    chan_op: int = 0
    skip: bool = False
    cmin: float = 1e-6
    cmax: float = 10.0
    eps: float = 1e-6

    def __hash__(self):   # computed once (on first use, so that Dynamo can build a configuration): it keys the plan cache
        try:
            return self._hash
        except AttributeError:
            h = hash((self.N, self.C, self.steps, self.dt, self.hx, self.hy, self.lie, self.smooth, self.has_max,
                      self.chan_op, self.skip, self.cmin, self.cmax, self.eps))
            object.__setattr__(self, "_hash", h)
            return h

    def desc(self, B: int, tuning: int = 0) -> "_cabi.AdiDesc":
        return _cabi.AdiDesc(B, self.C, self.N, self.steps, int(self.lie), int(self.smooth), int(self.has_max),
                             self.chan_op, int(self.skip), self.cmin, self.cmax, self.eps, tuning)


class _AdiPlan:
    """Everything about a call that depends only on (configuration, batch, tuning, device)."""
    __slots__ = ("cfg", "B", "desc", "dref", "sched", "sref", "tables_bytes", "ckpt_bytes", "ws_saved_bytes", "ws_bytes",
                 "grad_numel")

    def __init__(self, cfg: AdiConfig, B: int, tuning: int):
        L = _cabi.lib()
        self.cfg, self.B = cfg, B
        self.desc = cfg.desc(B, tuning)
        self.dref = byref(self.desc)
        self.tables_bytes = L.pde_adi_tables_bytes(self.dref)
        if self.tables_bytes == 0:
            raise _cabi.PdeB200Error(
                f"unsupported implicit-layer configuration (size={cfg.N}, channels={cfg.C}, steps={cfg.steps}); "
                "supported: size 2 ... 128 with channels * size * (size | 1) * 4 bytes <= 200 KB, "
                f"channels <= {_cabi.ADI_MAX_CHANNELS} (channels <= {_cabi.MAX_CHANNELS} also needs channels * size <= 384 "
                "unless size is 8, 12, ... 32), at most 64 Strang / 96 Lie steps")
        self.sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
        self.sref = byref(self.sched)
        self.ckpt_bytes = L.pde_adi_checkpoint_bytes(self.dref)
        self.ws_saved_bytes = L.pde_adi_backward_saved_workspace_bytes(self.dref)
        self.ws_bytes = L.pde_adi_backward_workspace_bytes(self.dref)
        self.grad_numel = 4 * cfg.C * cfg.N * cfg.N


@functools.lru_cache(maxsize=256)
def _adi_plan(cfg: AdiConfig, B: int, tuning: int, device_index: int) -> _AdiPlan:
    return _AdiPlan(cfg, B, tuning)


# Coefficient tables of inference calls, reused while the parameters have not changed.  An entry is valid
# only for the very tensor objects it was built from (weak references: an address reused by another tensor
# after the original died must not hit) at the versions it saw.  Never consulted under autograd or during
# CUDA-graph capture (a captured graph must contain its own prepare launch).
_TABLE_CACHE_SLOTS = 8
_table_cache: "dict" = {}


def _cached_tables(plan, params):
    key = (id(plan),) + tuple(id(p) for p in params)
    hit = _table_cache.get(key)
    if hit is None:
        return key, None
    tables, refs, versions = hit
    if all(r() is p for r, p in zip(refs, params)) and versions == tuple(p._version for p in params):
        return key, tables
    del _table_cache[key]
    return key, None


def _remember_tables(key, params, tables):
    if len(_table_cache) >= _TABLE_CACHE_SLOTS:
        _table_cache.pop(next(iter(_table_cache)))
    _table_cache[key] = (tables, tuple(weakref.ref(p) for p in params), tuple(p._version for p in params))


def _adi_tables_forward(u, params, chan, skipw, cfg: AdiConfig, tuning: int, training: bool, reuse_tables: bool):
    """The forward pass on the shared-memory kernels: coefficient tables (or the cached ones of an inference call
    while `reuse_tables`), then the forward kernel, writing step checkpoints while `training`.  Returns
    (out, tables, ckpt or None, plan, u, chan, skip), the last three as the kernels read them."""
    _require_cuda(u, "PDE layer input")
    L = _cabi.lib()
    u = _contig(u)
    maps = [_contig(p) for p in params]
    for p in maps:
        _require_cuda(p, "PDE layer parameter")
    chan_c = None if chan is None else _contig(chan.detach())
    skip_c = None if skipw is None else _contig(skipw.detach())
    dev = u.device
    with _guard(dev):
        # (the plan asks the library about the CURRENT device: built under the guard)
        plan = _adi_plan(cfg, u.shape[0], tuning, dev.index if dev.index is not None else torch.cuda.current_device())
        st = _stream(dev)
        tables, key = None, None
        if reuse_tables and not training and not torch.cuda.is_current_stream_capturing():
            key, tables = _cached_tables(plan, params)
        if tables is None:
            # a traced call's tables are an output of its op: zeroed, so that the bytes prepare leaves unwritten
            # (alignment padding) are the same in every run
            tables = _bytes(plan.tables_bytes, dev) if reuse_tables else torch.zeros(plan.tables_bytes, dtype=torch.uint8,
                                                                                     device=dev)
            _cabi.check(L.pde_adi_prepare(plan.dref, plan.sref, *[p.data_ptr() for p in maps], tables.data_ptr(), st),
                        "pde_adi_prepare")
            if key is not None:
                _remember_tables(key, params, tables)
        out = torch.empty_like(u)
        # under autograd the forward kernel also writes the state at the end of every step for
        # the backward kernel (0 bytes when the configuration is served by the kernels that
        # rebuild the trajectory on-chip).  PDE_B200_NO_CKPT=1 trades them for a recomputation
        # inside pde_adi_backward (saves num_steps x the input in memory between the passes)
        ck_bytes = plan.ckpt_bytes if training and not os.environ.get("PDE_B200_NO_CKPT") else 0
        ckpt = _bytes(ck_bytes, dev) if ck_bytes else None
        _cabi.check(L.pde_adi_forward_train(plan.dref, tables.data_ptr(), _ptr(u), _ptr(chan_c), _ptr(skip_c), _ptr(out),
                                            _ptr(ckpt), st), "pde_adi_forward_train")
    return out, tables, ckpt, plan, u, chan_c, skip_c


def _adi_grad_buffers(cfg: AdiConfig, u, param_shape, has_chan: bool, has_skip: bool, need_gin: bool):
    """grad_input (or None), the four coefficient-map gradients in one allocation, g_chan and g_skip (or None)."""
    dev = u.device
    gin = torch.empty_like(u) if need_gin else None
    gm = torch.empty((4,) + tuple(param_shape), dtype=torch.float32, device=dev)
    gchan = torch.empty((cfg.C, cfg.C), dtype=torch.float32, device=dev) if has_chan else None
    gskip = torch.empty((), dtype=torch.float32, device=dev) if has_skip else None
    return gin, gm, gchan, gskip


def _float_grad(gout):
    gout = _contig(gout)
    return gout if gout.dtype == torch.float32 else gout.float()


def _adi_tables_backward(plan, u, tables, chan, skipw, ckpt, gout, param_shape, need_gin: bool):
    """The backward pass on the shared-memory kernels, from the checkpoints of the forward call or -- ckpt None --
    recomputing them in a batch-sized workspace.  Returns (gin or None, the four map gradients as one (4, ...)
    tensor, g_chan or None, g_skip or None)."""
    L = _cabi.lib()
    gout = _float_grad(gout)
    dev = u.device
    with _guard(dev):
        ws_bytes = plan.ws_saved_bytes if ckpt is not None else plan.ws_bytes
        ws = _bytes(ws_bytes, dev)
        gin, gm, gchan, gskip = _adi_grad_buffers(plan.cfg, u, param_shape, chan is not None, skipw is not None, need_gin)
        base, plane = gm.data_ptr(), plan.grad_numel
        _cabi.check(L.pde_adi_backward_saved(plan.dref, tables.data_ptr(), _ptr(u), _ptr(gout), _ptr(chan), _ptr(skipw),
                                             _ptr(ckpt), _ptr(gin), base, base + plane, base + 2 * plane, base + 3 * plane,
                                             _ptr(gchan), _ptr(gskip), ws.data_ptr(), ws_bytes, _stream(dev)),
                    "pde_adi_backward_saved")
    return gin, gm, gchan, gskip


class _AdiFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw, cfg: AdiConfig, grad_mode: bool = True):
        # needs_input_grad ignores torch.no_grad() and grad mode is always off inside forward(): the
        # caller passes the mode it saw
        training = grad_mode and any(ctx.needs_input_grad)
        params = (alpha_base, beta_base, alpha_tc, beta_tc)
        out, tables, ckpt, plan, u, chan_c, skip_c = _adi_tables_forward(u, params, chan, skipw, cfg, env_tuning(), training,
                                                                         True)
        ctx.plan = plan   # the descriptor (tuning included) the backward pass must use as well
        ctx.has_chan = chan is not None
        ctx.has_skip = skipw is not None
        ctx.has_ckpt = ckpt is not None
        ctx.save_for_backward(u, tables, *(t for t in (chan_c, skip_c, ckpt) if t is not None))
        ctx.param_shape = alpha_base.shape
        return out

    @staticmethod
    def backward(ctx, gout):
        _no_double_backward("PDE layer")
        saved = list(ctx.saved_tensors)
        u, tables = saved[0], saved[1]
        rest = saved[2:]
        chan = rest.pop(0) if ctx.has_chan else None
        skipw = rest.pop(0) if ctx.has_skip else None
        ckpt = rest.pop(0) if ctx.has_ckpt else None
        gin, gm, gchan, gskip = _adi_tables_backward(ctx.plan, u, tables, chan, skipw, ckpt, gout, ctx.param_shape,
                                                     ctx.needs_input_grad[0])
        gmaps = gm.unbind(0)
        return (gin, gmaps[0], gmaps[1], gmaps[2], gmaps[3], gchan, gskip, None, None)


# ------------------------------- implicit ADI beyond one block's shared memory (pde_adi_stream_*)
@functools.lru_cache(maxsize=256)
def adi_route(cfg: AdiConfig) -> str:
    """Which kernel family serves `cfg`: "tables" where the shared-memory kernels do (pde_adi_tables_bytes > 0: their
    plans, table cache and checkpoints), "stream" where only the streaming kernels do (planes beyond one block's
    shared memory).  Raises PdeB200Error outside both domains."""
    L = _cabi.lib()
    d = cfg.desc(1)
    if L.pde_adi_tables_bytes(byref(d)):
        return "tables"
    if L.pde_adi_stream_forward_workspace_bytes(byref(d)):
        return "stream"
    raise _cabi.PdeB200Error(
        f"unsupported implicit-layer configuration (size={cfg.N}, channels={cfg.C}, steps={cfg.steps}); supported: "
        f"size 2 ... 4096, channels <= {_cabi.ADI_MAX_CHANNELS}, at most 64 Strang / 96 Lie steps")


class _AdiStreamPlan:
    """Descriptor, schedule and workspace sizes of a stream-routed call: (configuration, batch, device)."""
    __slots__ = ("cfg", "desc", "dref", "sched", "sref", "fwd_bytes", "bwd_bytes")

    def __init__(self, cfg: AdiConfig, B: int):
        L = _cabi.lib()
        self.cfg = cfg
        self.desc = cfg.desc(B, 0)
        self.dref = byref(self.desc)
        self.sched = adi_schedule(cfg.steps, cfg.dt, cfg.hx, cfg.hy, cfg.lie)
        self.sref = byref(self.sched)
        self.fwd_bytes = L.pde_adi_stream_forward_workspace_bytes(self.dref)
        self.bwd_bytes = L.pde_adi_stream_backward_workspace_bytes(self.dref)


@functools.lru_cache(maxsize=256)
def _adi_stream_plan(cfg: AdiConfig, B: int, device_index: int) -> _AdiStreamPlan:
    return _AdiStreamPlan(cfg, B)


def _adi_stream_forward(u, params, chan, skipw, cfg: AdiConfig):
    """The forward pass on the streaming kernels.  Returns (out, plan, u, maps, chan, skip), the last four as the
    kernels read them."""
    _require_cuda(u, "PDE layer input")
    L = _cabi.lib()
    u = _contig(u)
    maps = [_contig(p.detach()) for p in params]
    for p in maps:
        _require_cuda(p, "PDE layer parameter")
    chan_c = None if chan is None else _contig(chan.detach())
    skip_c = None if skipw is None else _contig(skipw.detach())
    dev = u.device
    with _guard(dev):
        plan = _adi_stream_plan(cfg, u.shape[0], dev.index if dev.index is not None else torch.cuda.current_device())
        ws = _bytes(plan.fwd_bytes, dev)
        out = torch.empty_like(u)
        _cabi.check(L.pde_adi_stream_forward(plan.dref, plan.sref, *[p.data_ptr() for p in maps], _ptr(u), _ptr(chan_c),
                                             _ptr(skip_c), _ptr(out), ws.data_ptr(), plan.fwd_bytes, _stream(dev)),
                    "pde_adi_stream_forward")
    return out, plan, u, maps, chan_c, skip_c


def _adi_stream_backward(plan, u, maps, chan, skipw, gout, param_shape, need_gin: bool):
    """The backward pass on the streaming kernels (it replays the trajectory itself).  Returns what
    _adi_tables_backward returns."""
    L = _cabi.lib()
    gout = _float_grad(gout)
    dev = u.device
    with _guard(dev):
        ws = _bytes(plan.bwd_bytes, dev)
        gin, gm, gchan, gskip = _adi_grad_buffers(plan.cfg, u, param_shape, chan is not None, skipw is not None, need_gin)
        C, N = plan.cfg.C, plan.cfg.N
        base, plane = gm.data_ptr(), 4 * C * N * N
        _cabi.check(L.pde_adi_stream_backward(plan.dref, plan.sref, *[m.data_ptr() for m in maps], _ptr(u), _ptr(gout),
                                              _ptr(chan), _ptr(skipw), _ptr(gin), base, base + plane, base + 2 * plane,
                                              base + 3 * plane, _ptr(gchan), _ptr(gskip), ws.data_ptr(), plan.bwd_bytes,
                                              _stream(dev)), "pde_adi_stream_backward")
    return gin, gm, gchan, gskip


class _AdiStreamFunction(torch.autograd.Function):
    """The implicit layer on the streaming kernels: the factor tables are built inside each call, and the backward
    pass replays the trajectory itself, so only the input and the parameters are kept between the passes."""

    @staticmethod
    def forward(ctx, u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw, cfg: AdiConfig):
        out, plan, u, maps, chan_c, skip_c = _adi_stream_forward(u, (alpha_base, beta_base, alpha_tc, beta_tc), chan, skipw,
                                                                 cfg)
        ctx.plan = plan
        ctx.has_chan = chan is not None
        ctx.has_skip = skipw is not None
        ctx.save_for_backward(u, *maps, *(t for t in (chan_c, skip_c) if t is not None))
        ctx.param_shape = alpha_base.shape
        return out

    @staticmethod
    def backward(ctx, gout):
        _no_double_backward("PDE layer")
        saved = list(ctx.saved_tensors)
        u, maps, rest = saved[0], saved[1:5], saved[5:]
        chan = rest.pop(0) if ctx.has_chan else None
        skipw = rest.pop(0) if ctx.has_skip else None
        gin, gm, gchan, gskip = _adi_stream_backward(ctx.plan, u, maps, chan, skipw, gout, ctx.param_shape,
                                                     ctx.needs_input_grad[0])
        gmaps = gm.unbind(0)
        return (gin, gmaps[0], gmaps[1], gmaps[2], gmaps[3], gchan, gskip, None)


def adi_layer(u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw, cfg: AdiConfig):
    u = _autocast_to_fp32(u)
    if _traced(u):
        # the condition under which _AdiFunction writes checkpoints: it also selects the forward kernel
        training = torch.is_grad_enabled() and any(t is not None and t.requires_grad
                                                   for t in (u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw))
        return torch.ops.pde_b200.adi_fwd(u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw, cfg.N, cfg.C, cfg.steps,
                                          cfg.dt, cfg.hx, cfg.hy, cfg.lie, cfg.smooth, cfg.has_max, cfg.chan_op, cfg.skip,
                                          cfg.cmin, cfg.cmax, cfg.eps, _traced_tuning(), training)[0]
    if isinstance(u, torch.Tensor) and u.is_cuda and adi_route(cfg) == "stream":
        return _AdiStreamFunction.apply(u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw, cfg)
    return _AdiFunction.apply(u, alpha_base, beta_base, alpha_tc, beta_tc, chan, skipw, cfg, torch.is_grad_enabled())


# ------------------------------------------- several implicit layers on the same input, one launch per pass
def _ptr_array(ptrs):
    arr = (ctypes.c_void_p * len(ptrs))(*[p if p else None for p in ptrs])
    return arr


class _AdiMultiPlan:
    """Descriptor / schedule arrays and buffer sizes of a multi-branch call: (configurations, batch, tuning, device)."""
    __slots__ = ("plans", "n", "descs", "scheds", "ok")

    def __init__(self, cfgs, B, tuning, device_index):
        self.plans = [_adi_plan(c, B, tuning, device_index) for c in cfgs]
        self.n = len(cfgs)
        self.descs = (_cabi.AdiDesc * self.n)(*[p.desc for p in self.plans])
        self.scheds = (_cabi.AdiSchedule * self.n)(*[p.sched for p in self.plans])
        # the library decides whether the layers can share a launch: with compatible descriptors and no
        # buffers it answers "invalid argument", with incompatible ones "unsupported"
        self.ok = False
        if 2 <= self.n <= _cabi.MAX_BRANCHES and B > 0 and all(p.ckpt_bytes > 0 for p in self.plans):
            rc = _cabi.lib().pde_adi_multi_prepare(self.n, ctypes.addressof(self.descs), None, None, None, None, None, None, None)
            self.ok = rc == _cabi.ERR_INVALID


@functools.lru_cache(maxsize=64)
def _adi_multi_plan(cfgs, B, tuning, device_index):
    return _AdiMultiPlan(cfgs, B, tuning, device_index)


class _AdiMultiFunction(torch.autograd.Function):
    """n implicit layers applied to one input: inputs (u, cfgs, ab_0, bb_0, atc_0, btc_0, chan_0, skip_0, ab_1, ...),
    outputs (out_0, ..., out_{n-1}).  One prepare, one forward and one backward (+ one finish) launch for all of
    them (include/pde_b200.h: pde_adi_multi_*)."""

    @staticmethod
    def forward(ctx, u, cfgs, *flat):
        _require_cuda(u, "PDE layer input")
        L = _cabi.lib()
        n = len(cfgs)
        u = _contig(u)
        per = [flat[6 * i:6 * i + 6] for i in range(n)]
        dev = u.device
        with _guard(dev):
            mp = _adi_multi_plan(cfgs, u.shape[0], env_tuning(), dev.index if dev.index is not None else torch.cuda.current_device())
        maps = [[_contig(p) for p in br[:4]] for br in per]
        chans = [None if br[4] is None else _contig(br[4].detach()) for br in per]
        skips = [None if br[5] is None else _contig(br[5].detach()) for br in per]
        keep = []   # the pointer arrays must outlive the calls that read them

        def arr(ptrs):
            a = _ptr_array(ptrs)
            keep.append(a)
            return ctypes.addressof(a)

        with _guard(dev):
            st = _stream(dev)
            tables = [_bytes(p.tables_bytes, dev) for p in mp.plans]
            tab = arr([t.data_ptr() for t in tables])
            _cabi.check(L.pde_adi_multi_prepare(n, ctypes.addressof(mp.descs), ctypes.addressof(mp.scheds),
                                                *[arr([m[k].data_ptr() for m in maps]) for k in range(4)], tab, st),
                        "pde_adi_multi_prepare")
            outs = [torch.empty_like(u) for _ in range(n)]
            ckpts = [_bytes(p.ckpt_bytes, dev) for p in mp.plans]
            _cabi.check(L.pde_adi_multi_forward_train(
                n, ctypes.addressof(mp.descs), tab, _ptr(u), arr([_ptr(c) for c in chans]), arr([_ptr(s) for s in skips]),
                arr([o.data_ptr() for o in outs]), arr([c.data_ptr() for c in ckpts]), st), "pde_adi_multi_forward_train")
        ctx.mp = mp
        ctx.has = [(c is not None, s is not None) for c, s in zip(chans, skips)]
        ctx.param_shapes = [br[0].shape for br in per]
        ctx.save_for_backward(u, *tables, *ckpts, *[t for t in chans + skips if t is not None])
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        _no_double_backward("PDE layers")
        L = _cabi.lib()
        mp = ctx.mp
        n = mp.n
        saved = list(ctx.saved_tensors)
        u, tables, ckpts, rest = saved[0], saved[1:1 + n], saved[1 + n:1 + 2 * n], saved[1 + 2 * n:]
        chans = [rest.pop(0) if h[0] else None for h in ctx.has]
        skips = [rest.pop(0) if h[1] else None for h in ctx.has]
        gouts = [_contig(g if g.dtype == torch.float32 else g.float()) for g in gouts]
        dev = u.device
        keep = []   # the pointer arrays must outlive the call that reads them

        def _keep(a):
            keep.append(a)
            return a

        arr = lambda ts: ctypes.addressof(_keep(_ptr_array([_ptr(t) for t in ts])))   # noqa: E731
        with _guard(dev):
            wss = [_bytes(p.ws_saved_bytes, dev) for p in mp.plans]
            wsb = _keep((ctypes.c_size_t * n)(*[p.ws_saved_bytes for p in mp.plans]))
            need_gin = ctx.needs_input_grad[0]
            gins = [torch.empty_like(u) for _ in range(n)] if need_gin else [None] * n
            gms = [torch.empty((4,) + tuple(s), dtype=torch.float32, device=dev) for s in ctx.param_shapes]
            plane = [4 * p.cfg.C * p.cfg.N * p.cfg.N for p in mp.plans]
            gch = [torch.empty((p.cfg.C, p.cfg.C), dtype=torch.float32, device=dev) if c is not None else None
                   for p, c in zip(mp.plans, chans)]
            gsk = [torch.empty((), dtype=torch.float32, device=dev) if s is not None else None for s in skips]
            gp = lambda k: ctypes.addressof(_keep(_ptr_array([g.data_ptr() + k * pl for g, pl in zip(gms, plane)])))   # noqa: E731
            _cabi.check(L.pde_adi_multi_backward_saved(
                n, ctypes.addressof(mp.descs), arr(tables), _ptr(u), arr(gouts), arr(chans), arr(skips), arr(ckpts), arr(gins),
                gp(0), gp(1), gp(2), gp(3), arr(gch), arr(gsk), arr(wss), ctypes.addressof(wsb), _stream(dev)),
                "pde_adi_multi_backward_saved")
        gin = None
        if need_gin:
            gin = gins[0]
            for g in gins[1:]:
                gin = gin + g
        grads = []
        for i in range(n):
            grads += list(gms[i].unbind(0)) + [gch[i], gsk[i]]
        return (gin, None, *grads)


def adi_multi_layer(u, branches):
    """Apply n implicit layers to the same input.  branches: sequence of (alpha_base, beta_base,
    alpha_time_coeff, beta_time_coeff, chan, skip_weight, cfg).  Returns the n outputs.  Falls back to n
    single-layer calls when the layers cannot share a launch (different shapes / channel ops, plane sizes the
    half-line kernels do not serve, planes on the streaming kernels, inference)."""
    u = _autocast_to_fp32(u)
    cfgs = tuple(b[6] for b in branches)
    # (a traced call takes one op per layer: whether the layers can share a launch is a library query)
    fused = not _traced(u) and u.is_cuda and torch.is_grad_enabled() and any(t is not None and t.requires_grad for b in branches for t in b[:6])
    # the multi-branch launches are built on the shared-memory kernels: a stream-routed branch means one call per layer
    fused = fused and all(adi_route(c) == "tables" for c in cfgs)
    if fused:
        dev = u.device
        with _guard(dev):
            mp = _adi_multi_plan(cfgs, u.shape[0], env_tuning(), dev.index if dev.index is not None else torch.cuda.current_device())
        fused = mp.ok and u.shape[0] > 0
    if not fused:
        return tuple(adi_layer(u, *b[:6], b[6]) for b in branches)
    flat = [t for b in branches for t in b[:6]]
    return _AdiMultiFunction.apply(u, cfgs, *flat)


# ------------------------------------------------------------------- explicit, frozen ghost ring
@dataclass(frozen=True)
class EmoConfig:
    N: int
    Nt: int
    dt: float
    dx: float
    dy: float

    def desc(self, B: int) -> "_cabi.EmoDesc":
        import numpy as np
        f = lambda v: float(np.float32(v))
        return _cabi.EmoDesc(B, self.N, self.Nt, f(0.5 * self.dt), f(self.dt), f(self.dx ** 2), f(self.dy ** 2), 0)


def _emo_check(rc: int, d, what: str):
    if rc == _cabi.ERR_UNSUPPORTED:
        raise _cabi.PdeB200Error(
            f"unsupported emotion PDELayer configuration (N={d.N}, Nt={d.Nt}); supported: N <= 64 with any Nt (the "
            "backward pass while a sample's step states fit a block's shared memory); 65 ... 4096 with Nt <= 16")
    _cabi.check(rc, what)


@functools.lru_cache(maxsize=256)
def _emo_plan(cfg: EmoConfig, B: int, generic: bool, device_index: int):
    """(descriptor, its byref, backward workspace bytes) of a call: depends on nothing else."""
    d = cfg.desc(B)
    d.tuning = _cabi.EMO_TUNE_GENERIC if generic else 0
    return d, byref(d), _cabi.lib().pde_emotion_backward_workspace_bytes(byref(d))


def _emotion_forward(u0, w6, xs, ys, cfg: EmoConfig, generic: bool):
    """The emotion layer's forward pass.  Returns (out, plan, u0, w6, xs, ys), the last four as the kernels read them."""
    _require_cuda(u0, "PDELayer input")
    L = _cabi.lib()
    dev = u0.device
    plan = _emo_plan(cfg, u0.shape[0], generic, dev.index if dev.index is not None else torch.cuda.current_device())
    u0 = _contig(u0)
    w6c, xs, ys = _contig(w6.detach()), _contig(xs), _contig(ys)
    with _guard(u0.device):
        out = torch.empty_like(u0)
        _emo_check(L.pde_emotion_forward(plan[1], _ptr(u0), _ptr(w6c), _ptr(xs), _ptr(ys), _ptr(out), _stream(u0.device)),
                   plan[0], "pde_emotion_forward")
    return out, plan, u0, w6c, xs, ys


def _emotion_backward(plan, u0, w6, xs, ys, gout, need_gin: bool):
    """The emotion layer's backward pass.  Returns (gin or None, g_w6)."""
    L = _cabi.lib()
    gout = _float_grad(gout)
    d, dref, ws_bytes = plan
    if ws_bytes == 0:
        raise _tiny_refused(d)
    with _guard(u0.device):
        ws = _bytes(ws_bytes, u0.device)
        gin = torch.empty_like(u0) if need_gin else None
        gw = torch.empty(6, dtype=torch.float32, device=u0.device)
        _emo_check(L.pde_emotion_backward(dref, _ptr(u0), _ptr(gout), _ptr(w6), _ptr(xs), _ptr(ys), _ptr(gin),
                                          _ptr(gw), _ptr(ws), ws_bytes, _stream(u0.device)), d, "pde_emotion_backward")
    return gin, gw


def _emo_generic() -> bool:
    return os.environ.get("PDE_B200_EMO_TILED") == "0"


class _EmotionFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, u0, w6, xs, ys, cfg: EmoConfig):
        out, plan, u0, w6c, xs, ys = _emotion_forward(u0, w6, xs, ys, cfg, _emo_generic())
        ctx.plan = plan   # the backward pass uses the same descriptor (tuning included)
        ctx.save_for_backward(u0, w6c, xs, ys)
        return out

    @staticmethod
    def backward(ctx, gout):
        _no_double_backward("PDELayer")
        u0, w6, xs, ys = ctx.saved_tensors
        gin, gw = _emotion_backward(ctx.plan, u0, w6, xs, ys, gout, ctx.needs_input_grad[0])
        return gin, gw, None, None, None


@torch.compiler.assume_constant_result
def _traced_emo_generic() -> bool:
    return _emo_generic()


def emotion_layer(u0, w6, xs, ys, cfg: EmoConfig):
    u0, w6 = _autocast_to_fp32(u0), _autocast_to_fp32(w6)
    if _traced(u0):
        return torch.ops.pde_b200.emotion_fwd(u0, w6, xs, ys, cfg.N, cfg.Nt, cfg.dt, cfg.dx, cfg.dy, _traced_emo_generic())
    return _EmotionFunction.apply(u0, w6, xs, ys, cfg)


# ----------------------------------------------------------------------- explicit, zero ghosts
@dataclass(frozen=True)
class TinyConfig:
    steps: int
    dt: float
    cmin: float
    cmax: float
    blend: float = 0.1


def _tiny_refused(d) -> "_cabi.PdeB200Error":
    return _cabi.PdeB200Error(
        f"unsupported tiny_imagenet diffusion configuration (channels={d.C}, H={d.H}, W={d.W}, steps={d.steps}); "
        "supported: any H, W 1 ... 4096 with at most 16 steps and channels <= 1024 (smaller planes take more steps "
        "while a sample's plane and its step states fit a block's shared memory)")


def _tiny_check(rc: int, d, what: str):
    if rc == _cabi.ERR_UNSUPPORTED:
        raise _tiny_refused(d)
    _cabi.check(rc, what)


@functools.lru_cache(maxsize=256)
def _tiny_plan(cfg: TinyConfig, shape, device_index: int):
    B, C, H, W = shape
    d = _cabi.TinyDesc(B, C, H, W, cfg.steps, cfg.dt, cfg.cmin, cfg.cmax, cfg.blend)
    # 0 where no backward pass serves d; the forward may still be served (small planes beyond 16 steps), so only
    # the backward refuses on it
    return d, byref(d), _cabi.lib().pde_tiny_backward_workspace_bytes(byref(d))


def _tiny_forward(u, alpha_base, channel_scaling, cfg: TinyConfig):
    """The tiny_imagenet layer's forward pass, fp32 or bf16 planes after the input's dtype.  Returns
    (out, plan, u, alpha_base, channel_scaling), the last three as the kernels read them."""
    bf16 = isinstance(u, torch.Tensor) and u.is_cuda and u.dtype == torch.bfloat16
    if not bf16:
        _require_cuda(u, "ImprovedDiffusionLayer input")
    L = _cabi.lib()
    u = _contig(u)
    al, sc = _contig(alpha_base.detach()), _contig(channel_scaling.detach())
    if al.dtype != torch.float32 or sc.dtype != torch.float32:   # a module converted with .bfloat16(): the kernels take fp32 scalars
        al, sc = al.float(), sc.float()
    dev = u.device
    plan = _tiny_plan(cfg, tuple(u.shape), dev.index if dev.index is not None else torch.cuda.current_device())
    fwd = L.pde_tiny_forward_bf16 if bf16 else L.pde_tiny_forward
    with _guard(u.device):
        out = torch.empty_like(u)
        _tiny_check(fwd(plan[1], _ptr(u), _ptr(al), _ptr(sc), _ptr(out), _stream(u.device)), plan[0], "pde_tiny_forward")
    return out, plan, u, al, sc


def _tiny_backward(plan, u, al, sc, gout, need_gin: bool):
    """The tiny_imagenet layer's backward pass in u's dtype.  Returns (gin or None, g_alpha_base, g_channel_scaling)."""
    L = _cabi.lib()
    gout = _contig(gout)
    if gout.dtype != u.dtype:
        gout = gout.to(u.dtype)
    C = u.shape[1]
    d, dref, ws_bytes = plan
    if ws_bytes == 0:
        raise _tiny_refused(d)
    with _guard(u.device):
        ws = _bytes(ws_bytes, u.device)
        gin = torch.empty_like(u) if need_gin else None
        ga = torch.empty(C, dtype=torch.float32, device=u.device)
        gs = torch.empty(C, dtype=torch.float32, device=u.device)
        bwd = L.pde_tiny_backward_bf16 if u.dtype == torch.bfloat16 else L.pde_tiny_backward
        _tiny_check(bwd(dref, _ptr(u), _ptr(gout), _ptr(al), _ptr(sc), _ptr(gin), _ptr(ga),
                        _ptr(gs), _ptr(ws), ws_bytes, _stream(u.device)), d, "pde_tiny_backward")
    return gin, ga, gs


class _TinyFunction(torch.autograd.Function):
    """fp32 planes in, fp32 planes out -- or bfloat16 in, bfloat16 out (pde_tiny_*_bf16: the arithmetic, the
    parameters and their gradients stay fp32; the one bandwidth-bound layer of the reference moves half the bytes)."""

    @staticmethod
    def forward(ctx, u, alpha_base, channel_scaling, cfg: TinyConfig):
        out, plan, u, al, sc = _tiny_forward(u, alpha_base, channel_scaling, cfg)
        ctx.plan = plan
        ctx.save_for_backward(u, al, sc)
        return out

    @staticmethod
    def backward(ctx, gout):
        _no_double_backward("ImprovedDiffusionLayer")
        u, al, sc = ctx.saved_tensors
        return (*_tiny_backward(ctx.plan, u, al, sc, gout, ctx.needs_input_grad[0]), None)


def tiny_layer(u, alpha_base, channel_scaling, cfg: TinyConfig):
    u = _autocast_to_fp32(u)
    if _traced(u):
        return torch.ops.pde_b200.tiny_fwd(u, alpha_base, channel_scaling, cfg.steps, cfg.dt, cfg.cmin, cfg.cmax, cfg.blend)
    return _TinyFunction.apply(u, alpha_base, channel_scaling, cfg)


# --------------------------------------------- tiny_imagenet's dormant scalar-coefficient methods
TINY_SPLIT_MODES = {"implicit_diffusion_step": 0, "solve_implicit_x": 1, "solve_implicit_y": 2,
                    "diffuse_x_explicit": 3, "diffuse_y_explicit": 4}


def _tiny_split_desc(mode: int, B: int, H: int, W: int, coeff_x: float, coeff_y: float, dt: float, eps: float):
    """Band values exactly as the reference produces them: Python-double arithmetic
    (`r = coeff * dt / (1.0 ** 2)`, `1 + 2 * r`, `1 + r`: tiny_imagenet.py:109,113-121; `coeff * self.dt`:
    :207), rounded to fp32 where torch.full / the scalar multiply round them."""
    import numpy as np
    f = lambda v: float(np.float32(v))   # noqa: E731

    def bands(coeff, step):
        r = coeff * step / (1.0 ** 2)
        return (f(-r), f(1 + 2 * r), f(1 + r))

    if mode == 0:
        cx, cy = bands(coeff_x, dt / 2), bands(coeff_y, dt / 2)     # implicit_diffusion_step: :96,99
    elif mode in (1, 2):
        cx, cy = bands(coeff_x, dt), bands(coeff_y, dt)
    else:
        cx, cy = (f(coeff_x * dt), 0.0, 0.0), (f(coeff_y * dt), 0.0, 0.0)
    d = _cabi.TinySplitDesc(B, H, W, mode)
    for i in range(3):
        d.cx[i], d.cy[i] = cx[i], cy[i]
    d.eps = f(eps)
    return d


def _tiny_split_run(desc, u, what: str):
    """One pde_tiny_split call on planes u; the forward pass and (on the upstream gradient) the backward pass."""
    _require_cuda(u, what)
    u = _contig(u)
    out = torch.empty_like(u)
    with _guard(u.device):
        _cabi.check(_cabi.lib().pde_tiny_split(byref(desc), _ptr(u), _ptr(out), _stream(u.device)), "pde_tiny_split")
    return out


class _TinySplitFunction(torch.autograd.Function):
    """All five maps are linear in u with symmetric bands: backward is the same kernel on the gradient."""

    @staticmethod
    def forward(ctx, u, desc):
        ctx.desc = desc
        return _tiny_split_run(desc, u, "ImprovedDiffusionLayer dormant-path input")

    @staticmethod
    def backward(ctx, gout):
        _no_double_backward("ImprovedDiffusionLayer dormant path")
        return _tiny_split_run(ctx.desc, _float_grad(gout), "ImprovedDiffusionLayer dormant-path gradient"), None


def tiny_split(method: str, u, coeff_x: float = 0.0, coeff_y: float = 0.0, dt: float = 0.01, eps: float = 1e-6):
    """One of ImprovedDiffusionLayer's dormant methods (tiny_imagenet.py:88-233) on planes u (B, H, W).
    The coefficients are Python numbers, as the reference requires (it hands them to torch.full)."""
    if u.dim() != 3:
        raise ValueError(f"{method}: expected (B, H, W) planes, got shape {tuple(u.shape)}")
    B, H, W = u.shape
    if H > 4096 or W > 4096:
        raise _cabi.PdeB200Error(f"{method}: planes up to 4096 x 4096 are built, got {H} x {W}")
    u = _autocast_to_fp32(u)
    if _traced(u):
        return torch.ops.pde_b200.tiny_split(u, TINY_SPLIT_MODES[method], float(coeff_x), float(coeff_y), float(dt),
                                             float(eps))
    d = _tiny_split_desc(TINY_SPLIT_MODES[method], B, H, W, float(coeff_x), float(coeff_y), float(dt), float(eps))
    return _TinySplitFunction.apply(u, d)
