"""ctypes binding of libpde_b200.so (include/pde_b200.h).

This is the only place Python touches native code: plain pointers (tensor.data_ptr()), sizes
and a cudaStream_t.  There is no CPU fallback -- if the library is missing or the tensors are
not CUDA tensors the call raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, byref, c_char_p, c_float, c_int, c_int32, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# PDE_B200_LIB points at another build of the same library (A/B timing of kernel variants)
LIB_PATH = os.environ.get("PDE_B200_LIB") or os.path.join(_HERE, "libpde_b200.so")
MAX_SWEEPS = 192
MAX_CHANNELS = 4          # channels of the register-resident implicit kernels
ADI_MAX_CHANNELS = 64     # bound of AdiDesc.C (implicit family)
MAX_BRANCHES = 4
ABI_VERSION = 3
ERR_INVALID, ERR_UNSUPPORTED, ERR_WORKSPACE = -1, -2, -3   # include/pde_b200.h

# pde_adi_desc.tuning / pde_emo_desc.tuning (include/pde_b200.h)
TUNE_IMPL_HALF_LINE = 1
TUNE_IMPL_WHOLE_LINE = 2
EMO_TUNE_GENERIC = 1


def adi_tuning(impl: int = 0, pairs: int = 0, qf: int = 0, np_: int = 0) -> int:
    return (impl & 3) | ((pairs & 7) << 2) | ((qf & 7) << 5) | ((np_ & 3) << 8)

EXPORTS = (
    "pde_b200_abi_version", "pde_b200_error_string", "pde_b200_device_info",
    "pde_adi_tables_bytes", "pde_adi_backward_workspace_bytes", "pde_adi_prepare",
    "pde_adi_forward", "pde_adi_backward",
    "pde_adi_checkpoint_bytes", "pde_adi_backward_saved_workspace_bytes", "pde_adi_forward_train",
    "pde_adi_backward_saved",
    "pde_adi_multi_prepare", "pde_adi_multi_forward_train", "pde_adi_multi_backward_saved",
    "pde_adi_stream_forward_workspace_bytes", "pde_adi_stream_backward_workspace_bytes", "pde_adi_stream_forward",
    "pde_adi_stream_backward",
    "pde_emotion_backward_workspace_bytes", "pde_emotion_forward", "pde_emotion_backward",
    "pde_tiny_backward_workspace_bytes", "pde_tiny_forward", "pde_tiny_backward",
    "pde_tiny_split", "pde_tiny_forward_bf16", "pde_tiny_backward_bf16",
    "pde_emotion_backward_workspace_bytes_bf16", "pde_emotion_forward_bf16", "pde_emotion_backward_bf16",
)


class AdiDesc(Structure):
    _fields_ = [(n, c_int32) for n in ("B", "C", "N", "steps", "lie", "smooth", "has_max", "chan_op", "skip")] + \
               [(n, c_float) for n in ("cmin", "cmax", "eps")] + [("tuning", c_int32)]


class AdiSchedule(Structure):
    _fields_ = [("t", c_float * MAX_SWEEPS), ("dts", c_float * MAX_SWEEPS), ("h2", c_float * MAX_SWEEPS)]


class EmoDesc(Structure):
    _fields_ = [(n, c_int32) for n in ("B", "N", "Nt")] + [(n, c_float) for n in ("half_dt", "dt", "dx2", "dy2")] + \
               [("tuning", c_int32)]


class TinyDesc(Structure):
    _fields_ = [(n, c_int32) for n in ("B", "C", "H", "W", "steps")] + \
               [(n, c_float) for n in ("dt", "cmin", "cmax", "blend")]


class TinySplitDesc(Structure):
    _fields_ = [(n, c_int32) for n in ("B", "H", "W", "mode")] + [("cx", c_float * 3), ("cy", c_float * 3), ("eps", c_float)]


class PdeB200Error(RuntimeError):
    pass


_lib = None


def lib():
    """Load libpde_b200.so (built by build.py / __graft_entry__.build()).  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PdeB200Error(
            f"{LIB_PATH} is missing: build it with `python cnn-with-pde_b200/build.py` "
            "(nvcc, sm_100a).  There is no CPU fallback for the PDE layers.")
    L = ctypes.CDLL(LIB_PATH)
    vp, fp = c_void_p, c_void_p  # device pointers travel as integers
    L.pde_b200_abi_version.restype = c_int
    L.pde_b200_error_string.restype = c_char_p
    L.pde_b200_error_string.argtypes = [c_int]
    L.pde_b200_device_info.restype = c_int
    L.pde_b200_device_info.argtypes = [POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_size_t)]
    L.pde_adi_tables_bytes.restype = c_size_t
    L.pde_adi_tables_bytes.argtypes = [POINTER(AdiDesc)]
    L.pde_adi_backward_workspace_bytes.restype = c_size_t
    L.pde_adi_backward_workspace_bytes.argtypes = [POINTER(AdiDesc)]
    L.pde_adi_prepare.restype = c_int
    L.pde_adi_prepare.argtypes = [POINTER(AdiDesc), POINTER(AdiSchedule), fp, fp, fp, fp, vp, vp]
    L.pde_adi_forward.restype = c_int
    L.pde_adi_forward.argtypes = [POINTER(AdiDesc), vp, fp, fp, fp, fp, vp]
    L.pde_adi_backward.restype = c_int
    L.pde_adi_backward.argtypes = [POINTER(AdiDesc), vp, fp, fp, fp, fp, fp, fp, fp, fp, fp, fp, fp, vp, c_size_t, vp]
    L.pde_adi_checkpoint_bytes.restype = c_size_t
    L.pde_adi_checkpoint_bytes.argtypes = [POINTER(AdiDesc)]
    L.pde_adi_backward_saved_workspace_bytes.restype = c_size_t
    L.pde_adi_backward_saved_workspace_bytes.argtypes = [POINTER(AdiDesc)]
    L.pde_adi_forward_train.restype = c_int
    L.pde_adi_forward_train.argtypes = [POINTER(AdiDesc), vp, fp, fp, fp, fp, vp, vp]
    L.pde_adi_backward_saved.restype = c_int
    L.pde_adi_backward_saved.argtypes = [POINTER(AdiDesc), vp, fp, fp, fp, fp, vp, fp, fp, fp, fp, fp, fp, fp, vp,
                                         c_size_t, vp]
    pp = c_void_p   # arrays of pointers / descriptors travel as their address
    L.pde_adi_multi_prepare.restype = c_int
    L.pde_adi_multi_prepare.argtypes = [c_int, pp, pp, pp, pp, pp, pp, pp, vp]
    L.pde_adi_multi_forward_train.restype = c_int
    L.pde_adi_multi_forward_train.argtypes = [c_int, pp, pp, fp, pp, pp, pp, pp, vp]
    L.pde_adi_multi_backward_saved.restype = c_int
    L.pde_adi_multi_backward_saved.argtypes = [c_int, pp, pp, fp, pp, pp, pp, pp, pp, pp, pp, pp, pp, pp, pp, pp, pp, vp]
    L.pde_adi_stream_forward_workspace_bytes.restype = c_size_t
    L.pde_adi_stream_forward_workspace_bytes.argtypes = [POINTER(AdiDesc)]
    L.pde_adi_stream_backward_workspace_bytes.restype = c_size_t
    L.pde_adi_stream_backward_workspace_bytes.argtypes = [POINTER(AdiDesc)]
    L.pde_adi_stream_forward.restype = c_int
    L.pde_adi_stream_forward.argtypes = [POINTER(AdiDesc), POINTER(AdiSchedule), fp, fp, fp, fp, fp, fp, fp, fp, vp, c_size_t,
                                         vp]
    L.pde_adi_stream_backward.restype = c_int
    L.pde_adi_stream_backward.argtypes = [POINTER(AdiDesc), POINTER(AdiSchedule), fp, fp, fp, fp, fp, fp, fp, fp, fp, fp, fp,
                                          fp, fp, fp, fp, vp, c_size_t, vp]
    L.pde_emotion_backward_workspace_bytes.restype = c_size_t
    L.pde_emotion_backward_workspace_bytes.argtypes = [POINTER(EmoDesc)]
    L.pde_emotion_forward.restype = c_int
    L.pde_emotion_forward.argtypes = [POINTER(EmoDesc), fp, fp, fp, fp, fp, vp]
    L.pde_emotion_backward.restype = c_int
    L.pde_emotion_backward.argtypes = [POINTER(EmoDesc), fp, fp, fp, fp, fp, fp, fp, vp, c_size_t, vp]
    L.pde_emotion_backward_workspace_bytes_bf16.restype = c_size_t
    L.pde_emotion_backward_workspace_bytes_bf16.argtypes = [POINTER(EmoDesc)]
    L.pde_emotion_forward_bf16.restype = c_int
    L.pde_emotion_forward_bf16.argtypes = [POINTER(EmoDesc), fp, fp, fp, fp, fp, vp]
    L.pde_emotion_backward_bf16.restype = c_int
    L.pde_emotion_backward_bf16.argtypes = [POINTER(EmoDesc), fp, fp, fp, fp, fp, fp, fp, vp, c_size_t, vp]
    L.pde_tiny_backward_workspace_bytes.restype = c_size_t
    L.pde_tiny_backward_workspace_bytes.argtypes = [POINTER(TinyDesc)]
    L.pde_tiny_forward.restype = c_int
    L.pde_tiny_forward.argtypes = [POINTER(TinyDesc), fp, fp, fp, fp, vp]
    L.pde_tiny_backward.restype = c_int
    L.pde_tiny_backward.argtypes = [POINTER(TinyDesc), fp, fp, fp, fp, fp, fp, fp, vp, c_size_t, vp]
    L.pde_tiny_forward_bf16.restype = c_int
    L.pde_tiny_forward_bf16.argtypes = [POINTER(TinyDesc), fp, fp, fp, fp, vp]
    L.pde_tiny_backward_bf16.restype = c_int
    L.pde_tiny_backward_bf16.argtypes = [POINTER(TinyDesc), fp, fp, fp, fp, fp, fp, fp, vp, c_size_t, vp]
    L.pde_tiny_split.restype = c_int
    L.pde_tiny_split.argtypes = [POINTER(TinySplitDesc), fp, fp, vp]
    if L.pde_b200_abi_version() != ABI_VERSION:
        raise PdeB200Error("libpde_b200.so ABI version mismatch; rebuild it")
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().pde_b200_error_string(rc).decode()
        raise PdeB200Error(f"{what} failed: {msg} (code {rc})")


def device_info():
    sm, mj, mn, l2 = c_int(), c_int(), c_int(), c_size_t()
    check(lib().pde_b200_device_info(byref(sm), byref(mj), byref(mn), byref(l2)), "pde_b200_device_info")
    return {"sm_count": sm.value, "cc": (mj.value, mn.value), "l2_bytes": l2.value}
