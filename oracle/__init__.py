"""oracle -- TEST INFRASTRUCTURE, NOT PRODUCT.

ctypes/numpy front end of ``libpde_oracle.so`` (built from ``pde_oracle.c`` by
``oracle/Makefile``): a plain-C CPU restatement of the seven PDE layers of
MariMamgo/CNN-with-PDE, forward and adjoint, in fp32 (reference op order) and fp64.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / --impl
reference legs may import this package.  The product (``cnn-with-pde_b200/``) never does.

Parity pinning: the reference has no tests or golden vectors of its own, so this oracle
is pinned against fixtures generated from the reference's Python modules imported
unmodified (``tests/golden/make_golden.py``).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from dataclasses import dataclass, field
from typing import Dict, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpde_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile libpde_oracle.so with gcc (recipe: oracle/Makefile)."""
    src = os.path.join(_HERE, "pde_oracle.c")
    hdr = os.path.join(_HERE, "pde_oracle.h")
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(p) > os.path.getmtime(_LIB_PATH) for p in (src, hdr)
    )
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-s", "clean"], check=True)
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return _LIB_PATH


class _AdiDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in
                ("B", "C", "N", "steps", "lie", "smooth", "has_max", "chan_op", "skip", "nthreads")] + \
               [(n, ctypes.c_double) for n in ("dt", "hx", "hy", "cmin", "cmax", "eps")]


class _EmoDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("B", "N", "Nt", "nthreads")] + \
               [(n, ctypes.c_double) for n in ("dt", "dx", "dy")]


class _TinyDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("B", "C", "H", "W", "steps", "nthreads")] + \
               [(n, ctypes.c_double) for n in ("dt", "cmin", "cmax", "blend")]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = ctypes.CDLL(_LIB_PATH)
        for name in ("adi_forward", "adi_backward", "emotion_forward", "emotion_backward",
                     "tiny_forward", "tiny_backward", "tiny_split"):
            for suf in ("f32", "f64"):
                getattr(_lib, f"oracle_{name}_{suf}").restype = ctypes.c_int
    return _lib


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _as(a, dt):
    return None if a is None else np.ascontiguousarray(np.asarray(a), dtype=dt)


def _suffix(dtype) -> str:
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        return "f32"
    if dtype == np.float64:
        return "f64"
    raise TypeError(f"oracle supports float32/float64, got {dtype}")


# --------------------------------------------------------------------------------------
# Variant descriptions (what each reference class does; SURVEY.md section 8a)
# --------------------------------------------------------------------------------------

@dataclass
class AdiSpec:
    """Static description of one implicit layer instance."""
    N: int
    C: int
    steps: int
    dt: float
    hx: float
    hy: float
    lie: bool = False
    smooth: bool = False
    has_max: bool = False
    chan_op: int = 0          # 0 none, 1 pre-step mix, 2 post-step coupling
    skip: bool = False
    cmin: float = 1e-6
    cmax: float = 10.0
    eps: float = 1e-6

    def desc(self, B: int, nthreads: int = 0) -> _AdiDesc:
        return _AdiDesc(B, self.C, self.N, self.steps, int(self.lie), int(self.smooth),
                        int(self.has_max), self.chan_op, int(self.skip), nthreads,
                        self.dt, self.hx, self.hy, self.cmin, self.cmax, self.eps)


def spec_mnist(size=28, dt=0.001, dx=1.0, dy=1.0, num_steps=10) -> AdiSpec:
    """mnist_test.DiffusionLayer (mnist_test.py:11-65)."""
    return AdiSpec(N=size, C=1, steps=num_steps, dt=dt, hx=dx, hy=dy, smooth=True)


def spec_fashion(size=28, dt=0.3, dx=1.0, num_steps=4) -> AdiSpec:
    """fashion_mnist.DiffusionLayer: y sweeps use dx (fashion_mnist.py:63)."""
    return AdiSpec(N=size, C=1, steps=num_steps, dt=dt, hx=dx, hy=dx, smooth=True)


def spec_svhn(size=32, channels=3, dt=0.01, dx=1.0, num_steps=10) -> AdiSpec:
    """SVHN.DiffusionLayer: smoothing, post-step coupling, sigmoid skip (SVHN.py:49-86)."""
    return AdiSpec(N=size, C=channels, steps=num_steps, dt=dt, hx=dx, hy=dx, smooth=True,
                   chan_op=2, skip=True)


def spec_cifar10(size=32, channels=3, dt=0.001, dx=1.0, dy=1.0, num_steps=10) -> AdiSpec:
    """cifar10.EnhancedDiffusionLayer: clamp max 10, pre-step mixing (cifar10.py:53-114)."""
    return AdiSpec(N=size, C=channels, steps=num_steps, dt=dt, hx=dx, hy=dy, has_max=True, chan_op=1)


def spec_cifar2(size=32, channels=3, dt=0.001, dx=1.0, dy=1.0, num_steps=10) -> AdiSpec:
    """cifar_2version.LearnableDiffusionLayer: Lie splitting (cifar_2version.py:70-104)."""
    return AdiSpec(N=size, C=channels, steps=num_steps, dt=dt, hx=dx, hy=dy, has_max=True,
                   chan_op=1, lie=True)


def adi_forward(spec: AdiSpec, u, alpha_base, beta_base, alpha_tc, beta_tc, chan=None, skipw=None,
                nthreads: int = 0) -> np.ndarray:
    dt = np.asarray(u).dtype
    suf = _suffix(dt)
    u = _as(u, dt)
    B = u.shape[0]
    assert u.shape[1:] == (spec.C, spec.N, spec.N), u.shape
    args = [_as(a, dt).reshape(spec.C, spec.N, spec.N) for a in (alpha_base, beta_base, alpha_tc, beta_tc)]
    chan = _as(chan, dt)
    skipw = None if skipw is None else _as(skipw, dt).reshape(1)
    out = np.empty_like(u)
    d = spec.desc(B, nthreads)
    rc = getattr(lib(), f"oracle_adi_forward_{suf}")(ctypes.byref(d), _p(u), *[_p(a) for a in args],
                                                      _p(chan), _p(skipw), _p(out))
    if rc:
        raise RuntimeError(f"oracle_adi_forward_{suf} failed rc={rc}")
    return out


def adi_backward(spec: AdiSpec, u, gout, alpha_base, beta_base, alpha_tc, beta_tc, chan=None, skipw=None,
                 need_gin: bool = True, nthreads: int = 0) -> Dict[str, np.ndarray]:
    """Returns dict with gin (dtype of u, or None) and float64 parameter gradients."""
    dt = np.asarray(u).dtype
    suf = _suffix(dt)
    u, gout = _as(u, dt), _as(gout, dt)
    B = u.shape[0]
    shp = (spec.C, spec.N, spec.N)
    assert u.shape[1:] == shp and gout.shape == u.shape
    args = [_as(a, dt).reshape(shp) for a in (alpha_base, beta_base, alpha_tc, beta_tc)]
    chan = _as(chan, dt)
    skipw = None if skipw is None else _as(skipw, dt).reshape(1)
    gin = np.empty_like(u) if need_gin else None
    g = {k: np.zeros(shp, np.float64) for k in ("alpha_base", "beta_base", "alpha_time_coeff", "beta_time_coeff")}
    gchan = np.zeros((spec.C, spec.C), np.float64) if spec.chan_op else None
    gskip = np.zeros(1, np.float64) if spec.skip else None
    d = spec.desc(B, nthreads)
    rc = getattr(lib(), f"oracle_adi_backward_{suf}")(
        ctypes.byref(d), _p(u), _p(gout), *[_p(a) for a in args], _p(chan), _p(skipw), _p(gin),
        _p(g["alpha_base"]), _p(g["beta_base"]), _p(g["alpha_time_coeff"]), _p(g["beta_time_coeff"]),
        _p(gchan), _p(gskip))
    if rc:
        raise RuntimeError(f"oracle_adi_backward_{suf} failed rc={rc}")
    g["gin"] = gin
    if gchan is not None:
        g["chan"] = gchan
    if gskip is not None:
        g["skip_weight"] = gskip.reshape(())
    return g


# --------------------------------------------------------------------------------------

@dataclass
class EmoSpec:
    """emotion_recognition.PDELayer (emotion_recognition.py:56-97)."""
    Nx: int = 48
    Ny: int = 48
    Lx: float = 1.0
    Ly: float = 1.0
    T: float = 0.01
    dt: float = 0.001
    dx: float = field(init=False)
    dy: float = field(init=False)
    Nt: int = field(init=False)

    def __post_init__(self):
        self.dx = self.Lx / self.Nx
        self.dy = self.Ly / self.Ny
        self.Nt = int(self.T / self.dt)

    def desc(self, B, nthreads=0):
        assert self.Nx == self.Ny, "reference broadcasting requires Nx == Ny"
        return _EmoDesc(B, self.Nx, self.Nt, nthreads, self.dt, self.dx, self.dy)


def emotion_forward(spec: EmoSpec, u0, w, xs, ys, nthreads=0) -> np.ndarray:
    dt = np.asarray(u0).dtype
    suf = _suffix(dt)
    u0 = _as(u0, dt)
    B = u0.shape[0]
    assert u0.shape[1:] == (1, spec.Nx, spec.Ny)
    w, xs, ys = _as(w, dt).reshape(6), _as(xs, dt), _as(ys, dt)
    out = np.empty_like(u0)
    d = spec.desc(B, nthreads)
    rc = getattr(lib(), f"oracle_emotion_forward_{suf}")(ctypes.byref(d), _p(u0), _p(w), _p(xs), _p(ys), _p(out))
    if rc:
        raise RuntimeError(f"oracle_emotion_forward failed rc={rc}")
    return out


def emotion_backward(spec: EmoSpec, u0, gout, w, xs, ys, need_gin=True, nthreads=0):
    dt = np.asarray(u0).dtype
    suf = _suffix(dt)
    u0, gout = _as(u0, dt), _as(gout, dt)
    B = u0.shape[0]
    w, xs, ys = _as(w, dt).reshape(6), _as(xs, dt), _as(ys, dt)
    gin = np.empty_like(u0) if need_gin else None
    gw = np.zeros(6, np.float64)
    d = spec.desc(B, nthreads)
    rc = getattr(lib(), f"oracle_emotion_backward_{suf}")(ctypes.byref(d), _p(u0), _p(gout), _p(w), _p(xs),
                                                           _p(ys), _p(gin), _p(gw))
    if rc:
        raise RuntimeError(f"oracle_emotion_backward failed rc={rc}")
    return {"gin": gin, "w": gw}


# --------------------------------------------------------------------------------------

@dataclass
class TinySpec:
    """tiny_imagenet.ImprovedDiffusionLayer live path (tiny_imagenet.py:14-72)."""
    size: int = 64
    channels: int = 3
    dt: float = 0.01
    num_steps: int = 1
    cmin: float = 1e-6
    cmax: float = 0.15
    blend: float = 0.1

    def desc(self, B, H, W, nthreads=0):
        return _TinyDesc(B, self.channels, H, W, self.num_steps, nthreads, self.dt, self.cmin, self.cmax, self.blend)


def tiny_forward(spec: TinySpec, u, alpha_base, scaling, nthreads=0) -> np.ndarray:
    dt = np.asarray(u).dtype
    suf = _suffix(dt)
    u = _as(u, dt)
    B, C, H, W = u.shape
    assert C == spec.channels
    out = np.empty_like(u)
    d = spec.desc(B, H, W, nthreads)
    rc = getattr(lib(), f"oracle_tiny_forward_{suf}")(ctypes.byref(d), _p(u), _p(_as(alpha_base, dt)),
                                                       _p(_as(scaling, dt)), _p(out))
    if rc:
        raise RuntimeError(f"oracle_tiny_forward failed rc={rc}")
    return out


def tiny_backward(spec: TinySpec, u, gout, alpha_base, scaling, need_gin=True, nthreads=0):
    dt = np.asarray(u).dtype
    suf = _suffix(dt)
    u, gout = _as(u, dt), _as(gout, dt)
    B, C, H, W = u.shape
    gin = np.empty_like(u) if need_gin else None
    ga, gs = np.zeros(C, np.float64), np.zeros(C, np.float64)
    d = spec.desc(B, H, W, nthreads)
    rc = getattr(lib(), f"oracle_tiny_backward_{suf}")(ctypes.byref(d), _p(u), _p(gout), _p(_as(alpha_base, dt)),
                                                        _p(_as(scaling, dt)), _p(gin), _p(ga), _p(gs))
    if rc:
        raise RuntimeError(f"oracle_tiny_backward failed rc={rc}")
    return {"gin": gin, "alpha_base": ga, "channel_scaling": gs}


# tiny_imagenet.py:88-233 -- the dormant scalar-coefficient methods of ImprovedDiffusionLayer
TINY_SPLIT_MODES = {"implicit_diffusion_step": 0, "solve_implicit_x": 1, "solve_implicit_y": 2,
                    "diffuse_x_explicit": 3, "diffuse_y_explicit": 4}


def tiny_split_coefficients(mode: int, coeff_x: float, coeff_y: float, dt: float, dtype):
    """The constants the reference hands to ATen, computed in Python double exactly as it does and
    rounded to the tensor dtype the way torch.full / a Python-scalar multiply round them.
    Implicit (tiny_imagenet.py:109,113-121): r = coeff * dt / (1.0 ** 2); bands -r, 1 + 2 r, 1 + r
    (implicit_diffusion_step passes dt / 2 to both solves, :96,99).  Explicit (:207): coeff * dt."""
    dtype = np.dtype(dtype)

    def bands(coeff, step):
        r = coeff * step / (1.0 ** 2)
        return np.array([-r, 1 + 2 * r, 1 + r], dtype=dtype)

    if mode == 0:
        return bands(coeff_x, dt / 2), bands(coeff_y, dt / 2)
    if mode in (1, 2):
        return bands(coeff_x, dt), bands(coeff_y, dt)
    return np.array([coeff_x * dt, 0, 0], dtype=dtype), np.array([coeff_y * dt, 0, 0], dtype=dtype)


def tiny_split(method: str, u, coeff_x: float = 0.0, coeff_y: float = 0.0, dt: float = 0.01, eps: float = 1e-6,
               nthreads=0) -> np.ndarray:
    """One of the dormant methods on planes u (B, H, W); `dt` is the argument the method receives
    (solve_implicit_x / _y take it explicitly, the others use the layer's dt)."""
    mode = TINY_SPLIT_MODES[method]
    dtp = np.asarray(u).dtype
    suf = _suffix(dtp)
    u = _as(u, dtp)
    B, H, W = u.shape
    cx, cy = tiny_split_coefficients(mode, coeff_x, coeff_y, dt, dtp)
    out = np.empty_like(u)
    fn = getattr(lib(), f"oracle_tiny_split_{suf}")
    ct = ctypes.c_float if suf == "f32" else ctypes.c_double
    fn.argtypes = [ctypes.c_int] * 4 + [ctypes.c_void_p, ctypes.c_void_p, ct, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    rc = fn(B, H, W, mode, _p(cx), _p(cy), ct(dtp.type(eps)), nthreads, _p(u), _p(out))
    if rc:
        raise RuntimeError(f"oracle_tiny_split failed rc={rc}")
    return out
