"""CPU oracle of the MSE observer's clipping-range search -- TEST INFRASTRUCTURE ONLY.

NumPy wrapper around ``mse_oracle/mse_oracle.c``; only tests/, __graft_entry__.smoke() and tools/mse_bench.py use it,
as the checker.  The library is compiled with gcc on first use (``build()``, also run by __graft_entry__.build()) into
``mse_oracle/_build``, or into a temporary directory when the tree is read-only.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "mse_oracle.c")
_f32p = ctypes.POINTER(ctypes.c_float)
_f64p = ctypes.POINTER(ctypes.c_double)
_i64 = ctypes.c_int64
STATE_WIDTH = 10
_lib = None


def _compile(out: str) -> None:
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-o", out,
                    _SRC, "-lm"], check=True)


def build(force: bool = False) -> str:
    """Compile the oracle (seconds); returns the path of the shared library."""
    so = os.path.join(_HERE, "_build", "libmse_oracle.so")
    if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(_SRC):
        return so
    try:
        os.makedirs(os.path.dirname(so), exist_ok=True)
        _compile(so)
        return so
    except (OSError, subprocess.CalledProcessError):
        so = os.path.join(tempfile.mkdtemp(prefix="mse_oracle_"), "libmse_oracle.so")
        _compile(so)
        return so


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        L.mse_oracle_search.argtypes = [_f32p, _i64, _i64, _i64, _f64p, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                        ctypes.c_int, _f64p, _f64p]
        L.mse_oracle_search.restype = None
        L.mse_oracle_qparams.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                         _f64p, _f64p]
        L.mse_oracle_qparams.restype = None
        _lib = L
    return _lib


def layout(shape, ch_axis: Optional[int]):
    """(outer, C, inner) of a contiguous tensor quantised along ``ch_axis`` (None = per tensor)."""
    n = int(np.prod(shape, dtype=np.int64)) if len(shape) else 1
    if ch_axis is None:
        return 1, 1, n
    outer = int(np.prod(shape[:ch_axis], dtype=np.int64)) if ch_axis > 0 else 1
    C = int(shape[ch_axis])
    return outer, C, n // (outer * C)


def new_state(channels: int) -> np.ndarray:
    """Fresh [C, 10] state: range 0, scale 1 (ops.new_observer_state's convention), no calls."""
    st = np.zeros((channels, STATE_WIDTH), dtype=np.float64)
    st[:, 2] = 1.0
    return st


def search(x, ch_axis, state: np.ndarray, bits: int, symmetric: bool, eps: float = 1e-8, n_candidates: int = 100):
    """One MSEObserver.observe(x) call on the logical (NCHW / OIHW) array x: updates ``state`` [C, 10] in place and
    returns (E [C, K], chosen alpha [C])."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    outer, C, inner = layout(x.shape, ch_axis)
    if state.shape != (C, STATE_WIDTH) or state.dtype != np.float64 or not state.flags.c_contiguous:
        raise ValueError("state must be a C-contiguous float64 [channels, 10] array")
    K = int(n_candidates)
    err = np.zeros((C, K), dtype=np.float64)
    alpha = np.zeros(C, dtype=np.float64)
    lib().mse_oracle_search(x.ctypes.data_as(_f32p), outer, C, inner, state.ctypes.data_as(_f64p), int(bits),
                            int(bool(symmetric)), float(eps), K, err.ctypes.data_as(_f64p), alpha.ctypes.data_as(_f64p))
    return err, alpha


def qparams(mn: float, mx: float, bits: int, symmetric: bool, eps: float = 1e-8):
    s, z = ctypes.c_double(), ctypes.c_double()
    lib().mse_oracle_qparams(float(mn), float(mx), int(bits), int(bool(symmetric)), float(eps), ctypes.byref(s),
                             ctypes.byref(z))
    return s.value, z.value


def relative_error(w, bits: int, symmetric: bool, n_candidates: int, eps: float = 1e-8) -> float:
    """||fq(W) - W||^2 / ||W||^2 of a per-channel (ch_axis 0) quantiser calibrated on W alone with K candidates
    (K = 1: the MinMax observer's qparams)."""
    w = np.ascontiguousarray(w, dtype=np.float32)
    C = w.shape[0]
    st = new_state(C)
    err, alpha = search(w, 0, st, bits, symmetric, eps, n_candidates)
    k = np.rint(alpha * n_candidates).astype(np.int64) - 1
    num = float(np.sum(err[np.arange(C), k]))
    return num / float(np.sum(w.astype(np.float64) ** 2))
