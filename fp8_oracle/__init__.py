"""CPU oracle of the FP8 fake-quantisers -- TEST INFRASTRUCTURE ONLY.

torch-on-CPU and NumPy: the definition of include/vsiq.h's vsiq_fp8_* entry points restated plainly.  Only tests/ and
tools/fp8_bench.py use it, as the checker; nothing under vsiquantization_b200/ imports it.

Per element (F = 448 for E4M3, 57344 for E5M2; s an fp32 tensor, so every CPU op below is one IEEE fp32 operation):
    v = x / s;  c = v.clamp(-F, F);  q = c.to(fp8).float();  y = q * s;  m = (c == v)
    dx = where(m, g * s, 0) / s;  ds = gs * sum g * (q - m * v)  (here in fp64; m * v is NaN for infinite v)
``encode`` is an independent round-to-nearest-even encoder built from the 256 codes, to check torch's cast itself.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

E4M3, E5M2 = 1, 2
FMAX = {E4M3: 448.0, E5M2: 57344.0}
DTYPE = {E4M3: torch.float8_e4m3fn, E5M2: torch.float8_e5m2}


def _scale_tensor(scale, shape, ch_axis: Optional[int]) -> torch.Tensor:
    s = torch.as_tensor(np.asarray(scale, dtype=np.float64)).to(torch.float32).reshape(-1)
    if ch_axis is None or s.numel() == 1:
        return s.reshape(())
    view = [1] * len(shape)
    view[ch_axis] = s.numel()
    return s.reshape(view)


def _pieces(x, scale, fmt, ch_axis, relu):
    xt = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))
    if relu:  # the kernels' fused ReLU, max(x, 0) with NaN propagated: -0.0 becomes +0.0 (ATen's CPU relu keeps -0.0)
        xt = torch.where(torch.isnan(xt) | (xt > 0), xt, torch.zeros((), dtype=torch.float32))
    st = _scale_tensor(scale, xt.shape, ch_axis)
    F = FMAX[fmt]
    v = xt / st
    c = v.clamp(-F, F)
    code = c.to(DTYPE[fmt])
    q = code.float()
    return xt, st, v, c, code, q


def forward(x, scale, fmt: int, ch_axis: Optional[int] = None, relu: bool = False):
    """(y, codes as uint8) as NumPy arrays."""
    _, st, _, _, code, q = _pieces(x, scale, fmt, ch_axis, relu)
    return (q * st).numpy(), code.view(torch.uint8).numpy()


def backward(x, g, scale, fmt: int, ch_axis: Optional[int] = None, relu: bool = False, grad_scale: float = 1.0):
    """(dx, ds as fp64 per channel, sum |terms| per channel) of the STE / LSQ backward."""
    xr = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))
    _, st, v, c, _, q = _pieces(x, scale, fmt, ch_axis, relu)
    gt = torch.as_tensor(np.ascontiguousarray(g, dtype=np.float32))
    m = c == v
    dx = torch.where(m, gt * st, torch.zeros((), dtype=torch.float32)) / st
    if relu:
        dx = torch.where(xr > 0, dx, torch.zeros((), dtype=torch.float32))
    # m * v as a product, like the autograd graph (and the kernels): an infinite x gives 0 * inf = NaN
    term = gt.double() * (q.double() - v.double() * m.double())
    if ch_axis is None:
        ds, mag = term.sum().reshape(1), term.abs().sum().reshape(1)
    else:
        dims = [d for d in range(term.dim()) if d != ch_axis]
        ds, mag = term.sum(dim=dims), term.abs().sum(dim=dims)
    return dx.numpy(), (ds * grad_scale).numpy(), (mag * abs(grad_scale)).numpy()


def grad_scale(fmt: int, numel: int, channels: int = 1) -> float:
    """The LSQ rule with Qp = F."""
    return float((FMAX[fmt] * (numel / channels)) ** -0.5) if channels > 1 else float((FMAX[fmt] * numel) ** -0.5)


# ---- the independent encoder -----------------------------------------------------------------------------------------
def decode_all(fmt: int) -> np.ndarray:
    """float64 value of each of the 256 codes from the bit fields (NaN for the NaN codes, +-inf for E5M2's)."""
    ebits, mbits = (4, 3) if fmt == E4M3 else (5, 2)
    bias = (1 << (ebits - 1)) - 1
    out = np.empty(256, dtype=np.float64)
    for code in range(256):
        sign = -1.0 if code & 0x80 else 1.0
        e = (code >> mbits) & ((1 << ebits) - 1)
        m = code & ((1 << mbits) - 1)
        if fmt == E4M3 and e == 15 and m == 7:
            val = np.nan
        elif fmt == E5M2 and e == 31:
            val = np.inf if m == 0 else np.nan
        elif e == 0:
            val = m / (1 << mbits) * 2.0 ** (1 - bias)
        else:
            val = (1 + m / (1 << mbits)) * 2.0 ** (e - bias)
        out[code] = sign * val
    return out


def encode(a: np.ndarray, fmt: int) -> np.ndarray:
    """uint8 codes of float32 values |a| <= F (or NaN): nearest finite value, ties to the even mantissa (the even code),
    the sign of zero kept.  Midpoints are compared exactly: they are dyadic with few bits, so float64 holds them."""
    vals = decode_all(fmt)
    pos = vals[:128]
    finite = np.isfinite(pos)
    pos = pos[finite]  # codes 0 .. last finite, ascending
    a = np.asarray(a, dtype=np.float32)
    with np.errstate(invalid="ignore"):
        mag = np.abs(a.astype(np.float64))
    hi = np.clip(np.searchsorted(pos, mag, side="left"), 0, len(pos) - 1)
    lo = np.clip(hi - 1, 0, len(pos) - 1)
    mid = (pos[lo] + pos[hi]) / 2.0
    pick = np.where(mag >= pos[hi], hi, np.where(mag < mid, lo, np.where(mag > mid, hi, np.where(lo % 2 == 0, lo, hi))))
    pick = np.where(mag <= pos[0], 0, pick)
    codes = pick.astype(np.uint8) | np.where(np.signbit(a), 0x80, 0).astype(np.uint8)
    return np.where(np.isnan(a), np.uint8(0x7F) | np.where(np.signbit(a), 0x80, 0).astype(np.uint8), codes)
