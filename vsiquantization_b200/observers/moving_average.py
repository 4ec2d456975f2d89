"""MovingAverageMinMaxObserver / MovingAveragePerChannelMinMaxObserver: the observer phase of the reference's
LSQFakeQuantize (quantizers/lsq_module.py:73-91 takes ``observer=MovingAverageMinMaxObserver`` from torch.quantization;
its forward runs ``self.activation_post_process(X.detach())`` and ``self.calculate_qparams()``, lsq_module.py:113-121).

The arithmetic lives in PyTorch (torch/ao/quantization/observer.py: MovingAverageMinMaxObserver.forward,
MovingAveragePerChannelMinMaxObserver.forward, UniformQuantizationObserverBase._calculate_qparams); it is restated here
on top of the one-pass CUDA observer:

    batch extrema       one read of x by the observer kernel (per tensor, per channel NCHW or channels_last) -- torch runs
                        ``torch.aminmax`` after a permute + flatten copy of the tensor
    running extrema     first call: the batch extrema; then  m <- m + c * (m_batch - m)   (fp32, c = averaging_constant)
    scale / zero-point  symmetric: s = max(-min(m_lo, 0), max(m_hi, 0)) / ((qmax - qmin) / 2), z = 0 (signed range)
                        affine:    s = (max(m_hi, 0) - min(m_lo, 0)) / (qmax - qmin),
                                   z = clamp(qmin - round(min(m_lo, 0) / s), qmin, qmax);   s = max(s, eps) in both

The per-channel vectors are tiny, so the running update is a handful of torch elementwise ops on the device (no host
synchronisation); ``ema_update_`` is device-agnostic and is checked bit for bit against torch's own observers on the CPU
(tests/test_abi_and_host.py).  The state layout is the one of MinMaxObserver ([C, 8] fp64), so the manager's sync-free
paths (device_qparams, lsq_init_scale, sync_observers' SUM columns) work unchanged.  Note that a MIN/MAX all-reduce is
NOT the right exchange for moving averages: their merge (parallel.reduce_moving_average_states) averages the running
extrema over the ranks that have observed something, and scale / zero-point are recomputed with the formula above."""
from __future__ import annotations

from typing import Optional

import torch

from .. import ops, parallel
from ..utils.registry import register_class
from .minmax import MinMaxObserver, _as_cuda

_F32_EPS = float(torch.finfo(torch.float32).eps)


def torch_qparams(min_val: torch.Tensor, max_val: torch.Tensor, quant_min: int, quant_max: int, symmetric: bool,
                  eps: float = _F32_EPS):
    """UniformQuantizationObserverBase._calculate_qparams for the signed-symmetric and the affine schemes (fp32 in,
    fp32 scale and int64 zero-point out, any device)."""
    min_neg = torch.min(min_val, torch.zeros_like(min_val))
    max_pos = torch.max(max_val, torch.zeros_like(max_val))
    eps_t = torch.tensor([eps], dtype=torch.float32, device=min_val.device)
    # divisors are TENSORS: ATen-on-CUDA turns division by a Python scalar into a multiplication by its reciprocal (one
    # ulp off the CPU result); tensor / tensor is the IEEE division on both devices, so CUDA reproduces torch-on-CPU
    if symmetric:
        half = torch.tensor([float(quant_max - quant_min) / 2], dtype=torch.float32, device=min_val.device)
        max_pos = torch.max(-min_neg, max_pos)
        scale = max_pos / half
        scale = torch.max(scale, eps_t)
        zero_point = torch.zeros(min_neg.size(), dtype=torch.int64, device=min_val.device)
    else:
        levels = torch.tensor([float(quant_max - quant_min)], dtype=torch.float32, device=min_val.device)
        scale = (max_pos - min_neg) / levels
        scale = torch.max(scale, eps_t)
        zero_point = quant_min - torch.round(min_neg / scale).to(torch.int)
        zero_point = torch.clamp(zero_point, quant_min, quant_max).to(torch.int64)
    return scale, zero_point


def ema_update_(state: torch.Tensor, batch_min: torch.Tensor, batch_max: torch.Tensor, averaging_constant: float,
                quant_min: int, quant_max: int, symmetric: bool, eps: float = _F32_EPS) -> None:
    """Advance a [C, 8] fp64 observer state by one batch (columns: run_min, run_max, scale, zero_point, n_calls, ...).
    batch_min / batch_max: [C] fp32.  The first call (n_calls == 0) adopts the batch extrema, like torch's
    ``min_val.numel() == 0`` branch; no host synchronisation."""
    first = state[:, 4] == 0
    lo, hi = state[:, 0].to(torch.float32), state[:, 1].to(torch.float32)
    bmin, bmax = batch_min.to(torch.float32), batch_max.to(torch.float32)
    new_lo = torch.where(first, bmin, lo + averaging_constant * (bmin - lo))
    new_hi = torch.where(first, bmax, hi + averaging_constant * (bmax - hi))
    scale, zp = torch_qparams(new_lo, new_hi, quant_min, quant_max, symmetric, eps)
    state[:, 0] = new_lo.to(torch.float64)
    state[:, 1] = new_hi.to(torch.float64)
    state[:, 2] = scale.to(torch.float64)
    state[:, 3] = zp.to(torch.float64)
    state[:, 4] += 1.0


@register_class
class MovingAverageMinMaxObserver(MinMaxObserver):
    """torch.quantization.MovingAverageMinMaxObserver semantics (``ch_axis=None``) or
    MovingAveragePerChannelMinMaxObserver (``ch_axis`` given) on the CUDA observer kernel.  Constructor follows the
    registry convention ``(symmetric, num_bits)``; the integer range is the UniformQuantizer's for the same arguments
    (signed for symmetric, unsigned for affine)."""

    def __init__(self, symmetric=True, num_bits=8, eps=_F32_EPS, ch_axis: Optional[int] = None,
                 averaging_constant: float = 0.01):
        super().__init__(symmetric, num_bits, eps, ch_axis)
        self.averaging_constant = averaging_constant
        if symmetric:
            self.quant_min, self.quant_max = -(2 ** (num_bits - 1)), 2 ** (num_bits - 1) - 1
        else:
            self.quant_min, self.quant_max = 0, 2 ** num_bits - 1

    def observe(self, x):
        x = _as_cuda(x.detach())
        st = self._ensure_state(x)
        stats = ops.observe(x, self.ch_axis, None, self.num_bits, self.symmetric, self.eps, want_stats=True)
        self.last_stats = stats
        self.last_count = x.numel() // st.shape[0]
        ema_update_(st, stats[:, 0], stats[:, 1], self.averaging_constant, self.quant_min, self.quant_max,
                    bool(self.symmetric), self.eps)
        n = float(self.last_count)
        mean = stats[:, 3] / n
        var = (stats[:, 4] - n * mean * mean) / (n - 1.0) if n > 1 else torch.full_like(mean, float("nan"))
        st[:, 5] += stats[:, 2] / n                      # the manager's LSQ-initialisation statistics
        st[:, 6] += mean
        st[:, 7] += torch.sqrt(torch.clamp(var, min=0.0))
        self._host = None

    def sync_key(self) -> tuple:
        return ("ema",)

    @classmethod
    def merge_states(cls, arena: torch.Tensor, observers: list, group=None) -> None:
        parallel.reduce_moving_average_states(arena, group)

    def after_merge(self) -> None:
        """Scale / zero-point from the averaged running extrema with torch's formula, then drop the host copies."""
        st = self._state
        s, z = torch_qparams(st[:, 0].to(torch.float32), st[:, 1].to(torch.float32), self.quant_min, self.quant_max,
                             bool(self.symmetric), float(self.eps))
        st[:, 2], st[:, 3] = s.to(st.dtype), z.to(st.dtype)
        super().after_merge()


@register_class
class MovingAveragePerChannelMinMaxObserver(MovingAverageMinMaxObserver):
    """Per-channel form (torch's default ch_axis is 0: weights; pass ``ch_axis=1`` for NCHW / channels_last
    activations)."""

    def __init__(self, symmetric=True, num_bits=8, eps=_F32_EPS, ch_axis: Optional[int] = 0,
                 averaging_constant: float = 0.01):
        super().__init__(symmetric, num_bits, eps, ch_axis, averaging_constant)
