"""PercentileObserver: activation ranges clipped at a percentile of exact-bin histograms, for low-bit (A4) quantisers.

With 15 levels, one outlier in 10^4 values sets the step for every other value.  On each ``observe(x)`` this observer
keeps MinMaxObserver's running range and statistics, and per channel two one-sided histograms anchored at 0 (``n_bins``
bins per side, bin width a power of two, integer counts) of every finite value seen.  The clip is recomputed from the
accumulated histogram on every call: the smallest bin edge above which at most (1 - percentile / 100) of all values lie,
on each side, capped by the running range; scale / zero-point come from the clipped range with the MinMax formula
(observers/minmax.py:67-74).  ``percentile=100`` gives MinMaxObserver's qparams bit for bit.

Integer counts in power-of-two bins make the histogram depend only on the multiset of values observed: the order of the
calls, how they were split, and how batches were sharded over ranks make no difference, so a data-parallel calibration
(parallel.sync_observers) ends with the single-GPU state.  A channel that saw +-inf keeps the MinMax result.  Everything
runs on the device (csrc/hist_observer.cu); observe() never synchronises.

Register by name like any plugin: ``FuseConfig(observer_a_name="PercentileObserver")`` or ``observer_a_name:
PercentileObserver`` in YAML.  QuantizationManager builds it at the quantiser's bit width (``needs_quantizer_bits``).
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import ops
from .._lib import HIST_STATE_HEAD
from ..utils.registry import register_class
from .minmax import MinMaxObserver, _as_cuda


@register_class
class PercentileObserver(MinMaxObserver):
    """State: [C, 12 + 2 * n_bins] fp64 on the device -- MinMaxObserver's eight columns (scale / zero-point those of the
    clipped range), the clipped lo / hi, the bin exponents of the negative and positive side, then the counts of x < 0
    and of x >= 0 (see include/vsiq.h, vsiq_hist_observe)."""

    needs_quantizer_bits = True  # QuantizationManager passes bits_width (the clip's qparams are at the quantiser's width)
    observe_epilogue = None      # no fused form: fused layers run their separate calibration passes
    keeps_histogram = True       # parallel.sync_observers merges the counts (reduce_percentile_states)

    def __init__(self, symmetric=True, num_bits=8, eps=1e-8, ch_axis: Optional[int] = None, percentile: float = 99.99,
                 n_bins: int = 2048):
        super().__init__(symmetric, num_bits, eps, ch_axis)
        n_bins = int(n_bins)
        if not (256 <= n_bins <= 4096 and n_bins & (n_bins - 1) == 0):
            raise ValueError("n_bins must be a power of two in 256..4096")
        if not 0.0 < float(percentile) <= 100.0:
            raise ValueError("percentile must be in (0, 100]")
        self.n_bins = n_bins
        self.percentile = float(percentile)

    @property
    def state_width(self) -> int:
        return HIST_STATE_HEAD + 2 * self.n_bins

    def load_state(self, state: torch.Tensor) -> None:
        """Restore a saved [C, 12 + 2 * n_bins] state.  A [C, 8] min/max state cannot be taken: a percentile needs the
        histogram."""
        if state.dim() != 2 or state.shape[1] != self.state_width:
            raise ValueError(f"percentile observer state must be [channels, {self.state_width}] (n_bins = {self.n_bins})")
        state = state.detach().to(torch.float64)
        dev = self._state.device if self._state is not None else (torch.device("cuda") if torch.cuda.is_available()
                                                                   else state.device)
        if self._state is not None and self._state.shape == state.shape:
            self._state.copy_(state)
        else:
            self._state = state.to(dev).contiguous().clone()
        self._host = None

    def _ensure_state(self, x: torch.Tensor) -> torch.Tensor:
        C = 1 if self.ch_axis is None else x.shape[self.ch_axis]
        if self._state is None:
            self._state = ops.new_percentile_state(C, self.n_bins, x.device)
        elif self._state.shape[0] != C:
            raise ValueError(f"observer saw {self._state.shape[0]} channels before, now {C}")
        elif self._state.device != x.device:
            self._state = self._state.to(x.device)
        return self._state

    @property
    def min_val(self):
        """Running minimum (the unclipped range, as MinMaxObserver reports it)."""
        return self._scalar(0, 0)

    @property
    def max_val(self):
        return self._scalar(1, 0)

    def observe(self, x):
        x = _as_cuda(x.detach())
        st = self._ensure_state(x)
        self.last_stats = ops.hist_observe(x, self.ch_axis, st, self.n_bins, self.percentile, self.num_bits,
                                           self.symmetric, self.eps)
        self.last_count = x.numel() // st.shape[0]
        self._host = None

    def set_percentile(self, percentile: float) -> None:
        """Clip at another percentile of the histogram already gathered: scale / zero-point are recomputed on the device,
        no data is needed (sweep percentiles after one calibration pass)."""
        if not 0.0 < float(percentile) <= 100.0:
            raise ValueError("percentile must be in (0, 100]")
        self.percentile = float(percentile)
        self.recompute_clip()

    def recompute_clip(self) -> None:
        """Columns 8, 9 (clip) and 2, 3 (scale / zero-point) from the stored counts at the current percentile."""
        if self._state is not None:
            ops.hist_clip(self._state, self.n_bins, self.percentile, self.num_bits, self.symmetric, self.eps)
        self._host = None
        if self._on_change is not None:
            self._on_change()

    def lsq_init_scale(self, bits: int, out: Optional[torch.Tensor] = None, dtype=torch.float64) -> torch.Tensor:
        """The reference rule on the call statistics (columns 4..7), unchanged by the clip."""
        if self._state is None:
            raise RuntimeError("PercentileObserver.lsq_init_scale() before any observe()")
        C = self._state.shape[0]
        if out is None:
            out = torch.empty(C, dtype=dtype, device=self._state.device)
        return ops.lsq_init_scale(self._state[:, :8].contiguous(), bits, out)
