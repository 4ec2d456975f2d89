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

from .. import ops, parallel
from .._lib import HIST_STATE_HEAD
from ..utils.registry import register_class
from .minmax import MinMaxObserver, _as_cuda


class HistogramObserver(MinMaxObserver):
    """What the histogram observers share: MinMaxObserver's running state plus per-channel exact-bin histograms, in a
    [C, 12 + 2 * n_bins] fp64 state on the device -- MinMaxObserver's eight columns (scale / zero-point those of the
    clipped range), the clipped lo / hi, the bin exponents of the negative and positive side, then the counts of x < 0
    and of x >= 0 (see include/vsiq.h, vsiq_hist_observe).  Subclasses choose the clip (recompute_clip); the histogram
    and its cross-rank merge are the same, so one subclass's checkpoint loads into another."""

    needs_quantizer_bits = True  # QuantizationManager passes bits_width (the clip's qparams are at the quantiser's width)
    observe_epilogue = None      # no fused form: fused layers run their separate calibration passes
    _kind = "histogram observer"

    def __init__(self, symmetric=True, num_bits=8, eps=1e-8, ch_axis: Optional[int] = None, n_bins: int = 2048):
        super().__init__(symmetric, num_bits, eps, ch_axis)
        ops._check_hist_args(n_bins, 100.0)
        self.n_bins = int(n_bins)

    @property
    def state_width(self) -> int:
        return HIST_STATE_HEAD + 2 * self.n_bins

    def _new_state(self, channels: int, device) -> torch.Tensor:
        return ops.new_percentile_state(channels, self.n_bins, device)

    def _adapt_state(self, state: torch.Tensor) -> torch.Tensor:
        """A [C, 8] min/max state cannot be taken: the clip needs the histogram."""
        if state.dim() != 2 or state.shape[1] != self.state_width:
            raise ValueError(f"{self._kind} state must be [channels, {self.state_width}] (n_bins = {self.n_bins})")
        return state

    # getters only, so that assigning raises: MinMaxObserver's setters would recompute qparams from the unclipped range
    @property
    def min_val(self):
        """Running minimum (the unclipped range, as MinMaxObserver reports it)."""
        return self._scalar(0, 0)

    @property
    def max_val(self):
        return self._scalar(1, 0)

    def recompute_clip(self) -> None:
        raise NotImplementedError

    def device_range(self):
        """(lo, hi) views of the device state (fp64): the clipped range (columns 8, 9)."""
        st = self._state
        return st[:, 8], st[:, 9]

    def sync_key(self) -> tuple:
        return ("percentile", self.n_bins)

    @classmethod
    def merge_states(cls, arena: torch.Tensor, observers: list, group=None) -> None:
        """Range and call statistics as MinMaxObserver, histograms merged exactly; each observer re-clips in
        after_merge, by its own rule."""
        parallel.reduce_percentile_states(arena, observers[0].n_bins, group)

    def after_merge(self) -> None:
        self.recompute_clip()  # also drops the host copies (_on_change)


@register_class
class PercentileObserver(HistogramObserver):
    """Clip at a percentile of the histogram (see the module docstring)."""

    _kind = "percentile observer"

    def __init__(self, symmetric=True, num_bits=8, eps=1e-8, ch_axis: Optional[int] = None, percentile: float = 99.99,
                 n_bins: int = 2048):
        super().__init__(symmetric, num_bits, eps, ch_axis, n_bins)
        ops._check_hist_args(n_bins, percentile)
        self.percentile = float(percentile)

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
        ops._check_hist_args(self.n_bins, percentile)
        self.percentile = float(percentile)
        self.recompute_clip()

    def recompute_clip(self) -> None:
        """Columns 8, 9 (clip) and 2, 3 (scale / zero-point) from the stored counts at the current percentile."""
        if self._state is not None:
            ops.hist_clip(self._state, self.n_bins, self.percentile, self.num_bits, self.symmetric, self.eps)
        self._host = None
        if self._on_change is not None:
            self._on_change()
