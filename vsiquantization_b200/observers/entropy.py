"""EntropyObserver: activation ranges clipped where the KL divergence of the quantised histogram is smallest.

Entropy calibration is TensorRT's default INT8 calibrator and the ``entropy`` method of pytorch-quantization's
HistogramCalibrator (next to ``mse`` and ``percentile``).  This observer keeps exactly PercentileObserver's state: the
running range and statistics of MinMaxObserver and, per channel, the exact-bin histograms of everything seen (integer
counts, power-of-two bin widths, independent of call order and sharding).  After every ``observe(x)`` it searches the
accumulated counts on the device: both sides folded into one magnitude histogram, every candidate threshold i from
max(start_bin, nq) to the highest non-zero bin scored by KL(P || Q) -- P the histogram below i with the outliers added
into its last bin, Q that histogram quantised to nq levels -- and the clip is the threshold with the smallest divergence
(ties to the larger one), capped by the running range.  Scale / zero-point come from the clipped range with the MinMax
formula.  ``start_bin = n_bins`` gives MinMaxObserver's qparams bit for bit.  The rule is spelled out in include/vsiq.h
(vsiq_hist_entropy_clip); the search is csrc/hist_entropy.cu.

Register by name like any plugin: ``FuseConfig(observer_a_name="EntropyObserver")`` or ``observer_a_name:
EntropyObserver`` in YAML.  QuantizationManager builds it at the quantiser's bit width (``needs_quantizer_bits``): nq is
2^(bits-1), or 2^bits for an asymmetric quantiser whose range starts at 0.
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import ops
from ..utils.registry import register_class
from .minmax import _as_cuda
from .percentile import HistogramObserver


@register_class
class EntropyObserver(HistogramObserver):
    """State: PercentileObserver's [C, 12 + 2 * n_bins] fp64 layout; columns 8, 9 hold the entropy clip."""

    _kind = "entropy observer"

    def __init__(self, symmetric=True, num_bits=8, eps=1e-8, ch_axis: Optional[int] = None, n_bins: int = 2048,
                 start_bin: int = 128):
        super().__init__(symmetric, num_bits, eps, ch_axis, n_bins)
        ops._check_entropy_args(n_bins, start_bin, num_bits)
        self.start_bin = int(start_bin)

    def observe(self, x):
        x = _as_cuda(x.detach())
        st = self._ensure_state(x)
        # percentile 100: the histogram pass leaves the min/max clip, which the search below replaces
        self.last_stats = ops.hist_observe(x, self.ch_axis, st, self.n_bins, 100.0, self.num_bits, self.symmetric,
                                           self.eps)
        ops.hist_entropy_clip(st, self.n_bins, self.start_bin, self.num_bits, self.symmetric, self.eps)
        self.last_count = x.numel() // st.shape[0]
        self._host = None

    def divergences(self) -> Optional[torch.Tensor]:
        """[C, n_bins + 1] fp64: the divergence D_i of every candidate threshold i over the counts gathered so far (NaN
        where i is no candidate).  Re-runs the search, which leaves the state as it is."""
        if self._state is None:
            return None
        d = torch.empty(self._state.shape[0], self.n_bins + 1, dtype=torch.float64, device=self._state.device)
        return ops.hist_entropy_clip(self._state, self.n_bins, self.start_bin, self.num_bits, self.symmetric, self.eps,
                                     divergences=d)

    def recompute_clip(self) -> None:
        """Columns 8, 9 (clip) and 2, 3 (scale / zero-point) from the stored counts by the entropy search."""
        if self._state is not None:
            ops.hist_entropy_clip(self._state, self.n_bins, self.start_bin, self.num_bits, self.symmetric, self.eps)
        self._host = None
        if self._on_change is not None:
            self._on_change()
