"""MSEObserver: min/max calibration with a GPU search over clipped ranges, for low-bit (W2 / W4) quantisers.

With 3 or 15 levels, one outlier per channel sets the step size of every other value.  On each ``observe(x)`` this
observer keeps MinMaxObserver's running range and statistics, then scores ``n_candidates`` clipped ranges
(alpha_k * run_min, alpha_k * run_max), alpha_k = k / K, by the squared error of the quantiser that will run, at the
quantiser's bit width, and keeps the best one per channel (ties to the larger alpha; a channel with a non-finite range or
error keeps alpha = 1, i.e. the MinMax result).  The chosen clipped extrema are averaged over calls and scale /
zero-point come from that mean range with the MinMax formula (observers/minmax.py:67-74).  Everything runs on the device
(csrc/mse_search.cu); observe() never synchronises.

Register by name like any plugin: ``FuseConfig(observer_w_name="MSEObserver")`` or ``observer_w_name: MSEObserver`` in
YAML.  QuantizationManager builds it at the quantiser's bit width (``needs_quantizer_bits``).
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import ops, parallel
from .._lib import MSE_STATE_WIDTH, STATE_WIDTH
from ..utils.registry import register_class
from .minmax import MinMaxObserver, _as_cuda, qparam_args


@register_class
class MSEObserver(MinMaxObserver):
    """State: [C, 10] fp64 on the device -- MinMaxObserver's eight columns (running range, scale, zero-point, call
    statistics), then the running means of the chosen clipped min / max."""

    needs_quantizer_bits = True  # QuantizationManager passes bits_width (the search must run at the quantiser's width)
    observe_epilogue = None      # no fused form: fused layers run their separate calibration passes

    def __init__(self, symmetric=True, num_bits=8, eps=1e-8, ch_axis: Optional[int] = None, n_candidates: int = 100):
        super().__init__(symmetric, num_bits, eps, ch_axis)
        if not 1 <= int(n_candidates) <= 256:
            raise ValueError("n_candidates must be in 1..256")
        self.n_candidates = int(n_candidates)
        self.last_err: Optional[torch.Tensor] = None
        self.last_alpha: Optional[torch.Tensor] = None
        self.keep_errors = False  # True: keep each call's E [C, K] and chosen alpha [C] on the device (diagnostics)

    def _new_state(self, channels: int, device) -> torch.Tensor:
        return ops.new_mse_state(channels, device)

    def _adapt_state(self, state: torch.Tensor) -> torch.Tensor:
        """A [C, 8] MinMax state is taken as a range whose clipped means are the range."""
        if state.dim() != 2 or state.shape[1] not in (STATE_WIDTH, MSE_STATE_WIDTH):
            raise ValueError("MSE observer state must be [channels, 10] (or a [channels, 8] min/max state)")
        if state.shape[1] == STATE_WIDTH:
            state = torch.cat([state, state[:, 0:2]], dim=1)
        return state

    # getters only, so that assigning raises: MinMaxObserver's setters would recompute qparams from the unclipped range
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
        self.last_stats, err, alpha = ops.mse_search(x, self.ch_axis, st, self.num_bits, self.symmetric, self.eps,
                                                     self.n_candidates, want_err=self.keep_errors)
        if self.keep_errors:
            self.last_err, self.last_alpha = err, alpha
        self.last_count = x.numel() // st.shape[0]
        self._host = None

    def sync_key(self) -> tuple:
        return ("mse",)

    @classmethod
    def merge_states(cls, arena: torch.Tensor, observers: list, group=None) -> None:
        """Range and call statistics as MinMaxObserver, clipped means weighted by call counts; scale / zero-point of
        every row from the merged means in one launch."""
        parallel.reduce_mse_states(arena, group)
        means = arena[:, :STATE_WIDTH].clone()
        means[:, 0:2] = arena[:, 8:10]
        ops.qparams_from_minmax(means, *qparam_args(observers))
        arena[:, 2:4] = means[:, 2:4]
