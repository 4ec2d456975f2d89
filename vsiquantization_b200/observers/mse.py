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

from .. import ops
from ..utils.registry import register_class
from .minmax import MinMaxObserver, _as_cuda


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

    def load_state(self, state: torch.Tensor) -> None:
        """Restore a saved [C, 10] state; a [C, 8] MinMax state is taken as a range whose clipped means are the range."""
        if state.dim() != 2 or state.shape[1] not in (8, 10):
            raise ValueError("MSE observer state must be [channels, 10] (or a [channels, 8] min/max state)")
        state = state.detach().to(torch.float64)
        if state.shape[1] == 8:
            state = torch.cat([state, state[:, 0:2]], dim=1)
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
            self._state = ops.new_mse_state(C, x.device)
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
        self.last_stats, err, alpha = ops.mse_search(x, self.ch_axis, st, self.num_bits, self.symmetric, self.eps,
                                                     self.n_candidates, want_err=self.keep_errors)
        if self.keep_errors:
            self.last_err, self.last_alpha = err, alpha
        self.last_count = x.numel() // st.shape[0]
        self._host = None

    def lsq_init_scale(self, bits: int, out: Optional[torch.Tensor] = None, dtype=torch.float64) -> torch.Tensor:
        """The reference rule on the call statistics (columns 4..7), unchanged by the search."""
        if self._state is None:
            raise RuntimeError("MSEObserver.lsq_init_scale() before any observe()")
        C = self._state.shape[0]
        if out is None:
            out = torch.empty(C, dtype=dtype, device=self._state.device)
        return ops.lsq_init_scale(self._state[:, :8].contiguous(), bits, out)
