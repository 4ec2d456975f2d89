"""MinMaxObserver / LSQObserver on the one-pass CUDA observer kernel.

Reference: observers/minmax.py:6-88.  Same constructor, attributes (symmetric, eps, min_val, max_val, num_bits)
and methods (observe, get_scale_zero_point, forward -> (Python float, Python int)), but:
  * one kernel pass produces min, max, sum|x|, sum x, sum x^2 and updates the running state, scale and zero-point
    on the device (fp64, bit-identical to the reference's Python-double formula) -- observe() never synchronises;
  * min_val / max_val / get_scale_zero_point() read the device state back on demand (one small D2H copy).
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import ops, parallel
from .._lib import STATE_WIDTH
from ..utils.registry import register_class
from .base import BaseObserver


def _as_cuda(x: torch.Tensor) -> torch.Tensor:
    if x.is_cuda:
        return x
    if not torch.cuda.is_available():
        raise RuntimeError("vsiquantization_b200 needs a CUDA device: there is no CPU fallback")
    return x.cuda()


def qparam_args(observers) -> tuple:
    """(bits, symmetric, eps) for one ops.qparams_from_minmax launch over the concatenated states of ``observers``."""
    bits = torch.cat([torch.full((o.state.shape[0],), int(o.num_bits), dtype=torch.int32) for o in observers])
    sym = torch.cat([torch.full((o.state.shape[0],), int(bool(o.symmetric)), dtype=torch.int32) for o in observers])
    eps = {float(o.eps) for o in observers}
    if len(eps) != 1:
        raise ValueError("observers with different eps cannot be recomputed in one launch")
    return bits, sym, eps.pop()


@register_class
class MinMaxObserver(BaseObserver):
    """Running min/max observer (state starts at 0, never reset -- observers/minmax.py:28-29).

    ``ch_axis`` (extension, default None = per tensor like the reference) selects per-channel statistics."""

    def __init__(self, symmetric=True, num_bits=8, eps=1e-8, ch_axis: Optional[int] = None):
        self.symmetric = symmetric
        self.eps = eps
        self.num_bits = num_bits
        self.ch_axis = ch_axis
        self._state: Optional[torch.Tensor] = None  # [C, W] fp64 on the device, see _new_state
        self._host = None                            # cached host copy of the state
        self.last_stats: Optional[torch.Tensor] = None
        self.last_count = 0
        self._on_change = None                       # set by the owning QuantizationManager (cache invalidation)

    # -- device state -----------------------------------------------------------------------------
    def _new_state(self, channels: int, device) -> torch.Tensor:
        """A fresh [channels, W] state in this observer's layout."""
        return ops.new_observer_state(channels, device)

    def _adapt_state(self, state: torch.Tensor) -> torch.Tensor:
        """A loaded fp64 state in this observer's layout, or ValueError when it cannot be one."""
        if state.dim() != 2 or state.shape[1] != STATE_WIDTH:
            raise ValueError("observer state must be [channels, 8]")
        return state

    def load_state(self, state: torch.Tensor) -> None:
        """Restore a saved state (checkpoints; QuantizationManager.set_extra_state).  It goes to the GPU when there is
        one; without one it stays on the host and the first kernel call fails loudly."""
        state = self._adapt_state(state.detach().to(torch.float64))
        dev = self._state.device if self._state is not None else (torch.device("cuda") if torch.cuda.is_available()
                                                                   else state.device)
        if self._state is not None and self._state.shape == state.shape:
            # in place: kernels hold pointers into the state (device_qparams() in bank.WeightBank's pointer table, CUDA
            # graphs captured with fixed qparams), which a new tensor would leave stale
            self._state.copy_(state)
        else:
            self._state = state.to(dev).contiguous().clone()
        self._host = None

    def _ensure_state(self, x: torch.Tensor) -> torch.Tensor:
        C = 1 if self.ch_axis is None else x.shape[self.ch_axis]
        if self._state is None:
            self._state = self._new_state(C, x.device)
        elif self._state.shape[0] != C:
            raise ValueError(f"observer saw {self._state.shape[0]} channels before, now {C}")
        elif self._state.device != x.device:
            self._state = self._state.to(x.device)
        return self._state

    @property
    def state(self) -> Optional[torch.Tensor]:
        return self._state

    def _host_state(self):
        if self._state is None:
            return None
        if self._host is None:
            self._host = self._state.detach().cpu()  # the only synchronisation point
        return self._host

    def _scalar(self, col: int, default):
        h = self._host_state()
        if h is None:
            return default
        return float(h[0, col]) if h.shape[0] == 1 else h[:, col].clone()

    @property
    def min_val(self):
        return self._scalar(0, 0)

    @min_val.setter
    def min_val(self, v):
        self._poke(0, v)

    @property
    def max_val(self):
        return self._scalar(1, 0)

    @max_val.setter
    def max_val(self, v):
        self._poke(1, v)

    def _poke(self, col: int, v) -> None:
        if self._state is None:
            if not torch.cuda.is_available():
                raise RuntimeError("vsiquantization_b200 needs a CUDA device: there is no CPU fallback")
            self._state = ops.new_observer_state(1, torch.device("cuda"))
        self._state[:, col] = torch.as_tensor(v, dtype=torch.float64)
        # scale / zero-point follow the extrema on every read in the reference (observers/minmax.py:67-74): recompute the
        # cached columns now and let the owning manager drop its host copies
        n = self._state.shape[0]
        ops.qparams_from_minmax(self._state, torch.full((n,), int(self.num_bits), dtype=torch.int32),
                                torch.full((n,), int(bool(self.symmetric)), dtype=torch.int32), float(self.eps))
        self._host = None
        if self._on_change is not None:
            self._on_change()

    # -- reference interface ------------------------------------------------------------------------
    def observe(self, x):
        """Update the running extrema (and scale / zero-point) from x: observers/minmax.py:32-47, no host sync."""
        x = _as_cuda(x.detach())
        st = self._ensure_state(x)
        self.last_stats = ops.observe(x, self.ch_axis, st, self.num_bits, self.symmetric, self.eps, want_stats=True)
        self.last_count = x.numel() // st.shape[0]
        self._host = None

    def observe_epilogue(self, pre, act=None, bias=None, bn=None):
        """observe(act(pre + bias)) / observe(act(BatchNorm_eval(pre))) with the activated tensor written by the SAME
        pass (ops.ci_epilogue_observe): returns it, or None when this observer / tensor has no such form (per-channel
        statistics, NCHW memory) and the caller must run its separate passes."""
        if type(self).observe is not MinMaxObserver.observe:
            return None  # a subclass with its own update rule (moving averages): its observe() must see the tensor
        if self.ch_axis is not None or not ops.ci_supported(pre):
            return None
        st = self._ensure_state(pre)
        operands = (pre, bias) + (tuple(bn[:4]) if bn is not None else ())
        if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in operands):
            # a calibration loop with autograd on (the reference's data_calib): same kernel behind an autograd node
            sink: list = []
            m, v, w, b, e = bn if bn is not None else (None, None, None, None, 0.0)
            y = ops.EpilogueObserve.apply(pre, bias, m, v, w, b, float(e), act, st, self.num_bits, self.symmetric,
                                          self.eps, sink)
            self.last_stats = sink[0]
        else:
            y, self.last_stats = ops.ci_epilogue_observe(pre.detach(), st, self.num_bits, self.symmetric, self.eps, act,
                                                         bias, bn)
        self.last_count = pre.numel()
        self._host = None
        return y

    def get_scale_zero_point(self):
        """(scale, zero_point) as Python float / int like observers/minmax.py:49-74 (per tensor), or two
        [C] tensors (per channel).  Before anything was observed the state is min = max = 0."""
        h = self._host_state()
        if h is None:
            return 0.0, 0  # min = max = 0: 0 / levels; asymmetric: round(-0 / eps)
        if h.shape[0] == 1:
            return float(h[0, 2]), int(h[0, 3])
        return h[:, 2].clone(), h[:, 3].clone()

    def forward(self, x):
        self.observe(x)
        return self.get_scale_zero_point()

    def lsq_init_scale(self, bits: int, out: Optional[torch.Tensor] = None, dtype=torch.float64) -> torch.Tensor:
        """The reference rule on the call statistics (columns 4..7), whatever columns follow them."""
        if self._state is None:
            raise RuntimeError(f"{type(self).__name__}.lsq_init_scale() before any observe()")
        C = self._state.shape[0]
        if out is None:
            out = torch.empty(C, dtype=dtype, device=self._state.device)
        return ops.lsq_init_scale(self._state[:, :STATE_WIDTH].contiguous(), bits, out)

    # device-side access for the sync-free manager path
    def device_qparams(self):
        """(scale, zero_point) views of the device state (fp64): usable directly as kernel qparams."""
        st = self._state
        return st[:, 2], st[:, 3]

    def device_range(self):
        """(lo, hi) views of the device state (fp64): the range this observer chose -- the running extrema here.  The
        FP8 quantisers derive their scale from it (QuantizationManager)."""
        st = self._state
        return st[:, 0], st[:, 1]

    # -- data-parallel merge (parallel.sync_observers) ------------------------------------------------
    def sync_key(self) -> tuple:
        """Observers with equal keys are merged together: their states are concatenated into one merge_states arena."""
        return ("minmax",)

    @classmethod
    def merge_states(cls, arena: torch.Tensor, observers: list, group=None) -> None:
        """Merge an arena (the concatenated states of ``observers``) over the ranks of ``group`` in place: running
        extrema by MIN / MAX, call statistics summed, then scale / zero-point of every row from the merged range in one
        launch."""
        parallel.reduce_observer_states(arena, group)
        ops.qparams_from_minmax(arena, *qparam_args(observers))

    def after_merge(self) -> None:
        """Runs once the merged rows are back in this observer's state: drop the host copies of the old ones."""
        self._host = None
        if self._on_change is not None:
            self._on_change()


@register_class
class LSQObserver(MinMaxObserver):
    """Observer for LSQ quantisers.  The reference names it (README.md:105-106, modules/fuse_config.py:182) but never
    defines it; here it is the MinMax observer (same min/max-derived scale / zero-point while calibrating) that also
    hands out the LSQ step-size initialisation 2*mean|x|/sqrt(Qp) (quantizers/quantization_manager.py:112) computed
    on the device from the statistics the same kernel pass already gathers (``lsq_init_scale``, inherited: the
    reference's manager uses that initialisation whatever the observer class is)."""
