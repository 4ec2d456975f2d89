"""QuantizationManager: per-tensor state machine between a fused layer and its observer / quantizer plugins.

Reference: quantizers/quantization_manager.py:10-114.  Same constructor, attributes (quantizer, observer, bits_width,
scale, zero_point, is_observer_qparam, is_learning_scale, is_quantize, is_symmetric, mean_abs_x, mean_x, std) and
methods (collect_qparameter, quantize, make_learn_qparameter, init_scaling_factor_for_learning); plugins are built
from the registry by name exactly like :41-42 (so the observer is always 8-bit unless ``observer_bits`` is given --
SURVEY.md 0.4).  What differs is WHERE the numbers live:

  * calibration (collect_qparameter) is one kernel launch and NO host synchronisation per call: min/max, the three
    statistics, the running state, scale and zero-point all stay on the device (the reference does 5 reductions and
    5 ``.item()`` syncs, :66-69).  ``scale`` / ``zero_point`` / ``mean_abs_x`` / ``mean_x`` / ``std`` are read back
    lazily, only when host code asks for them;
  * with fixed qparams the kernels read scale / zero-point straight from the observer state on the device;
  * init_scaling_factor_for_learning + make_learn_qparameter build the learnable Parameter on the device.

Checkpoints (SURVEY.md 5, 8(f).4): the reference's calibrated scale / zero-point are plain Python attributes and its
observer extrema live outside any nn.Module, so ``state_dict()`` loses them and only the learned ``scale`` Parameters
survive (yolov8_qat.py:299,309).  Here the same keys are kept (``...weight_quantizer.scale`` / ``.zero_point`` for
learned qparams) and everything else -- observer state, fixed qparams, the mode flags -- travels in the module's
``_extra_state`` entry; loading a checkpoint that has learned qparams into a freshly fused model re-creates the
Parameters, and a reference checkpoint without ``_extra_state`` still loads.

Deliberate fixes where the reference cannot run (SURVEY.md Appendix B): the constructor's ``is_symmetric`` is stored
(the reference hard-codes True, :50, so an asymmetric learnable zero-point is unreachable and crashes, uniform.py:50-52);
asymmetric managers therefore get the learnable zero-point the code at :100-101 intends.  Symmetric flows -- every
flow the reference can execute -- are unchanged.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.nn as nn

from .._lib import STATE_WIDTH
from ..observers.entropy import EntropyObserver  # noqa: F401  (registers the plugin classes)
from ..observers.minmax import MinMaxObserver  # noqa: F401
from ..observers.moving_average import MovingAverageMinMaxObserver  # noqa: F401
from ..observers.mse import MSEObserver  # noqa: F401
from ..observers.percentile import PercentileObserver  # noqa: F401
from ..quantizers.fp8 import FP8Quantizer  # noqa: F401
from ..quantizers.uniform import UniformQuantizer  # noqa: F401
from ..utils.registry import CLASS_REGISTRY

_LAZY = ("scale", "zero_point")


class QuantizationManager(nn.Module):
    def __init__(self, quantizer_name: str, observer_name: str, bits_width: int, is_symmetric: bool,
                 is_learning_scale: bool = True, observer_bits: Optional[int] = None, ch_axis: Optional[int] = None,
                 param_dtype: torch.dtype = torch.float64) -> None:
        super().__init__()
        self.quantizer = CLASS_REGISTRY[quantizer_name](bits_width, is_symmetric)
        if observer_bits is None and getattr(CLASS_REGISTRY[observer_name], "needs_quantizer_bits", False):
            observer_bits = bits_width  # an observer whose result depends on the quantiser's width (MSE, the histograms)
        if observer_bits is None:
            self.observer = CLASS_REGISTRY[observer_name](is_symmetric)  # num_bits stays 8, like the reference
        else:
            self.observer = CLASS_REGISTRY[observer_name](is_symmetric, observer_bits)
        if ch_axis is not None:
            self.quantizer.ch_axis = ch_axis
            self.observer.ch_axis = ch_axis
        self.ch_axis = ch_axis
        # FP8 quantisers: scale = amax / F of the observer's range, kept in a persistent device buffer (_fp8_refresh)
        self._fp8 = int(getattr(self.quantizer, "fp8_format", 0))
        self._fp8_scale: Optional[torch.Tensor] = None
        if self._fp8 and isinstance(self.observer, (MSEObserver, EntropyObserver)):
            raise ValueError(f"{type(self.observer).__name__} searches the best integer grid; it cannot calibrate "
                             f"{type(self.quantizer).__name__} (use MinMaxObserver or PercentileObserver)")
        if hasattr(self.observer, "_on_change"):
            self.observer._on_change = self._invalidate  # host code poking min_val / max_val drops the cached qparams
        self.bits_width = bits_width
        self.param_dtype = param_dtype  # the reference's learned scale is a 0-dim float64 Parameter (SURVEY 0.6)
        self.scale = 1
        self.zero_point = 0
        self.is_observer_qparam = True
        self.is_learning_scale = is_learning_scale
        self.is_quantize = True
        self.is_symmetric = is_symmetric
        self._call_stats: List = []   # (device stats [C,5], elements per channel) per calibration call
        self._calibrated = False      # the observer state on the device is the source of scale / zero_point

    # ---- lazily materialised host views ---------------------------------------------------------------
    def __getattr__(self, name):
        # reached only when normal lookup fails: scale / zero_point were invalidated by a calibration call
        if name in _LAZY and "_calibrated" in self.__dict__ and self.__dict__["_calibrated"]:
            if self.__dict__.get("_fp8"):
                s = self.__dict__["_fp8_scale"].cpu()  # one D2H copy
                s, z = (float(s[0]), 0) if s.numel() == 1 else (s.clone(), 0)
            else:
                s, z = self.observer.get_scale_zero_point()  # one D2H copy
            self.__dict__["scale"], self.__dict__["zero_point"] = s, z
            return self.__dict__[name]
        return super().__getattr__(name)

    def _invalidate(self) -> None:
        """The observer state changed (calibration call, load_state, a host poke, sync_observers' merge)."""
        self.__dict__.pop("scale", None)
        self.__dict__.pop("zero_point", None)
        self._fp8_refresh()

    def _fp8_refresh(self) -> None:
        """Rewrite the FP8 scale from the observer's range IN PLACE (no host sync): CUDA graphs captured with the fixed
        qparams and cached pointers keep seeing the current value."""
        st = getattr(self.observer, "state", None)
        if not self.__dict__.get("_fp8") or not isinstance(st, torch.Tensor) or not st.is_cuda:
            return
        from .. import ops
        buf = self._fp8_scale
        if buf is None or buf.numel() != st.shape[0] or buf.device != st.device:
            buf = self._fp8_scale = torch.empty(st.shape[0], dtype=torch.float64, device=st.device)
        lo, hi = self.observer.device_range()
        ops.fp8_scale_from_range(lo, hi, self._fp8, buf)

    def _device_qparams(self):
        """Calibrated fixed qparams on the device: the FP8 scale buffer and 0, or the observer's scale / zero-point."""
        if self._fp8:
            if self._fp8_scale is None:
                self._fp8_refresh()
            return self._fp8_scale, 0
        return self.observer.device_qparams()

    def _stats_host(self):
        if not self._call_stats:
            return []
        st = torch.stack([s[0] for s, _ in self._call_stats]).cpu()  # per-tensor view: channel 0
        return [(st[i], n) for i, (_, n) in enumerate(self._call_stats)]

    @property
    def mean_abs_x(self):
        """Per-call mean|x| (reference: a list of floats, :66)."""
        return [float(s[2]) / n for s, n in self._stats_host()]

    @property
    def mean_x(self):
        return [float(s[3]) / n for s, n in self._stats_host()]

    @property
    def std(self):
        out = []
        for s, n in self._stats_host():
            mean = float(s[3]) / n
            var = (float(s[4]) - n * mean * mean) / (n - 1) if n > 1 else float("nan")
            out.append(max(var, 0.0) ** 0.5)
        return out

    # ---- checkpointing --------------------------------------------------------------------------------------
    # state_dict() must hold TENSORS only: training engines walk it blindly (ultralytics' ModelEMA tests
    # ``v.dtype.is_floating_point`` on every entry, the reference's load_partial_checkpoint reads ``.shape``,
    # utils/util.py:27-29, 401-405).  The extra state is therefore ONE packed float64 vector:
    #   [magic, version, is_observer_qparam, is_learning_scale, is_quantize, calibrated, C,
    #    scale kind, scale numel, zero_point kind, zero_point numel, calib_grad_scale kind, calib_grad_scale numel,
    #    observer state (C x 8) ..., scale ..., zero_point ..., calib_grad_scale ...]
    # kind: 0 absent (a learned Parameter: an ordinary state_dict entry), 1 Python int, 2 Python float, 3 0-dim tensor,
    # 4 1-D tensor; +10 when the tensor was float32 (else float64).
    # Version 3 (observers whose state is not [C, 8], e.g. MSEObserver's [C, 10]) appends the state width W to the header
    # and the observer state is C x W; [C, 8] states are still written as version 2, byte for byte.
    _MAGIC, _HEADER = 20477.0, 13

    @staticmethod
    def _pack_value(v):
        if v is None or isinstance(v, nn.Parameter):
            return 0, []
        if isinstance(v, torch.Tensor):
            t = v.detach().to("cpu", torch.float64)
            kind = (3 if t.dim() == 0 else 4) + (10 if v.dtype == torch.float32 else 0)
            return kind, t.reshape(-1).tolist()
        if isinstance(v, bool) or isinstance(v, int):
            return 1, [float(v)]
        return 2, [float(v)]

    @staticmethod
    def _unpack_value(kind: int, vals):
        if kind == 0:
            return None
        if kind == 1:
            return int(vals[0])
        if kind == 2:
            return float(vals[0])
        dtype = torch.float32 if kind >= 10 else torch.float64
        t = torch.tensor(vals, dtype=torch.float64).to(dtype)
        return t.reshape(()) if kind % 10 == 3 else t

    def get_extra_state(self):
        """Everything state_dict() would otherwise lose -- mode flags, the observer's running state, fixed qparams,
        calib_grad_scale -- as one float64 tensor (layout above)."""
        st = getattr(self.observer, "state", None)
        st = st.detach().to("cpu", torch.float64) if isinstance(st, torch.Tensor) else None
        C = st.shape[0] if st is not None else 0
        parts = [self._pack_value(self.__dict__.get("scale")), self._pack_value(self.__dict__.get("zero_point")),
                 self._pack_value(getattr(self.quantizer, "calib_grad_scale", 1))]
        W = st.shape[1] if st is not None else STATE_WIDTH
        head = [self._MAGIC, 2.0 if W == STATE_WIDTH else 3.0, float(bool(self.is_observer_qparam)),
                float(bool(self.is_learning_scale)), float(bool(self.is_quantize)), float(bool(self._calibrated)), float(C)]
        for kind, vals in parts:
            head += [float(kind), float(len(vals))]
        if W != STATE_WIDTH:
            head.append(float(W))
        body = st.reshape(-1).tolist() if st is not None else []
        for _, vals in parts:
            body += vals
        return torch.tensor(head + body, dtype=torch.float64)

    def _decode_extra_state(self, t: torch.Tensor):
        v = t.detach().to("cpu", torch.float64).reshape(-1).tolist()
        if len(v) < self._HEADER or v[0] != self._MAGIC:
            raise ValueError("unrecognised QuantizationManager extra state")
        C = int(v[6])
        kinds = [(int(v[7 + 2 * i]), int(v[8 + 2 * i])) for i in range(3)]
        off = self._HEADER
        W = STATE_WIDTH
        if v[1] == 3.0:
            W = int(v[off])
            off += 1
        elif v[1] != 2.0:
            raise ValueError(f"unsupported QuantizationManager extra state version {v[1]}")
        st = torch.tensor(v[off:off + W * C], dtype=torch.float64).reshape(C, W) if C else None
        off += W * C
        vals = []
        for kind, n in kinds:
            vals.append(self._unpack_value(kind, v[off:off + n]))
            off += n
        return {"flags": {"is_observer_qparam": bool(v[2]), "is_learning_scale": bool(v[3]), "is_quantize": bool(v[4])},
                "calibrated": bool(v[5]), "observer_state": st, "scale": vals[0], "zero_point": vals[1],
                "calib_grad_scale": vals[2]}

    def set_extra_state(self, state) -> None:
        if state is None or (isinstance(state, dict) and not state):
            return
        if isinstance(state, torch.Tensor):
            state = self._decode_extra_state(state)  # dicts: checkpoints written before the packed layout
        for k, v in state.get("flags", {}).items():
            setattr(self, k, v)
        st = state.get("observer_state")
        if st is not None and hasattr(self.observer, "load_state"):
            self.observer.load_state(st)
        self._calibrated = bool(state.get("calibrated", False)) and st is not None
        self._invalidate()
        for name in _LAZY:
            v = state.get(name)
            if v is not None and name not in self._parameters:
                if isinstance(v, torch.Tensor) and st is not None:
                    v = v.to(self.observer.state.device)
                self.__dict__[name] = v
        if self._calibrated and (state.get("scale") is not None):
            self._calibrated = "scale" in self._parameters  # explicit host values win over the observer state
        cgs = state.get("calib_grad_scale")
        if cgs is not None and hasattr(self.quantizer, "calib_grad_scale"):
            self.quantizer.calib_grad_scale = cgs

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        # a checkpoint with learned qparams loaded into a freshly fused model: create the Parameters first
        for name in _LAZY:
            t = state_dict.get(prefix + name)
            if isinstance(t, torch.Tensor) and name not in self._parameters:
                self.__dict__.pop(name, None)
                st = getattr(self.observer, "state", None)
                dev = st.device if isinstance(st, torch.Tensor) else t.device
                self.register_parameter(name, nn.Parameter(torch.empty_like(t, device=dev), requires_grad=True))
                self._calibrated = False
        n_missing = len(missing_keys)
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)
        extra = prefix + "_extra_state"
        if extra in missing_keys[n_missing:]:  # checkpoints written by the reference have no extra state
            missing_keys.remove(extra)

    # ---- reference interface -----------------------------------------------------------------------------
    def collect_qparameter(self, x):
        """Observe x while calibrating (:55-71): one launch, no synchronisation."""
        if not self.is_learning_scale and self.is_observer_qparam:
            self.observer.observe(x)
            self._call_stats.append((self.observer.last_stats, self.observer.last_count))
            self._calibrated = True
            self._invalidate()

    def collect_epilogue(self, pre, act=None, bias=None, bn=None):
        """Calibration form of quantize(act(pre + bias)): while this manager only observes (no quantisation yet) the
        activation and the observer run as one pass over the conv output.  Returns the activated tensor, or None when
        the separate passes must run (quantising, not observing, a plugin observer without the fused form)."""
        collecting = (not self.is_learning_scale) and self.is_observer_qparam
        fused = getattr(self.observer, "observe_epilogue", None)
        if not collecting or self.is_quantize or fused is None:
            return None
        y = fused(pre, act, bias, bn)
        if y is None:
            return None
        self._call_stats.append((self.observer.last_stats, self.observer.last_count))
        self._calibrated = True
        self._invalidate()
        return y

    def can_fuse_relu(self) -> bool:
        """True when quantize(x, pre_relu=True) will run relu + fake-quant as ONE kernel pass."""
        collecting = (not self.is_learning_scale) and self.is_observer_qparam
        return bool(self.is_quantize and not collecting and getattr(self.quantizer, "supports_pre_relu", False))

    def can_fuse_act(self, act, x=None) -> bool:
        """Same question for either activation: "relu" everywhere, "silu" on tensors the NHWC kernels can walk."""
        if act == "relu":
            return self.can_fuse_relu()
        if act == "silu":
            from .. import ops
            return bool(self.can_fuse_relu() and getattr(self.quantizer, "supports_pre_silu", False)
                        and x is not None and ops.ci_supported(x))
        return False

    def _current_qparams(self):
        """(scale, zero_point) as quantize() hands them to the plugin: learned Parameters, never-calibrated defaults or
        host-set values as they are, calibrated fixed qparams from the observer state on the device (no sync)."""
        if "scale" in self._parameters or "zero_point" in self._parameters or not self._calibrated \
                or "scale" in self.__dict__:
            return self.scale, self.zero_point
        return self._device_qparams()

    def can_emit_second(self, act, x) -> bool:
        """True when quantize(x, pre_act=act, second=...) will run as the two-output channels_last epilogue."""
        from .. import ops
        q = self.quantizer
        return bool(act is not None and self.can_fuse_act(act, x) and ops.ci_supported(x) and hasattr(q, "kernel_args")
                    and getattr(q, "mask_mode", "rounded") == "rounded" and self.__dict__.get("_banked") is None
                    and not self._fp8)

    def prequant_plan(self, x):
        """(scale, zero_point, QSpec) for running THIS manager's quantise step as the second stage of another layer's
        epilogue over the channels_last tensor x (the producer of a ``quantize_inp`` layer's input), or None when it
        must run on its own: still observing, quantisation switched off, or a plugin / layout without that form."""
        collecting = (not self.is_learning_scale) and self.is_observer_qparam
        plan = getattr(self.quantizer, "kernel_args", None)
        if collecting or not self.is_quantize or plan is None or self.__dict__.get("_banked") is not None:
            return None
        s, z = self._current_qparams()
        return plan(x, s, z, self.is_learning_scale)

    def quantize_precomputed(self, x, y_pre):
        """quantize(x) whose forward result ``y_pre`` was already written by the producer's two-output epilogue: same
        autograd node (STE / LSQ backward at x), no forward launch."""
        from .. import ops
        s, z = self._current_qparams()
        return self.quantizer.quantize(x, s, z, self.is_learning_scale, precomputed=ops.Precomputed(y_pre))

    def quantize(self, x, pre_relu: bool = False, bias=None, pre_act=None, second=None):
        """collect (if calibrating) then fake-quantise (if enabled) -- :73-90.  ``pre_act`` ("relu" / "silu"; ``pre_relu``
        is the older spelling of "relu"): x is the pre-activation and the activation is applied here -- fused into the
        quantiser kernels when quantising, as a plain F.relu / F.silu otherwise.  ``bias`` (with an activation,
        channels_last x): the conv bias is added in the same pass and its gradient comes out of the backward kernel."""
        act = pre_act or ("relu" if pre_relu else None)
        banked = self.__dict__.get("_banked")
        if banked is not None:  # bank.WeightBank already fake-quantised this weight in its multi-tensor launch
            self.__dict__["_banked"] = None
            if banked[0] is x and act is None:
                return banked[1]
        if act is not None:
            if not self.can_fuse_act(act, x):
                if bias is not None:
                    x = x + bias.view(1, -1, 1, 1)
                fn = torch.nn.functional.relu if act == "relu" else torch.nn.functional.silu
                return self.quantize(fn(x))
            kw = {"pre_act": act}
            if bias is not None:
                kw["bias"] = bias
            if second is not None:
                kw["second"] = second
            if "scale" in self._parameters or "zero_point" in self._parameters or not self._calibrated \
                    or "scale" in self.__dict__:
                return self.quantizer.quantize(x, self.scale, self.zero_point, self.is_learning_scale, **kw)
            s, z = self._device_qparams()
            return self.quantizer.quantize(x, s, z, self.is_learning_scale, **kw)
        self.collect_qparameter(x)
        if not self.is_quantize:
            return x
        if "scale" in self._parameters or "zero_point" in self._parameters or not self._calibrated \
                or "scale" in self.__dict__:
            # learned Parameters, never-calibrated defaults, or values host code has set / read back
            return self.quantizer.quantize(x, self.scale, self.zero_point, self.is_learning_scale)
        # calibrated, fixed qparams: feed the kernels from the observer state on the device (no sync)
        s, z = self._device_qparams()
        return self.quantizer.quantize(x, s, z, self.is_learning_scale)

    def init_scaling_factor_for_learning(self):
        """scale = 2*mean(mean|x|)/sqrt(2^(b-1)-1) (:105-114), computed on the device; becomes a 0-dim (per tensor)
        or [C] tensor of ``param_dtype``.  FP8 quantisers start from the calibrated scale amax / F instead.  Without
        calibration data the current scale is kept."""
        st = self.observer.state
        if st is None or not self._call_stats:
            return
        if self._fp8:
            self._fp8_refresh()
            out = self._fp8_scale.to(self.param_dtype, copy=True)
        else:
            out = torch.empty(st.shape[0], dtype=self.param_dtype, device=st.device)
            self.observer.lsq_init_scale(self.bits_width, out)
        self._calibrated = False
        if "scale" in self._parameters:
            # already learnable (a second activate_learning_qparam / deactivate_learning_qparam): re-initialise the
            # registered Parameter IN PLACE -- a plain attribute of the same name would shadow it, the optimizer would keep
            # training an orphan (the reference raises TypeError here: nn.Module refuses a non-Parameter for that name)
            p = self._parameters["scale"]
            with torch.no_grad():
                p.copy_(out.reshape(p.shape).to(device=p.device, dtype=p.dtype))
            return
        self.__dict__.pop("zero_point", None)
        self.__dict__["scale"] = out.reshape(()) if out.numel() == 1 else out
        if "zero_point" not in self._parameters:
            self.__dict__["zero_point"] = self._current_zero_point()

    def _current_zero_point(self):
        st = self.observer.state
        if st is None or self._fp8:
            return 0
        z = st[:, 3]
        return z.reshape(()) if z.numel() == 1 else z.clone()

    def make_learn_qparameter(self):
        """scale -> nn.Parameter; asymmetric: zero_point -> float nn.Parameter initialised at zp + 1e-9 (:92-103);
        symmetric: zero_point = 0."""
        scale = self.scale
        zp_now = self.zero_point
        self._calibrated = False  # from here on the Parameters (not the observer state) are the source of truth
        if isinstance(scale, nn.Parameter):
            pass
        elif isinstance(scale, torch.Tensor):
            self.__dict__.pop("scale", None)
            self.scale = nn.Parameter(scale.detach().clone().to(self.param_dtype), requires_grad=True)
        else:
            dev = self.observer.state.device if self.observer.state is not None else None
            self.__dict__.pop("scale", None)
            # torch.tensor(python float) is float32, torch.tensor(np.float64) is float64 -- the reference gets fp64
            # after init_scaling_factor_for_learning and fp32 otherwise (:99); param_dtype decides here.
            self.scale = nn.Parameter(torch.tensor(float(scale), dtype=self.param_dtype, device=dev), requires_grad=True)
        if not self.is_symmetric:
            zp = zp_now
            if not isinstance(zp, nn.Parameter):
                self.__dict__.pop("zero_point", None)
                if isinstance(zp, torch.Tensor):
                    z0 = zp.detach().to(torch.float32) + 1e-9
                else:
                    z0 = torch.tensor(float(zp) + 1e-9, dtype=torch.float32, device=self.scale.device)
                self.zero_point = nn.Parameter(z0.to(self.scale.device).reshape(self.scale.shape), requires_grad=True)
        else:
            self.__dict__.pop("zero_point", None)
            if "zero_point" not in self._parameters:
                self.zero_point = 0
        self._calibrated = False
