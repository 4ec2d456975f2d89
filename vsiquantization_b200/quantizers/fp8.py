"""FP8Quantizer (E4M3) / FP8E5M2Quantizer: fake quantisation onto an FP8 value grid, for QAT toward FP8 deployment.

Per element, with F the format's largest finite value (448 for E4M3, 57344 for E5M2):

    v = x / s;  c = clamp(v, -F, F);  q = fp8_rne(c);  y = q * s

i.e. ``(x / s).clamp(-F, F).to(torch.float8_e4m3fn).float() * s`` with every step rounded once in fp32.  Gradients: the
straight-through estimator inside the clamp (dx = g where -F <= v <= F) and the LSQ step-size gradient
``gs * sum g * (q - m * v)`` with gs = (F * numel / channels) ** -0.5 * calib_grad_scale.  Symmetric only: the zero-point is
always 0.  The same kernels as the integer quantisers run it (the rounding step is the only difference, csrc/common.cuh);
the scale comes from the observer's range as amax / F (QuantizationManager).

These classes deliberately do not derive from UniformQuantizer: the multi-tensor weight bank (bank.WeightBank) and the
two-output channels_last epilogue know integer grids only, and leave FP8 layers on their own launches.
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import _lib, ops
from ..utils.registry import register_class
from .base import BaseQuantizer
from .uniform import UniformQuantizer, _as_cuda


@register_class
class FP8Quantizer(BaseQuantizer):
    """FP8 E4M3 (float8_e4m3fn) fake-quantiser.  ``(num_bits, symmetric)`` as the registry builds every quantiser: only
    (8, True) is an FP8 format.  ``ch_axis`` as UniformQuantizer (None = per tensor)."""

    fp8_format = _lib.FP8_E4M3
    supports_pre_relu = True   # quantize(..., pre_relu=True) fuses the preceding ReLU into the kernels
    supports_pre_silu = True   # quantize(..., pre_act="silu") fuses SiLU on channels_last tensors (ops.ci_supported)

    def __init__(self, num_bits=8, symmetric=True, ch_axis: Optional[int] = None):
        if num_bits != 8:
            raise ValueError(f"{type(self).__name__} is an 8-bit format, got num_bits={num_bits}")
        if not symmetric:
            raise ValueError(f"{type(self).__name__} is symmetric only (the zero-point is always 0)")
        self.num_bits = 8
        self.symmetric = True
        self.fmax = _lib.FP8_MAX[self.fp8_format]
        self.qmin = -self.fmax
        self.qmax = self.fmax
        self.calib_grad_scale = 1
        self.ch_axis = ch_axis

    @property
    def codes_dtype(self) -> torch.dtype:
        return torch.float8_e4m3fn if self.fp8_format == _lib.FP8_E4M3 else torch.float8_e5m2

    def calculate_grad_scale(self, quant_tensor, channels: int = 1):
        """The LSQ rule with Qp = F: 1/sqrt(F * numel / C)."""
        return ops.lsq_grad_scale(self.qmax, quant_tensor.numel(), channels)

    _resolve_axis = UniformQuantizer._resolve_axis

    def _spec(self, ch_axis, pre_relu=False) -> ops.QSpec:
        return ops.QSpec(0, 0, ch_axis=ch_axis, pre_relu=pre_relu, fp8_format=self.fp8_format)

    @staticmethod
    def _check_zero_point(zero_point) -> None:
        if isinstance(zero_point, torch.Tensor):
            nonzero = zero_point.numel() > 0 and bool(torch.count_nonzero(zero_point.detach()))
        else:
            nonzero = float(zero_point) != 0.0
        if nonzero:
            raise ValueError("FP8 quantisers are symmetric: the zero-point must be 0")

    def kernel_args(self, x, scale, zero_point, is_learning_scale=False):
        """None: an FP8 quantiser never rides along as the second stage of another layer's two-output epilogue."""
        return None

    def quantize(self, x, scale, zero_point=0, is_learning_scale=False, pre_relu=False, bias=None, pre_act=None,
                 second=None, precomputed=None):
        """Fake-quantise x onto the FP8 grid; the result is autograd-connected to x and to a scale that requires grad.
        ``pre_relu`` / ``pre_act="relu"``: quantise relu(x) in the same pass.  ``bias`` / ``pre_act="silu"``: the
        channels_last epilogue, fq(act(x + bias[c])) in one pass (ops.FakeQuantEpilogue)."""
        if pre_act not in (None, "relu", "silu"):
            raise ValueError("pre_act must be None, 'relu' or 'silu'")
        if second is not None:
            raise ValueError("FP8 quantisers have no two-output epilogue")
        self._check_zero_point(zero_point)
        pre_relu = bool(pre_relu) or pre_act == "relu"
        pre_silu = pre_act == "silu"
        if not x.is_cuda:
            if precomputed is not None:
                raise ValueError("precomputed results are for CUDA tensors")
            y = self.quantize(_as_cuda(x), scale, 0, is_learning_scale, pre_relu, bias, "silu" if pre_silu else None)
            return y.to(x.device)
        ch_axis = self._resolve_axis(x, scale)
        if bias is not None or pre_silu:
            # fq(act(x + bias[c])) on a channels_last conv output: one forward pass, dx / dbias / dscale from one backward
            if precomputed is not None:
                raise ValueError("a precomputed result replaces a plain fake-quant launch, not an epilogue")
            if not ops.ci_supported(x):
                raise ValueError("bias / SiLU fusion needs a channels_last float32 CUDA tensor with C % 4 == 0 and C <= 1024")
            spec = ops.QSpec(0, 0, ch_axis=ch_axis, pre_relu=pre_relu, pre_silu=pre_silu, fp8_format=self.fp8_format)
            learn = isinstance(scale, torch.Tensor) and scale.requires_grad and torch.is_grad_enabled()
            gs_host, gs_dev = self._grad_scale(x, scale, is_learning_scale)
            s_arg = scale if learn else (scale.detach() if isinstance(scale, torch.Tensor) else scale)
            return ops.FakeQuantEpilogue.apply(x, bias, s_arg, 0, spec, gs_host, gs_dev, None)
        spec = self._spec(ch_axis, pre_relu)
        if not (isinstance(scale, torch.Tensor) and scale.requires_grad and torch.is_grad_enabled()):
            s = scale.detach() if isinstance(scale, torch.Tensor) else scale
            return ops.FakeQuantFixed.apply(x, s, 0, spec, precomputed)
        gs_host, gs_dev = self._grad_scale(x, scale, is_learning_scale)
        return ops.FakeQuantLearned.apply(x, scale, 0, spec, gs_host, gs_dev, precomputed)

    def _grad_scale(self, x, scale, is_learning_scale):
        """(host factor, device factor or None) of the LSQ gradient scale, as UniformQuantizer applies it."""
        gs_host, gs_dev = 1.0, None
        if is_learning_scale and isinstance(scale, torch.Tensor):
            gs_host = self.calculate_grad_scale(x, scale.numel())
            cgs = self.calib_grad_scale
            if isinstance(cgs, torch.Tensor):
                gs_dev = cgs.detach().to(device=x.device, dtype=torch.float32).sum().reshape(1)
            else:
                gs_host *= float(cgs)
        return gs_host, gs_dev

    def quantize_codes(self, x, scale, zero_point=0, want_y: bool = True):
        """(fake-quantised tensor or None, codes): codes is a float8_e4m3fn / float8_e5m2 tensor of x's shape holding
        (x / s).clamp(-F, F) in that format -- the deployable FP8 weights."""
        self._check_zero_point(zero_point)
        x = _as_cuda(x)
        s = scale.detach() if isinstance(scale, torch.Tensor) else scale
        return ops.quantize_codes(x.detach(), s, 0, self._spec(self._resolve_axis(x, scale)), want_y=want_y)


@register_class
class FP8E5M2Quantizer(FP8Quantizer):
    """FP8 E5M2 (float8_e5m2) fake-quantiser: F = 57344, two mantissa bits."""

    fp8_format = _lib.FP8_E5M2
