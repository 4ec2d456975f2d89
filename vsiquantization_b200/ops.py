"""Tensor-level wrappers over the C ABI and the torch.autograd.Functions built on them.

Everything here takes/returns CUDA fp32 tensors and launches on torch's current stream.  PyTorch is
used for device memory, streams and autograd bookkeeping only; all arithmetic happens in libvsiq.so.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Optional, Tuple, Union

import torch

from . import _lib
from ._lib import F32, F64, Layout, QParams, check, lib

Number = Union[int, float]


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} lives on {t.device}; vsiquantization_b200 runs on CUDA only (no CPU fallback)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


# Slow-path bookkeeping: every time a wrapper has to COPY a tensor before the kernels can walk it (a layout conversion the
# fast paths avoid) or hands the kernels a pointer that forces the scalar (V = 1) instantiation, a counter moves.  Benchmarks
# read them (slow_path_counters()) to show that the measured step took none of these detours.
_slow = {"layout_conversion_copies": 0, "layout_conversion_elements": 0, "grad_layout_copies": 0,
         "unaligned_scalar_launches": 0, "workspace_resets": 0}


def slow_path_counters(reset: bool = False) -> dict:
    out = dict(_slow)
    if reset:
        for k in _slow:
            _slow[k] = 0
    return out


def _note_conversion(t: torch.Tensor) -> None:
    _slow["layout_conversion_copies"] += 1
    _slow["layout_conversion_elements"] += t.numel()


def _note_alignment(*tensors) -> None:
    if any(t is not None and t.data_ptr() % 32 for t in tensors):
        _slow["unaligned_scalar_launches"] += 1


def _dense_for(t: torch.Tensor, name: str, ch_axis: Optional[int]) -> torch.Tensor:
    """CUDA fp32 tensor the kernels can walk WITHOUT a copy.

    The kernels only need memory order, not logical order: per-tensor work (ch_axis None) and weight rows (ch_axis 0,
    the output channel is outermost in both formats) run on channels_last memory as it is, so cuDNN's native NHWC layout
    on sm_100 never has to be converted for the quantiser.  Per-channel ACTIVATION quantisation (ch_axis 1) needs the
    channel to own contiguous rows, i.e. NCHW: anything else is converted."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} lives on {t.device}; vsiquantization_b200 runs on CUDA only (no CPU fallback)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if t.is_contiguous():
        return t
    if ch_axis in (None, 0):
        if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
            return t
        if t.dim() == 5 and t.is_contiguous(memory_format=torch.channels_last_3d):
            return t
    _note_conversion(t)  # e.g. per-channel activation quantisation of an NHWC tensor with C % 4 != 0 or C > 1024
    return t.contiguous()


def _match_layout(g: torch.Tensor, x: torch.Tensor, name: str) -> torch.Tensor:
    """grad_output walked in the same memory order as x (elementwise kernels pair elements by address)."""
    if not g.is_cuda or g.dtype != torch.float32:
        _dense_for(g, name, None)  # raises the right error
    if g.shape != x.shape:
        raise ValueError(f"{name} has shape {tuple(g.shape)}, expected {tuple(x.shape)}")
    if g.stride() == x.stride():
        return g
    out = torch.empty_like(x)  # preserve_format: x's strides
    out.copy_(g)
    _slow["grad_layout_copies"] += 1
    return out


def layout_of(shape, ch_axis: Optional[int]) -> Tuple[int, int, int]:
    """(outer, channels, inner) of a contiguous tensor quantised along ch_axis (None = per tensor)."""
    n = 1
    for d in shape:
        n *= int(d)
    if ch_axis is None:
        return 1, 1, n
    if ch_axis < 0:
        ch_axis += len(shape)
    outer = 1
    for d in shape[:ch_axis]:
        outer *= int(d)
    C = int(shape[ch_axis])
    inner = n // (outer * C) if outer * C else 0
    return outer, C, inner


_workspaces = {}
_WS_PARANOID = os.environ.get("VSIQ_WS_PARANOID", "0") not in ("", "0")


def _workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    """Zero-initialised scratch, one per (device, stream).  The reducing kernels keep a ticket and a tile counter in its
    256-byte header and leave both zero when they finish; a launch that never completed would leave them non-zero and
    the NEXT launch would silently skip work, so the header is cleared again (vsiq_workspace_reset, asynchronous on the
    stream) whenever a library call fails (`check`), on request (reset_workspaces), and -- with VSIQ_WS_PARANOID=1 -- before
    every use (a debugging aid: one extra memset node per reducing launch)."""
    key = (device.index, _stream_ptr())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(nbytes, 1 << 16), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    elif _WS_PARANOID:
        lib.vsiq_workspace_reset(ws.data_ptr(), ws.numel(), _stream_ptr())
        _slow["workspace_resets"] += 1
    return ws


def reset_workspaces() -> int:
    """Clear the header of every cached workspace (each on the stream it belongs to); returns how many were reset.
    Called automatically when a library call reports an error."""
    n = 0
    for (dev_index, stream_ptr), ws in list(_workspaces.items()):
        with torch.cuda.device(dev_index):
            lib.vsiq_workspace_reset(ws.data_ptr(), ws.numel(), stream_ptr)
        n += 1
    _slow["workspace_resets"] += n
    return n


_lib.on_error = reset_workspaces


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise TypeError(f"quantisation parameters must be float32 or float64 tensors, got {t.dtype}")


@dataclass
class QSpec:
    """How one quantiser maps onto the ABI: integer range, channel axis and the qparam sources."""
    qmin: int
    qmax: int
    ch_axis: Optional[int] = None
    zp_learned: bool = False
    mask_mode: int = _lib.MASK_ROUNDED
    pre_relu: bool = False  # quantise relu(x); the backward also applies relu's mask (one pass instead of two)
    pre_silu: bool = False  # quantise silu(x) (ATen-CUDA's op order); channels_last tensors only (ci_forward / ci_backward)
    fp8_format: int = 0     # 0: the integer grid [qmin, qmax]; _lib.FP8_E4M3 / FP8_E5M2: that FP8 grid (qmin = qmax = 0)


def _make_qparams(spec: QSpec, scale, zero_point, channels: int, device: torch.device, keep: list) -> QParams:
    qp = QParams()
    qp.qmin, qp.qmax = (0, 0) if spec.fp8_format else (int(spec.qmin), int(spec.qmax))
    qp.zp_learned = 1 if spec.zp_learned else 0
    qp.pre_op = _lib.PRE_SILU if spec.pre_silu else (_lib.PRE_RELU if spec.pre_relu else _lib.PRE_NONE)
    qp.scale_dtype = qp.zp_dtype = F32
    if isinstance(scale, torch.Tensor):
        s = scale.detach()
        if s.device != device:
            s = s.to(device)
        if s.numel() != channels:
            raise ValueError(f"scale has {s.numel()} entries, the layout has {channels} channels")
        s = s.contiguous()
        keep.append(s)
        qp.scale = s.data_ptr()
        qp.scale_dtype = _dtype_code(s)
    else:
        if channels != 1:
            raise ValueError("a scalar scale needs a per-tensor layout")
        qp.scale = None
        qp.scale_host = float(scale)  # ctypes rounds the double to fp32 (RN), like ATen's scalar cast
    if isinstance(zero_point, torch.Tensor):
        z = zero_point.detach()
        if z.device != device:
            z = z.to(device)
        if not z.is_floating_point():
            z = z.to(torch.float32)
        if z.numel() != channels:
            raise ValueError(f"zero_point has {z.numel()} entries, the layout has {channels} channels")
        z = z.contiguous()
        keep.append(z)
        qp.zero_point = z.data_ptr()
        qp.zp_dtype = _dtype_code(z)
    else:
        qp.zero_point = None
        qp.zp_host = float(zero_point)
        if channels != 1 and isinstance(scale, torch.Tensor) and not spec.fp8_format:
            # scalar zero-point with per-channel scales: broadcast it
            z = torch.full((channels,), float(zero_point), dtype=torch.float32, device=device)
            keep.append(z)
            qp.zero_point = z.data_ptr()
    return qp


def _count_launch(n: int = 1) -> None:
    _lib.launch_count += n


# ----------------------------------------------------------------------------------------------
# raw ops
# ----------------------------------------------------------------------------------------------
def _out_like(x: torch.Tensor, out: Optional[torch.Tensor], name: str) -> torch.Tensor:
    if out is None:
        return torch.empty_like(x)
    if out.shape != x.shape or out.dtype != torch.float32 or out.device != x.device or out.stride() != x.stride():
        raise ValueError(f"{name} must be a float32 tensor with the input's shape and strides, on the same device")
    if out.data_ptr() == x.data_ptr():
        raise ValueError(f"{name} must not alias the input")
    return out


def code_bits_for(spec: QSpec) -> int:
    """Smallest supported code width (8 or 16 bits) that holds [qmin, qmax]; 4-bit packing is opt-in (quantize_codes)."""
    for bits in (8, 16):
        lo, hi = (-(1 << (bits - 1)), (1 << (bits - 1)) - 1) if spec.qmin < 0 else (0, (1 << bits) - 1)
        if spec.qmin >= lo and spec.qmax <= hi:
            return bits
    raise ValueError(f"integer range [{spec.qmin}, {spec.qmax}] does not fit 16-bit codes")


def quantize_codes(x: torch.Tensor, scale, zero_point, spec: QSpec, code_bits: Optional[int] = None, want_y: bool = True,
                   codes_out: Optional[torch.Tensor] = None):
    """(y or None, integer codes) in one pass: codes = clamp(rint(x/s + z), qmin, qmax)  [uniform.py:54,95 keeps them as
    floats].  code_bits 8 / 16 -> int8 / uint8 / int16 / uint16 tensors shaped like x; 4 -> uint8 tensor with HALF the last
    dimension, two codes per byte (element 2k in the low nibble, two's complement when qmin < 0)."""
    if spec.pre_relu or spec.pre_silu:
        raise ValueError("code export has no fused activation")
    if spec.fp8_format:
        return _fp8_codes(x, scale, spec, want_y, codes_out)
    x = _dense_for(x, "x", spec.ch_axis)
    if not x.is_contiguous():
        x = x.contiguous()  # codes are laid out in logical (row-major) order
    if x.data_ptr() % 32:
        x = x.clone()
    bits = code_bits_for(spec) if code_bits is None else int(code_bits)
    outer, C, inner = layout_of(x.shape, spec.ch_axis)
    lay = Layout(outer, C, inner)
    keep: list = []
    with torch.cuda.device(x.device):
        qp = _make_qparams(spec, scale, zero_point, max(C, 1), x.device, keep)
        y = torch.empty_like(x) if want_y else None
        if bits == 4:
            if x.dim() == 0 or x.shape[-1] % 2:
                raise ValueError("int4 packing needs an even last dimension")
            c_shape, dt = x.shape[:-1] + (x.shape[-1] // 2,), torch.uint8
        else:
            signed = spec.qmin < 0
            c_shape = x.shape
            dt = {(8, True): torch.int8, (8, False): torch.uint8, (16, True): torch.int16, (16, False): torch.uint16}[(bits, signed)]
        if codes_out is not None:
            if tuple(codes_out.shape) != tuple(c_shape) or codes_out.dtype != dt or codes_out.device != x.device \
                    or not codes_out.is_contiguous():
                raise ValueError(f"codes_out must be a contiguous {dt} tensor of shape {tuple(c_shape)} on {x.device}")
            codes = codes_out
        else:
            codes = torch.empty(c_shape, dtype=dt, device=x.device)
        check(lib.vsiq_quantize_codes(x.data_ptr(), y.data_ptr() if want_y else None, codes.data_ptr(), bits,
                                      ctypes.byref(lay), ctypes.byref(qp), _stream_ptr()), "vsiq_quantize_codes")
        _count_launch()
    return y, codes


_FP8_DTYPES = {_lib.FP8_E4M3: torch.float8_e4m3fn, _lib.FP8_E5M2: torch.float8_e5m2}


def _fp8_codes(x, scale, spec: QSpec, want_y: bool, codes_out: Optional[torch.Tensor]):
    """(y or None, FP8 codes): codes is a float8_e4m3fn / float8_e5m2 tensor shaped like x holding
    (x / s).clamp(-F, F) rounded to that format -- the deployable weights (vsiq_fp8_fake_quant_fwd with codes)."""
    x = _dense_for(x, "x", spec.ch_axis)
    if not x.is_contiguous():
        x = x.contiguous()  # codes are laid out in logical (row-major) order
    if x.data_ptr() % 32:
        x = x.clone()
    outer, C, inner = layout_of(x.shape, spec.ch_axis)
    lay = Layout(outer, C, inner)
    dt = _FP8_DTYPES[spec.fp8_format]
    keep: list = []
    with torch.cuda.device(x.device):
        qp = _make_qparams(spec, scale, 0, max(C, 1), x.device, keep)
        y = torch.empty_like(x) if want_y else None
        if codes_out is not None:
            if tuple(codes_out.shape) != tuple(x.shape) or codes_out.dtype != dt or codes_out.device != x.device \
                    or not codes_out.is_contiguous():
                raise ValueError(f"codes_out must be a contiguous {dt} tensor of shape {tuple(x.shape)} on {x.device}")
            codes = codes_out
        else:
            codes = torch.empty(x.shape, dtype=dt, device=x.device)
        check(lib.vsiq_fp8_fake_quant_fwd(x.data_ptr(), y.data_ptr() if want_y else None, codes.data_ptr(),
                                          ctypes.byref(lay), ctypes.byref(qp), int(spec.fp8_format), _stream_ptr()),
              "vsiq_fp8_fake_quant_fwd")
        _count_launch()
    return y, codes


def fake_quant_forward(x: torch.Tensor, scale, zero_point, spec: QSpec, want_codes: bool = False,
                       out: Optional[torch.Tensor] = None):
    """y = (clamp(rint(x/s + z), qmin, qmax) - z) * s  [reference: quantizers/uniform.py:54-55,95].
    want_codes: also the integer codes, int8 / uint8 when the range fits 8 bits, else int16 / uint16 (never wrapped)."""
    if want_codes:
        if out is not None:
            raise ValueError("want_codes allocates its own outputs")
        return quantize_codes(x, scale, zero_point, spec)
    if spec.ch_axis == 1 and ci_supported(x):
        return ci_forward(x, None, scale, zero_point, spec, out=out)  # per-channel qparams on NHWC memory, no conversion
    x = _dense_for(x, "x", spec.ch_axis)
    outer, C, inner = layout_of(x.shape, spec.ch_axis)
    lay = Layout(outer, C, inner)
    keep: list = []
    with torch.cuda.device(x.device):
        qp = _make_qparams(spec, scale, zero_point, max(C, 1), x.device, keep)
        y = _out_like(x, out, "out")
        _note_alignment(x, y)
        if spec.fp8_format:
            check(lib.vsiq_fp8_fake_quant_fwd(x.data_ptr(), y.data_ptr(), None, ctypes.byref(lay), ctypes.byref(qp),
                                              int(spec.fp8_format), _stream_ptr()), "vsiq_fp8_fake_quant_fwd")
        else:
            check(lib.vsiq_fake_quant_fwd(x.data_ptr(), y.data_ptr(), None, ctypes.byref(lay), ctypes.byref(qp),
                                          _stream_ptr()), "vsiq_fake_quant_fwd")
        _count_launch()
    return y


def fake_quant_backward_ste(x: torch.Tensor, g: torch.Tensor, scale, zero_point, spec: QSpec,
                            out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dx of the forward through the straight-through estimator [uniform.py:258-271 + clamp backward]."""
    if spec.ch_axis == 1 and out is None and ci_supported(x):
        return ci_backward(x, None, g, scale, zero_point, spec, want_ds=False, want_dbias=False)[0]
    x = _dense_for(x, "x", spec.ch_axis)
    g = _match_layout(g, x, "grad_output")
    outer, C, inner = layout_of(x.shape, spec.ch_axis)
    lay = Layout(outer, C, inner)
    keep: list = []
    with torch.cuda.device(x.device):
        qp = _make_qparams(spec, scale, zero_point, C, x.device, keep)
        dx = _out_like(x, out, "out")
        _note_alignment(x, g, dx)
        if spec.fp8_format:
            check(lib.vsiq_fp8_fake_quant_bwd_ste(x.data_ptr(), g.data_ptr(), dx.data_ptr(), ctypes.byref(lay),
                                                  ctypes.byref(qp), int(spec.fp8_format), _stream_ptr()),
                  "vsiq_fp8_fake_quant_bwd_ste")
        else:
            check(lib.vsiq_fake_quant_bwd_ste(x.data_ptr(), g.data_ptr(), dx.data_ptr(), ctypes.byref(lay),
                                              ctypes.byref(qp), _stream_ptr()), "vsiq_fake_quant_bwd_ste")
        _count_launch()
    return dx


def fake_quant_forward_backward(x, g, scale, zero_point, spec: QSpec, y_out=None, dx_out=None):
    """Fused forward + STE backward sweep (16 B/element) -- used by the host pipeline and the bench."""
    x = _dense_for(x, "x", spec.ch_axis)
    g = _match_layout(g, x, "grad_output")
    outer, C, inner = layout_of(x.shape, spec.ch_axis)
    lay = Layout(outer, C, inner)
    keep: list = []
    with torch.cuda.device(x.device):
        qp = _make_qparams(spec, scale, zero_point, C, x.device, keep)
        y, dx = _out_like(x, y_out, "y_out"), _out_like(x, dx_out, "dx_out")
        check(lib.vsiq_fake_quant_fwd_bwd(x.data_ptr(), g.data_ptr(), y.data_ptr(), dx.data_ptr(), ctypes.byref(lay),
                                          ctypes.byref(qp), _stream_ptr()), "vsiq_fake_quant_fwd_bwd")
        _count_launch()
    return y, dx


def lsq_backward(x, g, scale, zero_point, spec: QSpec, grad_scale: float, grad_scale_dev: Optional[torch.Tensor] = None,
                 ds_out: Optional[torch.Tensor] = None, dz_out: Optional[torch.Tensor] = None, want_dz: bool = False,
                 ds_dtype: torch.dtype = torch.float32, dz_dtype: torch.dtype = torch.float32,
                 dx_out: Optional[torch.Tensor] = None):
    """dx + per-channel dscale (+ dzero_point) in one pass [uniform.py:47-55,242-255; lsq_module.py:147-173,317-340].

    ds_out / dz_out let the caller point the kernel at slices of a flat gradient buffer (parallel.py)."""
    if (spec.ch_axis == 1 and ds_out is None and dz_out is None and dx_out is None and ci_supported(x)
            and spec.mask_mode == _lib.MASK_ROUNDED):
        dx, ds, dz, _ = ci_backward(x, None, g, scale, zero_point, spec, grad_scale, grad_scale_dev, True, want_dz,
                                    False, ds_dtype, dz_dtype)
        return dx, ds, dz
    x = _dense_for(x, "x", spec.ch_axis)
    g = _match_layout(g, x, "grad_output")
    outer, C, inner = layout_of(x.shape, spec.ch_axis)
    lay = Layout(outer, C, inner)
    keep: list = []
    with torch.cuda.device(x.device):
        qp = _make_qparams(spec, scale, zero_point, C, x.device, keep)
        dx = _out_like(x, dx_out, "dx_out")
        ds = ds_out if ds_out is not None else torch.empty(C, dtype=ds_dtype, device=x.device)
        dz = dz_out if dz_out is not None else (torch.empty(C, dtype=dz_dtype, device=x.device) if want_dz else None)
        if ds.numel() != C or (dz is not None and dz.numel() != C):
            raise ValueError("gradient outputs must have one entry per channel")
        nbytes = lib.vsiq_lsq_bwd_workspace_bytes(ctypes.byref(lay))
        ws = _workspace(nbytes, x.device)
        _note_alignment(x, g, dx)
        gsd = None
        if grad_scale_dev is not None:
            gsd = grad_scale_dev.detach().to(device=x.device, dtype=torch.float32).contiguous()
            keep.append(gsd)
        if spec.fp8_format:
            check(lib.vsiq_fp8_lsq_bwd(x.data_ptr(), g.data_ptr(), dx.data_ptr(), ds.data_ptr(), _dtype_code(ds),
                                       dz.data_ptr() if dz is not None else None, _dtype_code(dz) if dz is not None else F32,
                                       ctypes.byref(lay), ctypes.byref(qp), int(spec.fp8_format), float(grad_scale),
                                       gsd.data_ptr() if gsd is not None else None, int(spec.mask_mode), ws.data_ptr(),
                                       ws.numel(), _stream_ptr()), "vsiq_fp8_lsq_bwd")
        else:
            check(lib.vsiq_lsq_bwd(x.data_ptr(), g.data_ptr(), dx.data_ptr(), ds.data_ptr(), _dtype_code(ds),
                                   dz.data_ptr() if dz is not None else None, _dtype_code(dz) if dz is not None else F32,
                                   ctypes.byref(lay), ctypes.byref(qp), float(grad_scale),
                                   gsd.data_ptr() if gsd is not None else None, int(spec.mask_mode), ws.data_ptr(),
                                   ws.numel(), _stream_ptr()), "vsiq_lsq_bwd")
        _count_launch()
    return dx, ds, dz


def ci_supported(x: torch.Tensor) -> bool:
    """True when x is a channels_last (NHWC-in-memory) activation the channel-innermost kernels can walk in place."""
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
            and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last)
            and x.shape[1] % 4 == 0 and x.shape[1] <= 1024 and x.data_ptr() % 16 == 0)


def _ci_qparams(spec: QSpec, scale, zero_point, C: int, device, keep: list):
    qpc = C if spec.ch_axis == 1 else 1
    if spec.ch_axis not in (None, 1):
        raise ValueError("channel-innermost activations are quantised per tensor or along dim 1")
    return _make_qparams(spec, scale, zero_point, qpc, device, keep), qpc


def ci_forward(x: torch.Tensor, bias: Optional[torch.Tensor], scale, zero_point, spec: QSpec,
               out: Optional[torch.Tensor] = None, second: Optional[tuple] = None):
    """y = fq(act(x + bias[c])) on a channels_last tensor, in place of layout conversions (vsiq_ci_fake_quant_fwd).

    second = (scale2, zero_point2, spec2): also y2 = fq2(y), the next layer's ``quantize_inp`` result
    (fake_quantize.py:44-45), written by the same pass (vsiq_ci_fake_quant_fwd2); returns (y, y2)."""
    if not ci_supported(x):
        raise ValueError("ci_forward needs a float32 CUDA channels_last tensor with C % 4 == 0 and C <= 1024")
    N, C, H, W = x.shape
    rows = N * H * W
    keep: list = []
    with torch.cuda.device(x.device):
        qp, qpc = _ci_qparams(spec, scale, zero_point, C, x.device, keep)
        b = None
        if bias is not None:
            b = bias.detach().to(device=x.device, dtype=torch.float32).contiguous()
            if b.numel() != C:
                raise ValueError("bias must have one entry per channel")
        y = _out_like(x, out, "out")
        ws = _workspace(lib.vsiq_ci_workspace_bytes(rows, C), x.device)
        if second is not None:
            s2, z2, spec2 = second
            if spec.fp8_format or spec2.fp8_format:
                raise ValueError("the two-output epilogue has integer grids only")
            if spec2.pre_relu or spec2.pre_silu:
                raise ValueError("the second quantiser of a two-output pass has no activation of its own")
            qp2, qpc2 = _ci_qparams(spec2, s2, z2, C, x.device, keep)
            y2 = torch.empty_like(x)
            check(lib.vsiq_ci_fake_quant_fwd2(x.data_ptr(), b.data_ptr() if b is not None else None, y.data_ptr(),
                                              y2.data_ptr(), rows, C, ctypes.byref(qp), qpc, ctypes.byref(qp2), qpc2,
                                              ws.data_ptr(), ws.numel(), _stream_ptr()), "vsiq_ci_fake_quant_fwd2")
            _count_launch()
            return y, y2
        if spec.fp8_format:
            check(lib.vsiq_ci_fp8_fake_quant_fwd(x.data_ptr(), b.data_ptr() if b is not None else None, y.data_ptr(), rows,
                                                 C, ctypes.byref(qp), qpc, int(spec.fp8_format), ws.data_ptr(), ws.numel(),
                                                 _stream_ptr()), "vsiq_ci_fp8_fake_quant_fwd")
        else:
            check(lib.vsiq_ci_fake_quant_fwd(x.data_ptr(), b.data_ptr() if b is not None else None, y.data_ptr(), rows,
                                             C, ctypes.byref(qp), qpc, ws.data_ptr(), ws.numel(), _stream_ptr()),
                  "vsiq_ci_fake_quant_fwd")
        _count_launch()
    return y


def ci_backward(x: torch.Tensor, bias: Optional[torch.Tensor], g: torch.Tensor, scale, zero_point, spec: QSpec,
                grad_scale: float = 1.0, grad_scale_dev: Optional[torch.Tensor] = None, want_ds: bool = True,
                want_dz: bool = False, want_dbias: bool = True, ds_dtype=torch.float32, dz_dtype=torch.float32):
    """dx, dscale, dzero_point, dbias of ci_forward in one pass (vsiq_ci_lsq_bwd); dscale None = plain STE."""
    if not ci_supported(x):
        raise ValueError("ci_backward needs a float32 CUDA channels_last tensor with C % 4 == 0 and C <= 1024")
    N, C, H, W = x.shape
    rows = N * H * W
    # grad_output as a channel slice of a wider NHWC tensor (torch.cat's backward): read it in place through a row pitch
    pitch = 0
    if (g.is_cuda and g.dtype == torch.float32 and g.shape == x.shape and g.stride() != x.stride() and g.stride(1) == 1
            and g.stride(3) % 4 == 0 and g.stride(3) >= C and g.stride(2) == W * g.stride(3)
            and g.stride(0) == H * W * g.stride(3) and g.data_ptr() % 16 == 0):
        pitch = g.stride(3)
    else:
        g = _match_layout(g, x, "grad_output")
    keep: list = []
    with torch.cuda.device(x.device):
        qp, qpc = _ci_qparams(spec, scale, zero_point, C, x.device, keep)
        b = None
        if bias is not None:
            b = bias.detach().to(device=x.device, dtype=torch.float32).contiguous()
        dx = torch.empty_like(x)
        ds = torch.empty(qpc, dtype=ds_dtype, device=x.device) if want_ds else None
        dz = torch.empty(qpc, dtype=dz_dtype, device=x.device) if (want_ds and want_dz) else None
        db = torch.empty(C, dtype=torch.float32, device=x.device) if (b is not None and want_dbias) else None
        gsd = None
        if grad_scale_dev is not None:
            gsd = grad_scale_dev.detach().to(device=x.device, dtype=torch.float32).contiguous()
            keep.append(gsd)
        ws = _workspace(lib.vsiq_ci_workspace_bytes(rows, C), x.device)
        bwd_args = (x.data_ptr(), b.data_ptr() if b is not None else None, g.data_ptr(), dx.data_ptr(),
                    ds.data_ptr() if ds is not None else None, _dtype_code(ds) if ds is not None else F32,
                    dz.data_ptr() if dz is not None else None, _dtype_code(dz) if dz is not None else F32,
                    db.data_ptr() if db is not None else None, rows, C, ctypes.byref(qp), qpc)
        tail = (float(grad_scale), gsd.data_ptr() if gsd is not None else None, pitch, ws.data_ptr(), ws.numel(),
                _stream_ptr())
        if spec.fp8_format:
            check(lib.vsiq_ci_fp8_lsq_bwd(*bwd_args, int(spec.fp8_format), *tail), "vsiq_ci_fp8_lsq_bwd")
        else:
            check(lib.vsiq_ci_lsq_bwd(*bwd_args, *tail), "vsiq_ci_lsq_bwd")
        _count_launch()
    return dx, ds, dz, db


def new_observer_state(channels: int = 1, device=None) -> torch.Tensor:
    """[channels, 8] fp64: run_min, run_max, scale, zero_point, n_calls, sum mean|x|, sum mean x, sum std.
    Running extrema start at 0 like the reference's observer (observers/minmax.py:28-29); scale starts at the
    manager's default 1 (quantization_manager.py:45)."""
    st = torch.zeros(channels, _lib.STATE_WIDTH, dtype=torch.float64, device=device)
    st[:, 2] = 1.0
    return st


def observe(x: torch.Tensor, ch_axis: Optional[int] = None, state: Optional[torch.Tensor] = None, bits: int = 8,
            symmetric: bool = True, eps: float = 1e-8, want_stats: bool = True) -> Optional[torch.Tensor]:
    """One pass: per-channel {min, max, sum|x|, sum x, sum x^2} (+ running observer state, scale, zero-point).

    Replaces observers/minmax.py:42-47,67-74 and quantization_manager.py:66-68.  No host sync."""
    if ch_axis == 1 and ci_supported(x):
        return _ci_observe(x, state, bits, symmetric, eps, want_stats)  # per-channel statistics on NHWC memory in place
    x = _dense_for(x, "x", ch_axis)
    outer, C, inner = layout_of(x.shape, ch_axis)
    lay = Layout(outer, C, inner)
    with torch.cuda.device(x.device):
        stats = torch.empty(C, _lib.STATS_WIDTH, dtype=torch.float64, device=x.device) if want_stats else None
        if state is not None:
            if state.dtype != torch.float64 or not state.is_cuda or state.numel() != C * _lib.STATE_WIDTH \
                    or not state.is_contiguous():
                raise ValueError("observer state must be a contiguous CUDA float64 tensor [channels, 8]")
        ws = _workspace(lib.vsiq_observe_workspace_bytes(ctypes.byref(lay)), x.device)
        check(lib.vsiq_observe(x.data_ptr(), ctypes.byref(lay), stats.data_ptr() if want_stats else None,
                               state.data_ptr() if state is not None else None, int(bits), int(bool(symmetric)),
                               float(eps), ws.data_ptr(), ws.numel(), _stream_ptr()), "vsiq_observe")
        _count_launch()
    return stats


def _ci_observe(x, state, bits, symmetric, eps, want_stats):
    N, C, H, W = x.shape
    rows = N * H * W
    with torch.cuda.device(x.device):
        stats = torch.empty(C, _lib.STATS_WIDTH, dtype=torch.float64, device=x.device) if want_stats else None
        if state is not None:
            if state.dtype != torch.float64 or not state.is_cuda or state.numel() != C * _lib.STATE_WIDTH \
                    or not state.is_contiguous():
                raise ValueError("observer state must be a contiguous CUDA float64 tensor [channels, 8]")
        ws = _workspace(lib.vsiq_ci_observe_workspace_bytes(rows, C), x.device)
        check(lib.vsiq_ci_observe(x.data_ptr(), rows, C, stats.data_ptr() if want_stats else None,
                                  state.data_ptr() if state is not None else None, int(bits), int(bool(symmetric)),
                                  float(eps), ws.data_ptr(), ws.numel(), _stream_ptr()), "vsiq_ci_observe")
        _count_launch(2)
    return stats


def ci_epilogue_observe(x: torch.Tensor, state: torch.Tensor, bits: int = 8, symmetric: bool = True, eps: float = 1e-8,
                        act: Optional[str] = None, bias: Optional[torch.Tensor] = None, bn: Optional[tuple] = None,
                        want_stats: bool = True):
    """(y, stats): y = act(x + bias[c]) or act(BatchNorm_eval(x)) or act(x) on a channels_last conv output, written and
    observed PER TENSOR in the same pass (vsiq_ci_epilogue_observe): the calibration forward of a fused layer
    (modules/fused.py:124-134 then quantization_manager.py:55-71) at 8 bytes per element.
    bn = (running_mean, running_var, weight, bias, eps); act = None / "relu" / "silu"."""
    if not ci_supported(x):
        raise ValueError("ci_epilogue_observe needs a float32 CUDA channels_last tensor with C % 4 == 0 and C <= 1024")
    if bias is not None and bn is not None:
        raise ValueError("one pre-op: a bias add or a BatchNorm, not both")
    N, C, H, W = x.shape
    rows = N * H * W
    code = {None: _lib.PRE_NONE, "relu": _lib.PRE_RELU, "silu": _lib.PRE_SILU}[act]
    f32 = lambda t: None if t is None else t.detach().to(device=x.device, dtype=torch.float32).contiguous()  # noqa: E731
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    with torch.cuda.device(x.device):
        if state.dtype != torch.float64 or not state.is_cuda or state.numel() != _lib.STATE_WIDTH or not state.is_contiguous():
            raise ValueError("a per-tensor observer state is a contiguous CUDA float64 tensor [1, 8]")
        stats = torch.empty(1, _lib.STATS_WIDTH, dtype=torch.float64, device=x.device) if want_stats else None
        b = f32(bias)
        mean = var = gamma = beta = None
        bn_eps = 0.0
        if bn is not None:
            mean, var, gamma, beta = (f32(t) for t in bn[:4])
            bn_eps = float(bn[4])
            if mean is None or var is None:
                raise ValueError("BatchNorm pre-op needs running_mean and running_var")
        for t in (b, mean, var, gamma, beta):
            if t is not None and t.numel() != C:
                raise ValueError("per-channel operands need one entry per channel")
        y = torch.empty_like(x)
        ws = _workspace(lib.vsiq_ci_observe_workspace_bytes(rows, C), x.device)
        check(lib.vsiq_ci_epilogue_observe(x.data_ptr(), ptr(b), ptr(mean), ptr(var), ptr(gamma), ptr(beta), bn_eps, code,
                                           y.data_ptr(), rows, C, ptr(stats), state.data_ptr(), int(bits),
                                           int(bool(symmetric)), float(eps), ws.data_ptr(), ws.numel(), _stream_ptr()),
              "vsiq_ci_epilogue_observe")
        _count_launch()
    return y, stats


def _check_state(state: torch.Tensor, C: int, width: int, what: str, device) -> None:
    if state.dtype != torch.float64 or not state.is_cuda or tuple(state.shape) != (C, width) \
            or not state.is_contiguous() or state.device != device:
        raise ValueError(f"{what} state must be a contiguous float64 tensor [{C}, {width}] on {device}")


def _observe_first(x: torch.Tensor, ch_axis: Optional[int], state: torch.Tensor, width: int, what: str, bits: int,
                   symmetric: bool, eps: float):
    """The head of an observer call that reads x again after the min/max pass (mse_search, hist_observe): channels_last
    activations quantised along dim 1 are read in place, anything else as _dense_for leaves it; the [C, width] state is
    checked; then the min/max pass gives this call's statistics.  Returns (x as read, Layout, stats [C, 5])."""
    ci = ch_axis == 1 and ci_supported(x)
    if ci:
        N, C, H, W = x.shape
        outer, inner = N * H * W, 1
    else:
        x = _dense_for(x, "x", ch_axis)
        outer, C, inner = layout_of(x.shape, ch_axis)
    _check_state(state, C, width, what, x.device)
    stats = _ci_observe(x, None, bits, symmetric, eps, True) if ci else observe(x, ch_axis, None, bits, symmetric, eps)
    return x, Layout(outer, C, inner), stats


def new_mse_state(channels: int = 1, device=None) -> torch.Tensor:
    """[channels, 10] fp64 MSE observer state: new_observer_state's eight columns, then the running means of the chosen
    clipped min / max."""
    st = torch.zeros(channels, _lib.MSE_STATE_WIDTH, dtype=torch.float64, device=device)
    st[:, 2] = 1.0
    return st


def mse_search(x: torch.Tensor, ch_axis: Optional[int], state: torch.Tensor, bits: int, symmetric: bool = True,
               eps: float = 1e-8, n_candidates: int = 100, want_err: bool = False):
    """One calibration call of the MSE observer (vsiq_mse_search): the min/max pass for this call's statistics, then the
    search over n_candidates clipped ranges and the state update, all on the device (no host sync).  channels_last
    activations quantised along dim 1 are searched in place (no layout conversion).
    Returns (stats [C, 5], err [C, K] or None, alpha [C] or None)."""
    K = int(n_candidates)
    if not 1 <= K <= 256:
        raise ValueError("n_candidates must be in 1..256")
    x, lay, stats = _observe_first(x, ch_axis, state, _lib.MSE_STATE_WIDTH, "MSE observer", bits, symmetric, eps)
    C = lay.channels
    with torch.cuda.device(x.device):
        err = torch.empty(C, K, dtype=torch.float64, device=x.device) if want_err else None
        alpha = torch.empty(C, dtype=torch.float64, device=x.device) if want_err else None
        ws = _workspace(lib.vsiq_mse_search_workspace_bytes(ctypes.byref(lay), K), x.device)
        check(lib.vsiq_mse_search(x.data_ptr(), ctypes.byref(lay), stats.data_ptr(), state.data_ptr(), int(bits),
                                  int(bool(symmetric)), float(eps), K, err.data_ptr() if want_err else None,
                                  alpha.data_ptr() if want_err else None, ws.data_ptr(), ws.numel(), _stream_ptr()),
              "vsiq_mse_search")
        _count_launch(2)
    return stats, err, alpha


def _check_hist_args(n_bins: int, percentile: float) -> None:
    n_bins = int(n_bins)
    if not (256 <= n_bins <= 4096 and n_bins & (n_bins - 1) == 0):
        raise ValueError("n_bins must be a power of two in 256..4096")
    if not 0.0 < float(percentile) <= 100.0:
        raise ValueError("percentile must be in (0, 100]")


def new_percentile_state(channels: int, n_bins: int = 2048, device=None) -> torch.Tensor:
    """[channels, 12 + 2 * n_bins] fp64 percentile observer state: new_observer_state's eight columns, the clipped lo / hi,
    the bin exponents e_neg / e_pos (-149: the finest width, 2^-149), then n_bins counts of x < 0 and n_bins of x >= 0."""
    _check_hist_args(n_bins, 100.0)
    st = torch.zeros(channels, _lib.HIST_STATE_HEAD + 2 * int(n_bins), dtype=torch.float64, device=device)
    st[:, 2] = 1.0
    st[:, 10:12] = -149.0
    return st


def hist_observe(x: torch.Tensor, ch_axis: Optional[int], state: torch.Tensor, n_bins: int = 2048,
                 percentile: float = 99.99, bits: int = 8, symmetric: bool = True, eps: float = 1e-8) -> torch.Tensor:
    """One calibration call of the percentile observer (vsiq_hist_observe): the min/max pass for this call's statistics,
    then one histogram pass over x and the state update with the clip at `percentile`, all on the device (no host sync).
    channels_last activations quantised along dim 1 are read in place (no layout conversion).  Returns stats [C, 5]."""
    _check_hist_args(n_bins, percentile)
    x, lay, stats = _observe_first(x, ch_axis, state, _lib.HIST_STATE_HEAD + 2 * int(n_bins), "percentile observer",
                                   bits, symmetric, eps)
    with torch.cuda.device(x.device):
        ws = _workspace(lib.vsiq_hist_observe_workspace_bytes(ctypes.byref(lay), int(n_bins)), x.device)
        check(lib.vsiq_hist_observe(x.data_ptr(), ctypes.byref(lay), stats.data_ptr(), state.data_ptr(), int(n_bins),
                                    float(percentile), int(bits), int(bool(symmetric)), float(eps), ws.data_ptr(),
                                    ws.numel(), _stream_ptr()), "vsiq_hist_observe")
        _count_launch(2)
    return stats


def hist_clip(state: torch.Tensor, n_bins: int, percentile: float, bits: int, symmetric: bool = True,
              eps: float = 1e-8) -> None:
    """Recompute the clip (columns 8, 9) and scale / zero-point (2, 3) of a percentile observer state in place from its
    stored counts at `percentile` (vsiq_hist_clip): no new data, no host sync."""
    _check_hist_args(n_bins, percentile)
    if state.dim() != 2:
        raise ValueError("percentile observer state must be [channels, 12 + 2 * n_bins]")
    _check_state(state, state.shape[0], _lib.HIST_STATE_HEAD + 2 * int(n_bins), "percentile observer", state.device)
    with torch.cuda.device(state.device):
        check(lib.vsiq_hist_clip(state.data_ptr(), state.shape[0], int(n_bins), float(percentile), int(bits),
                                 int(bool(symmetric)), float(eps), _stream_ptr()), "vsiq_hist_clip")
        _count_launch()


def _check_entropy_args(n_bins: int, start_bin: int, bits: int) -> None:
    _check_hist_args(n_bins, 100.0)
    if not 1 <= int(start_bin) <= int(n_bins):
        raise ValueError("start_bin must be in 1..n_bins")
    if not 2 <= int(bits) <= 8:
        raise ValueError("bits must be in 2..8")


def hist_entropy_clip(state: torch.Tensor, n_bins: int, start_bin: int, bits: int, symmetric: bool = True,
                      eps: float = 1e-8, divergences: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
    """Recompute the clip (columns 8, 9) and scale / zero-point (2, 3) of a percentile / entropy observer state in place
    by the KL-divergence search over its stored counts (vsiq_hist_entropy_clip): no new data, no host sync.
    divergences: an optional [C, n_bins + 1] float64 tensor on the state's device that receives D_i of every candidate
    threshold i (NaN where i is no candidate); returned."""
    _check_entropy_args(n_bins, start_bin, bits)
    if state.dim() != 2:
        raise ValueError("entropy observer state must be [channels, 12 + 2 * n_bins]")
    C = state.shape[0]
    _check_state(state, C, _lib.HIST_STATE_HEAD + 2 * int(n_bins), "entropy observer", state.device)
    if divergences is not None:
        if divergences.dtype != torch.float64 or tuple(divergences.shape) != (C, int(n_bins) + 1) \
                or not divergences.is_contiguous() or divergences.device != state.device:
            raise ValueError(f"divergences must be a contiguous float64 tensor [{C}, {int(n_bins) + 1}] on {state.device}")
    with torch.cuda.device(state.device):
        ws = _workspace(lib.vsiq_hist_entropy_workspace_bytes(C, int(n_bins)), state.device)
        check(lib.vsiq_hist_entropy_clip(state.data_ptr(), C, int(n_bins), int(start_bin), int(bits),
                                         int(bool(symmetric)), float(eps),
                                         divergences.data_ptr() if divergences is not None else None, ws.data_ptr(),
                                         ws.numel(), _stream_ptr()), "vsiq_hist_entropy_clip")
        _count_launch(2)
    return divergences


def qparams_from_minmax(states: torch.Tensor, bits: torch.Tensor, symmetric: torch.Tensor, eps: float = 1e-8) -> None:
    """Recompute scale / zero-point of n observers in place from their running extrema [minmax.py:67-74]."""
    n = states.numel() // _lib.STATE_WIDTH
    if states.dtype != torch.float64 or not states.is_cuda or not states.is_contiguous():
        raise ValueError("states must be a contiguous CUDA float64 tensor [n, 8]")
    bits = bits.to(device=states.device, dtype=torch.int32).contiguous()
    symmetric = symmetric.to(device=states.device, dtype=torch.int32).contiguous()
    if bits.numel() != n or symmetric.numel() != n:
        raise ValueError("bits / symmetric need one entry per observer")
    with torch.cuda.device(states.device):
        check(lib.vsiq_qparams_from_minmax(states.data_ptr(), n, bits.data_ptr(), symmetric.data_ptr(), float(eps),
                                           _stream_ptr()), "vsiq_qparams_from_minmax")
        _count_launch()


def fp8_scale_from_range(lo: torch.Tensor, hi: torch.Tensor, fp8_format: int, out: torch.Tensor) -> torch.Tensor:
    """out[c] = max(|lo[c]|, |hi[c]|) / F, or 1.0 where that is zero or not finite (vsiq_fp8_scale_from_range), written
    IN PLACE: lo / hi are equally strided fp64 device views (an observer's device_range()), out a contiguous fp64 [C]."""
    C = lo.numel()
    if lo.dtype != torch.float64 or hi.dtype != torch.float64 or lo.dim() != 1 or hi.shape != lo.shape \
            or lo.stride() != hi.stride() or not lo.is_cuda or hi.device != lo.device:
        raise ValueError("lo / hi must be equally strided 1-D float64 CUDA views")
    if out.dtype != torch.float64 or out.numel() != C or not out.is_contiguous() or out.device != lo.device:
        raise ValueError(f"out must be a contiguous float64 tensor with {C} entries on {lo.device}")
    with torch.cuda.device(lo.device):
        check(lib.vsiq_fp8_scale_from_range(lo.data_ptr(), hi.data_ptr(), max(lo.stride(0), 1), C, int(fp8_format),
                                            out.data_ptr(), _stream_ptr()), "vsiq_fp8_scale_from_range")
        _count_launch()
    return out


def lsq_init_scale(state: torch.Tensor, bits: int, out: torch.Tensor) -> torch.Tensor:
    """2 * mean(mean|x|) / sqrt(2^(bits-1) - 1) per channel, written into `out` [quantization_manager.py:112]."""
    C = state.numel() // _lib.STATE_WIDTH
    if out.numel() != C or not out.is_cuda:
        raise ValueError("out must be a CUDA tensor with one entry per channel")
    with torch.cuda.device(state.device):
        check(lib.vsiq_lsq_init_scale(state.data_ptr(), C, int(bits), out.data_ptr(), _dtype_code(out), _stream_ptr()),
              "vsiq_lsq_init_scale")
        _count_launch()
    return out


def bn_fold(W, bias, gamma, beta, mean, var, eps: float, scale=None, zero_point=0, spec: Optional[QSpec] = None,
            want_stats: bool = False):
    """W' = W * gamma/sqrt(var+eps), b' = beta + (b - mean) * gamma/sqrt(var+eps)  [modules/fused.py:98-108,292-300].

    With `spec` also returns the fake-quantised W' from the same pass; with want_stats the per-tensor
    {min,max,sum|x|,sum x,sum x^2} of W'.  Returns (W', b', Wq or None, stats or None)."""
    W = _dense_for(W, "weight", 0)
    C = W.shape[0]
    inner = W.numel() // C
    dev = W.device
    vecs = [_require_cuda_f32(t.detach(), n) for t, n in ((gamma, "gamma"), (beta, "beta"), (mean, "mean"), (var, "var"))]
    for v in vecs:
        if v.numel() != C:
            raise ValueError("BN vectors must have one entry per output channel")
    b = _require_cuda_f32(bias.detach(), "bias") if bias is not None else None
    keep: list = []
    with torch.cuda.device(dev):
        Wf = torch.empty_like(W)
        bf = torch.empty(C, dtype=torch.float32, device=dev)
        Wq = None
        qp = None
        qpc = 1
        if spec is not None:
            if spec.ch_axis not in (None, 0):
                raise ValueError("weight fake-quant in the fold supports per-tensor or ch_axis 0")
            qpc = C if spec.ch_axis == 0 else 1
            qp = _make_qparams(spec, scale, zero_point, qpc, dev, keep)
            Wq = torch.empty_like(W)
        stats = torch.empty(1, _lib.STATS_WIDTH, dtype=torch.float64, device=dev) if want_stats else None
        ws = _workspace(lib.vsiq_bn_fold_workspace_bytes(C, inner), dev) if want_stats else None
        check(lib.vsiq_bn_fold(W.data_ptr(), b.data_ptr() if b is not None else None, vecs[0].data_ptr(),
                               vecs[1].data_ptr(), vecs[2].data_ptr(), vecs[3].data_ptr(), float(eps), C, inner,
                               Wf.data_ptr(), bf.data_ptr(), Wq.data_ptr() if Wq is not None else None,
                               ctypes.byref(qp) if qp is not None else None, qpc,
                               stats.data_ptr() if want_stats else None, ws.data_ptr() if ws is not None else None,
                               ws.numel() if ws is not None else 0, _stream_ptr()), "vsiq_bn_fold")
        _count_launch()
    return Wf, bf, Wq, stats


def bn_batch_moments(x: torch.Tensor, mean_sum: Optional[torch.Tensor] = None, var_sum: Optional[torch.Tensor] = None):
    """Per-channel batch mean, biased and unbiased variance of an [N,C,...] tensor in one pass, optionally
    accumulating mean / unbiased var into running sums (utils/estimate_bn.py:82,86-87).

    For SyncBN-style multi-GPU re-estimation call observe(x, ch_axis=1), all-reduce(SUM) the stats and pass the
    global per-channel count to bn_moments_finalize() instead."""
    x = _require_cuda_f32(x, "x")
    C = x.shape[1]
    stats = observe(x, ch_axis=1)
    return bn_moments_finalize(stats, float(x.numel() // C), mean_sum, var_sum)


def bn_moments_finalize(stats: torch.Tensor, count: float, mean_sum=None, var_sum=None):
    C = stats.shape[0]
    dev = stats.device
    with torch.cuda.device(dev):
        m = torch.empty(C, dtype=torch.float32, device=dev)
        vb = torch.empty(C, dtype=torch.float32, device=dev)
        vu = torch.empty(C, dtype=torch.float32, device=dev)
        check(lib.vsiq_bn_moments_finalize(stats.data_ptr(), float(count), C, m.data_ptr(), vb.data_ptr(), vu.data_ptr(),
                                           mean_sum.data_ptr() if mean_sum is not None else None,
                                           var_sum.data_ptr() if var_sum is not None else None, _stream_ptr()),
              "vsiq_bn_moments_finalize")
        _count_launch()
    return m, vb, vu


def ci_bn_normalize(x: torch.Tensor, mean, var, gamma, beta, eps: float, relu: bool = False) -> torch.Tensor:
    """act((x - mean) / sqrt(var + eps) * gamma + beta) on a channels_last tensor in one pass (vsiq_ci_bn_normalize):
    training-mode BatchNorm's normalisation with known batch moments, ReLU folded in (estimate_bn.py:79-91, fused.py:131-134)."""
    if not ci_supported(x):
        raise ValueError("ci_bn_normalize needs a float32 CUDA channels_last tensor with C % 4 == 0 and C <= 1024")
    N, C, H, W = x.shape
    f = lambda t: None if t is None else t.detach().to(device=x.device, dtype=torch.float32).contiguous()  # noqa: E731
    mean, var, gamma, beta = f(mean), f(var), f(gamma), f(beta)
    with torch.cuda.device(x.device):
        y = torch.empty_like(x)
        ws = _workspace(256, x.device)
        check(lib.vsiq_ci_bn_normalize(x.data_ptr(), mean.data_ptr(), var.data_ptr(),
                                       gamma.data_ptr() if gamma is not None else None,
                                       beta.data_ptr() if beta is not None else None, float(eps), y.data_ptr(),
                                       N * H * W, C, int(bool(relu)), ws.data_ptr(), ws.numel(), _stream_ptr()),
              "vsiq_ci_bn_normalize")
        _count_launch()
    return y


def bn_reestimate_finish(mean_sum, var_sum, batch_count: int, running_mean, running_var) -> None:
    """running = sum / batch_count  [utils/estimate_bn.py:96-97]."""
    C = mean_sum.numel()
    with torch.cuda.device(mean_sum.device):
        check(lib.vsiq_bn_reestimate_finish(mean_sum.data_ptr(), var_sum.data_ptr(), int(batch_count),
                                            running_mean.data_ptr(), running_var.data_ptr(), C, _stream_ptr()),
              "vsiq_bn_reestimate_finish")
        _count_launch()


def selftest_division(scale: float, mode: int = 0, device=None) -> int:
    """Mismatches between the kernels' fast arithmetic and the IEEE sequences over all 2^32 inputs (expect 0).
    mode 0: x / s;  mode 1: RN(RN(g*s) / s)."""
    dev = torch.device(device or "cuda")
    with torch.cuda.device(dev):
        out = torch.zeros(1, dtype=torch.int64, device=dev)
        check(lib.vsiq_selftest_division(float(scale), int(mode), out.data_ptr(), _stream_ptr()),
              "vsiq_selftest_division")
        _count_launch()
        return int(out.item())


class HostPipeline:
    """Forward + STE backward over HOST (ideally pinned) buffers, chunked; H2D, kernel and D2H overlap on three
    event-linked streams through ``n_slots`` sets of staging buffers (csrc/host_pipeline.cu)."""

    def __init__(self, chunk_elems: int = 1 << 23, n_slots: int = 4, device=None):
        self._h = ctypes.c_void_p()
        self.device = torch.device(device or "cuda")
        with torch.cuda.device(self.device):
            check(lib.vsiq_host_pipeline_create(ctypes.byref(self._h), int(chunk_elems), int(n_slots)),
                  "vsiq_host_pipeline_create")

    def fwd_bwd(self, x: torch.Tensor, g: torch.Tensor, scale: float, zero_point: float, qmin: int, qmax: int,
                y: Optional[torch.Tensor] = None, dx: Optional[torch.Tensor] = None):
        for t, n in ((x, "x"), (g, "g")):
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"{n} must be a contiguous float32 HOST tensor")
        y = torch.empty_like(x, pin_memory=True) if y is None else y
        dx = torch.empty_like(x, pin_memory=True) if dx is None else dx
        with torch.cuda.device(self.device):
            check(lib.vsiq_host_pipeline_fwd_bwd(self._h, x.data_ptr(), g.data_ptr(), y.data_ptr(), dx.data_ptr(),
                                                 x.numel(), float(scale), float(zero_point), int(qmin), int(qmax)),
                  "vsiq_host_pipeline_fwd_bwd")
        _count_launch(int(lib.vsiq_host_pipeline_last_launches(self._h)))
        return y, dx

    @property
    def last_submit_ms(self) -> float:
        """Host time the last fwd_bwd call spent submitting copies and launches (before waiting for them)."""
        return lib.vsiq_host_pipeline_last_enqueue_ns(self._h) / 1e6

    def close(self):
        if self._h:
            lib.vsiq_host_pipeline_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ----------------------------------------------------------------------------------------------
# autograd
# ----------------------------------------------------------------------------------------------
class Precomputed:
    """Holder for a forward result some other kernel already produced (the two-output epilogue): handed to
    FakeQuantFixed / FakeQuantLearned in place of a launch.  Not a tensor argument, so autograd sees a fresh output."""
    __slots__ = ("tensor",)

    def __init__(self, tensor: torch.Tensor):
        self.tensor = tensor

    def take(self, x: torch.Tensor) -> torch.Tensor:
        t, self.tensor = self.tensor, None
        if t is None or t.shape != x.shape or t.dtype != x.dtype or t.device != x.device:
            raise ValueError("precomputed fake-quant result does not match the tensor it stands for")
        return t


class FakeQuantFixed(torch.autograd.Function):
    """Fake-quant with constant qparams; STE backward.  (uniform.py:54-55 with is_learning_scale=False)"""

    @staticmethod
    def forward(ctx, x, scale, zero_point, spec: QSpec, pre: Optional[Precomputed] = None):
        ctx.spec, ctx.scale, ctx.zero_point = spec, scale, zero_point
        ctx.save_for_backward(x)
        return pre.take(x) if pre is not None else fake_quant_forward(x, scale, zero_point, spec)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        dx = fake_quant_backward_ste(x, g, ctx.scale, ctx.zero_point, ctx.spec) if ctx.needs_input_grad[0] else None
        return dx, None, None, None, None


class FakeQuantLearned(torch.autograd.Function):
    """Fake-quant with learnable step size (and optionally zero-point); LSQ backward in one pass.

    scale: tensor with `channels` entries of any shape (0-dim fp64 Parameter in the reference's per-tensor
    path, [1,C,1,1] fp32 in lsq_module.py); zero_point: same-shaped float tensor, or a Python number."""

    @staticmethod
    def forward(ctx, x, scale, zero_point, spec: QSpec, grad_scale: float, grad_scale_dev,
                pre: Optional[Precomputed] = None):
        ctx.spec, ctx.grad_scale, ctx.grad_scale_dev = spec, grad_scale, grad_scale_dev
        ctx.zp_is_tensor = isinstance(zero_point, torch.Tensor)
        ctx.zp_const = None if ctx.zp_is_tensor else zero_point
        if ctx.zp_is_tensor:
            ctx.save_for_backward(x, scale, zero_point)
        else:
            ctx.save_for_backward(x, scale)
        return pre.take(x) if pre is not None else fake_quant_forward(x, scale, zero_point, spec)

    @staticmethod
    def backward(ctx, g):
        if ctx.zp_is_tensor:
            x, scale, zp = ctx.saved_tensors
        else:
            x, scale = ctx.saved_tensors
            zp = ctx.zp_const
        want_dz = ctx.zp_is_tensor and ctx.needs_input_grad[2]
        dx, ds, dz = lsq_backward(x, g, scale, zp, ctx.spec, ctx.grad_scale, ctx.grad_scale_dev, want_dz=want_dz,
                                  ds_dtype=scale.dtype, dz_dtype=zp.dtype if ctx.zp_is_tensor else torch.float32)
        ds = ds.view(scale.shape).to(scale.device) if ctx.needs_input_grad[1] else None
        dz = dz.view(zp.shape).to(zp.device) if want_dz else None
        return (dx if ctx.needs_input_grad[0] else None), ds, dz, None, None, None, None


class FakeQuantEpilogue(torch.autograd.Function):
    """y = fq(act(x + bias[c])) on a channels_last conv output: the fused layer's bias add, activation and output
    quantiser as one forward pass, and dx, dbias (the conv's bias gradient), dscale, dzero_point as one backward pass."""

    @staticmethod
    def forward(ctx, x, bias, scale, zero_point, spec: QSpec, grad_scale: float, grad_scale_dev, second=None):
        """second = (scale2, zero_point2, spec2, sink): the pass also writes y2 = fq2(y) -- the next layer's
        quantize_inp result -- and appends it to the list ``sink`` (a plain buffer; its autograd node is the second
        quantiser's own Function, fed through ops.Precomputed)."""
        ctx.spec, ctx.grad_scale, ctx.grad_scale_dev = spec, grad_scale, grad_scale_dev
        ctx.scale_is_tensor = isinstance(scale, torch.Tensor)
        ctx.zp_is_tensor = isinstance(zero_point, torch.Tensor)
        ctx.scale_const = None if ctx.scale_is_tensor else scale
        ctx.zp_const = None if ctx.zp_is_tensor else zero_point
        ctx.has_bias = bias is not None
        saved = [x] + ([bias] if ctx.has_bias else []) + ([scale] if ctx.scale_is_tensor else []) + \
            ([zero_point] if ctx.zp_is_tensor else [])
        ctx.save_for_backward(*saved)
        if second is not None:
            s2, z2, spec2, sink = second
            y, y2 = ci_forward(x, bias, scale, zero_point, spec, second=(s2, z2, spec2))
            sink.append(y2)
            return y
        return ci_forward(x, bias, scale, zero_point, spec)

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        x = saved[0]
        bias = saved[1] if ctx.has_bias else None
        k = 2 if ctx.has_bias else 1
        scale = saved[k] if ctx.scale_is_tensor else ctx.scale_const
        k += 1 if ctx.scale_is_tensor else 0
        zp = saved[k] if ctx.zp_is_tensor else ctx.zp_const
        want_ds = ctx.scale_is_tensor and ctx.needs_input_grad[2]
        want_dz = want_ds and ctx.zp_is_tensor and ctx.needs_input_grad[3]
        dx, ds, dz, db = ci_backward(x, bias, g, scale, zp, ctx.spec, ctx.grad_scale, ctx.grad_scale_dev, want_ds, want_dz,
                                     ctx.has_bias and ctx.needs_input_grad[1], scale.dtype if ctx.scale_is_tensor else torch.float32,
                                     zp.dtype if ctx.zp_is_tensor else torch.float32)
        ds = ds.view(scale.shape).to(scale.device) if want_ds else None
        dz = dz.view(zp.shape).to(zp.device) if want_dz else None
        db = db.view(bias.shape) if db is not None else None
        return (dx if ctx.needs_input_grad[0] else None), db, ds, dz, None, None, None, None


class EpilogueObserve(torch.autograd.Function):
    """ci_epilogue_observe with an autograd node, for calibration loops that do not switch autograd off (the reference's
    data_calib, yolov8_qat.py:42-52, runs model(imgs) with grad mode on).  Nobody back-propagates through a calibration
    pass; if someone does, the backward re-runs the ATen composition the kernel stands for (bias add or inference-mode
    batch_norm, then relu / silu) under autograd -- correct, and never on a hot path."""

    @staticmethod
    def forward(ctx, pre, bias, bn_mean, bn_var, bn_weight, bn_bias, bn_eps, act, state, bits, symmetric, eps, sink):
        bn = None if bn_mean is None else (bn_mean, bn_var, bn_weight, bn_bias, bn_eps)
        y, stats = ci_epilogue_observe(pre, state, bits, symmetric, eps, act, bias, bn)
        sink.append(stats)
        ctx.act, ctx.bn_eps, ctx.has_bn = act, bn_eps, bn is not None
        ctx.save_for_backward(pre, bias, bn_mean, bn_var, bn_weight, bn_bias)
        return y

    @staticmethod
    def backward(ctx, g):
        pre, bias, mean, var, w, b = ctx.saved_tensors
        F = torch.nn.functional
        with torch.enable_grad():
            leaves = [t.detach().requires_grad_(True) if (t is not None and need) else t
                      for t, need in zip((pre, bias, w, b), (ctx.needs_input_grad[0], ctx.needs_input_grad[1],
                                                             ctx.needs_input_grad[4], ctx.needs_input_grad[5]))]
            p_, bias_, w_, b_ = leaves
            if ctx.has_bn:
                y = F.batch_norm(p_, mean, var, w_, b_, False, 0.0, ctx.bn_eps)
            else:
                y = p_ if bias_ is None else p_ + bias_.view(1, -1, 1, 1)
            y = F.relu(y) if ctx.act == "relu" else (F.silu(y) if ctx.act == "silu" else y)
            wanted = [t for t in leaves if t is not None and t.requires_grad]
            got = iter(torch.autograd.grad(y, wanted, g, allow_unused=True)) if wanted else iter(())
        out = [next(got) if (t is not None and t.requires_grad) else None for t in leaves]
        return (out[0], out[1], None, None, out[2], out[3]) + (None,) * 7


def lsq_grad_scale(qmax: int, numel: int, channels: int = 1) -> float:
    """(qmax * numel / channels) ** -0.5  [uniform.py:69-71; lsq_module.py:327-340]."""
    return float((qmax * (numel / channels)) ** -0.5) if channels > 1 else float((qmax * numel) ** -0.5)
