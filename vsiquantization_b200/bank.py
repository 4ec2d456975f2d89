"""WeightBank: every weight quantiser of a model in ONE kernel launch each way (SURVEY.md 8(f).1).

The reference fake-quantises each fused layer's weight inside that layer's forward (quantizers/fake_quantize.py:43-51,
62-63 -> quantization_manager.py:73-90 -> uniform.py:34-56): for YOLOv8 that is 57..97 tiny forward launches and as
many backward launches per step, each behind its own autograd node.  The bank runs them as one multi-tensor launch
(csrc/multi_tensor.cu) before the model's forward and hands every layer its fake-quantised weight when the layer asks
for it; the backward is one streaming launch plus one combine launch and produces dW of all layers (views of one flat
buffer) and the LSQ dscale / dzero_point of all layers (views of one flat fp64 / fp32 buffer).  Values are
bit-identical to the per-layer path (same element code); per-layer is still what runs whenever a quantiser is not in
a bankable state (calibrating, quantisation switched off, CPU tensors, exotic strides).

    bank = WeightBank(model).install()      # forward pre-hook on `model`
    ...train as usual...
    bank.remove()

``backward="per_layer"`` keeps the single forward launch but gives every layer its own backward node (one LSQ / STE
launch per layer, as without the bank).  That is the right mode under DistributedDataParallel: a weight's gradient is
then ready as soon as its layer's backward has run, so DDP's bucketed all-reduce still overlaps the rest of the
backward pass; the one-launch backward can only run after the LAST weight gradient exists.
"""
from __future__ import annotations

import ctypes
from typing import List

import torch

from . import _lib, ops
from ._lib import MtEntry, check, lib


def _dense_in_memory(w: torch.Tensor) -> bool:
    if w.is_contiguous():
        return True
    if w.dim() == 4 and w.is_contiguous(memory_format=torch.channels_last):
        return True
    return w.dim() == 5 and w.is_contiguous(memory_format=torch.channels_last_3d)


class _Plan:
    """Device table + bookkeeping for one bankable state of the model (rebuilt when the signature changes)."""

    def __init__(self, items, device):
        self.items = items                      # [(manager, weight, scale, zero_point, spec, learn, gs_host, gs_dev)]
        self.device = device
        n = len(items)
        self.host = (MtEntry * n)()
        self.keep: list = []
        out_off = q_off = 0
        self.out_offsets: List[int] = []
        self.q_offsets: List[int] = []
        for i, (mgr, w, scale, zp, spec, learn, gs_host, gs_dev) in enumerate(items):
            rows = int(w.shape[0])
            inner = w.numel() // rows if rows else 0
            qpc = rows if spec.ch_axis == 0 else 1
            e = self.host[i]
            e.x = w.data_ptr()
            e.rows, e.inner = rows, inner
            e.out_offset, e.qp_offset, e.qp_channels = out_off, q_off, qpc
            e.qp = ops._make_qparams(spec, scale, zp, qpc, device, self.keep)
            e.grad_scale = float(gs_host)
            e.grad_scale_dev = gs_dev.data_ptr() if gs_dev is not None else None
            if gs_dev is not None:
                self.keep.append(gs_dev)
            e.learn = learn
            self.out_offsets.append(out_off)
            self.q_offsets.append(q_off)
            out_off += (w.numel() + 7) // 8 * 8
            q_off += qpc
        self.total_out, self.total_q = out_off, q_off
        tiles = ctypes.c_uint32(0)
        check(lib.vsiq_mt_plan(self.host, n, ctypes.byref(tiles)), "vsiq_mt_plan")
        self.total_tiles = int(tiles.value)
        raw = torch.frombuffer(bytearray(bytes(self.host)), dtype=torch.uint8)
        self.dev = raw.to(device)
        self.learns = any(it[5] for it in items)
        self.ws_bytes = int(lib.vsiq_mt_workspace_bytes(self.total_tiles))
        # what vsiq_mt_* launch: nothing for a table without tiles, one streaming launch per pack of MT_PACK tensors
        # that has tiles, one combine launch when a learning entry has qparam channels
        self.fwd_launches = 1 if self.total_tiles else 0
        packs = sum(1 for lo in range(0, n, _lib.MT_PACK)
                    if any(self.host[i].n_tiles for i in range(lo, min(lo + _lib.MT_PACK, n))))
        self.bwd_launches = packs + (1 if self.learns and self.total_q else 0)

    def view(self, flat: torch.Tensor, i: int) -> torch.Tensor:
        w = self.items[i][1]
        return torch.as_strided(flat, w.shape, w.stride(), self.out_offsets[i])


class _BankFunction(torch.autograd.Function):
    """inputs: plan, n weights, then the qparam tensors that require grad (scales first, then zero-points)."""

    @staticmethod
    def forward(ctx, plan: _Plan, n_w: int, *tensors):
        ctx.plan, ctx.n_w = plan, n_w
        dev = plan.device
        with torch.cuda.device(dev):
            y_flat = torch.empty(plan.total_out, dtype=torch.float32, device=dev)
            check(lib.vsiq_mt_fake_quant_fwd(plan.host, plan.dev.data_ptr(), len(plan.items), y_flat.data_ptr(),
                                             ops._stream_ptr()), "vsiq_mt_fake_quant_fwd")
            ops._count_launch(plan.fwd_launches)
        return tuple(plan.view(y_flat, i) for i in range(len(plan.items)))

    @staticmethod
    def backward(ctx, *grads):
        plan: _Plan = ctx.plan
        n = len(plan.items)
        dev = plan.device
        keep = []
        gptrs = (ctypes.c_void_p * n)()
        for i, g in enumerate(grads):
            w = plan.items[i][1]
            if g is None:
                g = torch.zeros_like(w)
            else:
                g = ops._match_layout(g, w, "grad_output")
            keep.append(g)
            gptrs[i] = g.data_ptr()
        with torch.cuda.device(dev):
            dx_flat = torch.empty(plan.total_out, dtype=torch.float32, device=dev)
            ds_flat = torch.empty(plan.total_q, dtype=torch.float64, device=dev) if plan.learns else None
            dz_flat = torch.empty(plan.total_q, dtype=torch.float32, device=dev) if plan.learns else None
            ws = ops._workspace(plan.ws_bytes, dev) if plan.learns else None
            check(lib.vsiq_mt_lsq_bwd(plan.host, plan.dev.data_ptr(), n, gptrs, dx_flat.data_ptr(),
                                      ds_flat.data_ptr() if ds_flat is not None else None,
                                      dz_flat.data_ptr() if dz_flat is not None else None,
                                      ws.data_ptr() if ws is not None else None, ws.numel() if ws is not None else 0,
                                      ops._stream_ptr()), "vsiq_mt_lsq_bwd")
            ops._count_launch(plan.bwd_launches)
        out: list = [None, None]
        for i in range(n):
            out.append(plan.view(dx_flat, i) if ctx.needs_input_grad[2 + i] else None)
        k = 2 + n
        for i, (mgr, w, scale, zp, spec, learn, _, _) in enumerate(plan.items):  # scales that require grad
            if learn >= 1:
                q0, C = plan.q_offsets[i], scale.numel()
                ds = ds_flat[q0:q0 + C].view(scale.shape)
                out.append(ds if scale.dtype == torch.float64 else ds.to(scale.dtype))
                k += 1
        for i, (mgr, w, scale, zp, spec, learn, _, _) in enumerate(plan.items):  # zero-points that require grad
            if learn >= 2:
                q0, C = plan.q_offsets[i], zp.numel()
                dz = dz_flat[q0:q0 + C].view(zp.shape)
                out.append(dz if zp.dtype == torch.float32 else dz.to(zp.dtype))
                k += 1
        return tuple(out)


class _BankedLayer(torch.autograd.Function):
    """backward="per_layer": the forward value comes from the bank's launch, the backward is this layer's own."""

    @staticmethod
    def forward(ctx, w, scale, zero_point, wq, spec, learn, gs_host, gs_dev):
        ctx.spec, ctx.learn, ctx.gs_host, ctx.gs_dev = spec, learn, gs_host, gs_dev
        ctx.s_t, ctx.z_t = isinstance(scale, torch.Tensor), isinstance(zero_point, torch.Tensor)
        ctx.consts = (None if ctx.s_t else scale, None if ctx.z_t else zero_point)
        ctx.save_for_backward(w, *([scale] if ctx.s_t else []), *([zero_point] if ctx.z_t else []))
        return wq.detach()

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        w = saved.pop(0)
        scale = saved.pop(0) if ctx.s_t else ctx.consts[0]
        zp = saved.pop(0) if ctx.z_t else ctx.consts[1]
        if ctx.learn == 0:
            dw = ops.fake_quant_backward_ste(w, g, scale, zp, ctx.spec) if ctx.needs_input_grad[0] else None
            return dw, None, None, None, None, None, None, None
        dw, ds, dz = ops.lsq_backward(w, g, scale, zp, ctx.spec, ctx.gs_host, ctx.gs_dev, want_dz=ctx.learn == 2,
                                      ds_dtype=scale.dtype, dz_dtype=zp.dtype if ctx.z_t else torch.float32)
        ds = ds.view(scale.shape) if ctx.needs_input_grad[1] else None
        dz = dz.view(zp.shape) if (ctx.learn == 2 and ctx.needs_input_grad[2]) else None
        return (dw if ctx.needs_input_grad[0] else None), ds, dz, None, None, None, None, None


class WeightBank:
    def __init__(self, model: torch.nn.Module, backward: str = "bank"):
        if backward not in ("bank", "per_layer"):
            raise ValueError("backward must be 'bank' or 'per_layer'")
        self.backward = backward
        self.model = model
        self.layers = [m for m in model.modules() if hasattr(m, "weight_quantizer") and hasattr(m, "get_weight_bias")]
        self._plans: dict = {}  # signature -> _Plan (train / eval states alternate; a handful at most)
        self._hook = None
        self.enabled = True
        self.last_used = False  # did the last forward go through the multi-tensor launch?

    # ---- wiring ---------------------------------------------------------------------------------------
    def install(self) -> "WeightBank":
        if self._hook is None:
            self._hook = self.model.register_forward_pre_hook(self._pre_forward)
        return self

    def _pre_forward(self, module, args) -> None:  # a pre-hook's return value would replace the inputs: return None
        self.prepare()

    def remove(self) -> None:
        if self._hook is not None:
            self._hook.remove()
            self._hook = None
        for layer in self.layers:
            layer.weight_quantizer.__dict__.pop("_banked", None)

    # ---- per step -------------------------------------------------------------------------------------
    def _collect(self):
        """[(manager, weight, scale, zero_point, spec, learn, gs_host, gs_dev)] of every layer but the FP8 ones, or None
        when one of those is not bankable (or there is none)."""
        items, sig = [], []
        grad_on = torch.is_grad_enabled()
        device = None
        for layer in self.layers:
            mgr = layer.weight_quantizer
            w, _ = layer.get_weight_bias()
            q = mgr.quantizer
            if getattr(q, "fp8_format", 0):
                continue  # the multi-tensor kernels know integer grids only: FP8 weights keep their per-layer launch
            collecting = (not mgr.is_learning_scale) and mgr.is_observer_qparam
            if (not mgr.is_quantize or collecting or not isinstance(w, torch.Tensor) or not w.is_cuda
                    or w.dtype != torch.float32 or w.dim() < 2 or not _dense_in_memory(w)
                    or getattr(q, "mask_mode", "rounded") != "rounded" or not hasattr(q, "_spec")):
                return None, None
            if device is None:
                device = w.device
            elif w.device != device:
                return None, None
            if "scale" in mgr._parameters or "zero_point" in mgr._parameters or not mgr._calibrated \
                    or "scale" in mgr.__dict__:
                scale, zp = mgr.scale, mgr.zero_point
            else:
                scale, zp = mgr.observer.device_qparams()
            try:
                ch_axis = q._resolve_axis(w, scale)
            except ValueError:
                return None, None
            if ch_axis not in (None, 0):
                return None, None
            s_t, z_t = isinstance(scale, torch.Tensor), isinstance(zp, torch.Tensor)
            # the table holds raw pointers: qparams must live on the device, densely (a strided view would be copied
            # and the copy would go stale)
            if (s_t and (scale.device != device or not scale.is_contiguous())) \
                    or (z_t and (zp.device != device or not zp.is_contiguous() or not zp.is_floating_point())):
                return None, None
            learning = mgr.is_learning_scale
            scale_learn = s_t and scale.requires_grad and grad_on
            zp_round = z_t and learning and not q.symmetric and zp.is_floating_point()
            zp_learn = zp_round and zp.requires_grad and grad_on
            if zp_learn and not scale_learn:
                return None, None
            spec = q._spec(ch_axis, zp_learned=zp_round)
            gs_host, gs_dev = 1.0, None
            if (scale_learn or zp_learn) and learning:
                gs_host = q.calculate_grad_scale(w, scale.numel()) * float(q.grad_boost)
                cgs = q.calib_grad_scale
                if isinstance(cgs, torch.Tensor):
                    gs_dev = cgs.detach().to(device=device, dtype=torch.float32).sum().reshape(1)
                else:
                    gs_host *= float(cgs)
            learn = 2 if zp_learn else (1 if scale_learn else 0)
            items.append((mgr, w, scale, zp, spec, learn, gs_host, gs_dev))
            sig.append((w.data_ptr(), tuple(w.stride()), scale.data_ptr() if s_t else float(scale),
                        zp.data_ptr() if z_t else float(zp), learn, gs_host, spec.qmin, spec.qmax, spec.zp_learned,
                        gs_dev is not None))
        if not items:
            return None, None
        return items, (tuple(sig), str(device))

    def prepare(self) -> bool:
        """Quantise every weight now (one launch) and park the results on the managers; False = per-layer path."""
        self.last_used = False
        if not self.enabled or not self.layers:
            return False
        items, sig = self._collect()
        if items is None:
            for layer in self.layers:
                layer.weight_quantizer.__dict__.pop("_banked", None)
            return False
        plan = self._plans.get(sig)
        if plan is None or any(it[7] is not None for it in items):  # a device-side calib_grad_scale is re-summed
            if len(self._plans) >= 8:
                self._plans.clear()
            plan = self._plans[sig] = _Plan(items, items[0][1].device)
        weights = [it[1] for it in plan.items]
        if self.backward == "per_layer" and torch.is_grad_enabled():
            with torch.no_grad():
                flat = _BankFunction.apply(plan, len(weights), *weights)
            outs = [_BankedLayer.apply(w, scale, zp, wq, spec, learn, gs_host, gs_dev)
                    for (_, w, scale, zp, spec, learn, gs_host, gs_dev), wq in zip(plan.items, flat)]
        else:
            scales = [it[2] for it in plan.items if it[5] >= 1]
            zps = [it[3] for it in plan.items if it[5] >= 2]
            outs = _BankFunction.apply(plan, len(weights), *weights, *scales, *zps)
        for (mgr, w, *_), wq in zip(plan.items, outs):
            mgr.__dict__["_banked"] = (w, wq)
        self.last_used = True
        return True
