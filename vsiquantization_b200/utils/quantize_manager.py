"""QAT control API (reference: utils/quantize_manager.py:4-118): mode switches over every module that owns a
``weight_quantizer`` / ``activation_quantizer``.  Same names, arguments and semantics."""
from __future__ import annotations


def _managers(model, layer_names=None):
    for name, module in model.named_modules():
        for attr in ("weight_quantizer", "activation_quantizer"):
            if hasattr(module, attr) and (layer_names is None or name in layer_names):
                yield name, getattr(module, attr)


def calibrate_qat_model(model, dataloader, data_calib, device=None):
    """Observer mode on, learning and quantisation off, model.eval(), then ``data_calib(model, dataloader, device)``
    runs the forward passes (quantize_manager.py:4-31).  Each observed tensor costs one kernel launch and no host
    synchronisation; scales / zero-points are read back lazily afterwards."""
    for _, q in _managers(model):
        q.is_observer_qparam = True
        q.is_learning_scale = False
        q.is_quantize = False
    model.eval()
    data_calib(model, dataloader, device)


def activate_learning_qparam(model, layer_names=None, use_init=True, active=True):
    """Switch (selected) layers to learnable qparams: optional LSQ initialisation from the calibration statistics, then
    scale (and, for asymmetric quantisers, zero-point) become nn.Parameters (quantize_manager.py:34-66)."""
    for _, q in _managers(model, layer_names):
        q.is_learning_scale = active
        if use_init:
            q.init_scaling_factor_for_learning()
        if active:
            q.make_learn_qparameter()


def deactivate_learning_qparam(model, layer_names=None):
    activate_learning_qparam(model, layer_names=layer_names, active=False)


def activate_quantizer(model, layer_names=None, active=True):
    """Enable / disable fake quantisation in the forward pass (quantize_manager.py:83-103)."""
    for _, q in _managers(model, layer_names):
        q.is_quantize = active


def deactivate_quantizer(model, layer_names=None):
    activate_quantizer(model, layer_names=layer_names, active=False)


def link_quantize_inp(model, example_input=None, forward=None) -> int:
    """Find the layers whose output goes straight into a ``quantize_inp=True`` layer and link each such pair
    (FakeQuantize.feed_input_quantizer_of): the producer's output epilogue then also writes the consumer's input
    quantisation (fake_quantize.py:44-45) in the same pass.  Discovery is one forward pass of ``model(example_input)``
    (or ``forward(model)``) under no_grad with hooks comparing tensor identities; pairs whose tensors are re-packed on
    the way (cat, chunk, add) are not linked and keep their own launch.  Returns the number of links made; existing
    links are dropped first.  Extension: the reference has no counterpart, its model runs unchanged without it."""
    import torch

    fused = [m for m in model.modules() if hasattr(m, "activation_quantizer") and hasattr(m, "feed_input_quantizer_of")]
    for m in fused:
        m.feed_input_quantizer_of(None)
    producer_of, alive, pairs, handles = {}, [], [], []

    def after(mod, args, out):
        if isinstance(out, torch.Tensor):
            producer_of[id(out)] = mod
            alive.append(out)  # keep ids unique for the duration of the pass

    def before(mod, args):
        if getattr(mod, "quantize_inp", False) and args and isinstance(args[0], torch.Tensor):
            src = producer_of.get(id(args[0]))
            if src is not None and src is not mod:
                pairs.append((src, mod))

    for m in fused:
        handles.append(m.register_forward_pre_hook(before))
        handles.append(m.register_forward_hook(after))
    try:
        with torch.no_grad():
            forward(model) if forward is not None else model(example_input)
    finally:
        for h in handles:
            h.remove()
    def fp8(m):
        return bool(getattr(getattr(m.activation_quantizer, "quantizer", None), "fp8_format", 0))

    linked, seen = 0, set()
    for src, dst in pairs:
        if id(src) in seen:  # one second stage per producer: the first consumer found keeps the link
            continue
        if fp8(src) or fp8(dst):  # the two-output epilogue has integer grids only
            continue
        seen.add(id(src))
        src.feed_input_quantizer_of(dst)
        linked += 1
    return linked
