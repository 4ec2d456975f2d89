"""Drop this implementation into a checkout of the reference.

Tier 1 -- registry tier: the reference's own managers, fused layers, control API and drivers stay untouched; only the
two plugin classes they build by name (quantizers/quantization_manager.py:41-42) are replaced:

    import vsiquantization_b200.dropin as dropin
    dropin.install_plugins()          # after the reference's packages are importable (its repo root on sys.path)

Tier 2 -- package tier: the reference's module paths resolve to this package, so ``from modules.fuse import
fuse_modules_unified`` etc. run the B200-native host code (sync-free calibration, device-resident qparams):

    dropin.install_modules()          # before importing the reference's drivers
"""
from __future__ import annotations

import importlib
import sys

_TIER2 = {
    "utils.registry": "vsiquantization_b200.utils.registry",
    "utils.quantize_manager": "vsiquantization_b200.utils.quantize_manager",
    "utils.estimate_bn": "vsiquantization_b200.utils.estimate_bn",
    "observers.base": "vsiquantization_b200.observers.base",
    "observers.minmax": "vsiquantization_b200.observers.minmax",
    "observers.mse": "vsiquantization_b200.observers.mse",
    "observers.percentile": "vsiquantization_b200.observers.percentile",
    "observers.entropy": "vsiquantization_b200.observers.entropy",
    "quantizers.base": "vsiquantization_b200.quantizers.base",
    "quantizers.uniform": "vsiquantization_b200.quantizers.uniform",
    "quantizers.quantization_manager": "vsiquantization_b200.quantizers.quantization_manager",
    "quantizers.fake_quantize": "vsiquantization_b200.quantizers.fake_quantize",
    "quantizers.lsq_module": "vsiquantization_b200.quantizers.lsq_module",
    "modules.fused": "vsiquantization_b200.modules.fused",
    "modules.fuse": "vsiquantization_b200.modules.fuse",
    "modules.fuse_config": "vsiquantization_b200.modules.fuse_config",
}


def install_plugins(registry=None, mse_observer: bool = False, percentile_observer: bool = False,
                    entropy_observer: bool = False):
    """Register UniformQuantizer / LSQQuantizer / MinMaxObserver / LSQObserver (and this package's moving-average
    observers) in the REFERENCE's CLASS_REGISTRY (utils/registry.py:2; a later registration overwrites, :26).  Returns the
    registry dict.  mse_observer=True also registers MSEObserver, percentile_observer=True PercentileObserver,
    entropy_observer=True EntropyObserver; the reference's own QuantizationManager builds every observer at 8 bits
    (quantization_manager.py:41-42), so under Tier 1 they search / clip at 8 bits -- Tier 2's manager hands them the
    quantiser's width."""
    from .observers.entropy import EntropyObserver
    from .observers.minmax import LSQObserver, MinMaxObserver
    from .observers.moving_average import MovingAverageMinMaxObserver, MovingAveragePerChannelMinMaxObserver
    from .observers.mse import MSEObserver
    from .observers.percentile import PercentileObserver
    from .quantizers.uniform import LSQQuantizer, UniformQuantizer
    if registry is None:
        registry = importlib.import_module("utils.registry").CLASS_REGISTRY  # the reference's module
    for cls in (UniformQuantizer, LSQQuantizer, MinMaxObserver, LSQObserver, MovingAverageMinMaxObserver,
                MovingAveragePerChannelMinMaxObserver) + ((MSEObserver,) if mse_observer else ()) \
            + ((PercentileObserver,) if percentile_observer else ()) + ((EntropyObserver,) if entropy_observer else ()):
        registry[cls.__name__] = cls
    return registry


def install_modules():
    """Alias the reference's module paths to this package (sys.modules), so its drivers import the native host code."""
    for ref_name, ours in _TIER2.items():
        sys.modules[ref_name] = importlib.import_module(ours)
    return sorted(_TIER2)
