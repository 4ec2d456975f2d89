"""FP8 quantisers without a GPU: torch's CPU fp32 -> fp8 cast (the oracle of tests/test_gpu_fp8_quantizer.py) against an
independent nearest-even encoder built from the 256 codes, the validation errors of the quantisers, the manager and the C
ABI (argument checks that fail before any launch), and the FuseConfig / YAML wiring."""
import ctypes

import numpy as np
import pytest
import torch

import fp8_oracle

FMTS = [fp8_oracle.E4M3, fp8_oracle.E5M2]


def _interesting(fmt):
    """Every code value, every midpoint of neighbouring values, both +-1 ulp (fp32), zeros, fp32 denormals, +-F and the
    first values above F (which the definition clamps to F)."""
    vals = fp8_oracle.decode_all(fmt)
    pos = np.sort(vals[np.isfinite(vals) & (vals >= 0)])
    mids = (pos[:-1] + pos[1:]) / 2
    base = np.concatenate([pos, mids]).astype(np.float32)
    F = np.float32(fp8_oracle.FMAX[fmt])
    above = [np.nextafter(F, np.float32(np.inf)), F * np.float32(1.0625), F * 2, np.float32(3e38), np.float32(np.inf)]
    ext = np.concatenate([base, np.nextafter(base, np.float32(np.inf)), np.nextafter(base, np.float32(0)),
                          np.array([0.0, 1e-45, 1e-40, 1.17e-38, 2 ** -149, 2 ** -126] + above, dtype=np.float32)])
    rng = np.random.default_rng(fmt)
    rand = np.concatenate([rng.standard_normal(200000).astype(np.float32) * s for s in (1e-4, 1e-2, 1, 50, 3000)])
    rand_bits = rng.integers(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    allv = np.concatenate([ext, rand, rand_bits])
    return np.concatenate([allv, -allv, np.array([np.nan, -np.nan], dtype=np.float32)])


@pytest.mark.parametrize("fmt", FMTS)
def test_torch_cast_matches_the_independent_encoder(fmt):
    x = _interesting(fmt)
    F = fp8_oracle.FMAX[fmt]
    c = torch.from_numpy(x).clamp(-F, F)
    got = c.to(fp8_oracle.DTYPE[fmt]).view(torch.uint8).numpy()
    want = fp8_oracle.encode(c.numpy(), fmt)
    vals = fp8_oracle.decode_all(fmt)
    nan = np.isnan(c.numpy())
    assert np.isnan(vals[got[nan]]).all()
    bad = np.nonzero(got[~nan] != want[~nan])[0]
    assert bad.size == 0, [(float(c.numpy()[~nan][i]), int(got[~nan][i]), int(want[~nan][i])) for i in bad[:5]]
    # the decoded values agree with torch's fp8 -> fp32 conversion on every code
    codes = torch.arange(256, dtype=torch.int32).to(torch.uint8).view(fp8_oracle.DTYPE[fmt]).float().double().numpy()
    fin = np.isfinite(vals)
    assert np.array_equal(codes[fin], vals[fin]) and np.isnan(codes[np.isnan(vals)]).all()
    assert np.array_equal(np.signbit(codes[fin]), np.signbit(vals[fin]))


def test_oracle_forward_keeps_negative_zero_and_clamps():
    y, codes = fp8_oracle.forward(np.array([-0.0, 1e-30, -1e-30, 1e9, -np.inf], np.float32), 1.0, fp8_oracle.E4M3)
    assert np.signbit(y[0]) and y[0] == 0 and codes[0] == 0x80
    assert y[1] == 0 and not np.signbit(y[1]) and np.signbit(y[2])
    assert y[3] == 448.0 and y[4] == -448.0


def test_quantizer_construction_errors_and_attributes():
    from vsiquantization_b200.quantizers.fp8 import FP8E5M2Quantizer, FP8Quantizer
    from vsiquantization_b200.utils.registry import CLASS_REGISTRY
    assert CLASS_REGISTRY["FP8Quantizer"] is FP8Quantizer and CLASS_REGISTRY["FP8E5M2Quantizer"] is FP8E5M2Quantizer
    with pytest.raises(ValueError, match="8-bit"):
        FP8Quantizer(4, True)
    with pytest.raises(ValueError, match="symmetric"):
        FP8Quantizer(8, False)
    q = FP8Quantizer(8, True, ch_axis=0)
    assert (q.fmax, q.qmin, q.qmax, q.ch_axis, q.calib_grad_scale) == (448.0, -448.0, 448.0, 0, 1)
    assert q.codes_dtype == torch.float8_e4m3fn and q.supports_pre_relu and q.kernel_args(None, 1.0, 0) is None
    assert FP8E5M2Quantizer().fmax == 57344.0 and FP8E5M2Quantizer().codes_dtype == torch.float8_e5m2
    x = torch.zeros(2, 3)
    assert q.calculate_grad_scale(x, 1) == pytest.approx((448 * 6) ** -0.5)
    assert q.calculate_grad_scale(x, 2) == pytest.approx((448 * 3) ** -0.5)
    with pytest.raises(ValueError, match="zero-point"):
        q.quantize(x, 1.0, 3)
    with pytest.raises(ValueError, match="pre_act"):
        q.quantize(x, 1.0, 0, pre_act="gelu")
    assert q.supports_pre_silu
    from vsiquantization_b200.quantizers.uniform import UniformQuantizer
    assert not isinstance(q, UniformQuantizer)


@pytest.mark.parametrize("obs", ["MSEObserver", "EntropyObserver"])
@pytest.mark.parametrize("qname", ["FP8Quantizer", "FP8E5M2Quantizer"])
def test_manager_refuses_integer_grid_searches(obs, qname):
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager
    with pytest.raises(ValueError) as e:
        QuantizationManager(qname, obs, 8, True)
    assert obs in str(e.value) and qname in str(e.value)


@pytest.mark.parametrize("obs", ["MinMaxObserver", "LSQObserver", "PercentileObserver", "MovingAverageMinMaxObserver"])
def test_manager_accepts_range_observers(obs):
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager
    m = QuantizationManager("FP8Quantizer", obs, 8, True)
    assert m._fp8 == fp8_oracle.E4M3 and m.zero_point == 0
    assert hasattr(m.observer, "device_range")


def test_fuse_config_and_yaml(tmp_path):
    from vsiquantization_b200.modules.fuse_config import FuseConfig, load_fuse_config_from_yaml
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager
    cfg = FuseConfig(quantizer_w_name="FP8Quantizer", quantizer_a_name="FP8E5M2Quantizer")
    assert cfg.quantizer_w_name == "FP8Quantizer"
    p = tmp_path / "fp8.yaml"
    p.write_text("default:\n  quantizer_w_name: FP8Quantizer\n  quantizer_a_name: FP8Quantizer\n"
                 "  observer_a_name: PercentileObserver\n")
    mgr = load_fuse_config_from_yaml(str(p))
    d = mgr.default_config
    assert (d.quantizer_w_name, d.quantizer_a_name, d.observer_a_name) == ("FP8Quantizer", "FP8Quantizer",
                                                                         "PercentileObserver")
    qm = QuantizationManager(d.quantizer_a_name, d.observer_a_name, d.bits_a, d.a_symmetric)
    assert qm.quantizer.fmax == 448.0


def test_abi_argument_checks_before_any_launch():
    from vsiquantization_b200 import _lib
    from vsiquantization_b200._lib import Layout, QParams
    lib = _lib.lib
    lay = Layout(1, 1, 0)  # empty tensor: valid calls return before touching the device
    qp = QParams()
    qp.qmin = qp.qmax = 0
    qp.scale_host = 1.0
    ok = lib.vsiq_fp8_fake_quant_fwd(None, None, None, ctypes.byref(lay), ctypes.byref(qp), 1, None)
    assert ok == 0
    assert lib.vsiq_fp8_fake_quant_fwd(None, None, None, ctypes.byref(lay), ctypes.byref(qp), 3, None) == -1
    assert lib.vsiq_fp8_fake_quant_bwd_ste(None, None, None, ctypes.byref(lay), ctypes.byref(qp), 0, None) == -1
    bad = QParams()
    bad.qmin, bad.qmax = -128, 127  # an integer range: the grid comes from fp8_format
    assert lib.vsiq_fp8_fake_quant_fwd(None, None, None, ctypes.byref(lay), ctypes.byref(bad), 1, None) == -1
    zp = QParams()
    zp.zp_host = 1.0
    assert lib.vsiq_fp8_fake_quant_fwd(None, None, None, ctypes.byref(lay), ctypes.byref(zp), 2, None) == -3
    zl = QParams()
    zl.zp_learned = 1
    assert lib.vsiq_fp8_fake_quant_bwd_ste(None, None, None, ctypes.byref(lay), ctypes.byref(zl), 1, None) == -3
    silu = QParams()
    silu.pre_op = _lib.PRE_SILU
    assert lib.vsiq_fp8_fake_quant_fwd(None, None, None, ctypes.byref(lay), ctypes.byref(silu), 1, None) == -3
    ds = ctypes.c_float()
    args = lambda dzp, mask, fmt: (None, None, None, ctypes.byref(ds), 0, dzp, 0, ctypes.byref(lay),  # noqa: E731
                                   ctypes.byref(qp), fmt, 1.0, None, mask, None, 0, None)
    assert lib.vsiq_fp8_lsq_bwd(*args(None, _lib.MASK_FUNLSQ, 1)) == -3
    assert lib.vsiq_fp8_lsq_bwd(*args(ctypes.byref(ds), _lib.MASK_ROUNDED, 1)) == -3
    assert lib.vsiq_fp8_lsq_bwd(*args(None, 7, 1)) == -1
    assert lib.vsiq_fp8_lsq_bwd(*args(None, _lib.MASK_ROUNDED, 5)) == -1
    assert lib.vsiq_fp8_lsq_bwd(*args(None, _lib.MASK_ROUNDED, 1)) == -2  # no workspace
    ci = lambda fmt, dzp: lib.vsiq_ci_fp8_lsq_bwd(None, None, None, None, None, 0, dzp, 0, None, 0, 16,  # noqa: E731
                                                ctypes.byref(qp), 1, fmt, 1.0, None, 0, None, 0, None)
    assert ci(1, None) == 0 and ci(4, None) == -1 and ci(1, ctypes.byref(ds)) == -3
    assert lib.vsiq_ci_fp8_fake_quant_fwd(None, None, None, 0, 16, ctypes.byref(qp), 1, 2, None, 0, None) == 0
    assert lib.vsiq_ci_fp8_fake_quant_fwd(None, None, None, 0, 16, ctypes.byref(qp), 1, 0, None, 0, None) == -1
    assert lib.vsiq_ci_fp8_fake_quant_fwd(None, None, None, 0, 16, ctypes.byref(bad), 1, 1, None, 0, None) == -1
    assert lib.vsiq_fp8_scale_from_range(None, None, 1, 0, 1, None, None) == 0
    assert lib.vsiq_fp8_scale_from_range(None, None, 1, 4, 1, None, None) == -1
    assert lib.vsiq_fp8_scale_from_range(None, None, 1, 4, 9, None, None) == -1
