"""Percentile observer on the GPU (csrc/hist_observer.cu) against the NumPy oracle (hist_oracle/): the whole state bit for
bit (counts, exponents, clip, scale / zero-point; the call statistics, columns 5..7, to 1e-5 as for every observer) over
every layout the kernel walks, bit widths 2 / 3 / 4 / 8, symmetric and asymmetric, three percentiles, three calls of
growing range (coarsening), inputs salted with NaN, +-inf, denormals, +-0.0 and all-zero channels; the min/max
equivalence at percentile 100, order independence, determinism, a red-zone check, set_percentile, checkpoints and
YOLOv8n end to end."""
import ctypes

import numpy as np
import pytest
import torch

import hist_oracle

pytestmark = pytest.mark.gpu


def _salted(shape, ch_axis, seed, call):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * 0.7).astype(np.float32)
    x.reshape(-1)[::97] = np.float32(3e-39)    # denormals
    x.reshape(-1)[5::89] = np.float32(-0.0)    # negative zeros
    x.reshape(-1)[13] = 4.5                    # an outlier
    if ch_axis is not None:
        sl = [slice(None)] * len(shape)
        sl[ch_axis] = 0
        x[tuple(sl)] = 0.0  # an all-zero channel
        idx = [0] * len(shape)
        if call == 1:
            idx[ch_axis] = 1
            x[tuple(idx)] = np.nan  # this call is skipped for channel 1
            idx[ch_axis] = 2
            x[tuple(idx)] = np.inf  # channel 2 is frozen from here on
        if call == 2:
            idx[ch_axis] = 3
            x[tuple(idx)] = -np.inf
    elif call == 1:
        x.reshape(-1)[1000] = np.nan
    return x * np.float32(1.0 if call == 0 else 5.0 * call)  # growing range: the stored counts are coarsened


_LAYOUTS = {  # name: (shape, ch_axis, channels_last)
    "tensor": ((3, 5, 37, 41), None, False),
    "weight": ((16, 8, 3, 3), 0, False),
    "nchw": ((4, 8, 24, 24), 1, False),
    "nhwc": ((4, 16, 20, 20), 1, True),
}


def _same_bits(a, b):
    """Bitwise equality of fp64 arrays, all NaNs equal (their payloads differ between the GPU and the host)."""
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint64), b[~nan].view(np.uint64))


def _check(st_gpu, st_o):
    st = st_gpu.cpu().numpy()
    cols = [0, 1, 2, 3, 4] + list(range(8, st.shape[1]))
    assert _same_bits(st[:, cols], st_o[:, cols])
    np.testing.assert_allclose(st[:, 5:8], st_o[:, 5:8], rtol=1e-5, atol=1e-8, equal_nan=True)


def _cuda(xn, cl):
    x = torch.from_numpy(xn).cuda()
    return x.contiguous(memory_format=torch.channels_last) if cl else x


@pytest.mark.parametrize("percentile", [99.0, 99.99, 100.0])
@pytest.mark.parametrize("bits,symmetric", [(2, True), (2, False), (3, True), (3, False), (4, True), (4, False),
                                            (8, True), (8, False)])
@pytest.mark.parametrize("layout", sorted(_LAYOUTS))
def test_state_matches_oracle(layout, bits, symmetric, percentile):
    from vsiquantization_b200 import ops
    shape, ch_axis, cl = _LAYOUTS[layout]
    C = 1 if ch_axis is None else shape[ch_axis]
    st = ops.new_percentile_state(C, 2048, torch.device("cuda"))
    st_o = hist_oracle.new_state(C, 2048)
    for call in range(3):
        xn = _salted(shape, ch_axis, 100 * bits + int(symmetric), call)
        x = _cuda(xn, cl)
        if cl:
            assert ops.ci_supported(x)
        ops.slow_path_counters(reset=True)
        ops.hist_observe(x, ch_axis, st, 2048, percentile, bits, symmetric, 1e-8)
        assert ops.slow_path_counters()["layout_conversion_copies"] == 0  # NHWC read in place
        hist_oracle.observe(xn, ch_axis, st_o, 2048, percentile, bits, symmetric, 1e-8)
        _check(st, st_o)


@pytest.mark.parametrize("n_bins", [256, 512, 4096])
@pytest.mark.parametrize("layout", ["tensor", "nhwc"])
def test_bin_counts(layout, n_bins):
    from vsiquantization_b200 import ops
    shape, ch_axis, cl = _LAYOUTS[layout]
    C = 1 if ch_axis is None else shape[ch_axis]
    st = ops.new_percentile_state(C, n_bins, torch.device("cuda"))
    st_o = hist_oracle.new_state(C, n_bins)
    for call in range(3):
        xn = _salted(shape, ch_axis, n_bins, call)
        ops.hist_observe(_cuda(xn, cl), ch_axis, st, n_bins, 99.9, 4, False)
        hist_oracle.observe(xn, ch_axis, st_o, n_bins, 99.9, 4, False)
        _check(st, st_o)


def test_relu_output_large_tensor_matches_oracle():
    """Half exact zeros (positive bin 0 counted in registers), tens of CTAs per channel, both channel-group widths."""
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(7)
    xn = np.maximum(rng.standard_normal((8, 32, 64, 64)).astype(np.float32), np.float32(0))
    xn[3, 5, 7, 9] = 60.0
    for ch_axis, cl in ((None, False), (1, True), (1, False)):
        C = 1 if ch_axis is None else 32
        st = ops.new_percentile_state(C, 2048, torch.device("cuda"))
        ops.hist_observe(_cuda(xn, cl), ch_axis, st, 2048, 99.99, 4, False)
        st_o = hist_oracle.new_state(C, 2048)
        hist_oracle.observe(xn, ch_axis, st_o, 2048, 99.99, 4, False)
        _check(st, st_o)


@pytest.mark.parametrize("layout", sorted(_LAYOUTS))
def test_percentile_100_is_minmax_call_after_call(layout):
    from vsiquantization_b200.observers.minmax import MinMaxObserver
    from vsiquantization_b200.observers.percentile import PercentileObserver
    shape, ch_axis, cl = _LAYOUTS[layout]
    for bits, symmetric in ((4, True), (3, False)):
        a = MinMaxObserver(symmetric, bits, ch_axis=ch_axis)
        b = PercentileObserver(symmetric, bits, ch_axis=ch_axis, percentile=100)
        for call in range(3):
            x = _cuda(_salted(shape, ch_axis, 9, call), cl)
            a.observe(x)
            b.observe(x)
            assert _same_bits(a.state.cpu().numpy()[:, :4], b.state.cpu().numpy()[:, :4])


def test_order_and_split_independence_and_determinism():
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(3)
    xs = (rng.standard_normal((12, 16, 20, 20)) * rng.uniform(0.01, 50, (12, 1, 1, 1))).astype(np.float32)
    xs[4, 2, 3, 3] = 900.0
    dev = torch.device("cuda")

    def run(pieces):
        st = ops.new_percentile_state(16, 2048, dev)
        for p in pieces:
            ops.hist_observe(_cuda(np.ascontiguousarray(xs[p]), True), 1, st, 2048, 99.9, 4, True)
        return st.cpu().numpy()

    ref = run([slice(i, i + 1) for i in range(12)])
    cols = [0, 1, 2, 3] + list(range(8, ref.shape[1]))  # 4..7 count and average per call: they depend on the split
    for pieces in ([slice(i, i + 1) for i in (11, 3, 7, 0, 5, 9, 1, 10, 2, 8, 6, 4)],
                   [slice(0, 5), slice(5, 6), slice(6, 12)], [slice(8, 12), slice(0, 8)]):
        assert _same_bits(run(pieces)[:, cols], ref[:, cols])
    assert _same_bits(run([slice(i, i + 1) for i in range(12)]), ref)  # a repeat: identical bits


def test_outlier_is_clipped():
    from vsiquantization_b200.observers.minmax import MinMaxObserver
    from vsiquantization_b200.observers.percentile import PercentileObserver
    x = torch.randn(4, 64, 32, 32, device="cuda").contiguous(memory_format=torch.channels_last)
    x[1, 7, 3, 3] = 500.0
    a, b = MinMaxObserver(True, 4), PercentileObserver(True, 4)
    a.observe(x)
    b.observe(x)
    s_mm, _ = a.get_scale_zero_point()
    s_p, _ = b.get_scale_zero_point()
    assert b.max_val == 500.0 and s_p < 0.02 * s_mm
    assert float(b.state[0, 9]) < 10.0


def test_red_zone():
    """Nothing outside the state changes; x is untouched; the workspace header and everything past its size stay."""
    from vsiquantization_b200 import _lib, ops
    B = 512
    W = 12 + 2 * B
    xn = _salted((4, 16, 20, 20), 1, 5, 0)
    for cl in (False, True):
        x = _cuda(xn, cl)
        lay = _lib.Layout(4 * 20 * 20, 16, 1) if cl else _lib.Layout(4, 16, 400)
        x0 = x.clone()
        stats = ops.observe(x, 1)
        sentinel = -1234.5
        buf = torch.full((16 * W + 8192,), sentinel, dtype=torch.float64, device="cuda")
        st = buf[4096:4096 + 16 * W]
        st.copy_(ops.new_percentile_state(16, B, torch.device("cuda")).reshape(-1))
        nbytes = _lib.lib.vsiq_hist_observe_workspace_bytes(ctypes.byref(lay), B)
        ws = torch.full((nbytes + 4096,), 0x5A, dtype=torch.uint8, device="cuda")  # stale counts included
        ws[:256] = 0
        ws[nbytes:] = 0xA5
        rc = _lib.lib.vsiq_hist_observe(x.data_ptr(), ctypes.byref(lay), stats.data_ptr(), st.data_ptr(), B, 99.0, 4, 0,
                                        1e-8, ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        mask = torch.ones_like(buf, dtype=torch.bool)
        mask[4096:4096 + 16 * W] = False
        assert bool((buf[mask] == sentinel).all())
        assert bool((ws[:256] == 0).all()) and bool((ws[nbytes:] == 0xA5).all())
        assert torch.equal(x.contiguous().view(torch.int32), x0.contiguous().view(torch.int32))
        st_o = hist_oracle.new_state(16, B)
        hist_oracle.observe(xn, 1, st_o, B, 99.0, 4, False)
        _check(st.reshape(16, W), st_o)


def test_set_percentile_equals_a_fresh_calibration():
    from vsiquantization_b200.observers.percentile import PercentileObserver
    gen = torch.Generator(device="cuda").manual_seed(4)
    xs = [torch.randn(8, 32, 16, 16, device="cuda", generator=gen) * (1 + i) for i in range(3)]
    a = PercentileObserver(False, 4, ch_axis=1, percentile=99.99)
    for x in xs:
        a.observe(x)
    for p in (99.0, 99.9, 100.0):
        a.set_percentile(p)
        b = PercentileObserver(False, 4, ch_axis=1, percentile=p)
        for x in xs:
            b.observe(x)
        assert torch.equal(a.state, b.state)


# ---------------------------------------------------------------------------------------------- model level (YOLOv8n)
IMG = 96


def _yolo(cfg):
    from vsiquantization_b200.modules.fuse import fuse_modules_unified
    from vsiquantization_b200.modules.fuse_config import create_fuse_config_manager
    from vsiquantization_b200.nets import yolov8
    torch.manual_seed(0)
    model = yolov8.yolo_v8_n(num_classes=20)
    g = torch.Generator().manual_seed(1)
    for mod in model.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    model = fuse_modules_unified(model.cuda(), [["conv", "bn", "relu"]], config_manager=create_fuse_config_manager(cfg))
    return model.to(memory_format=torch.channels_last)


def _batches(n, seed=2):
    gc = torch.Generator().manual_seed(seed)
    return [(torch.randint(0, 256, (2, 3, IMG, IMG), generator=gc, dtype=torch.uint8), None) for _ in range(n)]


def _calibrate(model, batches):
    from vsiquantization_b200.utils.quantize_manager import calibrate_qat_model

    def data_calib(m, loader, dev):
        m.eval()
        with torch.no_grad():
            for imgs, _ in loader:
                m(imgs.to(dev).float().div(255.0).contiguous(memory_format=torch.channels_last))

    calibrate_qat_model(model, batches, data_calib, torch.device("cuda"))


def _act_managers(model):
    return [(n, m.activation_quantizer) for n, m in model.named_modules() if hasattr(m, "activation_quantizer")]


def test_yolov8n_percentile_100_scales_equal_minmax(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    a = _yolo(FuseConfig(bits_w=8, bits_a=4))
    b = _yolo(FuseConfig(bits_w=8, bits_a=4, observer_a_name="PercentileObserver"))
    for _, mgr in _act_managers(b):
        assert type(mgr.observer).__name__ == "PercentileObserver" and mgr.observer.num_bits == 4
        mgr.observer.percentile = 100.0
    for _, mgr in _act_managers(a):
        mgr.observer.num_bits = 4  # the MinMax observer at the quantiser's width, as the percentile observer runs
    batches = _batches(2)
    for model in (a, b):
        _calibrate(model, batches)
    ma, mb = _act_managers(a), _act_managers(b)
    assert len(ma) == 57
    for (n, qa), (_, qb) in zip(ma, mb):
        assert torch.equal(qa.observer.state[:, 2:4], qb.observer.state[:, 2:4]), n


def test_yolov8n_activation_states_equal_the_oracle_and_survive_a_checkpoint(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    cfg = FuseConfig(bits_w=8, bits_a=4, observer_a_name="PercentileObserver")
    model = _yolo(cfg)
    seen = {}
    for n, mgr in _act_managers(model):
        obs = mgr.observer

        def spy(x, obs=obs, n=n, f=obs.observe):
            seen.setdefault(n, []).append(x.detach().float().cpu().numpy())
            return f(x)
        obs.observe = spy
    batches = _batches(3)
    _calibrate(model, batches[:2])
    saved = {k: v.clone() for k, v in model.state_dict().items()}
    _calibrate(model, batches[2:])
    assert len(seen) == 57
    for n, mgr in _act_managers(model):
        assert len(seen[n]) == 3
        st_o = hist_oracle.new_state(1, 2048)
        for x in seen[n]:
            hist_oracle.observe(x, None, st_o, 2048, 99.99, 4, True)
        _check(mgr.observer.state, st_o)
    # mid-calibration checkpoint into a freshly fused model, then the rest of the data: the uninterrupted result
    fresh = _yolo(cfg)
    fresh.load_state_dict(saved)
    _calibrate(fresh, batches[2:])
    for (n, q1), (_, q2) in zip(_act_managers(model), _act_managers(fresh)):
        st1, st2 = q1.observer.state.cpu().numpy(), q2.observer.state.cpu().numpy()
        cols = [0, 1, 2, 3, 4] + list(range(8, st1.shape[1]))
        assert _same_bits(st1[:, cols], st2[:, cols]), n
        np.testing.assert_allclose(st1[:, 5:8], st2[:, 5:8], rtol=1e-12, atol=0)
