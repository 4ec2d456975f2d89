"""MSE observer on the GPU (csrc/mse_search.cu) against the C oracle (mse_oracle/): E[C, K] to 1e-12 relative (only the
summation order differs), the chosen alpha (or, on a near-tie, two oracle errors within that bound), scale / zero-point
bit for bit; every layout the kernel walks, bit widths 2 / 3 / 4 / 8, symmetric and asymmetric, inputs salted with NaN,
+-inf, denormals and all-zero channels; a red-zone check; YOLOv8n end to end."""
import ctypes

import numpy as np
import pytest
import torch

import mse_oracle

pytestmark = pytest.mark.gpu
RTOL = 1e-12


def _salted(shape, ch_axis, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * 0.7).astype(np.float32)
    x.reshape(-1)[::97] = np.float32(3e-39)  # denormals
    x.reshape(-1)[13] = 4.5                  # an outlier
    if ch_axis is not None:
        sl = [slice(None)] * len(shape)
        for c, v in ((0, 0.0), (1, np.nan), (2, np.inf), (3, -np.inf)):
            sl[ch_axis] = c
            if v == 0.0:
                x[tuple(sl)] = 0.0  # an all-zero channel
            else:
                idx = [0] * len(shape)
                idx[ch_axis] = c
                x[tuple(idx)] = v
    else:
        x.reshape(-1)[1000:1400] = 0.0
    return x


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


def _check_call(st_gpu, err, alpha, st_o, E_o, a_o):
    E = err.cpu().numpy()
    A = alpha.cpu().numpy()
    st = st_gpu.cpu().numpy()
    fin = np.isfinite(E_o)
    assert np.array_equal(fin, np.isfinite(E))
    np.testing.assert_allclose(E[fin], E_o[fin], rtol=RTOL, atol=0)
    K = E.shape[1]
    for c in range(E.shape[0]):
        if A[c] != a_o[c]:  # a near-tie: both oracle errors within the bound
            k1, k2 = int(round(A[c] * K)) - 1, int(round(a_o[c] * K)) - 1
            assert abs(E_o[c, k1] - E_o[c, k2]) <= RTOL * abs(E_o[c, k2]), (c, A[c], a_o[c])
            return False
    assert np.array_equal(st[:, [0, 1, 4]], st_o[:, [0, 1, 4]])
    assert _same_bits(st[:, 2:4], st_o[:, 2:4])  # scale / zero-point bit for bit
    assert _same_bits(st[:, 8:10], st_o[:, 8:10])
    # call statistics (LSQ initialisation): the min/max pass's fp64 sums of fp32 vector partials, as for every observer
    np.testing.assert_allclose(st[:, 5:8], st_o[:, 5:8], rtol=1e-5, atol=1e-8)
    return True


@pytest.mark.parametrize("bits,symmetric", [(2, True), (2, False), (3, True), (3, False), (4, True), (4, False),
                                            (8, True), (8, False)])
@pytest.mark.parametrize("layout", sorted(_LAYOUTS))
def test_search_matches_oracle(layout, bits, symmetric):
    from vsiquantization_b200 import ops
    shape, ch_axis, cl = _LAYOUTS[layout]
    C = 1 if ch_axis is None else shape[ch_axis]
    st = ops.new_mse_state(C, torch.device("cuda"))
    st_o = mse_oracle.new_state(C)
    for call in range(2):  # two calls: running range and running means of the clipped extrema
        xn = _salted(shape, ch_axis, 100 * bits + 10 * call + int(symmetric))
        xn *= np.float32(1.0 + call)
        x = torch.from_numpy(xn).cuda()
        if cl:
            x = x.contiguous(memory_format=torch.channels_last)
            assert ops.ci_supported(x)
        ops.slow_path_counters(reset=True)
        _, err, alpha = ops.mse_search(x, ch_axis, st, bits, symmetric, 1e-8, 100, want_err=True)
        assert ops.slow_path_counters()["layout_conversion_copies"] == 0  # NHWC searched in place
        E_o, a_o = mse_oracle.search(xn, ch_axis, st_o, bits, symmetric, 1e-8, 100)
        if not _check_call(st, err, alpha, st_o, E_o, a_o):
            return


@pytest.mark.parametrize("K", [1, 7, 37, 64, 65, 256])
@pytest.mark.parametrize("layout", ["tensor", "nhwc"])
def test_candidate_counts(layout, K):
    from vsiquantization_b200 import ops
    shape, ch_axis, cl = _LAYOUTS[layout]
    C = 1 if ch_axis is None else shape[ch_axis]
    xn = _salted(shape, ch_axis, K)
    x = torch.from_numpy(xn).cuda()
    if cl:
        x = x.contiguous(memory_format=torch.channels_last)
    st = ops.new_mse_state(C, torch.device("cuda"))
    _, err, alpha = ops.mse_search(x, ch_axis, st, 4, False, 1e-8, K, want_err=True)
    st_o = mse_oracle.new_state(C)
    E_o, a_o = mse_oracle.search(xn, ch_axis, st_o, 4, False, 1e-8, K)
    _check_call(st, err, alpha, st_o, E_o, a_o)


def test_observer_interface_and_deterministic_repeat():
    from vsiquantization_b200.observers.mse import MSEObserver
    w = torch.randn(32, 16, 3, 3, device="cuda") * 0.1
    w[3, 0, 0, 0] = 2.0
    a, b = MSEObserver(False, 4, ch_axis=0), MSEObserver(False, 4, ch_axis=0)
    s1, z1 = a.forward(w)
    b.observe(w)
    b.observe(w)  # the same tensor again: the single-call result
    s2, z2 = b.get_scale_zero_point()
    assert torch.equal(s1, s2) and torch.equal(z1, z2)
    st_o = mse_oracle.new_state(32)
    mse_oracle.search(w.cpu().numpy(), 0, st_o, 4, False, 1e-8, 100)
    assert np.array_equal(s1.numpy(), st_o[:, 2]) and np.array_equal(z1.numpy(), st_o[:, 3])
    assert torch.equal(a.min_val, torch.from_numpy(st_o[:, 0])) and torch.equal(a.max_val, torch.from_numpy(st_o[:, 1]))
    ds, dz = a.device_qparams()
    assert torch.equal(ds.cpu(), s1) and torch.equal(dz.cpu(), z1)
    init = a.lsq_init_scale(4)  # the reference rule on sum|x|, unchanged by the search
    want = 2 * w.abs().double().reshape(32, -1).mean(1) / 7 ** 0.5
    torch.testing.assert_close(init, want, rtol=1e-6, atol=0)  # fp64 sums of fp32 vector partials
    assert float(st_o[3, 2]) < (float(st_o[3, 1]) - float(st_o[3, 0])) / 15  # the outlier channel is clipped


def test_red_zone():
    """Nothing outside err / alpha / state changes; x is untouched; the workspace header is left zero."""
    from vsiquantization_b200 import _lib, ops
    xn = _salted((4, 16, 20, 20), 1, 5)
    for cl in (False, True):
        x = torch.from_numpy(xn).cuda()
        if cl:
            x = x.contiguous(memory_format=torch.channels_last)
            lay = _lib.Layout(4 * 20 * 20, 16, 1)
        else:
            lay = _lib.Layout(4, 16, 400)
        x0 = x.clone()
        stats = ops.observe(x, 1)
        C, K = 16, 100
        sentinel = -1234.5
        buf = torch.full((3 * 4096,), sentinel, dtype=torch.float64, device="cuda")
        st = buf[100:100 + C * 10]
        st.zero_()
        err = buf[4096 + 3:4096 + 3 + C * K]
        alpha = buf[8192 + 7:8192 + 7 + C]
        nbytes = _lib.lib.vsiq_mse_search_workspace_bytes(ctypes.byref(lay), K)
        ws = torch.zeros(nbytes + 4096, dtype=torch.uint8, device="cuda")
        ws[nbytes:] = 0xA5
        rc = _lib.lib.vsiq_mse_search(x.data_ptr(), ctypes.byref(lay), stats.data_ptr(), st.data_ptr(), 3, 0, 1e-8, K,
                                      err.data_ptr(), alpha.data_ptr(), ws.data_ptr(), nbytes,
                                      torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        mask = torch.ones_like(buf, dtype=torch.bool)
        mask[100:100 + C * 10] = False
        mask[4096 + 3:4096 + 3 + C * K] = False
        mask[8192 + 7:8192 + 7 + C] = False
        assert bool((buf[mask] == sentinel).all())
        assert bool((ws[:256] == 0).all()) and bool((ws[nbytes:] == 0xA5).all())
        assert torch.equal(x.contiguous().view(torch.int32), x0.contiguous().view(torch.int32))


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
    model = model.cuda()
    return fuse_modules_unified(model, [["conv", "bn", "relu"]], config_manager=create_fuse_config_manager(cfg))


def _calibrate(model, n_batches):
    from vsiquantization_b200.utils.quantize_manager import calibrate_qat_model
    gc = torch.Generator().manual_seed(2)
    calib = [(torch.randint(0, 256, (2, 3, IMG, IMG), generator=gc, dtype=torch.uint8), None) for _ in range(n_batches)]

    def data_calib(m, loader, dev):
        m.eval()
        with torch.no_grad():
            for imgs, _ in loader:
                m(imgs.to(dev).float() / 255.0)

    calibrate_qat_model(model, calib, data_calib, torch.device("cuda"))


def _fused(model):
    return [(n, m) for n, m in model.named_modules() if hasattr(m, "weight_quantizer")]


def _step(model, x):
    acts, hooks = {}, []
    for n, m in _fused(model):
        hooks.append(m.register_forward_hook(lambda mod, i, o, n=n: acts.__setitem__(n, o.detach())))
    x = x.clone().requires_grad_(True)
    model.zero_grad(set_to_none=True)
    loss = sum((o.float() ** 2).mean() for o in model(x))
    loss.backward()
    for h in hooks:
        h.remove()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return acts, loss.detach(), x.grad.detach(), grads


def test_yolov8n_one_candidate_is_bit_identical_to_minmax(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.utils.quantize_manager import activate_learning_qparam, activate_quantizer
    a = _yolo(FuseConfig(bits_w=8, bits_a=8))
    b = _yolo(FuseConfig(bits_w=8, bits_a=8, observer_w_name="MSEObserver", observer_a_name="MSEObserver"))
    for _, m in _fused(b):
        for mgr in (m.weight_quantizer, m.activation_quantizer):
            assert type(mgr.observer).__name__ == "MSEObserver"
            mgr.observer.n_candidates = 1
    for model in (a, b):
        _calibrate(model, 1)
    for (n, ma), (_, mb) in zip(_fused(a), _fused(b)):
        for attr in ("weight_quantizer", "activation_quantizer"):
            sa, sb = getattr(ma, attr).observer.state, getattr(mb, attr).observer.state
            assert torch.equal(sa[:, 2:4], sb[:, 2:4]), (n, attr)
    for model in (a, b):  # LSQ from the calibrated qparams (observers stop absorbing batches)
        activate_learning_qparam(model, use_init=False)
        activate_quantizer(model)
        model.train()
    x = torch.rand(2, 3, IMG, IMG, generator=torch.Generator().manual_seed(3)).cuda()
    ra, rb = _step(a, x), _step(b, x)
    assert len(ra[0]) == 57 and all(torch.equal(ra[0][k], rb[0][k]) for k in ra[0])
    assert torch.equal(ra[1], rb[1]) and torch.equal(ra[2], rb[2])
    assert set(ra[3]) == set(rb[3]) and all(torch.equal(ra[3][k], rb[3][k]) for k in ra[3])


def test_yolov8n_w4_per_channel_mse_weights_calibrate_and_train():
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.utils.quantize_manager import activate_quantizer
    cfg = FuseConfig(observer_w_name="MSEObserver", quantizer_w_name="LSQQuantizer", observer_a_name="LSQObserver",
                     quantizer_a_name="LSQQuantizer", w_symmetric=False, a_symmetric=False, bits_w=4, bits_a=8,
                     w_ch_axis=0, a_ch_axis=1)
    model = _yolo(cfg)
    _calibrate(model, 2)
    n_clipped = 0
    for n, m in _fused(model):
        obs = m.weight_quantizer.observer
        assert type(obs).__name__ == "MSEObserver" and obs.num_bits == 4
        w, _ = m.get_weight_bias()
        st_o = mse_oracle.new_state(w.shape[0])
        for _ in range(2):  # the weight is observed once per calibration batch
            mse_oracle.search(w.detach().cpu().numpy(), 0, st_o, 4, False, 1e-8, 100)
        st = obs.state.cpu().numpy()
        assert _same_bits(st[:, 2:4], st_o[:, 2:4]), n
        n_clipped += int((st_o[:, 8] > st_o[:, 0]).sum() + (st_o[:, 9] < st_o[:, 1]).sum())
    assert n_clipped > 0
    for _, m in _fused(model):  # weights: LSQ starts from the searched qparams; activations: the reference's LSQ init
        wq, aq = m.weight_quantizer, m.activation_quantizer
        wq.is_learning_scale = aq.is_learning_scale = True
        aq.init_scaling_factor_for_learning()
        wq.make_learn_qparameter()
        aq.make_learn_qparameter()
    activate_quantizer(model)
    model.train()
    opt = torch.optim.SGD([p for p in model.parameters() if p.requires_grad], lr=1e-4)
    gen = torch.Generator().manual_seed(4)
    for _ in range(3):
        x = torch.rand(2, 3, IMG, IMG, generator=gen).cuda()
        opt.zero_grad(set_to_none=True)
        loss = sum((o.float() ** 2).mean() for o in model(x))
        loss.backward()
        opt.step()
        assert bool(torch.isfinite(loss))
