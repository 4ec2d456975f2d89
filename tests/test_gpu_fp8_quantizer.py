"""FP8 fake-quantisers (E4M3 / E5M2) on the GPU against the CPU oracle (fp8_oracle/): every fp32 bit pattern through the
forward, y / dx / codes bit for bit and dscale to 2e-6 of the summed magnitudes over per-tensor, per-channel (weights and
NCHW), short-row, unaligned and pre-ReLU layouts with salted inputs and scales on both sides of the fast-division range,
a red-zone check, determinism, and the QuantizationManager / FuseConfig flow on YOLOv8n: calibrated scales, learned-scale
start, checkpoints, sync_observers, FP8 code export, mixed integer / FP8 models with the weight bank and input links."""
import numpy as np
import pytest
import torch

import fp8_oracle

pytestmark = pytest.mark.gpu

FMTS = [fp8_oracle.E4M3, fp8_oracle.E5M2]


def _spec(fmt, ch_axis=None, relu=False):
    from vsiquantization_b200 import ops
    return ops.QSpec(0, 0, ch_axis=ch_axis, pre_relu=relu, fp8_format=fmt)


def _same_bits(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    return bool(same.all()), int((~same).sum())


# ------------------------------------------------------------------------------------------ 1. every fp32 bit pattern
@pytest.mark.parametrize("fmt", FMTS)
def test_exhaustive_cast_matches_torch_cpu(fmt):
    from vsiquantization_b200 import ops
    F = fp8_oracle.FMAX[fmt]
    chunk = 1 << 28
    wrong = 0
    for k in range(1 << 4):
        bits = torch.arange(k * chunk, (k + 1) * chunk, dtype=torch.int64, device="cuda")
        bits = torch.where(bits >= (1 << 31), bits - (1 << 32), bits).to(torch.int32)
        x = bits.view(torch.float32)
        y = ops.fake_quant_forward(x, 1.0, 0, _spec(fmt)).cpu()
        del bits
        ref = x.cpu().clamp(-F, F).to(fp8_oracle.DTYPE[fmt]).float()
        same = (y.view(torch.int32) == ref.view(torch.int32)) | (torch.isnan(y) & torch.isnan(ref))
        wrong += int((~same).sum())
    assert wrong == 0


# ------------------------------------------------------------------------------------------ 2. bit-exact cases
def _salted(shape, ch_axis, scales, fmt, seed):
    """Values spread over the whole FP8 range of each channel's scale, salted with FP8 midpoints (times s), +-0, fp32
    denormals, +-inf, NaN, +-F*s and the next floats beyond."""
    rng = np.random.default_rng(seed)
    F = fp8_oracle.FMAX[fmt]
    n = int(np.prod(shape))
    C = 1 if ch_axis is None else shape[ch_axis]
    s = np.broadcast_to(np.asarray(scales, np.float32).reshape(-1), (C,)).astype(np.float32)
    view = [1] * len(shape)
    if ch_axis is not None:
        view[ch_axis] = C
    sb = np.broadcast_to(s.reshape(view), shape)
    mag = np.exp2(rng.uniform(-12 if fmt == fp8_oracle.E4M3 else -18, np.log2(F) + 1, n)).reshape(shape)
    x = (np.sign(rng.standard_normal(shape)) * mag * sb).astype(np.float32)
    vals = fp8_oracle.decode_all(fmt)
    pos = np.sort(vals[np.isfinite(vals) & (vals >= 0)])
    mids = ((pos[:-1] + pos[1:]) / 2).astype(np.float32)
    flat, sflat = x.reshape(-1), sb.reshape(-1)
    idx = rng.choice(n, size=min(n, 4000), replace=False)
    k = len(idx) // 2
    flat[idx[:k]] = mids[rng.integers(0, len(mids), k)] * sflat[idx[:k]] * np.where(rng.random(k) < 0.5, -1, 1)
    special = np.array([0.0, -0.0, 1e-40, -1e-40, 1e-45, np.inf, -np.inf, np.nan], np.float32)
    j = idx[k:k + 400]
    flat[j] = special[rng.integers(0, len(special), len(j))]
    j = idx[k + 400:k + 800]
    edge = np.array([1.0, -1.0, 1.0000001, -1.0000001, 0.99999994], np.float32)
    flat[j] = np.float32(F) * sflat[j] * edge[rng.integers(0, len(edge), len(j))]
    return x, s


CASES = [  # (shape, ch_axis, relu, unaligned)
    ((1 << 20) + 13, None, False, False),
    ((64, 3, 3, 3), 0, False, False),
    ((2, 16, 33, 17), 1, False, False),
    ((4, 24, 7, 5), 1, True, False),      # short rows: the warp-per-tile schedule
    ((3, 8, 300, 11), 1, False, True),    # unaligned view: the scalar instantiation
    ((40000,), None, True, True),
    ((256, 4096), None, False, False),
    ((96, 640), 0, True, False),
]
SCALES = {"pow2": lambda C, r: np.exp2(r.integers(-8, 4, C)).astype(np.float32),
          "random": lambda C, r: r.uniform(0.003, 2.0, C).astype(np.float32),
          "ieee_path": lambda C, r: np.where(np.arange(C) % 2 == 0, 2.0 ** -45, 2.0 ** 45).astype(np.float32)}


@pytest.mark.parametrize("scale_kind", list(SCALES))
@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("fmt", FMTS)
def test_bit_exact_against_oracle(fmt, case, scale_kind):
    from vsiquantization_b200 import ops
    shape, ch_axis, relu, unaligned = CASES[case]
    shape = shape if isinstance(shape, tuple) else (shape,)
    rng = np.random.default_rng(case * 7 + len(scale_kind))
    C = 1 if ch_axis is None else shape[ch_axis]
    x, s = _salted(shape, ch_axis, SCALES[scale_kind](C, rng), fmt, case)
    g = rng.standard_normal(shape).astype(np.float32)
    g.reshape(-1)[:50] = np.array([0.0, -0.0, 1e-40, np.inf, np.nan] * 10, np.float32)

    def dev(a):
        t = torch.from_numpy(a).cuda()
        if unaligned:
            buf = torch.empty(t.numel() + 1, device="cuda")
            buf[1:].copy_(t.reshape(-1))
            t = buf[1:].view(t.shape)
        return t

    xd, gd = dev(x), dev(g)
    sd = torch.from_numpy(s).cuda() if C > 1 else torch.from_numpy(s.reshape(())).cuda()
    spec = _spec(fmt, ch_axis if C > 1 else None, relu)
    y_o, codes_o = fp8_oracle.forward(x, s if C > 1 else s[0], fmt, ch_axis if C > 1 else None, relu)
    gs = fp8_oracle.grad_scale(fmt, x.size, C)
    dx_o, ds_o, mag = fp8_oracle.backward(x, g, s if C > 1 else s[0], fmt, ch_axis if C > 1 else None, relu, gs)

    y = ops.fake_quant_forward(xd, sd, 0, spec)
    ok, bad = _same_bits(y.cpu().numpy(), y_o)
    assert ok, f"y: {bad} mismatches"
    dx = ops.fake_quant_backward_ste(xd, gd, sd, 0, spec)
    ok, bad = _same_bits(dx.cpu().numpy(), dx_o)
    assert ok, f"STE dx: {bad} mismatches"
    dx2, ds, dz = ops.lsq_backward(xd, gd, sd, 0, spec, gs, ds_dtype=torch.float64)
    assert dz is None
    ok, bad = _same_bits(dx2.cpu().numpy(), dx_o)
    assert ok, f"LSQ dx: {bad} mismatches"
    ds = ds.cpu().numpy()
    fin = np.isfinite(ds_o)
    assert np.array_equal(np.isnan(ds), np.isnan(ds_o))
    assert (np.abs(ds[fin] - ds_o[fin]) <= 2e-6 * mag[fin] + 1e-300).all(), (ds[fin][:4], ds_o[fin][:4])
    if not relu:
        yc, codes = ops.quantize_codes(xd, sd, 0, spec)
        assert codes.dtype == fp8_oracle.DTYPE[fmt] and codes.shape == xd.shape
        ok, bad = _same_bits(yc.cpu().numpy(), y_o)
        assert ok, f"codes-path y: {bad} mismatches"
        c = codes.cpu().view(torch.uint8).numpy()
        nan = np.isnan(y_o)
        assert np.array_equal(c[~nan], codes_o[~nan])
        assert np.isnan(fp8_oracle.decode_all(fmt)[c[nan]]).all()
        _, only = ops.quantize_codes(xd, sd, 0, spec, want_y=False)
        assert torch.equal(only.view(torch.uint8), codes.view(torch.uint8))


# ------------------------------------------------------------------------------------------ 3. red zone, determinism
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("n,off", [(1000, 1), (65536 + 5, 8), (3 << 20, 3)])
def test_red_zone(fmt, n, off):
    from vsiquantization_b200 import ops
    torch.manual_seed(n)
    x = torch.randn(n, device="cuda") * 100
    g = torch.randn(n, device="cuda")
    spec = _spec(fmt)
    for fn in ("fwd", "ste"):
        buf = torch.full((n + 2 * off + 64,), 0x7FBADBAD, dtype=torch.int32, device="cuda").view(torch.float32)
        out = buf[off + 32:off + 32 + n]
        if fn == "fwd":
            ops.fake_quant_forward(x, 0.25, 0, spec, out=out)
        else:
            ops.fake_quant_backward_ste(x, g, 0.25, 0, spec, out=out)
        b = buf.view(torch.int32)
        assert (b[:off + 32] == 0x7FBADBAD).all() and (b[off + 32 + n:] == 0x7FBADBAD).all()
    cbuf = torch.full((n + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    codes = cbuf[32:32 + n].view(fp8_oracle.DTYPE[fmt])
    ops.quantize_codes(x, 0.25, 0, spec, codes_out=codes)
    assert (cbuf[:32] == 0xA5).all() and (cbuf[32 + n:] == 0xA5).all()


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("shape,ch_axis", [(((1 << 24) + 7,), None), ((64, 256, 40, 40), 1), ((512, 4096), 0)])
def test_lsq_backward_is_deterministic(fmt, shape, ch_axis):
    from vsiquantization_b200 import ops
    torch.manual_seed(3)
    x = torch.randn(shape, device="cuda") * 30
    g = torch.randn(shape, device="cuda")
    C = 1 if ch_axis is None else shape[ch_axis]
    s = torch.rand(C, device="cuda") + 0.05 if C > 1 else torch.tensor(0.07, device="cuda")
    runs = [ops.lsq_backward(x, g, s, 0, _spec(fmt, ch_axis if C > 1 else None), 1e-3, ds_dtype=torch.float64)
            for _ in range(3)]
    for dx, ds, _ in runs[1:]:
        assert torch.equal(dx.view(torch.int32), runs[0][0].view(torch.int32))
        assert torch.equal(ds.view(torch.int64), runs[0][1].view(torch.int64))


# ------------------------------------------------------------------------------------------ 4. managers and models
IMG = 96


def _yolo(cfg, swap=None):
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


def _fp8_cfg(obs_a="MinMaxObserver"):
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    return FuseConfig(quantizer_w_name="FP8Quantizer", quantizer_a_name="FP8Quantizer", observer_a_name=obs_a,
                      w_ch_axis=0)


def _batches(n, seed=2):
    gc = torch.Generator().manual_seed(seed)
    return [(torch.randint(0, 256, (2, 3, IMG, IMG), generator=gc, dtype=torch.uint8), None) for _ in range(n)]


def _img(b):
    return b[0].cuda().float().div(255.0).contiguous(memory_format=torch.channels_last)


def _calibrate(model, batches):
    from vsiquantization_b200.utils.quantize_manager import calibrate_qat_model

    def data_calib(m, loader, dev):
        m.eval()
        with torch.no_grad():
            for b in loader:
                m(_img(b))

    calibrate_qat_model(model, batches, data_calib, torch.device("cuda"))


def _managers(model):
    from vsiquantization_b200.parallel import quantization_managers
    return quantization_managers(model)


def _expected_scale(mgr):
    """amax / F from the observer's documented range, read through its public host accessors rather than device_range():
    MinMax: the running extrema (min_val / max_val); Percentile: the clip, state columns 8 / 9 (observers/percentile.py)."""
    from vsiquantization_b200.observers.percentile import HistogramObserver
    obs = mgr.observer
    if isinstance(obs, HistogramObserver):
        st = obs.state.detach().cpu().double()
        lo, hi = st[:, 8], st[:, 9]
        assert torch.all(hi <= st[:, 1]) and torch.all(lo >= st[:, 0])  # a clip, inside the running extrema
    else:
        lo = torch.as_tensor(obs.min_val, dtype=torch.float64).reshape(-1)
        hi = torch.as_tensor(obs.max_val, dtype=torch.float64).reshape(-1)
    amax = torch.maximum(lo.abs(), hi.abs())
    F = mgr.quantizer.fmax
    return torch.where((amax > 0) & torch.isfinite(amax), amax / F, torch.ones_like(amax))


def _loss(out):
    outs = out if isinstance(out, (list, tuple)) else [out]
    return sum(o.float().square().mean() for o in outs if isinstance(o, torch.Tensor))


@pytest.mark.parametrize("obs_a", ["MinMaxObserver", "PercentileObserver"])
def test_yolov8n_fp8_flow(obs_a):
    from vsiquantization_b200.utils.quantize_manager import activate_learning_qparam, activate_quantizer
    model = _yolo(_fp8_cfg(obs_a))
    _calibrate(model, _batches(2))
    mgrs = _managers(model)
    assert mgrs and all(m._fp8 for _, m in mgrs)
    for name, m in mgrs:
        assert torch.equal(m._fp8_scale.cpu(), _expected_scale(m)), name
        s, z = m._current_qparams()
        assert s is m._fp8_scale and z == 0
    # the lazy readback
    name, m = next((n, m) for n, m in mgrs if m.observer.state.shape[0] == 1)
    assert m.scale == float(_expected_scale(m)[0]) and m.zero_point == 0
    activate_learning_qparam(model)
    activate_quantizer(model)
    for name, m in mgrs:
        p = m._parameters["scale"]
        assert torch.equal(p.detach().reshape(-1).cpu(), _expected_scale(m)), name
    model.train()
    opt = torch.optim.SGD([p for p in model.parameters() if p.requires_grad], lr=1e-4)
    losses = []
    for b in _batches(3, seed=5):
        opt.zero_grad()
        loss = _loss(model(_img(b)))
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert all(np.isfinite(losses))
    grads = {n: m._parameters["scale"].grad for n, m in mgrs}
    bad = [n for n, gr in grads.items() if gr is None or not torch.isfinite(gr).all()]
    assert not bad, bad[:8]
    # FP8 weight export equals the CPU cast of W / s
    for layer in [mod for mod in model.modules() if hasattr(mod, "weight_quantizer")][:12]:
        wm = layer.weight_quantizer
        w, _ = layer.get_weight_bias()
        s = wm.scale.detach()
        y, codes = wm.quantizer.quantize_codes(w, s)
        sc = s.float().cpu().reshape(-1, *([1] * (w.dim() - 1)))
        ref = (w.detach().cpu().contiguous() / sc).clamp(-448, 448).to(torch.float8_e4m3fn)
        assert torch.equal(codes.cpu().view(torch.uint8), ref.view(torch.uint8))


def test_learned_step_matches_eager_composition():
    """One learned FP8 quantiser on the GPU against an eager torch composition on the same GPU: tensor-scale division,
    clamp, .to(fp8) with a straight-through estimator and the LSQ gradient scale."""
    from vsiquantization_b200.quantizers.fp8 import FP8Quantizer
    torch.manual_seed(7)
    q = FP8Quantizer(8, True, ch_axis=0)
    for layout in ("nchw", "channels_last"):
        x0 = torch.randn(8, 16, 12, 12, device="cuda") * 40
        x = x0.contiguous(memory_format=torch.channels_last) if layout == "channels_last" else x0
        s = torch.nn.Parameter(torch.rand(8, device="cuda", dtype=torch.float64) * 0.2 + 0.01)
        xa = x.clone().requires_grad_(True)
        y = q.quantize(xa, s, 0, is_learning_scale=True)
        g = torch.randn_like(y)
        y.backward(g)

        xb = x0.clone().requires_grad_(True)
        sb = s.detach().clone().requires_grad_(True)
        gs = q.calculate_grad_scale(xb, 8)  # the ScaleGradient factor, applied to the eager gradient below
        s32 = sb.float().view(-1, 1, 1, 1)
        v = xb / s32
        c = v.clamp(-448, 448)
        qc = c.to(torch.float8_e4m3fn).float()
        qv = c + (qc - c).detach()
        yb = qv * s32
        gc = g.contiguous()
        yb.backward(gc)
        assert torch.equal(y.detach().contiguous().view(torch.int32), yb.detach().view(torch.int32)), layout
        assert torch.equal(xa.grad.contiguous().view(torch.int32), xb.grad.contiguous().view(torch.int32)), layout
        mag = (gc.double().abs() * (qc.double().abs() + v.detach().double().abs())).sum(dim=(1, 2, 3)) * gs
        assert ((s.grad - sb.grad * gs).abs() <= 1e-5 * mag).all(), layout


def test_checkpoint_mid_calibration_and_sync_observers():
    from vsiquantization_b200.parallel import sync_observers
    model = _yolo(_fp8_cfg("PercentileObserver"))
    _calibrate(model, _batches(1))
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    want = {n: m._fp8_scale.clone() for n, m in _managers(model)}
    fresh = _yolo(_fp8_cfg("PercentileObserver"))
    fresh.load_state_dict(sd)
    for n, m in _managers(fresh):
        assert torch.equal(m._fp8_scale, want[n]), n
    # sync_observers at world size 1: the merge re-derives every FP8 scale in place
    ptrs = {n: m._fp8_scale.data_ptr() for n, m in _managers(fresh)}
    for _, m in _managers(fresh):
        m._fp8_scale.fill_(-1.0)
    sync_observers(fresh)
    for n, m in _managers(fresh):
        assert m._fp8_scale.data_ptr() == ptrs[n]
        assert torch.equal(m._fp8_scale, want[n]), n


def test_mixed_model_bank_and_links():
    from vsiquantization_b200.bank import WeightBank
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager
    from vsiquantization_b200.utils.quantize_manager import activate_learning_qparam, activate_quantizer, link_quantize_inp
    model = _yolo(FuseConfig(w_ch_axis=0))
    layers = [m for m in model.modules() if hasattr(m, "weight_quantizer") and hasattr(m, "get_weight_bias")]
    for i, layer in enumerate(layers):
        if i % 3 == 0:
            layer.weight_quantizer = QuantizationManager("FP8Quantizer", "MinMaxObserver", 8, True,
                                                         is_learning_scale=False, ch_axis=0).cuda()
            layer.activation_quantizer = QuantizationManager("FP8Quantizer", "MinMaxObserver", 8, True,
                                                             is_learning_scale=False).cuda()
    _calibrate(model, _batches(1))
    activate_learning_qparam(model)
    activate_quantizer(model)
    model.eval()  # no BatchNorm statistics move between the two runs
    x = _img(_batches(1, seed=4)[0])
    link_quantize_inp(model, x)
    fp8_layers = sum(1 for layer in layers if layer.weight_quantizer._fp8)

    def step(use_bank):
        bank = WeightBank(model).install() if use_bank else None
        for p in model.parameters():
            p.grad = None
        out = model(x)
        loss = _loss(out)
        loss.backward()
        grads = [p.grad.clone() if p.grad is not None else None for p in model.parameters()]
        items = None
        if bank is not None:
            items, _ = bank._collect()
            assert bank.last_used
            bank.remove()
        return out, grads, items

    out_b, g_b, items = step(True)
    assert len(items) == len(layers) - fp8_layers
    assert all(not it[0]._fp8 for it in items)
    out_u, g_u, _ = step(False)
    o1 = out_b if isinstance(out_b, (list, tuple)) else [out_b]
    o2 = out_u if isinstance(out_u, (list, tuple)) else [out_u]
    for a, b in zip(o1, o2):
        assert torch.equal(a, b)
    for a, b in zip(g_b, g_u):
        assert (a is None) == (b is None)
        if a is None:
            continue
        if a.dtype == torch.float32:  # weights and biases: bit for bit
            assert torch.equal(a, b)
        else:  # the learned scales: the bank sums each tensor's terms in another order (fp32 tiles, fp64 combine)
            assert ((a - b).abs() <= 1e-5 * b.abs().max() + 1e-30).all()


# ------------------------------------------------------------------------------------------ 5. channels_last epilogue
def _rows_reference(pre, b, g, s, spec_ci, gs):
    """y, dx and dscale of the rows kernels applied to act(x + b) on contiguous NCHW memory; SiLU as ATen's F.silu."""
    import torch.nn.functional as F
    from vsiquantization_b200 import ops
    xb = (pre + b.view(1, -1, 1, 1)).contiguous() if b is not None else pre.contiguous()
    spec = _spec(spec_ci.fp8_format, spec_ci.ch_axis, spec_ci.pre_relu)
    if spec_ci.pre_silu:
        xs = xb.clone().requires_grad_(True)
        a = F.silu(xs)
        y = ops.fake_quant_forward(a.detach(), s, 0, spec)
        dq, ds, _ = ops.lsq_backward(a.detach(), g.contiguous(), s, 0, spec, gs, ds_dtype=torch.float64)
        (dx,) = torch.autograd.grad(a, xs, dq)
        return y, dx, ds, a.detach()
    y = ops.fake_quant_forward(xb, s, 0, spec)
    dx, ds, _ = ops.lsq_backward(xb, g.contiguous(), s, 0, spec, gs, ds_dtype=torch.float64)
    return y, dx, ds, torch.relu(xb) if spec_ci.pre_relu else xb


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("C", [16, 64, 512])
@pytest.mark.parametrize("pcq", [False, True])
@pytest.mark.parametrize("act", [None, "relu", "silu"])
def test_channels_last_epilogue_matches_rows_kernels(fmt, C, pcq, act):
    from vsiquantization_b200 import ops
    torch.manual_seed(C + 7 * fmt)
    HW = {16: 40, 64: 20, 512: 12}[C]
    F = fp8_oracle.FMAX[fmt]
    s = (torch.rand(C, device="cuda") * 0.05 + 0.002) if pcq else torch.tensor(0.03, device="cuda")
    x = torch.randn(4, C, HW, HW, device="cuda") * (F * 0.02)
    x.view(-1)[:64] = torch.tensor([0.0, -0.0, 1e-40, float("inf"), -float("inf"), float("nan"), F * 0.03, -F * 0.03] * 8,
                                   device="cuda")
    x = x.contiguous(memory_format=torch.channels_last)
    b = torch.randn(C, device="cuda")
    # grad_output as a channel slice of a wider NHWC tensor (torch.cat's backward): the pitched / TMA path
    gw = torch.randn(4, C + 8, HW, HW, device="cuda").contiguous(memory_format=torch.channels_last)
    g = gw[:, :C]
    spec = ops.QSpec(0, 0, ch_axis=1 if pcq else None, pre_relu=act == "relu", pre_silu=act == "silu", fp8_format=fmt)
    gs = fp8_oracle.grad_scale(fmt, x.numel(), C if pcq else 1)
    y = ops.ci_forward(x, b, s, 0, spec)
    dx, ds, dz, db = ops.ci_backward(x, b, g, s, 0, spec, gs, None, True, False, True, torch.float64)
    dx_d, ds_d, _, db_d = ops.ci_backward(x, b, g.contiguous(memory_format=torch.channels_last), s, 0, spec, gs, None,
                                          True, False, True, torch.float64)
    assert dz is None
    y_r, dx_r, ds_r, a = _rows_reference(x.contiguous(), b, g, s, spec, gs)
    ok, bad = _same_bits(y.contiguous().cpu().numpy(), y_r.cpu().numpy())
    assert ok, f"y: {bad} mismatches"
    for d in (dx, dx_d):
        ok, bad = _same_bits(d.contiguous().cpu().numpy(), dx_r.cpu().numpy())
        assert ok, f"dx: {bad} mismatches"
    # dscale: within 2e-6 of the summed magnitudes of the fp64 oracle on the activated tensor
    _, ds_o, mag = fp8_oracle.backward(a.cpu().numpy(), g.contiguous().cpu().numpy(),
                                       s.cpu().numpy() if pcq else float(s), fmt, 1 if pcq else None, False, gs)
    for d in (ds, ds_d, ds_r):
        d = d.cpu().numpy()
        fin = np.isfinite(ds_o)
        assert np.array_equal(np.isnan(d), np.isnan(ds_o))
        assert (np.abs(d[fin] - ds_o[fin]) <= 2e-6 * mag[fin] + 1e-300).all()
    # dbias: the sum of dx over N, H, W (fp64 here)
    ref_db = dx_r.double().sum(dim=(0, 2, 3))
    mass = dx_r.double().abs().sum(dim=(0, 2, 3))
    for d in (db, db_d):
        fin = torch.isfinite(ref_db)
        assert torch.equal(torch.isnan(d.double()), torch.isnan(ref_db))
        assert ((d.double() - ref_db).abs()[fin] <= 1e-5 * mass[fin] + 1e-30).all()
    # the quantiser's own entry: FakeQuantEpilogue through FP8Quantizer.quantize
    from vsiquantization_b200.quantizers.fp8 import FP8E5M2Quantizer, FP8Quantizer
    q = (FP8Quantizer if fmt == fp8_oracle.E4M3 else FP8E5M2Quantizer)(8, True, ch_axis=1 if pcq else None)
    yq = q.quantize(x, s.reshape(1, C, 1, 1) if pcq else s, 0, bias=b, pre_act=act)
    assert torch.equal(yq.contiguous().view(torch.int32), y.contiguous().view(torch.int32))


# ------------------------------------------------------------------------------------------ 6. YOLOv8n against eager
class _RoundFP8(torch.autograd.Function):
    @staticmethod
    def forward(ctx, c, dtype):
        return c.to(dtype).float()

    @staticmethod
    def backward(ctx, g):
        return g, None


class EagerFP8Quantizer:
    """The FP8 definition as an eager torch composition: division by the scale tensor, clamp, .to(float8) with a
    straight-through estimator, times the scale; LSQ gradient scale on the scale.  No fused activation (the manager
    applies F.relu / F.silu and the bias add before it)."""

    def __init__(self, q):
        self.fmt, self.fmax, self.ch_axis = q.fp8_format, q.fmax, q.ch_axis
        self.qmax, self.num_bits, self.symmetric = q.qmax, 8, True
        self.calib_grad_scale = q.calib_grad_scale

    def quantize(self, x, scale, zero_point, is_learning_scale=False):
        from oracle.torch_port import _ScaleGrad
        C = scale.numel() if isinstance(scale, torch.Tensor) else 1
        shape = [1] * x.dim()
        if C > 1:
            shape[self.ch_axis] = C
        if isinstance(scale, torch.Tensor):
            scale = scale.to(torch.float32).reshape(shape if C > 1 else ())
            if is_learning_scale:
                scale = _ScaleGrad.apply(scale, (self.fmax * (x.numel() / C)) ** -0.5 * self.calib_grad_scale)
        c = (x / scale).clamp(-self.fmax, self.fmax)
        return _RoundFP8.apply(c, fp8_oracle.DTYPE[self.fmt]) * scale


def _build_fp8():
    from vsiquantization_b200.modules.fuse import fuse_modules_unified
    from vsiquantization_b200.modules.fuse_config import create_fuse_config_manager
    from vsiquantization_b200.nets import yolov8
    from vsiquantization_b200.utils.quantize_manager import activate_learning_qparam, activate_quantizer, calibrate_qat_model
    torch.manual_seed(0)
    model = yolov8.yolo_v8_n(num_classes=20)
    g = torch.Generator().manual_seed(1)
    for mod in model.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    model = fuse_modules_unified(model.cuda(), [["conv", "bn", "relu"]],
                                 config_manager=create_fuse_config_manager(_fp8_cfg()))
    gc = torch.Generator().manual_seed(2)
    calib = [(torch.randint(0, 256, (2, 3, IMG, IMG), generator=gc, dtype=torch.uint8), None) for _ in range(2)]

    def data_calib(m, loader, dev):
        m.eval()
        with torch.no_grad():
            for imgs, _ in loader:
                m(imgs.to(dev).float() / 255.0)

    calibrate_qat_model(model, calib, data_calib, torch.device("cuda"))
    activate_learning_qparam(model, use_init=True)
    activate_quantizer(model)
    return model.cuda().train()


def test_yolov8n_fp8_equals_eager_composition_and_graphed_steps(monkeypatch):
    """Per-channel FP8 weights, per-tensor FP8 activations: every fused layer's output, the input gradient and every
    weight gradient bit for bit against the eager composition (NCHW and channels_last, the latter through the fused bias +
    SiLU epilogue); scale gradients and the epilogue's bias gradients to 1e-5 of the summed magnitudes; three graphed SGD
    steps equal three eagerly launched ones."""
    import copy

    import torch.nn.functional as F
    from test_gpu_model_parity import _compare, _fused, _step
    from vsiquantization_b200.modules.fused import ConvBnReLU
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    model = _build_fp8()
    assert all(m.weight_quantizer._fp8 and m.activation_quantizer._fp8 for _, m in _fused(model))

    def eager_of(mdl, decomposed_bias):
        e = copy.deepcopy(mdl)
        for _, m in _fused(e):
            for mgr in (m.weight_quantizer, m.activation_quantizer):
                mgr.quantizer = EagerFP8Quantizer(mgr.quantizer)
            if decomposed_bias and isinstance(m, ConvBnReLU):
                def fwd(x, m=m):
                    w, b = m.get_weight_bias()
                    pre = m._conv(x, m.quantize_weights(w), None) + b.view(1, -1, 1, 1)
                    return m.quantize_activation(F.relu(pre) if m.is_relu else F.silu(pre))
                m.forward = fwd
        return e

    gx = torch.Generator().manual_seed(3)
    x = torch.randint(0, 256, (2, 3, IMG, IMG), generator=gx, dtype=torch.uint8).cuda().float() / 255.0
    n_q = 2 * 57
    mass = {}
    native = _step(copy.deepcopy(model), x, mass)
    assert _compare(native, _step(eager_of(model, False), x), mass, "NCHW native vs eager") == n_q
    xcl = x.contiguous(memory_format=torch.channels_last)
    mcl = copy.deepcopy(model).to(memory_format=torch.channels_last)
    mass_cl = {}
    native_cl = _step(copy.deepcopy(mcl), xcl, mass_cl)
    assert _compare(native_cl, _step(eager_of(mcl, True), xcl), mass_cl, "channels_last native vs eager",
                    bias_is_sum=True) == n_q

    from vsiquantization_b200.graph import GraphedQATStep
    loss_fn = lambda outs: sum((o.float() ** 2).mean() for o in outs)  # noqa: E731
    batches = [torch.randint(0, 256, (2, 3, IMG, IMG), generator=gx, dtype=torch.uint8).cuda().float().div(255.0)
               .contiguous(memory_format=torch.channels_last) for _ in range(3)]
    m1, m2 = copy.deepcopy(mcl), copy.deepcopy(mcl)
    o1 = torch.optim.SGD(m1.parameters(), lr=1e-3, momentum=0.9, nesterov=True)
    o2 = torch.optim.SGD(m2.parameters(), lr=1e-3, momentum=0.9, nesterov=True)
    for _ in range(3):  # the warm-up steps GraphedQATStep runs on its example input
        o1.zero_grad(set_to_none=True)
        loss_fn(m1(batches[0])).backward()
        o1.step()
    step = GraphedQATStep(m2, o2, loss_fn, batches[0], warmup=3)
    for b in batches:
        o1.zero_grad(set_to_none=True)
        l1 = loss_fn(m1(b))
        l1.backward()
        o1.step()
        l2 = step(b)
        assert float(l1.detach()) == float(l2), "graphed and eagerly launched steps diverge"
    for (n1, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(p1.detach().view(torch.int32) if p1.dtype == torch.float32 else p1.detach(),
                           p2.detach().view(torch.int32) if p2.dtype == torch.float32 else p2.detach()), n1


def test_link_quantize_inp_skips_fp8_consumers():
    """int -> int(quantize_inp) -> FP8(quantize_inp): the integer pair is linked, the FP8 consumer keeps its own launch,
    and the values equal the unlinked model's."""
    from vsiquantization_b200.modules.fused import ConvBnReLU
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager
    from vsiquantization_b200.utils.quantize_manager import activate_quantizer, calibrate_qat_model, link_quantize_inp
    torch.manual_seed(7)
    layers = []
    for cin, cout in ((8, 16), (16, 16), (16, 16)):
        cv, bn = torch.nn.Conv2d(cin, cout, 3, padding=1, bias=False), torch.nn.BatchNorm2d(cout)
        with torch.no_grad():
            bn.running_mean.normal_(0, 0.1)
            bn.running_var.uniform_(0.5, 1.5)
            bn.bias.normal_(0, 0.2)
        layers.append(ConvBnReLU(cv, bn, torch.nn.ReLU(), "MinMaxObserver", "UniformQuantizer", "MinMaxObserver",
                                 "UniformQuantizer", True, False, True, 8, 8))
    layers[1].quantize_inp = True
    layers[2].quantize_inp = True
    layers[2].activation_quantizer = QuantizationManager("FP8Quantizer", "MinMaxObserver", 8, True,
                                                         is_learning_scale=False)
    model = torch.nn.Sequential(*layers).cuda().to(memory_format=torch.channels_last)
    x = torch.randn(4, 8, 20, 20, device="cuda").contiguous(memory_format=torch.channels_last)
    calibrate_qat_model(model, [x], lambda m, loader, dev: [m(b) for b in loader])
    for m in model:
        for q in (m.weight_quantizer, m.activation_quantizer):
            q.is_learning_scale = False
            q.is_observer_qparam = False
    activate_quantizer(model)
    model.eval()
    with torch.no_grad():
        y0 = model(x)
    assert link_quantize_inp(model, x) == 1
    assert model[0].__dict__.get("_inp_consumer") is model[1]
    assert model[1].__dict__.get("_inp_consumer") is None
    with torch.no_grad():
        y1 = model(x)
    assert torch.equal(y0.view(torch.int32), y1.view(torch.int32))
