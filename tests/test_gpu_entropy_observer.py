"""Entropy observer on the GPU (csrc/hist_entropy.cu) against the NumPy oracle (hist_oracle.entropy_clip): every
candidate's divergence to rtol 1e-9 / atol 1e-12 with the same non-finite pattern, the chosen threshold (a near-tie
may go either way), the whole state bit for bit (the call statistics, columns 5..7, to 1e-5 as for every observer) over
every layout the histogram pass walks, bit widths 2 / 3 / 4 / 8, symmetric and asymmetric, three calls of growing range,
inputs salted with NaN, +-inf, denormals, +-0.0 and all-zero channels; other bin counts and start bins, determinism and
order independence, a red-zone check, an outlier, and YOLOv8n end to end (the MinMax equivalence at start_bin = n_bins,
the oracle over three batches with a mid-calibration checkpoint, a world-size-1 sync)."""

import numpy as np
import pytest
import torch

import hist_oracle
from test_gpu_percentile_observer import _LAYOUTS, _act_managers, _batches, _calibrate, _cuda, _salted, _same_bits, _yolo

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-9, 1e-12


def _last_argmin(d):
    """The search's choice over one divergence row: smallest D (NaN as +inf), ties to the larger i; -1: no candidate."""
    cand = np.flatnonzero(~np.isnan(d))
    if cand.size == 0:
        return -1
    v = d[cand]
    return int(cand[len(v) - 1 - int(np.argmin(v[::-1]))])


def _check_call(st_gpu, d_gpu, st_o, d_o, bits, symmetric):
    """Divergences within tolerance, the same threshold as the oracle unless its two divergences are within that
    tolerance (a near-tie), the state bit for bit (columns 2, 3, 8, 9 of a near-tie channel: those of the GPU's own
    threshold)."""
    st = st_gpu.cpu().numpy()
    d = d_gpu.cpu().numpy()
    assert np.array_equal(np.isnan(d), np.isnan(d_o)) and np.array_equal(np.isinf(d), np.isinf(d_o))
    fin = np.isfinite(d_o)
    np.testing.assert_allclose(d[fin], d_o[fin], rtol=RTOL, atol=ATOL)
    cols = [0, 1, 4] + list(range(10, st.shape[1]))
    assert _same_bits(st[:, cols], st_o[:, cols])
    np.testing.assert_allclose(st[:, 5:8], st_o[:, 5:8], rtol=1e-5, atol=1e-8, equal_nan=True)
    for c in range(st.shape[0]):
        i_g, i_o = _last_argmin(d[c]), _last_argmin(d_o[c])
        if i_g == i_o:
            assert _same_bits(st[c, [2, 3, 8, 9]], st_o[c, [2, 3, 8, 9]]), c
            continue
        a, b = d_o[c, i_g], d_o[c, i_o]
        assert np.isfinite(a) and abs(a - b) <= RTOL * abs(b) + ATOL, (c, i_g, i_o, a, b)
        e = int(max(st[c, 10], st[c, 11]))
        amax = i_g * 2.0 ** e
        lo, hi = max(st[c, 0], -amax), min(st[c, 1], amax)
        assert (st[c, 8], st[c, 9]) == (lo, hi) and (st[c, 2], st[c, 3]) == hist_oracle.qparams(lo, hi, bits, symmetric)


def _run_both(x, xn, ch_axis, st, st_o, n_bins, start_bin, bits, symmetric):
    from vsiquantization_b200 import ops
    ops.hist_observe(x, ch_axis, st, n_bins, 100.0, bits, symmetric, 1e-8)
    d = torch.empty(st.shape[0], n_bins + 1, dtype=torch.float64, device=st.device)
    ops.hist_entropy_clip(st, n_bins, start_bin, bits, symmetric, 1e-8, divergences=d)
    hist_oracle.observe(xn, ch_axis, st_o, n_bins, 100.0, bits, symmetric, 1e-8)
    d_o = hist_oracle.entropy_clip(st_o, n_bins, start_bin, bits, symmetric, 1e-8)
    _check_call(st, d, st_o, d_o, bits, symmetric)
    return d


@pytest.mark.parametrize("bits,symmetric", [(2, True), (2, False), (3, True), (3, False), (4, True), (4, False),
                                            (8, True), (8, False)])
@pytest.mark.parametrize("layout", sorted(_LAYOUTS))
def test_state_matches_oracle(layout, bits, symmetric):
    from vsiquantization_b200 import ops
    shape, ch_axis, cl = _LAYOUTS[layout]
    C = 1 if ch_axis is None else shape[ch_axis]
    st = ops.new_percentile_state(C, 2048, torch.device("cuda"))
    st_o = hist_oracle.new_state(C, 2048)
    for call in range(3):
        xn = _salted(shape, ch_axis, 100 * bits + int(symmetric), call)
        x = _cuda(xn, cl)
        ops.slow_path_counters(reset=True)
        _run_both(x, xn, ch_axis, st, st_o, 2048, 128, bits, symmetric)
        assert ops.slow_path_counters()["layout_conversion_copies"] == 0  # NHWC read in place


@pytest.mark.parametrize("n_bins", [256, 512, 4096])
@pytest.mark.parametrize("layout", ["tensor", "nhwc"])
def test_bin_counts_and_start_bins(layout, n_bins):
    from vsiquantization_b200 import ops
    shape, ch_axis, cl = _LAYOUTS[layout]
    C = 1 if ch_axis is None else shape[ch_axis]
    for start_bin in (1, 8, n_bins // 2, n_bins):
        st = ops.new_percentile_state(C, n_bins, torch.device("cuda"))
        st_o = hist_oracle.new_state(C, n_bins)
        for call in range(3):
            xn = _salted(shape, ch_axis, n_bins + start_bin, call)
            _run_both(_cuda(xn, cl), xn, ch_axis, st, st_o, n_bins, start_bin, 4, False)
        if start_bin == n_bins:  # the min/max result
            s = st.cpu().numpy()
            assert _same_bits(s[:, 8:10], s[:, 0:2])


def test_determinism_order_and_split_independence():
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(3)
    xs = (rng.standard_normal((12, 16, 20, 20)) * rng.uniform(0.01, 50, (12, 1, 1, 1))).astype(np.float32)
    xs[4, 2, 3, 3] = 900.0
    dev = torch.device("cuda")

    def run(pieces, ch_axis):
        C = 16 if ch_axis == 1 else 1
        st = ops.new_percentile_state(C, 2048, dev)
        d = torch.empty(C, 2049, dtype=torch.float64, device=dev)
        for p in pieces:
            ops.hist_observe(_cuda(np.ascontiguousarray(xs[p]), True), ch_axis, st, 2048, 100.0, 8, True)
            ops.hist_entropy_clip(st, 2048, 128, 8, True, 1e-8, divergences=d)
        return st.cpu().numpy(), d.cpu().numpy()

    for ch_axis in (None, 1):
        ref, dref = run([slice(i, i + 1) for i in range(12)], ch_axis)
        cols = [0, 1, 2, 3] + list(range(8, ref.shape[1]))  # 4..7 count and average per call: they depend on the split
        for pieces in ([slice(i, i + 1) for i in (11, 3, 7, 0, 5, 9, 1, 10, 2, 8, 6, 4)],
                       [slice(0, 5), slice(5, 6), slice(6, 12)], [slice(8, 12), slice(0, 8)]):
            st, d = run(pieces, ch_axis)
            assert _same_bits(st[:, cols], ref[:, cols]) and _same_bits(d, dref)
        st, d = run([slice(i, i + 1) for i in range(12)], ch_axis)  # a repeat: identical bits
        assert _same_bits(st, ref) and _same_bits(d, dref)


def test_red_zone():
    """Nothing outside the state and the divergence rows changes; the workspace header stays zero and nothing past the
    workspace's size is touched."""
    from vsiquantization_b200 import _lib, ops
    B, C = 512, 16
    W = 12 + 2 * B
    xn = _salted((4, C, 20, 20), 1, 5, 0)
    st0 = ops.new_percentile_state(C, B, torch.device("cuda"))
    ops.hist_observe(_cuda(xn, True), 1, st0, B, 100.0, 4, False)
    sentinel = -1234.5
    buf = torch.full((C * W + 8192,), sentinel, dtype=torch.float64, device="cuda")
    st = buf[4096:4096 + C * W]
    st.copy_(st0.reshape(-1))
    dbuf = torch.full((C * (B + 1) + 2048,), sentinel, dtype=torch.float64, device="cuda")
    d = dbuf[1024:1024 + C * (B + 1)]
    nbytes = _lib.lib.vsiq_hist_entropy_workspace_bytes(C, B)
    ws = torch.full((nbytes + 4096,), 0x5A, dtype=torch.uint8, device="cuda")  # stale records included
    ws[:256] = 0
    ws[nbytes:] = 0xA5
    rc = _lib.lib.vsiq_hist_entropy_clip(st.data_ptr(), C, B, 16, 4, 0, 1e-8, d.data_ptr(), ws.data_ptr(), nbytes,
                                         torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask[4096:4096 + C * W] = False
    assert bool((buf[mask] == sentinel).all())
    dmask = torch.ones_like(dbuf, dtype=torch.bool)
    dmask[1024:1024 + C * (B + 1)] = False
    assert bool((dbuf[dmask] == sentinel).all()) and not bool((d == sentinel).any())
    assert bool((ws[:256] == 0).all()) and bool((ws[nbytes:] == 0xA5).all())
    st_o = hist_oracle.new_state(C, B)
    hist_oracle.observe(xn, 1, st_o, B, 100.0, 4, False)
    d_o = hist_oracle.entropy_clip(st_o, B, 16, 4, False)
    _check_call(st.reshape(C, W), d.reshape(C, B + 1), st_o, d_o, 4, False)


def test_outlier_is_clipped():
    from vsiquantization_b200.observers.entropy import EntropyObserver
    from vsiquantization_b200.observers.minmax import MinMaxObserver
    gen = torch.Generator(device="cuda").manual_seed(6)
    x = torch.randn(4, 64, 32, 32, device="cuda", generator=gen).contiguous(memory_format=torch.channels_last)
    x[1, 7, 3, 3] = 20.0
    a, b = MinMaxObserver(True, 4), EntropyObserver(True, 4)
    a.observe(x)
    b.observe(x)
    s_mm, _ = a.get_scale_zero_point()
    s_e, _ = b.get_scale_zero_point()
    assert b.max_val == 20.0 and s_e < s_mm
    assert -20.0 < float(b.state[0, 8]) and float(b.state[0, 9]) < 20.0
    d = b.divergences()
    i = _last_argmin(d.cpu().numpy()[0])
    e = int(max(float(b.state[0, 10]), float(b.state[0, 11])))
    assert d.shape == (1, 2049) and float(b.state[0, 9]) == i * 2.0 ** e


# ---------------------------------------------------------------------------------------------- model level (YOLOv8n)
def test_yolov8n_start_bin_n_bins_scales_equal_minmax(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    a = _yolo(FuseConfig(bits_w=8, bits_a=4))
    b = _yolo(FuseConfig(bits_w=8, bits_a=4, observer_a_name="EntropyObserver"))
    for _, mgr in _act_managers(b):
        assert type(mgr.observer).__name__ == "EntropyObserver" and mgr.observer.num_bits == 4
        mgr.observer.start_bin = mgr.observer.n_bins
    for _, mgr in _act_managers(a):
        mgr.observer.num_bits = 4  # the MinMax observer at the quantiser's width, as the entropy observer runs
    batches = _batches(2)
    for model in (a, b):
        _calibrate(model, batches)
    ma, mb = _act_managers(a), _act_managers(b)
    assert len(ma) == 57
    for (n, qa), (_, qb) in zip(ma, mb):
        assert torch.equal(qa.observer.state[:, 2:4], qb.observer.state[:, 2:4]), n


def test_yolov8n_activation_states_equal_the_oracle_survive_a_checkpoint_and_a_sync(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.parallel import sync_observers
    cfg = FuseConfig(bits_w=8, bits_a=4, observer_a_name="EntropyObserver")
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
            hist_oracle.observe(x, None, st_o, 2048, 100.0, 4, True)
        d_o = hist_oracle.entropy_clip(st_o, 2048, 128, 4, True)
        _check_call(mgr.observer.state, mgr.observer.divergences(), st_o, d_o, 4, True)
    # mid-calibration checkpoint into a freshly fused model, then the rest of the data: the uninterrupted result
    fresh = _yolo(cfg)
    fresh.load_state_dict(saved)
    _calibrate(fresh, batches[2:])
    for (n, q1), (_, q2) in zip(_act_managers(model), _act_managers(fresh)):
        st1, st2 = q1.observer.state.cpu().numpy(), q2.observer.state.cpu().numpy()
        cols = [0, 1, 2, 3, 4] + list(range(8, st1.shape[1]))
        assert _same_bits(st1[:, cols], st2[:, cols]), n
        np.testing.assert_allclose(st1[:, 5:8], st2[:, 5:8], rtol=1e-12, atol=0)
    # one process: the merge changes nothing and after_merge's search lands on the same state
    before = [q.observer.state.clone() for _, q in _act_managers(model)]
    assert sync_observers(model) > 0
    for (n, q), b in zip(_act_managers(model), before):
        assert torch.equal(q.observer.state, b), n
