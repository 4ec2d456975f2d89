"""Percentile observer without a GPU: the NumPy oracle (hist_oracle/) against an independent restatement by sorting,
exactness of coarsening and order independence, the ABI entries, constructor validation, manager wiring, checkpoints at
W = 4108 and a two-rank state sync (gloo)."""
import numpy as np
import pytest
import torch

import hist_oracle
from test_parallel_gloo import _run


def _restated_clip(values, percentile, n_bins):
    """(lo, hi) from the definition, by sorting: the histogram at the final exponents holds every finite value, and the
    smallest j with at most T values in bins above j is the bin of the (T+1)-th largest value (0 if there are <= T)."""
    v = values[np.isfinite(values)].astype(np.float64)
    run_min, run_max = min(0.0, float(v.min())), max(0.0, float(v.max()))
    N = v.size
    T = int(np.floor((1.0 - percentile / 100.0) * float(N)))
    out = []
    for side, mag, m in ((0, -v[v < 0], -run_min), (1, v[v >= 0], run_max)):
        e = hist_oracle.exponent(m, n_bins)
        desc = np.sort(mag)[::-1]
        j = int(np.floor(desc[T] / 2.0 ** e)) if desc.size > T else 0
        out.append((j + 1) * 2.0 ** e)
    return max(run_min, -out[0]), min(run_max, out[1])


def _inputs(kind, rng, n):
    if kind == "random":
        return (rng.standard_normal(n) * 3).astype(np.float32)
    if kind == "heavy":
        return (rng.standard_t(1.5, n) * 0.01).astype(np.float32)
    x = (rng.standard_normal(n) * 1e-40).astype(np.float32)  # denormals
    x[::7] = 0.0
    x[::11] = -0.0
    return x


@pytest.mark.parametrize("percentile", [99.0, 99.9, 99.99, 100.0])
@pytest.mark.parametrize("kind", ["random", "heavy", "denormal"])
@pytest.mark.parametrize("n_bins", [256, 2048, 4096])
def test_oracle_clip_equals_sorting_restatement(kind, percentile, n_bins):
    rng = np.random.default_rng(len(kind) * 10000 + n_bins)
    calls = [_inputs(kind, rng, 3000) * np.float32(s) for s in (1.0, 3.0, 0.5)]
    st = hist_oracle.new_state(1, n_bins)
    for x in calls:
        hist_oracle.observe(x, None, st, n_bins, percentile, 4, False)
    lo, hi = _restated_clip(np.concatenate(calls), percentile, n_bins)
    assert (st[0, 8], st[0, 9]) == (lo, hi)
    assert (st[0, 2], st[0, 3]) == hist_oracle.qparams(lo, hi, 4, False)
    assert st[0, 12:].sum() == 9000
    if percentile == 100.0:  # the min/max result
        assert (lo, hi) == (st[0, 0], st[0, 1])


def test_coarsening_then_adding_equals_binning_at_the_final_exponent():
    rng = np.random.default_rng(1)
    for trial in range(20):
        B = int(rng.choice([256, 1024, 4096]))
        calls = [(rng.standard_normal(int(rng.integers(1, 500))) * 10.0 ** rng.uniform(-30, 30)).astype(np.float32)
                 for _ in range(int(rng.integers(1, 6)))]
        st = hist_oracle.new_state(1, B)
        for x in calls:
            hist_oracle.observe(x, None, st, B, 99.9, 8, True)
        allv = np.concatenate(calls)
        for side, sel, col in ((0, allv < 0, 10), (1, allv >= 0, 11)):
            e = int(st[0, col])
            assert e == hist_oracle.exponent(-st[0, 0] if side == 0 else st[0, 1], B)
            want = np.bincount(hist_oracle.bins(allv[sel], e), minlength=B)
            assert np.array_equal(st[0, 12 + side * B:12 + (side + 1) * B], want), trial


def test_state_is_independent_of_call_order_and_split():
    rng = np.random.default_rng(2)
    x = (rng.standard_normal((6, 8, 50)) * rng.uniform(0.01, 100, (6, 1, 1))).astype(np.float32)
    x[2, 3, 7] = 1e4
    ref = hist_oracle.new_state(8, 512)
    for i in range(6):
        hist_oracle.observe(x[i:i + 1], 1, ref, 512, 99.0, 4, True)
    for order in ([5, 4, 3, 2, 1, 0], [3, 0, 5, 1, 4, 2]):
        st = hist_oracle.new_state(8, 512)
        for i in order:
            hist_oracle.observe(x[i:i + 1], 1, st, 512, 99.0, 4, True)
        assert np.array_equal(st[:, :4], ref[:, :4]) and np.array_equal(st[:, 8:], ref[:, 8:])
    st = hist_oracle.new_state(8, 512)
    for sl in (slice(4, 6), slice(0, 1), slice(1, 4)):  # other call sizes
        hist_oracle.observe(x[sl], 1, st, 512, 99.0, 4, True)
    assert np.array_equal(st[:, :4], ref[:, :4]) and np.array_equal(st[:, 8:], ref[:, 8:])


def test_nan_calls_are_skipped_and_inf_freezes():
    st = hist_oracle.new_state(1, 256)
    hist_oracle.observe(np.array([1.0, -2.0, 3.0], np.float32), None, st, 256, 50.0, 8, True)
    before = st.copy()
    hist_oracle.observe(np.array([np.nan, 100.0], np.float32), None, st, 256, 50.0, 8, True)
    assert np.array_equal(st[:, [0, 1, 8, 9, 10, 11]], before[:, [0, 1, 8, 9, 10, 11]])
    assert np.array_equal(st[:, 12:], before[:, 12:])
    hist_oracle.observe(np.array([np.inf, 5.0], np.float32), None, st, 256, 50.0, 8, True)
    assert st[0, 1] == np.inf and (st[0, 8], st[0, 9]) == (st[0, 0], st[0, 1])
    assert np.array_equal(st[:, 10:], before[:, 10:])  # frozen


def test_an_outlier_is_clipped():
    rng = np.random.default_rng(3)
    x = rng.standard_normal(100000).astype(np.float32)
    x[17] = 1000.0
    st = hist_oracle.new_state(1)
    hist_oracle.observe(x, None, st, 2048, 99.99, 4, True)
    assert st[0, 1] == 1000.0 and st[0, 9] < 10.0
    assert st[0, 2] < 0.01 * hist_oracle.qparams(st[0, 0], st[0, 1], 4, True)[0]  # min/max: 1000 / 7


def test_abi_declares_and_exports_the_histogram():
    from vsiquantization_b200 import _lib
    for name in ("vsiq_hist_observe", "vsiq_hist_observe_workspace_bytes", "vsiq_hist_clip"):
        assert name in _lib.EXPORTED and hasattr(_lib.lib, name)
    lay = _lib.Layout(64, 32, 1)
    assert _lib.lib.vsiq_hist_observe_workspace_bytes(lay, 2048) == 256 + 32 * 2 * 2048 * 4
    for bad in (0, 128, 1000, 8192):
        assert _lib.lib.vsiq_hist_observe_workspace_bytes(lay, bad) == 0
    assert _lib.lib.vsiq_hist_observe(None, lay, None, None, 2048, 99.99, 4, 1, 1e-8, None, 0, None) == -1
    assert _lib.lib.vsiq_hist_clip(None, 4, 2048, 99.99, 4, 1, 1e-8, None) == -1
    with open(__import__("os").path.join(__import__("os").path.dirname(__file__), "..", "include", "vsiq.h")) as f:
        h = f.read()
    assert all(name + "(" in h for name in ("vsiq_hist_observe", "vsiq_hist_observe_workspace_bytes", "vsiq_hist_clip"))


def test_constructor_validation_and_manager_wiring():
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.observers.percentile import PercentileObserver
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    for kw in ({"n_bins": 128}, {"n_bins": 3000}, {"n_bins": 8192}, {"percentile": 0.0}, {"percentile": 100.5},
               {"percentile": -1}):
        with pytest.raises(ValueError):
            PercentileObserver(**kw)
    o = PercentileObserver(n_bins=256, percentile=100)
    assert o.n_bins == 256 and o.percentile == 100.0 and o.state_width == 12 + 512
    with pytest.raises(ValueError):
        o.set_percentile(0)
    m = M("UniformQuantizer", "PercentileObserver", 4, True)
    assert isinstance(m.observer, PercentileObserver) and m.observer.num_bits == 4 and m.observer.percentile == 99.99
    assert getattr(m.observer, "observe_epilogue", None) is None
    assert FuseConfig(observer_a_name="PercentileObserver").observer_a_name == "PercentileObserver"
    import vsiquantization_b200.dropin as dropin
    assert "PercentileObserver" not in dropin.install_plugins({})
    assert dropin.install_plugins({}, percentile_observer=True)["PercentileObserver"] is PercentileObserver
    assert "observers.percentile" in dropin._TIER2
    with pytest.raises(ValueError):  # a min/max state has no histogram
        PercentileObserver().load_state(torch.zeros(3, 8, dtype=torch.float64))


def test_checkpoint_packs_the_histogram_as_version_3():
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    a = M("UniformQuantizer", "PercentileObserver", 4, False, ch_axis=1)
    st = torch.from_numpy(hist_oracle.new_state(3, 2048))
    st[:, 12:] = torch.arange(3 * 4096, dtype=torch.float64).reshape(3, 4096)
    a.observer.load_state(st)
    a._calibrated = True
    a._invalidate()
    blob = a.get_extra_state()
    assert blob[1].item() == 3.0 and blob[13].item() == 4108.0 and blob.numel() == 14 + 3 * 4108 + 1
    b = M("UniformQuantizer", "PercentileObserver", 4, False, ch_axis=1)
    b.set_extra_state(blob)
    assert torch.equal(b.observer.state.cpu(), st) and b._calibrated
    with pytest.raises(ValueError):  # another width: another n_bins
        M("UniformQuantizer", "MinMaxObserver", 4, False, ch_axis=1).set_extra_state(blob)


def _batches():
    rng = np.random.default_rng(5)
    out = [(rng.standard_normal((2, 3, 300)) * (0.5 + i)).astype(np.float32) for i in range(5)]
    out[3][0, 1, 7] = 40.0
    out[1][1, 2, :] = np.maximum(out[1][1, 2, :], 0)
    return out


def _pct_sync_case(rank, world):
    from vsiquantization_b200.parallel import reduce_percentile_states
    st = hist_oracle.new_state(3, 256)
    for b in _batches()[rank::world]:
        hist_oracle.observe(b, 1, st, 256, 99.0, 4, False)
    t = torch.tensor(st)
    reduce_percentile_states(t, 256)
    return t.numpy()


def test_percentile_state_sync_two_ranks_equals_the_union():
    res = _run(_pct_sync_case)
    for r in res:
        hist_oracle.clip(r, 256, 99.0, 4, False)  # what ops.hist_clip does on the device after the sync
    assert np.array_equal(res[0].view(np.uint64), res[1].view(np.uint64))  # every rank: the same bits
    union = hist_oracle.new_state(3, 256)
    for b in _batches():
        hist_oracle.observe(b, 1, union, 256, 99.0, 4, False)
    got = res[0]
    assert np.array_equal(got[:, 0:2], union[:, 0:2]) and np.array_equal(got[:, 4], union[:, 4])
    assert np.array_equal(got[:, 10:], union[:, 10:])  # exponents and counts: the histogram of the union
    assert np.array_equal(got[:, [2, 3, 8, 9]], union[:, [2, 3, 8, 9]])
