"""Entropy observer without a GPU: the NumPy oracle's search (hist_oracle.entropy_clip) against a literal restatement of
pytorch-quantization's _compute_amax_entropy loop (linspace / digitize, stride 1), the fold and the cases that keep the
running range, the ABI entries, constructor validation, manager / FuseConfig / dropin wiring, checkpoints and a two-rank
state sync (gloo)."""
import ctypes
import os

import numpy as np
import pytest
import scipy.stats
import torch

import hist_oracle
from test_parallel_gloo import _run


def _literal_entropy(calib_hist, nq, start, stop):
    """pytorch-quantization's loop, restated with its linspace / digitize chunking and scipy's entropy, over thresholds
    start..stop: (divergences, last argmin)."""
    bins = calib_hist.astype(np.int64).copy()
    bins[0] = bins[1]
    divergences = []
    for i in range(start, stop + 1):
        space = np.linspace(0, i, num=nq + 1)
        digitized = np.digitize(range(i), space) - 1
        digitized[bins[:i] == 0] = -1
        keep = digitized != -1
        density_counts = np.zeros(nq, dtype=np.float64)
        np.add.at(density_counts, digitized[keep], bins[:i][keep])
        counter = np.bincount(digitized[keep], minlength=nq)
        density_counts[counter > 0] /= counter[counter > 0]
        new_density = np.zeros(i, dtype=np.float64)
        new_density[keep] = density_counts[digitized[keep]]
        with np.errstate(all="ignore"):
            new_density /= new_density.sum()
            reference = bins[:i].astype(np.float64)
            reference[-1] += np.sum(bins[i:])
            reference /= reference.sum()
            divergences.append(scipy.stats.entropy(reference, new_density))
    d = np.array(divergences)
    d[np.isnan(d)] = np.inf
    return d, start + len(d) - 1 - int(np.argmin(d[::-1]))


def _data(kind, rng, n):
    if kind == "relu":
        x = np.maximum(rng.standard_normal(n), 0.0)
    elif kind == "two_sided":
        x = rng.standard_normal(n)
        m = np.abs(x).max()
        x[0], x[1] = -m, m  # the same extent on both sides: one exponent
    else:  # a heavy outlier, 15 sigma out
        x = rng.standard_normal(n) * 2.0
        x[7] = 30.0
    return x.astype(np.float32)


# (nq, kind, bits, symmetric): nq = 2^(bits - 1), or 2^bits for an asymmetric quantiser of a ReLU output
_CASES = [(2, "two_sided", 2, True), (4, "relu", 2, False), (8, "two_sided", 4, True), (16, "relu", 4, False),
          (16, "outlier", 5, True), (128, "two_sided", 8, True), (128, "outlier", 8, False), (256, "relu", 8, False)]


@pytest.mark.parametrize("n_bins", [256, 2048, 4096])
@pytest.mark.parametrize("nq,kind,bits,symmetric", _CASES)
def test_oracle_equals_literal_restatement(nq, kind, bits, symmetric, n_bins):
    rng = np.random.default_rng(nq * 10 + n_bins)
    x = _data(kind, rng, 50000)
    st = hist_oracle.new_state(1, n_bins)
    hist_oracle.observe(x, None, st, n_bins, 100.0, bits, symmetric)
    e = int(max(st[0, 10], st[0, 11]))
    assert hist_oracle.entropy_levels(st[0, 0], bits, symmetric) == nq
    calib_hist = np.bincount(hist_oracle.bins(x, e), minlength=n_bins)  # |x| at the one exponent
    start_bin = 128 if n_bins > 256 else 16
    div = hist_oracle.entropy_clip(st, n_bins, start_bin, bits, symmetric)[0]
    n_used = int(np.flatnonzero(calib_hist)[-1]) + 1
    if max(start_bin, nq) > n_used:  # no candidate (nq = 256 levels in 256 bins): the running range
        assert np.isnan(div).all() and (st[0, 8], st[0, 9]) == (st[0, 0], st[0, 1])
        return
    lit, i_lit = _literal_entropy(calib_hist, nq, max(start_bin, nq), n_used)
    ours = div[max(start_bin, nq):n_used + 1]
    assert np.array_equal(np.isinf(ours), np.isinf(lit))
    fin = np.isfinite(lit)
    np.testing.assert_allclose(ours[fin], lit[fin], rtol=1e-9, atol=1e-12)
    amax = i_lit * 2.0 ** e
    assert (st[0, 8], st[0, 9]) == (max(st[0, 0], -amax), min(st[0, 1], amax))
    assert (st[0, 2], st[0, 3]) == hist_oracle.qparams(st[0, 8], st[0, 9], bits, symmetric)
    assert np.isnan(div[:max(start_bin, nq)]).all() and np.isnan(div[n_used + 1:]).all()
    if kind == "outlier" and n_bins >= 2048:  # the outlier is clipped (at 256 bins the bulk fills only 17)
        assert st[0, 9] < st[0, 1]


def test_fold_with_different_exponents():
    rng = np.random.default_rng(3)
    x = np.concatenate([-rng.uniform(0, 0.01, 3000), rng.uniform(0, 100, 3000)]).astype(np.float32)
    st = hist_oracle.new_state(1, 512)
    hist_oracle.observe(x, None, st, 512, 100.0, 4, True)
    assert st[0, 10] < st[0, 11]
    H, e = hist_oracle.entropy_fold(st[0], 512)
    want = np.bincount(hist_oracle.bins(x, e), minlength=512)
    want[0] = want[1]
    assert e == st[0, 11] and np.array_equal(H, want)
    before = st.copy()
    hist_oracle.entropy_clip(st, 512, 16, 4, True)
    assert np.array_equal(st[:, 10:], before[:, 10:])  # the counts are never modified


def test_cases_that_keep_the_running_range():
    # an all-zero channel, start_bin above n_used, a running range that is not finite
    st = hist_oracle.new_state(3, 256)
    rng = np.random.default_rng(4)
    x = rng.uniform(-1, 1, (2, 3, 500)).astype(np.float32)
    x[:, 0] = 0.0
    x[0, 1, :] *= 0.6  # channel 1: its top bins stay empty at the default exponent
    x[0, 1, 0] = 1.0
    x[0, 1, 1:] = np.clip(x[0, 1, 1:], -0.6, 0.6)
    x[1, 1, :] = 0.1
    x[1, 2, 3] = np.inf
    hist_oracle.observe(x, 1, st, 256, 100.0, 4, False)
    H, _ = hist_oracle.entropy_fold(st[1], 256)
    n_used = int(np.flatnonzero(H)[-1]) + 1
    assert n_used < 256
    for start_bin in (n_used + 1, 256):
        s = st.copy()
        div = hist_oracle.entropy_clip(s, 256, start_bin, 4, False)
        assert np.isnan(div).all()
        assert np.array_equal(s[:, 8:10], s[:, 0:2])
        for c in range(3):
            assert (s[c, 2], s[c, 3]) == hist_oracle.qparams(s[c, 0], s[c, 1], 4, False)
    assert st[2, 1] == np.inf


def test_abi_declares_and_exports_the_search():
    from vsiquantization_b200 import _lib
    names = ("vsiq_hist_entropy_clip", "vsiq_hist_entropy_workspace_bytes")
    for name in names:
        assert name in _lib.EXPORTED and hasattr(_lib.lib, name)
    with open(os.path.join(os.path.dirname(__file__), "..", "include", "vsiq.h")) as f:
        h = f.read()
    assert all(name + "(" in h for name in names)
    wsb = _lib.lib.vsiq_hist_entropy_workspace_bytes
    assert wsb(32, 2048) == 256 + 32 * 17 * 16  # one 16-byte record per scoring CTA, at most 17 CTAs per channel
    for C, B in ((0, 2048), (4, 128), (4, 1000), (4, 8192)):
        assert wsb(C, B) == 0
    fake = ctypes.c_void_p(4096)  # never dereferenced: the arguments are rejected first
    clip = _lib.lib.vsiq_hist_entropy_clip
    for B, start, bits in ((128, 16, 4), (1000, 16, 4), (8192, 16, 4), (2048, 0, 4), (2048, 2049, 4), (2048, 128, 1),
                           (2048, 128, 9)):
        assert clip(fake, 4, B, start, bits, 1, 1e-8, None, fake, 1 << 20, None) == -1
    assert clip(None, 4, 2048, 128, 4, 1, 1e-8, None, fake, 1 << 20, None) == -1


def test_constructor_validation_and_wiring():
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.observers.entropy import EntropyObserver
    from vsiquantization_b200.observers.percentile import HistogramObserver, PercentileObserver
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    for kw in ({"n_bins": 128}, {"n_bins": 3000}, {"n_bins": 8192}, {"start_bin": 0}, {"start_bin": 2049},
               {"n_bins": 256, "start_bin": 257}, {"num_bits": 1}, {"num_bits": 9}):
        with pytest.raises(ValueError):
            EntropyObserver(**kw)
    o = EntropyObserver(n_bins=256, start_bin=256)
    assert o.n_bins == 256 and o.start_bin == 256 and o.state_width == 12 + 512
    assert isinstance(o, HistogramObserver) and not isinstance(o, PercentileObserver)
    assert not hasattr(o, "set_percentile") and not hasattr(o, "percentile")
    m = M("UniformQuantizer", "EntropyObserver", 4, True)
    assert isinstance(m.observer, EntropyObserver) and m.observer.num_bits == 4 and m.observer.start_bin == 128
    assert m.observer.n_bins == 2048 and getattr(m.observer, "observe_epilogue", None) is None
    assert M("UniformQuantizer", "EntropyObserver", 3, False, ch_axis=1).observer.ch_axis == 1
    assert FuseConfig(observer_a_name="EntropyObserver").observer_a_name == "EntropyObserver"
    assert EntropyObserver().sync_key() == PercentileObserver().sync_key() == ("percentile", 2048)
    import vsiquantization_b200.dropin as dropin
    assert "EntropyObserver" not in dropin.install_plugins({})
    assert dropin.install_plugins({}, entropy_observer=True)["EntropyObserver"] is EntropyObserver
    assert "observers.entropy" in dropin._TIER2
    with pytest.raises(ValueError):  # a min/max state has no histogram
        EntropyObserver().load_state(torch.zeros(3, 8, dtype=torch.float64))


def test_fuse_config_yaml_key(tmp_path):
    from vsiquantization_b200.modules.fuse_config import load_fuse_config_from_yaml
    p = tmp_path / "cfg.yaml"
    p.write_text("default:\n  bits_a: 4\n  observer_a_name: EntropyObserver\n"
                 "layers:\n  head.*:\n    observer_a_name: PercentileObserver\n")
    mgr = load_fuse_config_from_yaml(str(p))
    assert mgr.get_config_for_layer("net.p1.0").observer_a_name == "EntropyObserver"
    assert mgr.get_config_for_layer("head.box.0").observer_a_name == "PercentileObserver"


def test_checkpoint_round_trip_and_percentile_checkpoint():
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    st = torch.from_numpy(hist_oracle.new_state(3, 2048))
    st[:, 12:] = torch.arange(3 * 4096, dtype=torch.float64).reshape(3, 4096)
    for src in ("EntropyObserver", "PercentileObserver"):
        a = M("UniformQuantizer", src, 4, False, ch_axis=1)
        a.observer.load_state(st)
        a._calibrated = True
        a._invalidate()
        blob = a.get_extra_state()
        assert blob[1].item() == 3.0 and blob[13].item() == 4108.0 and blob.numel() == 14 + 3 * 4108 + 1
        b = M("UniformQuantizer", "EntropyObserver", 4, False, ch_axis=1)
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


def _entropy_observe(x, st):
    hist_oracle.observe(x, 1, st, 256, 100.0, 4, False)
    hist_oracle.entropy_clip(st, 256, 16, 4, False)


def _entropy_sync_case(rank, world):
    from vsiquantization_b200.parallel import reduce_percentile_states
    st = hist_oracle.new_state(3, 256)
    for b in _batches()[rank::world]:
        _entropy_observe(b, st)
    t = torch.tensor(st)
    reduce_percentile_states(t, 256)
    return t.numpy()


def test_entropy_state_sync_two_ranks_equals_the_union():
    res = _run(_entropy_sync_case)
    for r in res:
        hist_oracle.entropy_clip(r, 256, 16, 4, False)  # what after_merge does on the device
    assert np.array_equal(res[0].view(np.uint64), res[1].view(np.uint64))  # every rank: the same bits
    union = hist_oracle.new_state(3, 256)
    for b in _batches():
        _entropy_observe(b, union)
    got = res[0]
    assert np.array_equal(got[:, 0:2], union[:, 0:2]) and np.array_equal(got[:, 4], union[:, 4])
    assert np.array_equal(got[:, 10:], union[:, 10:])
    assert np.array_equal(got[:, [2, 3, 8, 9]], union[:, [2, 3, 8, 9]])
