"""MSE observer without a GPU: the C oracle of the clipping-range search against a NumPy restatement over the pinned
fake-quant oracle, its K = 1 and clipping cases, the ABI entries, the two-rank state sync (gloo) and checkpoints."""
import numpy as np
import pytest
import torch

import mse_oracle
import oracle
from test_parallel_gloo import _run


def _numpy_errors(x, ch_axis, lo, hi, bits, symmetric, K, eps=1e-8):
    """E[c,k] by the definition: oracle.fake_quant_fwd (the pinned fq) per candidate, fp64 differences and squares."""
    outer, C, inner = oracle.layout(x.shape, ch_axis)
    qmin, qmax = (-(1 << (bits - 1)), (1 << (bits - 1)) - 1) if symmetric else (0, (1 << bits) - 1)
    xr = x.reshape(outer, C, inner)
    E = np.zeros((C, K))
    for c in range(C):
        xc = np.ascontiguousarray(xr[:, c, :]).reshape(-1)
        for k in range(1, K + 1):
            a = k / K
            s, z = oracle.qparams(a * lo[c], a * hi[c], bits, symmetric, eps)
            y = oracle.fake_quant_fwd(xc, s, z, qmin, qmax)
            d = y.astype(np.float64) - xc.astype(np.float64)
            E[c, k - 1] = np.sum(d * d)
    return E


@pytest.mark.parametrize("bits,symmetric", [(2, True), (3, False), (4, False), (8, True)])
@pytest.mark.parametrize("ch_axis", [None, 0, 1])
def test_oracle_errors_equal_numpy_restatement(bits, symmetric, ch_axis):
    rng = np.random.default_rng(bits * 7 + int(symmetric))
    x = (rng.standard_normal((3, 4, 5, 6)) * rng.uniform(0.1, 3, (1, 4, 1, 1))).astype(np.float32)
    x.reshape(-1)[5] = 9.0
    C = 1 if ch_axis is None else x.shape[ch_axis]
    st = mse_oracle.new_state(C)
    E, alpha = mse_oracle.search(x, ch_axis, st, bits, symmetric, 1e-8, 20)
    ref = _numpy_errors(x, ch_axis, st[:, 0], st[:, 1], bits, symmetric, 20)
    np.testing.assert_allclose(E, ref, rtol=1e-13, atol=0)
    best = np.array([np.flatnonzero(e == e.min()).max() + 1 for e in E]) / 20
    assert np.array_equal(alpha, best)


@pytest.mark.parametrize("bits,symmetric", [(2, True), (4, False), (8, True), (3, False)])
def test_one_candidate_is_the_minmax_observer(bits, symmetric):
    rng = np.random.default_rng(3)
    w = (rng.standard_normal((8, 3, 3, 3)) * 0.2).astype(np.float32)
    st = mse_oracle.new_state(8)
    for _ in range(2):  # repeated calls on the same tensor (weights while calibrating) keep the single-call result
        _, alpha = mse_oracle.search(w, 0, st, bits, symmetric, 1e-8, 1)
    assert np.all(alpha == 1.0)
    mm = oracle.minmax_stats(w, ch_axis=0)
    for c in range(8):
        lo, hi = min(mm[c, 0], 0.0), max(mm[c, 1], 0.0)
        assert (st[c, 0], st[c, 1], st[c, 8], st[c, 9]) == (lo, hi, lo, hi)
        assert (st[c, 2], st[c, 3]) == oracle.qparams(lo, hi, bits, symmetric)


def test_one_outlier_in_a_w2_channel_is_clipped():
    rng = np.random.default_rng(11)
    w = (rng.standard_normal((2, 4096)) * 0.05).astype(np.float32)
    w[0, 17] = 1.5  # one outlier: min/max would spend the whole 2-bit range on it
    st = mse_oracle.new_state(2)
    E, alpha = mse_oracle.search(w, 0, st, 2, True, 1e-8, 100)
    assert alpha[0] < 0.5 and E[0].min() < 0.5 * E[0, -1]
    assert st[0, 2] < 0.5 * oracle.qparams(st[0, 0], st[0, 1], 2, True)[0]
    # an all-zero channel keeps min/max (every candidate's scale is 0: non-finite error -> alpha = 1)
    z = np.zeros((1, 64), dtype=np.float32)
    st = mse_oracle.new_state(1)
    _, alpha = mse_oracle.search(z, 0, st, 4, False, 1e-8, 100)
    assert alpha[0] == 1.0 and (st[0, 2], st[0, 3]) == oracle.qparams(0.0, 0.0, 4, False)


def test_abi_declares_and_exports_the_search():
    from vsiquantization_b200 import _lib
    for name in ("vsiq_mse_search", "vsiq_mse_search_workspace_bytes"):
        assert name in _lib.EXPORTED and hasattr(_lib.lib, name)
    lay = _lib.Layout(64, 32, 1)
    assert _lib.lib.vsiq_mse_search_workspace_bytes(lay, 100) > 256
    assert _lib.lib.vsiq_mse_search_workspace_bytes(lay, 0) == 0 and _lib.lib.vsiq_mse_search_workspace_bytes(lay, 257) == 0
    assert _lib.lib.vsiq_mse_search(None, lay, None, None, 4, 1, 1e-8, 100, None, None, None, 0, None) == -1


def test_manager_builds_the_mse_observer_at_the_quantizer_width():
    from vsiquantization_b200.modules.fuse_config import FuseConfig
    from vsiquantization_b200.observers.mse import MSEObserver
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    m = M("UniformQuantizer", "MSEObserver", 4, False)
    assert isinstance(m.observer, MSEObserver) and m.observer.num_bits == 4 and m.observer.n_candidates == 100
    assert M("UniformQuantizer", "MinMaxObserver", 4, False).observer.num_bits == 8  # unchanged: always 8 bits
    assert M("UniformQuantizer", "LSQObserver", 2, True).observer.num_bits == 8
    assert FuseConfig(observer_w_name="MSEObserver").observer_w_name == "MSEObserver"
    assert getattr(m.observer, "observe_epilogue", None) is None
    import vsiquantization_b200.dropin as dropin
    assert dropin.install_plugins({}, mse_observer=True)["MSEObserver"] is MSEObserver
    assert "observers.mse" in dropin._TIER2


def _mse_sync_case(rank, world):
    from vsiquantization_b200.parallel import reduce_mse_states
    rng = np.random.default_rng(5)
    batches = [(rng.standard_normal((3, 400)) * (0.5 + i)).astype(np.float32) for i in range(5)]  # same on every rank
    for b in batches:
        b[1, 7 * (1 + len(b))] = 6.0
    st = mse_oracle.new_state(3)
    for b in batches[rank::world]:
        mse_oracle.search(b, 0, st, 2, True, 1e-8, 50)
    t = torch.tensor(st)
    reduce_mse_states(t)
    return t.numpy()


def test_mse_state_sync_two_ranks_matches_single_process():
    res = _run(_mse_sync_case)
    cols = [0, 1, 4, 5, 6, 7, 8, 9]  # scale / zero-point (2, 3) are recomputed from the means on the device afterwards
    assert np.array_equal(res[0][:, cols].view(np.uint64), res[1][:, cols].view(np.uint64))  # every rank: same bits
    rng = np.random.default_rng(5)
    batches = [(rng.standard_normal((3, 400)) * (0.5 + i)).astype(np.float32) for i in range(5)]
    for b in batches:
        b[1, 7 * (1 + len(b))] = 6.0
    # the union in one process: the same per-call choices (each call's candidates follow the running range of the rank
    # that saw it, so replay each rank's calls in its own state and merge by hand for the reference means)
    per_rank = []
    for r in range(2):
        st = mse_oracle.new_state(3)
        for b in batches[r::2]:
            mse_oracle.search(b, 0, st, 2, True, 1e-8, 50)
        per_rank.append(st)
    got = res[0]
    n = per_rank[0][:, 4] + per_rank[1][:, 4]
    assert np.array_equal(got[:, 0], np.minimum(per_rank[0][:, 0], per_rank[1][:, 0]))
    assert np.array_equal(got[:, 1], np.maximum(per_rank[0][:, 1], per_rank[1][:, 1]))
    assert np.array_equal(got[:, 4], n)
    for col in (8, 9):
        want = (per_rank[0][:, 4] * per_rank[0][:, col] + per_rank[1][:, 4] * per_rank[1][:, col]) / n
        np.testing.assert_allclose(got[:, col], want, rtol=1e-15, atol=0)
    # a single process whose calls made the same choices has the same running means to 1e-15
    alphas = []
    for r in range(2):
        st = mse_oracle.new_state(3)
        for b in batches[r::2]:
            _, a = mse_oracle.search(b, 0, st, 2, True, 1e-8, 50)
            alphas.append((a, st[:, 0].copy(), st[:, 1].copy()))
    m = np.zeros((3, 2))
    for i, (a, lo, hi) in enumerate(alphas):
        m[:, 0] += (a * lo - m[:, 0]) / (i + 1)
        m[:, 1] += (a * hi - m[:, 1]) / (i + 1)
    np.testing.assert_allclose(got[:, 8:10], m, rtol=1e-15, atol=0)


def _mgr_with_state(observer, width, C=3):
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    m = M("UniformQuantizer", observer, 4, False, ch_axis=0)
    st = torch.arange(C * width, dtype=torch.float64).reshape(C, width) / 7.0
    m.observer.load_state(st)
    m._calibrated = True
    m._invalidate()
    m.is_learning_scale, m.is_quantize = False, True
    return m


def test_checkpoint_round_trip_and_version_2_still_loads():
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M
    a = _mgr_with_state("MSEObserver", 10)
    blob = a.get_extra_state()
    assert blob[1].item() == 3.0 and blob[13].item() == 10.0 and blob.numel() == 14 + 30 + 1  # + calib_grad_scale
    b = M("UniformQuantizer", "MSEObserver", 4, False, ch_axis=0)
    b.set_extra_state(blob)
    assert torch.equal(b.observer.state.cpu(), a.observer.state.cpu()) and b._calibrated
    # min/max observers still write version 2, byte for byte the layout they always had
    mm = _mgr_with_state("MinMaxObserver", 8)
    v2 = mm.get_extra_state()
    assert v2[1].item() == 2.0 and v2.numel() == 13 + 24 + 1
    assert torch.equal(v2[13:37], mm.observer.state.cpu().reshape(-1))
    c = M("UniformQuantizer", "MinMaxObserver", 4, False, ch_axis=0)
    c.set_extra_state(v2)
    assert torch.equal(c.observer.state.cpu(), mm.observer.state.cpu())
    # a version-2 (min/max) checkpoint loaded into an MSE observer: the clipped means start at the range
    d = M("UniformQuantizer", "MSEObserver", 4, False, ch_axis=0)
    d.set_extra_state(v2)
    st = d.observer.state.cpu()
    assert st.shape == (3, 10) and torch.equal(st[:, :8], mm.observer.state.cpu()) and torch.equal(st[:, 8:], st[:, :2])
    with pytest.raises(ValueError):
        M("UniformQuantizer", "MinMaxObserver", 4, False, ch_axis=0).set_extra_state(blob)
