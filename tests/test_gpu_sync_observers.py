"""parallel.sync_observers end to end on the GPU: every observer kind the merge handles, states filled by the real
observe() kernels, then synchronised over a two-rank gloo group (both ranks on cuda:0) and, with no process group, at
world size 1.  After the merge every rank holds the state a single process would hold after seeing all batches (MinMax,
LSQ, percentile), the call-weighted clipped means (MSE) or the averaged running extrema (moving averages); the managers'
cached host qparams are gone, and the merge itself costs a fixed number of kernel launches."""
import os
import pickle
import tempfile

import numpy as np
import pytest
import torch

from test_parallel_gloo import _run

pytestmark = pytest.mark.gpu

N_BATCHES = 4
# (name, observer, quantiser bits, symmetric, ch_axis, observer keyword arguments, input shape, channels_last)
SPECS = [
    ("mm_t", "MinMaxObserver", 8, False, None, {}, (2, 8, 6, 6), False),
    ("mm_c", "MinMaxObserver", 8, True, 0, {}, (8, 4, 3, 3), False),
    ("lsq", "LSQObserver", 8, True, None, {}, (3, 50), False),
    ("mse", "MSEObserver", 4, True, 0, {}, (8, 4, 3, 3), False),
    ("pct256", "PercentileObserver", 4, False, 1, {"n_bins": 256, "percentile": 99.0}, (2, 8, 6, 6), True),
    ("pct2048", "PercentileObserver", 4, True, None, {"n_bins": 2048}, (4, 400), False),
    ("ema_t", "MovingAverageMinMaxObserver", 8, False, None, {}, (2, 8, 6, 6), False),
    ("ema_c", "MovingAveragePerChannelMinMaxObserver", 8, True, 0, {}, (8, 4, 3, 3), False),
]
# launches inside sync_observers: one qparams_from_minmax for the MinMax / LSQ rows, one for the MSE rows, one hist_clip
# per percentile observer; moving averages recompute their qparams with torch ops
SYNC_LAUNCHES = 1 + 1 + 2
ROWS = 1 + 8 + 1 + 8 + 8 + 1 + 1 + 8


def _batches():
    """The same seeded inputs in every process: one tensor per observer per batch, on the host."""
    g = torch.Generator().manual_seed(1234)
    out = []
    for i in range(N_BATCHES):
        b = {}
        for name, *_, shape, _cl in SPECS:
            x = torch.randn(shape, generator=g) * (0.5 + i)
            x.view(-1)[7 * (i + 1)] = 6.0 * (i + 1)  # an outlier the clipping observers should drop
            b[name] = x
        out.append(b)
    return out


def _model():
    from vsiquantization_b200.quantizers.quantization_manager import QuantizationManager as M

    class Layer(torch.nn.Module):
        def __init__(self, mgr):
            super().__init__()
            self.activation_quantizer = mgr

    layers = []
    for name, obs, bits, sym, ch_axis, kw, *_ in SPECS:
        m = M("UniformQuantizer", obs, bits, sym, is_learning_scale=False, ch_axis=ch_axis)
        if kw:  # the registry builds (symmetric, bits): set the observer's own options here
            o = type(m.observer)(sym, m.observer.num_bits, ch_axis=ch_axis, **kw)
            o._on_change = m._invalidate
            m.observer = o
        layers.append(Layer(m))
    return torch.nn.Sequential(*layers)


def _sync_case(rank, world):
    """Observe this rank's shard through the managers, sync, and report states before / after (host, fp64)."""
    from vsiquantization_b200 import _lib
    from vsiquantization_b200.parallel import sync_observers
    torch.cuda.set_device(0)
    model = _model()
    mgrs = {name: layer.activation_quantizer for (name, *_), layer in zip(SPECS, model)}
    for b in _batches()[rank::world]:
        for name, *_, cl in SPECS:
            x = b[name].cuda()
            if cl:
                x = x.contiguous(memory_format=torch.channels_last)
            mgrs[name].collect_qparameter(x)
    for m in mgrs.values():
        m.scale  # noqa: B018  (fill the host cache the sync must drop)
    before = {n: m.observer.state.cpu().numpy() for n, m in mgrs.items()}
    l0 = _lib.launch_count
    rows = sync_observers(model)
    launches = _lib.launch_count - l0
    after = {n: m.observer.state.cpu().numpy() for n, m in mgrs.items()}
    dropped = all("scale" not in m.__dict__ and m.observer._host is None for m in mgrs.values())
    scales = {n: torch.as_tensor(m.scale, dtype=torch.float64).reshape(-1).cpu().numpy() for n, m in mgrs.items()}
    return rank, rows, launches, before, after, dropped, scales


def _sync_rank(rank, world):
    """_sync_case in a spawned rank: the result goes through a file (a queue's pipe holds only 64 KB until read)."""
    fd, path = tempfile.mkstemp(suffix=".pkl")
    with os.fdopen(fd, "wb") as f:
        pickle.dump(_sync_case(rank, world), f)
    return path


def _collect(paths):
    out = []
    for path in paths:
        with open(path, "rb") as f:
            out.append(pickle.load(f))
        os.remove(path)
    return sorted(out, key=lambda r: r[0])  # the queue hands results back in arrival order


def _spec(name):
    return next(s for s in SPECS if s[0] == name)


def _qparams_from_minmax(state, lo_hi_cols, name):
    """Columns 2, 3 of ops.qparams_from_minmax applied to the range in columns lo_hi_cols of a host state."""
    from vsiquantization_b200 import ops
    _, _, bits, sym, _, _, _, _ = _spec(name)
    st = torch.tensor(state[:, :8]).cuda().contiguous()
    st[:, 0:2] = torch.tensor(state[:, lo_hi_cols]).cuda()
    n = st.shape[0]
    ops.qparams_from_minmax(st, torch.full((n,), bits, dtype=torch.int32), torch.full((n,), int(sym), dtype=torch.int32),
                            1e-8)
    return st[:, 2:4].cpu().numpy()


def _clipped(state, name):
    """The state after ops.hist_clip at the observer's percentile (what recompute_clip does)."""
    from vsiquantization_b200 import ops
    _, _, bits, sym, _, kw, _, _ = _spec(name)
    st = torch.tensor(state).cuda().contiguous()
    ops.hist_clip(st, kw["n_bins"], kw.get("percentile", 99.99), bits, sym, 1e-8)
    return st.cpu().numpy()


def _torch_qparams(state, name):
    from vsiquantization_b200.observers.moving_average import torch_qparams
    _, _, bits, sym, _, _, _, _ = _spec(name)
    qmin, qmax = (-(1 << (bits - 1)), (1 << (bits - 1)) - 1) if sym else (0, (1 << bits) - 1)
    lo, hi = (torch.tensor(state[:, c]).float().cuda() for c in (0, 1))  # on the device, like the sync
    s, z = torch_qparams(lo, hi, qmin, qmax, sym)
    return np.stack([s.double().cpu().numpy(), z.double().cpu().numpy()], axis=1)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _check_summed_columns(got, per_rank):
    assert np.array_equal(got[:, 4], sum(b[:, 4] for b in per_rank))  # call counts: exact
    np.testing.assert_allclose(got[:, 5:8], sum(b[:, 5:8] for b in per_rank), rtol=1e-12, atol=0)


def _check_merged(after, per_rank, union):
    """after: one rank's states after the sync; per_rank: every rank's states before it; union: one process's states
    after all batches (per_rank == [union] at world size 1)."""
    for name in ("mm_t", "mm_c", "lsq", "pct256", "pct2048"):
        got, want = after[name], union[name]
        assert np.array_equal(_bits(got[:, 0:2]), _bits(want[:, 0:2])), name  # extrema: exact
        _check_summed_columns(got, [want])
        if name.startswith("pct"):
            assert np.array_equal(_bits(got[:, 10:]), _bits(want[:, 10:])), name  # exponents and counts
            want = _clipped(want, name)
            assert np.array_equal(_bits(got[:, 8:10]), _bits(want[:, 8:10])), name
        assert np.array_equal(_bits(got[:, 2:4]), _bits(want[:, 2:4])), name
    got, ranks = after["mse"], [b["mse"] for b in per_rank]
    assert np.array_equal(_bits(got[:, 0]), _bits(np.minimum.reduce([b[:, 0] for b in ranks])))
    assert np.array_equal(_bits(got[:, 1]), _bits(np.maximum.reduce([b[:, 1] for b in ranks])))
    _check_summed_columns(got, ranks)
    if len(ranks) == 1:
        assert np.array_equal(_bits(got[:, 8:10]), _bits(ranks[0][:, 8:10]))
    else:  # clipped means weighted by each rank's call count
        n = sum(b[:, 4] for b in ranks)
        for col in (8, 9):
            want = sum(b[:, 4] * b[:, col] for b in ranks) / n
            np.testing.assert_allclose(got[:, col], want, rtol=1e-15, atol=0)
    assert np.array_equal(_bits(got[:, 2:4]), _bits(_qparams_from_minmax(got, [8, 9], "mse")))
    for name in ("ema_t", "ema_c"):  # both ranks observed: plain mean of the running extrema, rounded to fp32
        got, ranks = after[name], [b[name] for b in per_rank]
        want = (sum(b[:, 0:2] for b in ranks) / len(ranks)).astype(np.float32).astype(np.float64)
        assert np.array_equal(_bits(got[:, 0:2]), _bits(want)), name
        _check_summed_columns(got, ranks)
        assert np.array_equal(_bits(got[:, 2:4]), _bits(_torch_qparams(got, name))), name


def _check_caches(res):
    _, rows, launches, _, after, dropped, scales = res
    assert rows == ROWS
    assert launches == SYNC_LAUNCHES
    assert dropped
    for name, st in after.items():  # mgr.scale read after the sync is the new column 2
        assert np.array_equal(_bits(scales[name]), _bits(st[:, 2])), name


def test_sync_observers_two_ranks_equals_one_process():
    res = _collect(_run(_sync_rank))
    union = _sync_case(0, 1)[3]  # one process, every batch, before its (no-op) reduction
    for r in res:
        _check_caches(r)
        for name in res[0][4]:
            assert np.array_equal(_bits(r[4][name]), _bits(res[0][4][name])), name  # every rank: the same bits
    _check_merged(res[0][4], [r[3] for r in res], union)
    for name, st in res[0][3].items():
        assert not np.array_equal(st[:, 2], res[0][4][name][:, 2]), name  # the shards alone gave other scales


def test_sync_observers_world_size_one_only_recomputes():
    res = _sync_case(0, 1)
    _check_caches(res)
    before, after = res[3], res[4]
    _check_merged(after, [before], before)
    for name in before:  # nothing to reduce: the running ranges, statistics and histograms are untouched
        keep = [c for c in range(before[name].shape[1]) if c not in (2, 3, 8, 9)]
        assert np.array_equal(_bits(after[name][:, keep]), _bits(before[name][:, keep])), name
