"""Every host-side schedule of the record-and-combine reductions against the oracle.

vsiq_observe, vsiq_lsq_bwd and vsiq_bn_fold (with statistics) pick a streaming kernel and a combine step from the layout
and the SM count: channel-item records combined by the last CTA (thread, CTA or warp per channel) or by a finalize kernel
(modes 0 and 1), the per-tensor persistent kernel, or per-tile records (warp or CTA tiles, 256-bit or scalar loads)
combined by the last CTA or finalized in modes 0, 1 and 2.  The branch each shape takes on a 148-SM B200 is written next to
it (k: channel-item CTAs per channel, items: tile records per channel).

Bit-exact: min, max, dx, W', b', the running extrema and qparams, and a second run of the same call (of the persistent
per-tensor kernels only what their tile queue cannot change, see persistent()).  Tolerance (the sums' order differs from
the oracle's): sum|x|, sum x, sum x^2, dscale, dzero_point.
"""
import numpy as np
import pytest
import torch

import oracle
from conftest import bits_equal, first_mismatch

pytestmark = pytest.mark.gpu

# (outer, C, inner) of an [outer, C, inner] tensor observed / quantised along axis 1
OBSERVE_SHAPES = [
    ((33, 64, 1), "channel-item, ticket, thread per channel (k=5, grid=320)"),
    ((600, 4, 1), "channel-item, ticket, CTA per channel (k=75, grid=300)"),
    ((300, 8, 1), "channel-item, ticket, warp per channel (k=38, grid=304)"),
    ((9, 300, 1), "channel-item, finalize mode 0 (k=2, grid=600)"),
    ((600, 8, 1), "channel-item, finalize mode 1 (k=75, grid=600)"),
    ((1, 1, 100000), "per-tensor persistent (grid=13)"),
    ((1, 1, 3000000), "per-tensor persistent (grid=367)"),
    ((1, 1, 1), "tile G32, ticket, thread (items=1)"),
    ((33, 1, 1), "tile G32, ticket, CTA (items=33)"),
    ((33, 8, 1), "tile G32, ticket, warp (items=33)"),
    ((5, 1000, 1), "tile G32, finalize mode 0 (grid=625, items=5)"),
    ((4096, 1, 1600), "tile G32, finalize mode 2 (grid=1024, items=8192)"),
    ((2, 1, 2048), "tile G256, ticket, thread (items=2)"),
    ((33, 1, 2048), "tile G256, ticket, CTA (items=33)"),
    ((33, 8, 2048), "tile G256, ticket, warp (grid=264, items=33)"),
    ((600, 1, 2048), "tile G256, finalize mode 2 (grid=600, items=600)"),
]
# FunLSQ never takes the channel-item schedule, so its per-channel shapes reach the per-tile finalize modes that the
# channel-item schedule takes over for the observer and the rounded mask
FUNLSQ_SHAPES = [
    ((8, 600, 1), "tile G32, finalize mode 0 (grid=600, items=8)"),
    ((300, 16, 1), "tile G32, finalize mode 1 (grid=600, items=300)"),
    ((600, 8, 1), "tile G32, finalize mode 2 (grid=600, items=600)"),
    ((1, 600, 2048), "tile G256, finalize mode 0 (grid=600, items=1)"),
    ((33, 18, 2048), "tile G256, finalize mode 1 (grid=594, items=33)"),
    ((33, 8, 2048), "tile G256, ticket, warp (grid=264, items=33)"),
    ((1, 1, 100000), "per-tensor persistent (grid=13)"),
]
# W [C, inner]: warp tiles below 2048 elements per row, CTA tiles from there on; one record per warp / CTA
FOLD_SHAPES = [
    ((64, 27), "fold G32 (grid=8)"),
    ((3000, 9), "fold G32 (grid=375)"),
    ((16, 4096), "fold G256 (grid=16)"),
    ((300, 2304), "fold G256 (grid=600)"),
]


def persistent(shape):
    """The per-tensor persistent kernels take tiles from a dynamic queue: which CTA sums which tile, and so the grouping of
    the fp64 sums, depends on timing.  Their extrema, qparams and dx are still the same on every run."""
    return shape[0] == 1 and shape[1] == 1 and shape[2] >= 2048


def _ids(cases):
    return [f"{'x'.join(map(str, s))}" for s, _ in cases]


@pytest.fixture(scope="module")
def ops():
    from vsiquantization_b200 import ops as _ops
    return _ops


def on_device(a, vec8):
    """a copy of `a` on the GPU; vec8=False places it one element past a 32-byte boundary (scalar-load instantiation)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    off = 0 if vec8 else 1
    buf = torch.empty(a.size + 8, dtype=torch.float32, device="cuda")
    t = buf[off:off + a.size].view(a.shape)
    t.copy_(torch.from_numpy(a))
    assert (t.data_ptr() % 32 == 0) == vec8
    return t


def assert_sums_close(st, so, rel=1e-6):
    st, so = np.asarray(st, np.float64), np.asarray(so, np.float64)
    assert np.all(np.abs(st[:, 2] - so[:, 2]) <= rel * so[:, 2] + 1e-30), (st[:, 2], so[:, 2])
    assert np.all(np.abs(st[:, 3] - so[:, 3]) <= rel * so[:, 2] + 1e-30), (st[:, 3], so[:, 3])
    assert np.all(np.abs(st[:, 4] - so[:, 4]) <= rel * so[:, 4] + 1e-30), (st[:, 4], so[:, 4])


def sum_mass(x, g, s, z, qmin, qmax):
    with np.errstate(all="ignore"):
        v = x.astype(np.float32) / np.float32(s)
        q = np.clip(np.rint(v + np.float32(z)), qmin, qmax)
        return float(np.sum(np.abs(g.astype(np.float64) * (q - z))) + np.sum(np.abs(g.astype(np.float64) * v)))


def inputs(shape, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * 2 + 0.3).astype(np.float32)
    g = rng.standard_normal(shape).astype(np.float32)
    return x, g


@pytest.mark.parametrize("vec8", [True, False], ids=["v8", "v1"])
@pytest.mark.parametrize("shape", [s for s, _ in OBSERVE_SHAPES], ids=_ids(OBSERVE_SHAPES))
def test_observe_paths(ops, shape, vec8):
    x, _ = inputs(shape, sum(shape))
    C = shape[1]
    so = oracle.minmax_stats(x, ch_axis=1)
    xd = on_device(x, vec8)
    for with_state in (False, True):
        runs = []
        for _ in range(2):
            state = ops.new_observer_state(C, "cuda") if with_state else None
            for _ in range(2 if with_state else 1):  # twice: the running state carries over
                st = ops.observe(xd, ch_axis=1, state=state, bits=8, symmetric=False)
            runs.append((st.cpu().numpy(), None if state is None else state.cpu().numpy()))
        st, state = runs[0]
        assert np.array_equal(st[:, :2], so[:, :2]), first_mismatch(st[:, :2], so[:, :2])
        assert_sums_close(st, so)
        sums_fixed = not persistent(shape)
        assert bits_equal(runs[1][0] if sums_fixed else runs[1][0][:, :2], st if sums_fixed else st[:, :2])
        if with_state:
            assert bits_equal(runs[1][1] if sums_fixed else runs[1][1][:, :5], state if sums_fixed else state[:, :5])
            count = x.size // C
            for c in range(C):
                rmin, rmax = oracle.minmax_update(0.0, 0.0, so[c, 0], so[c, 1])
                assert (state[c, 0], state[c, 1]) == (rmin, rmax), c
                assert tuple(state[c, 2:4]) == oracle.qparams(rmin, rmax, 8, False), c
                assert state[c, 4] == 2.0
                assert state[c, 5] == pytest.approx(2 * so[c, 2] / count, rel=1e-6)
                assert state[c, 6] == pytest.approx(2 * so[c, 3] / count, rel=1e-6, abs=1e-6 * so[c, 2] / count)


def _lsq_case(ops, shape, vec8, mask_mode, want_dz):
    x, g = inputs(shape, 7 + sum(shape))
    C = shape[1]
    rng = np.random.default_rng(C)
    s = (0.02 * rng.uniform(0.5, 2.0, C)).astype(np.float32)
    zf = rng.uniform(100, 150, C).astype(np.float32) if mask_mode == 0 else np.zeros(C, np.float32)
    spec = ops.QSpec(0, 255, ch_axis=1, zp_learned=want_dz, mask_mode=mask_mode)
    gs = ops.lsq_grad_scale(255, x.size, C)
    dx_o, ds_o, dz_o = oracle.fake_quant_bwd(x, g, s, zf, 0, 255, ch_axis=1, zp_learned=want_dz, grad_scale=gs,
                                             want_dz=want_dz, mask_mode=mask_mode)
    xd, gd = on_device(x, vec8), on_device(g, True)
    s_t = torch.from_numpy(s).cuda().view(1, C, 1)
    z_t = torch.from_numpy(zf).cuda().view(1, C, 1)
    runs = []
    for _ in range(2):
        dx, ds, dz = ops.lsq_backward(xd, gd, s_t, z_t, spec, gs, want_dz=want_dz, ds_dtype=torch.float64,
                                      dz_dtype=torch.float64)
        runs.append([dx.cpu().numpy(), ds.cpu().numpy()] + ([dz.cpu().numpy()] if want_dz else []))
    for a, b in zip(*runs) if not persistent(shape) else [(runs[0][0], runs[1][0])]:
        assert bits_equal(a, b)
    dx, ds = runs[0][0], runs[0][1]
    assert bits_equal(dx, dx_o), first_mismatch(dx, dx_o)
    xm = np.moveaxis(x, 1, 0).reshape(C, -1)
    gm = np.moveaxis(g, 1, 0).reshape(C, -1)
    for c in range(C):
        zeff = float(np.clip(np.rint(zf[c]), 0, 255)) if want_dz else float(zf[c])
        mass = gs * sum_mass(xm[c], gm[c], s[c], zeff, 0, 255)
        assert abs(ds[c] - ds_o[c]) <= 2e-6 * mass + 1e-30, (c, ds[c], ds_o[c])
        if want_dz:
            zmass = gs * float(np.sum(np.abs(gm[c].astype(np.float64) * s[c])))
            assert abs(runs[0][2][c] - dz_o[c]) <= 2e-6 * zmass + 1e-30, (c, runs[0][2][c], dz_o[c])


@pytest.mark.parametrize("want_dz", [False, True], ids=["ds", "ds_dz"])
@pytest.mark.parametrize("vec8", [True, False], ids=["v8", "v1"])
@pytest.mark.parametrize("shape", [s for s, _ in OBSERVE_SHAPES], ids=_ids(OBSERVE_SHAPES))
def test_lsq_rounded_paths(ops, shape, vec8, want_dz):
    _lsq_case(ops, shape, vec8, 0, want_dz)


@pytest.mark.parametrize("vec8", [True, False], ids=["v8", "v1"])
@pytest.mark.parametrize("shape", [s for s, _ in FUNLSQ_SHAPES], ids=_ids(FUNLSQ_SHAPES))
def test_lsq_funlsq_paths(ops, shape, vec8):
    _lsq_case(ops, shape, vec8, 1, False)


@pytest.mark.parametrize("vec8", [True, False], ids=["v8", "v1"])
@pytest.mark.parametrize("shape", [s for s, _ in FOLD_SHAPES], ids=_ids(FOLD_SHAPES))
def test_bn_fold_stats_paths(ops, shape, vec8):
    C, inner = shape
    rng = np.random.default_rng(C + inner)
    W = (rng.standard_normal(shape) * 0.1).astype(np.float32)
    b = rng.standard_normal(C).astype(np.float32)
    gamma = rng.uniform(0.5, 1.5, C).astype(np.float32)
    beta = rng.standard_normal(C).astype(np.float32)
    mean = rng.standard_normal(C).astype(np.float32) * 0.1
    var = rng.uniform(0.5, 2.0, C).astype(np.float32)
    eps = 1e-5
    Wf_o, bf_o = oracle.bn_fold(W, b, gamma, beta, mean, var, eps)
    so = oracle.minmax_stats(Wf_o)[0]
    Wd = on_device(W, vec8)
    bn = [torch.from_numpy(v).cuda() for v in (b, gamma, beta, mean, var)]
    runs = []
    for _ in range(2):
        Wf, bf, _, st = ops.bn_fold(Wd, *bn, eps, want_stats=True)
        runs.append((Wf.cpu().numpy(), bf.cpu().numpy(), st.cpu().numpy()))
    for a, c in zip(*runs):
        assert bits_equal(a, c)
    Wf, bf, st = runs[0]
    assert bits_equal(Wf, Wf_o), first_mismatch(Wf, Wf_o)
    assert bits_equal(bf, bf_o), first_mismatch(bf, bf_o)
    assert st[0, 0] == so[0] and st[0, 1] == so[1]
    assert_sums_close(st[:, :5], so[None, :])
