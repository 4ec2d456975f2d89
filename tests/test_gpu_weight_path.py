"""The weight path of a QAT step against the C oracle, at the sizes a YOLOv8 step runs it.

bank.WeightBank fake-quantises every weight of the model in one multi-tensor launch and produces every dW, dscale and
dzero_point in one streaming launch per 120 tensors plus one combine launch (csrc/multi_tensor.cu); the BN fold
(csrc/bn_fold.cu) builds every fused layer's weight.  Checked here:

- whole YOLOv8 n ... x weight sets (63 .. 103 tensors, up to 68 M elements) in four quantiser configurations;
- table edges: sizes around the 120-tensor packs up to VSIQ_MT_MAX_TENSORS, empty entries, row lengths around the
  1024-element tile, misaligned views, special values and scales outside the fast-division window;
- the launches write their outputs and nothing else, need no workspace initialisation and are deterministic;
- the bank inside a fused YOLOv8n against the oracle, weight by weight;
- the BN fold at every YOLOv8 weight shape, both group instantiations, both vector widths.

y, dx, folded weights / biases, Wq and the statistics' min / max must equal the oracle bit for bit.  dscale is within
2e-6 x mass of the fp64 oracle (mass as in test_gpu_kernels.sum_mass, per channel), dzero_point within 2e-6 x
gs * sum |g * s|.
"""
import ctypes
import functools
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import oracle
from conftest import bits_equal, first_mismatch
from test_gpu_kernels import assert_sums_close

pytestmark = pytest.mark.gpu

MT_MAX_TENSORS = 4096  # VSIQ_MT_MAX_TENSORS (include/vsiq.h)
ERR_INVALID_ARG = -1   # VSIQ_ERR_INVALID_ARG
SUM_REL = 2e-6
_SENT32 = 0x7FC0DEAD              # fp32 NaN with a payload no kernel produces
_SENT64 = 0x7FF8DEADBEEFDEAD      # fp64 likewise


def _lib():
    from vsiquantization_b200 import _lib as L
    return L


def _round8(n):
    return (n + 7) // 8 * 8


# ------------------------------------------------------------------------------------------------ quantiser entries
class _Q:
    """One tensor of a table: its quantiser as the bank hands it to the kernels, and the same numbers for the oracle.

    s / z: fp64 arrays with one entry per qparam channel (rows when per channel, else 1).  s_kind: "host" (a Python
    float, scale_host), "f32" / "f64" ([C] device tensors) or "f64_0d" (the reference's 0-dim fp64 Parameter).
    z_kind: "host" or "f32".  gs_dev: None or the value of a one-element fp32 device factor."""

    def __init__(self, shape, qmin, qmax, pc, s, s_kind="f32", z=0.0, z_kind="host", zp_learned=False, learn=0,
                 gs=1.0, gs_dev=None):
        self.shape, self.qmin, self.qmax, self.pc = tuple(shape), int(qmin), int(qmax), bool(pc)
        self.numel = int(np.prod(self.shape))
        self.rows = int(self.shape[0])
        self.C = self.rows if self.pc else 1
        self.s = np.broadcast_to(np.asarray(s, np.float64), (self.C,)).copy()
        self.z = np.broadcast_to(np.asarray(z, np.float64), (self.C,)).copy()
        self.s_kind, self.z_kind, self.zp_learned, self.learn = s_kind, z_kind, bool(zp_learned), int(learn)
        self.gs, self.gs_dev = float(gs), gs_dev
        assert s_kind != "host" or self.C == 1

    def item(self, w):
        from vsiquantization_b200 import ops
        dev = w.device
        if self.s_kind == "host":
            scale = float(self.s[0])
        elif self.s_kind == "f64_0d":
            scale = torch.tensor(float(self.s[0]), dtype=torch.float64, device=dev)
        else:
            scale = torch.tensor(self.s, dtype=torch.float32 if self.s_kind == "f32" else torch.float64, device=dev)
        zp = float(self.z[0]) if self.z_kind == "host" else torch.tensor(self.z, dtype=torch.float32, device=dev)
        spec = ops.QSpec(self.qmin, self.qmax, ch_axis=0 if self.pc else None, zp_learned=self.zp_learned)
        gsd = None if self.gs_dev is None else torch.tensor([self.gs_dev], dtype=torch.float32, device=dev)
        return (None, w, scale, zp, spec, self.learn, self.gs, gsd)

    @property
    def gs_total(self):  # what the combine multiplies by: gs_host * float32(gs_dev), in fp64
        return self.gs * (1.0 if self.gs_dev is None else float(np.float32(self.gs_dev)))

    def z_eff(self):
        z = self.z.astype(np.float32)
        return np.clip(np.rint(z), self.qmin, self.qmax) if self.zp_learned else z

    def oracle(self, x, g):
        """(y, dx, ds, dz) of the oracle; x, g flat fp32 of this tensor."""
        ax = 0 if self.pc else None
        x2 = x.reshape(self.rows, -1) if self.pc else x
        g2 = g.reshape(self.rows, -1) if self.pc else g
        y = oracle.fake_quant_fwd(x2, self.s, self.z, self.qmin, self.qmax, ch_axis=ax, zp_learned=self.zp_learned)
        dx, ds, dz = oracle.fake_quant_bwd(x2, g2, self.s, self.z, self.qmin, self.qmax, ch_axis=ax,
                                           zp_learned=self.zp_learned, grad_scale=self.gs_total, want_ds=True,
                                           want_dz=True, mask_mode=_lib().MASK_ROUNDED)
        return y.reshape(-1), dx.reshape(-1), ds, dz

    def masses(self, x, g):
        """Per qparam channel: mass of dscale (test_gpu_kernels.sum_mass, times gs) and of dzero_point
        (gs * sum |g * s|), both in fp64."""
        x2 = x.reshape(self.C, -1).astype(np.float32)
        g2 = g.reshape(self.C, -1).astype(np.float64)
        s32 = self.s.astype(np.float32)[:, None]
        z = self.z_eff().astype(np.float32)[:, None]
        with np.errstate(all="ignore"):
            v = x2 / s32
            q = np.clip(np.rint(v + z), self.qmin, self.qmax)
            ms = np.sum(np.abs(g2 * (q - z)), axis=1) + np.sum(np.abs(g2 * v), axis=1)
            mz = np.sum(np.abs(g2), axis=1) * np.abs(s32[:, 0].astype(np.float64))
        return self.gs_total * ms, self.gs_total * mz


def _plan(qs, ws):
    from vsiquantization_b200.bank import _Plan
    return _Plan([q.item(w) for q, w in zip(qs, ws)], ws[0].device)


def _launch(plan, gs, y=None, dx=None, ds=None, dz=None, ws=None):
    """Forward, then backward, straight through the C ABI; outputs default to fresh flat buffers."""
    from vsiquantization_b200 import ops
    L = _lib()
    dev = plan.device
    n = len(plan.items)
    y = torch.empty(plan.total_out, device=dev) if y is None else y
    dx = torch.empty(plan.total_out, device=dev) if dx is None else dx
    ds = torch.empty(max(plan.total_q, 1), dtype=torch.float64, device=dev) if ds is None else ds
    dz = torch.empty(max(plan.total_q, 1), dtype=torch.float32, device=dev) if dz is None else dz
    ws = torch.zeros(max(plan.ws_bytes, 1), dtype=torch.uint8, device=dev) if ws is None else ws
    L.check(L.lib.vsiq_mt_fake_quant_fwd(plan.host, plan.dev.data_ptr(), n, y.data_ptr(), ops._stream_ptr()), "mt fwd")
    gptrs = (ctypes.c_void_p * n)(*[g.data_ptr() or None for g in gs])
    L.check(L.lib.vsiq_mt_lsq_bwd(plan.host, plan.dev.data_ptr(), n, gptrs, dx.data_ptr(), ds.data_ptr(), dz.data_ptr(),
                                  ws.data_ptr(), ws.numel(), ops._stream_ptr()), "mt bwd")
    return y, dx, ds, dz


def _sums_close(tag, got, ref, mass):
    got, ref, mass = (np.asarray(a, np.float64).reshape(-1) for a in (got, ref, mass))
    bad = ~(np.abs(got - ref) <= SUM_REL * mass + 1e-300)
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        return [f"{tag}: {int(bad.sum())}/{bad.size} channels off, first c={i}: {got[i]!r} vs oracle {ref[i]!r} "
                f"(mass {mass[i]!r})"]
    return []


def _check_entry(tag, q, x, g, y, dx, ds, dz, sums="strict"):
    """Failure messages of one tensor: y / dx bitwise, ds / dz against the oracle.  x, g: this tensor's input; y, dx:
    its slice of the flat outputs; ds, dz: its qparam slots."""
    if q.numel == 0:
        if q.learn >= 1 and q.C:  # a per-tensor quantiser of an empty tensor: the sums are empty, i.e. zero
            out = [] if ds[0] == 0 else [f"{tag}: dscale {ds[0]!r} of an empty tensor"]
            return out + ([] if q.learn < 2 or dz[0] == 0 else [f"{tag}: dzero_point {dz[0]!r} of an empty tensor"])
        return []
    yo, dxo, dso, dzo = q.oracle(x, g)
    out = []
    if not bits_equal(y, yo):
        out.append(f"{tag}: y {first_mismatch(y, yo)}")
    if not bits_equal(dx, dxo):
        out.append(f"{tag}: dx {first_mismatch(dx, dxo)}")
    if q.learn >= 1:
        ms, mz = q.masses(x, g)
        if sums == "strict":
            out += _sums_close(f"{tag} dscale", ds, dso, ms)
            if q.learn == 2:
                out += _sums_close(f"{tag} dzero_point", dz, dzo, mz)
        else:
            out += _special_sums(tag, q, x, g, ds, dso, ms, dz if q.learn == 2 else None, dzo, mz)
    return out


def _special_sums(tag, q, x, g, ds, dso, ms, dz, dzo, mz):
    """Sums over special values.

    dscale: a channel with a NaN or an infinity in x or g sums to a non-finite value on both sides.  A channel on which
    every fp32 intermediate of the reference's backward (x/s, g*s, (x/s)/s) is finite and whose mass stays far below
    FLT_MAX is held to the usual bar.  Elsewhere the reference's own fp32 intermediates overflow (scales like 1e-38 or
    3e38, inputs near FLT_MAX) and its sum is NaN or infinite where the kernels' fused form g * ((q - z) - m * x/s) is
    not; y and dx are still compared bit for bit there.
    dzero_point: a channel whose g and g*s are finite is held to the usual bar, special values in x included (a NaN or
    infinite x is clamped out on both sides).  With an infinite or NaN g the reference forms inf - inf."""
    out = []
    x2 = x.reshape(q.C, -1).astype(np.float32)
    g2 = g.reshape(q.C, -1).astype(np.float32)
    s32 = q.s.astype(np.float32)[:, None]
    with np.errstate(all="ignore"):
        special = ~np.isfinite(x2).all(1) | ~np.isfinite(g2).all(1)
        v = x2 / s32
        gs_ok = np.isfinite(g2 * s32).all(1)
        tame = np.isfinite(v).all(1) & gs_ok & np.isfinite(v / s32).all(1) & ~special & (ms < 2.0 ** 100)
    got, ref = np.asarray(ds, np.float64), np.asarray(dso, np.float64)
    for c in np.flatnonzero(special):
        if np.isfinite(got[c]) or np.isfinite(ref[c]):
            out.append(f"{tag} dscale[{c}]: {got[c]!r} vs oracle {ref[c]!r}, expected both non-finite")
            break
    if tame.any():
        out += _sums_close(f"{tag} dscale", got[tame], ref[tame], ms[tame])
    if dz is not None:
        ok = gs_ok & (mz < 2.0 ** 100)
        if ok.any():
            out += _sums_close(f"{tag} dzero_point", np.asarray(dz)[ok], dzo[ok], mz[ok])
    return out


def _check_table(qs, xs, gs, plan, y, dx, ds, dz, tag, sums="strict", threads=None):
    """Every tensor of a table against the oracle (in parallel: the oracle's backward is single-threaded per tensor)."""
    y, dx = y.cpu().numpy(), dx.cpu().numpy()
    ds, dz = ds.cpu().numpy(), dz.cpu().numpy()

    def one(i):
        oracle.set_threads(1)
        q, o, q0 = qs[i], plan.out_offsets[i], plan.q_offsets[i]
        return _check_entry(f"{tag} #{i} {q.shape}", q, xs[i], gs[i], y[o:o + q.numel], dx[o:o + q.numel],
                            ds[q0:q0 + q.C], dz[q0:q0 + q.C], sums)

    with ThreadPoolExecutor(threads or max(1, oracle.max_threads())) as ex:
        fails = [m for r in ex.map(one, range(len(qs))) for m in r]
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:12])


def _device_inputs(shapes, xs_host, gs_host, offsets=None, base_off=0):
    """Device copies of per-tensor inputs as views into two flat buffers (8-element aligned unless offsets say)."""
    if offsets is None:
        offsets, o = [], base_off
        for shp in shapes:
            offsets.append(o)
            o += _round8(int(np.prod(shp)))
    total = max(offsets[-1] + int(np.prod(shapes[-1])), 1) + 8 if shapes else 8
    xf, gf = np.zeros(total, np.float32), np.zeros(total, np.float32)
    for o, x, g in zip(offsets, xs_host, gs_host):
        xf[o:o + x.size], gf[o:o + g.size] = x, g
    xd, gd = torch.from_numpy(xf).cuda(), torch.from_numpy(gf).cuda()
    ws = [xd[o:o + int(np.prod(s))].view(s) for o, s in zip(offsets, shapes)]
    gs = [gd[o:o + int(np.prod(s))].view(s) for o, s in zip(offsets, shapes)]
    return ws, gs


# ------------------------------------------------------------------------------------------------ 1. YOLOv8 weight sets
@functools.lru_cache(maxsize=None)
def _yolo_shapes(variant):
    """Shapes of every convolution weight of yolo_v8_<variant> (built on the CPU, shapes only)."""
    from vsiquantization_b200.nets import yolov8
    model = getattr(yolov8, f"yolo_v8_{variant}")()
    return tuple(tuple(m.weight.shape) for m in model.modules() if isinstance(m, torch.nn.Conv2d))


@functools.lru_cache(maxsize=1)
def _yolo_data(variant):
    """Seeded weights at a Kaiming-like scale with a few outliers per tensor, seeded upstream gradients, flat on the host
    at the offsets the bank gives them (multiples of 8)."""
    shapes = _yolo_shapes(variant)
    offs, o = [], 0
    for shp in shapes:
        offs.append(o)
        o += _round8(int(np.prod(shp)))
    rng = np.random.default_rng(ord(variant))
    w = rng.standard_normal(o, dtype=np.float32)
    g = rng.standard_normal(o, dtype=np.float32)
    stds = []
    for off, shp in zip(offs, shapes):
        n = int(np.prod(shp))
        std = np.float32(np.sqrt(2.0 / (n // shp[0])))
        seg = w[off:off + n]
        seg *= std
        k = rng.integers(0, n, 4)
        seg[k] = (rng.choice([-1.0, 1.0], 4) * rng.uniform(6.0, 12.0, 4) * std).astype(np.float32)
        stds.append(float(std))
    return shapes, offs, w, g, stds


def _yolo_config(config, shapes, stds, rng):
    from vsiquantization_b200 import ops
    qs = []
    for i, (shp, std) in enumerate(zip(shapes, stds)):
        n, C = int(np.prod(shp)), shp[0]
        if config == "w8_per_tensor":
            qs.append(_Q(shp, -128, 127, False, 4.0 * std / 127, "f64_0d", learn=1, gs=ops.lsq_grad_scale(127, n)))
        elif config == "w4_per_channel_lsq":
            s = std * rng.uniform(0.25, 0.6, C)
            z = rng.uniform(4.0, 11.0, C)
            z[3::7], z[5::7], z[6::7] = -1.6, 15.7, 15.4  # rint: -2 and 16 lie outside [0, 15], 15 inside
            qs.append(_Q(shp, 0, 15, True, s, "f32", z, "f32", zp_learned=True, learn=2,
                         gs=ops.lsq_grad_scale(15, n, C)))
        elif config == "w2_w3_per_channel":
            qmin, qmax = (-2, 1) if i % 2 == 0 else (-4, 3)
            qs.append(_Q(shp, qmin, qmax, True, std * rng.uniform(0.5, 1.5, C), "f64", learn=1,
                         gs=ops.lsq_grad_scale(qmax, n, C)))
        else:  # mixed: learn cycles 0/1/2, the scale kind host float / fp32 / fp64 with period 9
            learn, kind = i % 3, ("host", "f32", "f64")[(i // 3) % 3]
            pc = kind != "host" and i % 2 == 1
            Cq = C if pc else 1
            if learn == 2:
                qmin, qmax, zl = 0, 15, True
                s = std * rng.uniform(0.25, 0.6, Cq)
                z = rng.uniform(-2.0, 17.0, Cq)
            elif i % 2:
                qmin, qmax, zl = 0, 255, False
                s, z = std * rng.uniform(0.03, 0.06, Cq), np.full(Cq, 128.0)
            else:
                qmin, qmax, zl = -128, 127, False
                s, z = std * rng.uniform(0.03, 0.06, Cq), np.zeros(Cq)
            zk = "host" if kind == "host" else ("f32" if learn == 2 or pc else "host")
            gs = ops.lsq_grad_scale(qmax, n, Cq) * (1.0 if i % 5 else 5000.0)
            qs.append(_Q(shp, qmin, qmax, pc, s, kind, z if zk == "f32" else z[0], zk, zp_learned=zl, learn=learn,
                         gs=gs, gs_dev=(0.37 + 0.01 * i) if (learn and i % 4 == 1) else None))
    return qs


@pytest.mark.parametrize("config", ["w8_per_tensor", "w4_per_channel_lsq", "w2_w3_per_channel", "mixed"])
@pytest.mark.parametrize("variant", ["n", "s", "m", "l", "x"])
def test_yolov8_weight_set_against_oracle(variant, config):
    """Every weight of a YOLOv8 variant as one table: forward and backward launches, every tensor against the oracle."""
    shapes, offs, w, g, stds = _yolo_data(variant)
    qs = _yolo_config(config, shapes, stds, np.random.default_rng(zlib.crc32(f"{variant}/{config}".encode())))
    xs = [w[o:o + q.numel] for o, q in zip(offs, qs)]
    gh = [g[o:o + q.numel] for o, q in zip(offs, qs)]
    wd, gd = torch.from_numpy(w).cuda(), torch.from_numpy(g).cuda()
    wts = [wd[o:o + q.numel].view(q.shape) for o, q in zip(offs, qs)]
    grads = [gd[o:o + q.numel].view(q.shape) for o, q in zip(offs, qs)]
    plan = _plan(qs, wts)
    assert plan.out_offsets == offs and len(qs) == {"n": 63, "s": 63, "m": 83, "l": 103, "x": 103}[variant]
    y, dx, ds, dz = _launch(plan, grads)
    _check_table(qs, xs, gh, plan, y, dx, ds, dz, f"yolov8{variant} {config}")


# ------------------------------------------------------------------------------------------------ 2. table edges
def _ragged(n, seed, empty_at=(), pack_learn=True):
    """n small ragged tensors (some per channel, learn cycling 0/1/2), their host inputs, qparams and device views."""
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(seed)
    qs, xs, gh = [], [], []
    for i in range(n):
        if i in empty_at:
            shp = ((0, 3, 3, 3), (5, 0), (0,), (0, 7))[i % 4]
        else:
            shp = (int(rng.integers(1, 6)), int(rng.integers(1, 300)))
        numel = int(np.prod(shp))
        learn = i % 3 if pack_learn else 0
        pc = i % 2 == 1 and shp[0] > 1 and numel > 0
        C = shp[0] if pc else 1
        if learn == 2:
            qmin, qmax, zl, z = 0, 15, True, rng.uniform(-2.0, 17.0, C)
        else:
            qmin, qmax, zl, z = -8, 7, False, np.zeros(C)
        s = rng.uniform(0.1, 0.5, C)
        qs.append(_Q(shp, qmin, qmax, pc, s, ("f32", "f64")[i % 2] if pc else ("host", "f64_0d", "f32")[i % 3],
                     z if (learn == 2 and (pc or i % 3)) else z[0], "f32" if (learn == 2 and (pc or i % 3)) else "host",
                     zp_learned=zl, learn=learn, gs=ops.lsq_grad_scale(qmax, max(numel, 1), C),
                     gs_dev=1.25 if (learn and i % 5 == 0) else None))
        xs.append((rng.standard_normal(numel) * 2).astype(np.float32))
        gh.append(rng.standard_normal(numel).astype(np.float32))
    return qs, xs, gh


def _kernel_counts(fn):
    """(forward launches, streaming backward launches, combine launches) that fn() makes, from the CUDA trace."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]  # kernel names appear on the kernels' own trace events only
    return tuple(sum(1 for nm in names if k in nm) for k in ("mt_fwd_kernel", "mt_bwd_kernel", "mt_combine_kernel"))


@pytest.mark.parametrize("n", [119, 120, 121, 240, 241, MT_MAX_TENSORS])
def test_table_sizes_around_the_gradient_packs(n):
    """Tables of up to VSIQ_MT_MAX_TENSORS tensors: one streaming launch per 120, every tensor checked (those on each side
    of a pack boundary included), the plan's launch count equal to what runs."""
    qs, xs, gh = _ragged(n, n)
    wts, grads = _device_inputs([q.shape for q in qs], xs, gh)
    plan = _plan(qs, wts)
    assert plan.bwd_launches == (n + 119) // 120 + 1
    out = {}
    counts = _kernel_counts(lambda: out.setdefault("r", _launch(plan, grads)))
    assert counts == (plan.fwd_launches, plan.bwd_launches - 1, 1), counts
    _check_table(qs, xs, gh, plan, *out["r"], f"n={n}")


def test_table_size_limit():
    """4097 tensors are refused by the planner and by both launchers, before anything runs."""
    from vsiquantization_b200 import _lib as L
    n = MT_MAX_TENSORS + 1
    table = (L.MtEntry * n)()
    w = torch.zeros(8, device="cuda")
    for i, e in enumerate(table):
        e.x, e.rows, e.inner, e.qp_channels, e.out_offset, e.qp_offset = w.data_ptr(), 1, 8, 1, 8 * i, i
        e.qp.scale_host, e.qp.qmin, e.qp.qmax = 0.1, -8, 7
    tiles = ctypes.c_uint32(0)
    assert L.lib.vsiq_mt_plan(table, n, ctypes.byref(tiles)) == ERR_INVALID_ARG
    assert L.lib.vsiq_mt_plan(table, n - 1, ctypes.byref(tiles)) == 0 and tiles.value == n - 1
    # the extra entry planned by hand like its identical predecessor: the table on the device is a valid one, so the
    # launchers are refused for its length alone
    ctypes.memmove(ctypes.byref(table[n - 1], L.MtEntry.first_tile.offset), ctypes.byref(table[n - 2], L.MtEntry.first_tile.offset),
                   ctypes.sizeof(L.MtEntry) - L.MtEntry.first_tile.offset)
    table[n - 1].first_tile = n - 1
    dev_table = torch.frombuffer(bytearray(bytes(table)), dtype=torch.uint8).cuda()
    y = torch.empty(8 * n, device="cuda")
    gptrs = (ctypes.c_void_p * n)(*([w.data_ptr()] * n))
    assert L.lib.vsiq_mt_fake_quant_fwd(table, dev_table.data_ptr(), n, y.data_ptr(), None) == ERR_INVALID_ARG
    assert L.lib.vsiq_mt_lsq_bwd(table, dev_table.data_ptr(), n, gptrs, y.data_ptr(), None, None, None, 0,
                                 None) == ERR_INVALID_ARG
    from vsiquantization_b200.bank import _Plan
    from vsiquantization_b200 import ops
    items = [(None, w, 0.1, 0, ops.QSpec(-8, 7), 0, 1.0, None)] * n
    with pytest.raises(L.VsiqError, match="code -1"):
        _Plan(items, w.device)


def test_empty_entries_anywhere_in_the_table():
    """Zero-element per-tensor entries first, in the middle, in a run, across pack boundaries (a whole pack of them
    included) and last: they write nothing (a learning one sums to zero) and every neighbour is right."""
    n = 300
    empty = {0, 1, 57, 58, 59, 118, 119, 120, 121, 299} | set(range(150, 300, 1)) - {200, 201, 298}
    qs, xs, gh = _ragged(n, 11, empty_at=empty)
    assert all(qs[i].numel == 0 and qs[i].C == 1 for i in empty)
    wts, grads = _device_inputs([q.shape for q in qs], xs, gh)
    plan = _plan(qs, wts)
    # every pack has tiles: [120, 240) in 122..149, 200 and 201, [240, 300) only in 298
    assert plan.bwd_launches == 3 + 1
    out = {}
    counts = _kernel_counts(lambda: out.setdefault("r", _launch(plan, grads)))
    assert counts == (1, 3, 1), counts
    _check_table(qs, xs, gh, plan, *out["r"], "empty entries")
    # a whole pack without tiles is skipped
    qs2, xs2, gh2 = _ragged(250, 12, empty_at=set(range(120, 240)))
    wts2, grads2 = _device_inputs([q.shape for q in qs2], xs2, gh2)
    plan2 = _plan(qs2, wts2)
    assert plan2.bwd_launches == 2 + 1
    out2 = {}
    assert _kernel_counts(lambda: out2.setdefault("r", _launch(plan2, grads2))) == (1, 2, 1)
    _check_table(qs2, xs2, gh2, plan2, *out2["r"], "empty pack")


def test_per_channel_entry_without_rows_produces_nothing():
    """A per-channel quantiser of a weight with zero output channels: the plan accepts it with qp_channels = 0; it owns no
    output element and no dscale / dzero_point slot, and the entry after it, which shares its qp_offset, gets its own
    sums.  Alone in a table it makes no launch and the backward succeeds."""
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(21)
    shapes = [(3, 40), (0, 16, 3, 3), (4, 1030), (0, 5), (2, 9)]
    qs = []
    for i, shp in enumerate(shapes):
        C = shp[0]
        qs.append(_Q(shp, 0, 15, True, rng.uniform(0.1, 0.3, C), "f32", rng.uniform(3.0, 12.0, C), "f32",
                     zp_learned=True, learn=2, gs=ops.lsq_grad_scale(15, max(int(np.prod(shp)), 1), max(C, 1))))
    xs = [(rng.standard_normal(q.numel) * 2).astype(np.float32) for q in qs]
    gh = [rng.standard_normal(q.numel).astype(np.float32) for q in qs]
    wts, grads = _device_inputs(shapes, xs, gh)
    plan = _plan(qs, wts)
    assert [plan.host[i].qp_channels for i in range(5)] == [3, 0, 4, 0, 2]
    assert plan.q_offsets == [0, 3, 3, 7, 7] and plan.total_q == 9
    assert plan.out_offsets == [0, 120, 120, 4240, 4240]
    y, dx, ds, dz = _launch(plan, grads)
    _check_table(qs, xs, gh, plan, y, dx, ds, dz, "rows == 0")
    # alone (or only with its own kind) in a table: nothing to launch, nothing to combine
    lone = [qs[1], qs[3]]
    plan1 = _plan(lone, [wts[1], wts[3]])
    assert plan1.total_tiles == 0 and plan1.total_q == 0 and plan1.bwd_launches == 0 and plan1.fwd_launches == 0
    assert _kernel_counts(lambda: _launch(plan1, [grads[1], grads[3]])) == (0, 0, 0)


@pytest.mark.parametrize("pc", [False, True], ids=["per_tensor", "per_channel"])
def test_row_lengths_around_the_tile(pc):
    """Rows of 1, 7 and around 1024 / 2048 elements (one, two, three tiles per row; ragged tails), rows = 1 with a
    per-channel quantiser among them."""
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(31 + pc)
    shapes = [(r, k) for k in (1, 7, 1023, 1024, 1025, 2047, 2048, 2049) for r in (1, 3)] + [(5, 3, 1, 683), (1, 1)]
    qs = []
    for i, shp in enumerate(shapes):
        C = shp[0] if pc else 1
        n = int(np.prod(shp))
        learn = (1, 2, 0)[i % 3]
        zl = learn == 2
        qs.append(_Q(shp, 0 if zl else -8, 15 if zl else 7, pc, rng.uniform(0.1, 0.4, C), "f32",
                     rng.uniform(-1.0, 16.0, C) if zl else np.zeros(C), "f32", zp_learned=zl, learn=learn,
                     gs=ops.lsq_grad_scale(15 if zl else 7, n, C)))
    xs = [(rng.standard_normal(q.numel) * 2).astype(np.float32) for q in qs]
    gh = [rng.standard_normal(q.numel).astype(np.float32) for q in qs]
    wts, grads = _device_inputs(shapes, xs, gh)
    plan = _plan(qs, wts)
    y, dx, ds, dz = _launch(plan, grads)
    _check_table(qs, xs, gh, plan, y, dx, ds, dz, "row lengths")


def test_misaligned_views():
    """x and g as views at element offsets 1..7, each misaligned on its own and both together (the streaming kernel
    picks the vector width from x, g and dx separately)."""
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(41)
    cases = [(o, 0) for o in range(1, 8)] + [(0, o) for o in range(1, 8)] + [(o, 8 - o) for o in range(1, 8)]
    base_x = torch.empty(1 << 20, device="cuda")
    base_g = torch.empty(1 << 20, device="cuda")
    qs, xs, gh, wts, grads = [], [], [], [], []
    px = pg = 64
    for i, (ox, og) in enumerate(cases):
        shp = (int(rng.integers(1, 5)), int(rng.integers(200, 3000)))
        n = int(np.prod(shp))
        pc = i % 2 == 0
        C = shp[0] if pc else 1
        learn = (2, 1, 0)[i % 3]
        zl = learn == 2
        qs.append(_Q(shp, 0 if zl else -8, 15 if zl else 7, pc, rng.uniform(0.1, 0.4, C), "f32",
                     rng.uniform(2.0, 13.0, C) if zl else np.zeros(C), "f32", zp_learned=zl, learn=learn,
                     gs=ops.lsq_grad_scale(15 if zl else 7, n, C)))
        xs.append((rng.standard_normal(n) * 2).astype(np.float32))
        gh.append(rng.standard_normal(n).astype(np.float32))
        wv = base_x[px + ox:px + ox + n]
        gv = base_g[pg + og:pg + og + n]
        wv.copy_(torch.from_numpy(xs[-1]))
        gv.copy_(torch.from_numpy(gh[-1]))
        assert (wv.data_ptr() % 32 != 0) == (ox != 0) and (gv.data_ptr() % 32 != 0) == (og != 0)
        wts.append(wv.view(shp))
        grads.append(gv.view(shp))
        px += _round8(n) + 64
        pg += _round8(n) + 64
    plan = _plan(qs, wts)
    y, dx, ds, dz = _launch(plan, grads)
    _check_table(qs, xs, gh, plan, y, dx, ds, dz, "misaligned")


_SPECIAL = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, 1.17549435e-38, np.inf, -np.inf, np.nan, 3.4e38, -3.4e38, 1e-30,
                     6e-39, 2.0 ** -61, 2.0 ** -60, 2.0 ** 60, 2.0 ** 61, 1.5, -2.5, 0.5, -0.5], dtype=np.float32)
_ODD_SCALES = (0.0236, 2.0 ** -41, 2.0 ** 41, 1e-38, 3e38, -0.05, 1.0)  # as test_gpu_kernels.test_special_values...


def test_special_values_and_odd_scales():
    """NaN, +-inf, +-0, denormals and +-3.4e38 in w (normal g), in g (normal w) and in both, per tensor and per
    channel, at scales inside and outside the fast-division window: y and dx bit for bit."""
    from vsiquantization_b200 import ops
    rng = np.random.default_rng(51)
    qs, xs, gh = [], [], []
    i = 0
    for s in _ODD_SCALES:
        for (qmin, qmax, z, zl, learn) in ((-128, 127, 0.0, False, 1), (0, 255, 128.0, False, 0), (0, 15, 7.6, True, 2)):
            for where in ("w", "g", "both"):
                for pc in (False, True):
                    shp = (3, 7 * _SPECIAL.size) if pc else (2, 5 * _SPECIAL.size + 3)
                    n = int(np.prod(shp))
                    x = (rng.standard_normal(n) * 2).astype(np.float32)
                    g = rng.standard_normal(n).astype(np.float32)
                    sp = np.resize(rng.permutation(_SPECIAL), n)
                    if where in ("w", "both"):
                        x = np.where(rng.random(n) < 0.5, sp, x).astype(np.float32)
                    if where in ("g", "both"):
                        g = np.where(rng.random(n) < 0.5, np.roll(sp, 3), g).astype(np.float32)
                    if pc and where == "w":
                        x[:7 * _SPECIAL.size] = (rng.standard_normal(7 * _SPECIAL.size) * 2).astype(np.float32)
                    C = shp[0] if pc else 1
                    qs.append(_Q(shp, qmin, qmax, pc, np.full(C, s), ("f32", "f64")[i % 2] if pc else
                                 ("host", "f32", "f64_0d")[i % 3], np.full(C, z) if pc else z, "f32" if pc else "host",
                                 zp_learned=zl, learn=learn, gs=ops.lsq_grad_scale(qmax, n, C)))
                    xs.append(x)
                    gh.append(g)
                    i += 1
    wts, grads = _device_inputs([q.shape for q in qs], xs, gh)
    plan = _plan(qs, wts)
    assert len(qs) > 120  # two packs
    y, dx, ds, dz = _launch(plan, grads)
    _check_table(qs, xs, gh, plan, y, dx, ds, dz, "special", sums="special")


# ------------------------------------------------------------------------------------------------ 3. writes only its outputs
class _Carved:
    """A flat output carved out of a sentinel-filled buffer at an element offset."""

    def __init__(self, n, off, dtype):
        self.n, self.off, self.pad = n, off, 64
        idt, sent = (torch.int32, _SENT32) if dtype == torch.float32 else (torch.int64, _SENT64)
        self.sent = sent
        self.raw = torch.full((self.pad + off + n + self.pad,), sent, dtype=idt, device="cuda")
        self.out = self.raw.view(dtype)[self.pad + off:self.pad + off + n]

    def untouched_except(self, ranges):
        """Positions of the carved output outside `ranges` ([lo, hi) pairs) and the pads that lost the sentinel."""
        keep = torch.ones(self.raw.numel(), dtype=torch.bool, device="cuda")
        base = self.pad + self.off
        for lo, hi in ranges:
            keep[base + lo:base + hi] = False
        bad = keep & (self.raw != self.sent)
        return torch.nonzero(bad).reshape(-1).tolist()[:8]


@pytest.mark.parametrize("off", [0, 1, 5])
def test_launches_write_only_their_outputs(off):
    """y / dx / dscale / dzero_point carved out of NaN-sentinel buffers at element offset `off` (0: aligned, 1 and 5:
    the unaligned-output path), workspace full of garbage: every word outside each tensor's [out_offset, out_offset +
    numel) keeps the sentinel -- the gaps that round each offset up to 8 included -- as do the dscale slots of
    non-learning tensors and the dzero_point slots of tensors that learn no zero-point.  The results equal those of a
    run with a zeroed workspace and of a second run bit for bit (both into buffers carved at the same offset: the
    streaming kernel's vector width, and with it the fp32 order of a tile's sum, follows the alignment of dx), and the
    oracle's."""
    qs, xs, gh = _ragged(131, 61 + off, empty_at={0, 64, 130})
    wts, grads = _device_inputs([q.shape for q in qs], xs, gh)
    plan = _plan(qs, wts)

    def carve():
        return [_Carved(plan.total_out, off, torch.float32), _Carved(plan.total_out, off, torch.float32),
                _Carved(plan.total_q, off, torch.float64), _Carved(plan.total_q, off, torch.float32)]
    bufs = carve()
    garbage = torch.randint(0, 256, (plan.ws_bytes,), dtype=torch.uint8, device="cuda",
                            generator=torch.Generator("cuda").manual_seed(off))
    y, dx, ds, dz = _launch(plan, grads, *[b.out for b in bufs], ws=garbage)
    torch.cuda.synchronize()
    spans = [(o, o + q.numel) for o, q in zip(plan.out_offsets, qs)]
    ds_spans = [(q0, q0 + q.C) for q0, q in zip(plan.q_offsets, qs) if q.learn >= 1]
    dz_spans = [(q0, q0 + q.C) for q0, q in zip(plan.q_offsets, qs) if q.learn >= 2]
    for name, b, rng_ in (("y", bufs[0], spans), ("dx", bufs[1], spans), ("dscale", bufs[2], ds_spans),
                          ("dzero_point", bufs[3], dz_spans)):
        assert b.untouched_except(rng_) == [], (name, b.untouched_except(rng_))
    zeroed = _launch(plan, grads, *[b.out for b in carve()])  # zero-filled workspace
    again = _launch(plan, grads, *[b.out for b in carve()], ws=garbage)  # the first run's leftovers in the workspace
    for k, (name, sp) in enumerate((("y", spans), ("dx", spans), ("dscale", ds_spans), ("dzero_point", dz_spans))):
        it = torch.int64 if k == 2 else torch.int32
        for other in (zeroed, again):
            for lo, hi in sp:
                u, v = (t[lo:hi].contiguous().view(it) for t in ((y, dx, ds, dz)[k], other[k]))
                assert torch.equal(u, v), (name, lo, hi)
    _check_table(qs, xs, gh, plan, y, dx, ds, dz, f"carved off={off}")


# ------------------------------------------------------------------------------------------------ 4. the bank in a model
def test_bank_at_model_scale_against_oracle(monkeypatch):
    """A fused QAT YOLOv8n with per-channel asymmetric W4 LSQ weights, bank installed: the loss equals the eager
    composition's, every banked dW is the oracle's dx of that weight and its upstream gradient (taken from the banked
    output), every dscale / dzero_point is within the bar of the oracle's."""
    from test_gpu_model_parity import _build, _fused, _make_eager
    from vsiquantization_b200.bank import WeightBank
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    model = _build(True)
    x = torch.randint(0, 256, (2, 3, 96, 96), generator=torch.Generator().manual_seed(3), dtype=torch.uint8)
    x = x.cuda().float() / 255.0
    eager = _make_eager(model, decomposed_bias=False)
    eager.zero_grad(set_to_none=True)
    loss_e = sum((o.float() ** 2).mean() for o in eager(x))

    layers = [m for _, m in _fused(model)]
    bank = WeightBank(model).install()
    upstream = {}

    def grab(module, args):  # runs after the bank's pre-hook: the banked outputs exist, not yet consumed
        for k, m in enumerate(layers):
            wq = m.weight_quantizer.__dict__["_banked"][1]
            wq.register_hook(lambda g, k=k: upstream.__setitem__(k, g.detach().clone()))
    h = model.register_forward_pre_hook(grab)
    model.zero_grad(set_to_none=True)
    loss = sum((o.float() ** 2).mean() for o in model(x))
    loss.backward()
    h.remove()
    assert bank.last_used and len(bank._plans) == 1
    plan = next(iter(bank._plans.values()))
    bank.remove()
    assert float(loss) == float(loss_e)
    assert len(upstream) == len(layers) == 57

    def one(k):
        oracle.set_threads(1)
        m = layers[k]
        mgr = m.weight_quantizer
        w, _ = m.get_weight_bias()
        C = w.shape[0]
        q = mgr.quantizer
        assert (q.qmin, q.qmax) == (0, 15)
        s = mgr.scale.detach().double().cpu().numpy().reshape(-1)
        z = mgr.zero_point.detach().double().cpu().numpy().reshape(-1)
        assert s.size == z.size == C
        qq = _Q(tuple(w.shape), 0, 15, True, s, "f32", z, "f32", zp_learned=True, learn=2,
                gs=oracle.grad_scale(15, w.numel(), C))
        it = plan.items[k]
        assert it[0] is mgr and it[1] is w and it[5] == 2 and it[7] is None
        assert abs(it[6] - qq.gs) <= 1e-15 * qq.gs, (k, it[6], qq.gs)  # the bank's gradient scale is the reference's
        xh = w.detach().cpu().numpy().reshape(-1)
        gh = upstream[k].contiguous().cpu().numpy().reshape(-1)
        _, dxo, dso, dzo = qq.oracle(xh, gh)
        out = []
        dw = w.grad.detach().cpu().numpy().reshape(-1)
        if not bits_equal(dw, dxo):
            out.append(f"layer {k} dW {first_mismatch(dw, dxo)}")
        ms, mz = qq.masses(xh, gh)
        out += _sums_close(f"layer {k} dscale", mgr.scale.grad.double().cpu().numpy().reshape(-1), dso, ms)
        out += _sums_close(f"layer {k} dzero_point", mgr.zero_point.grad.double().cpu().numpy().reshape(-1), dzo, mz)
        return out

    with ThreadPoolExecutor(max(1, oracle.max_threads())) as ex:
        fails = [msg for r in ex.map(one, range(len(layers))) for msg in r]
    assert not fails, "\n".join(fails[:12])


# ------------------------------------------------------------------------------------------------ 5. BN fold
def _fold_shapes():
    return sorted({shp for v in "nsmlx" for shp in _yolo_shapes(v)})


def test_bn_fold_at_yolov8_shapes():
    """ops.bn_fold at every distinct YOLOv8 n..x weight shape, with and without conv bias, on 32-byte aligned inputs and
    on inputs at an element offset: warp-per-tile (inner < 2048) and CTA-per-tile instantiations, each with 8-wide and
    scalar access.  W', b' equal oracle.bn_fold bit for bit; fused per-tensor and per-channel quantisation give the
    oracle's fake-quantised W'; the fused statistics give its exact min / max and sums within assert_sums_close."""
    from vsiquantization_b200 import ops
    shapes = _fold_shapes()
    inners = [int(np.prod(s[1:])) for s in shapes]
    assert min(inners) < 2048 <= max(inners) and sum(i >= 2048 for i in inners) >= 5
    rng = np.random.default_rng(71)
    eps = 1e-3
    fails = []
    for shp in shapes:
        C, n = shp[0], int(np.prod(shp))
        W = (rng.standard_normal(n) * np.sqrt(2.0 / (n // C))).astype(np.float32).reshape(shp)
        gamma = rng.uniform(0.3, 1.7, C).astype(np.float32)
        gamma[::5] *= -1
        beta = (rng.standard_normal(C) * 0.1).astype(np.float32)
        mean = (rng.standard_normal(C) * 0.1).astype(np.float32)
        var = np.exp(rng.uniform(np.log(1e-3), np.log(2.0), C)).astype(np.float32)
        bn = [torch.from_numpy(a).cuda() for a in (gamma, beta, mean, var)]
        Wbase = torch.empty(n + 16, device="cuda")
        for with_bias in (False, True):
            b = (rng.standard_normal(C) * 0.1).astype(np.float32) if with_bias else None
            bd = torch.from_numpy(b).cuda() if with_bias else None
            Wfo, bfo = oracle.bn_fold(W, b, gamma, beta, mean, var, eps)
            mx = float(np.abs(Wfo).max())
            s_t = mx / 7 * 0.8
            s_c = (np.abs(Wfo.reshape(C, -1)).max(1) / 7 * rng.uniform(0.6, 1.0, C)).astype(np.float32)
            s_c[s_c == 0] = 1.0
            yq_t = oracle.fake_quant_fwd(Wfo, s_t, 0, -8, 7)
            yq_c = oracle.fake_quant_fwd(Wfo.reshape(C, -1), s_c, 0, -8, 7, ch_axis=0).reshape(shp)
            so = oracle.minmax_stats(Wfo)
            for off in (0, 3):
                Wd = Wbase[8 + off:8 + off + n].view(shp)
                Wd.copy_(torch.from_numpy(W))
                tag = f"{shp} bias={with_bias} off={off}"
                Wf, bf, _, _ = ops.bn_fold(Wd, bd, *bn, eps)
                if not (bits_equal(Wf.cpu().numpy(), Wfo) and bits_equal(bf.cpu().numpy(), bfo)):
                    fails.append(f"{tag}: W' {first_mismatch(Wf.cpu().numpy(), Wfo)}; b' "
                                 f"{first_mismatch(bf.cpu().numpy(), bfo)}")
                    continue
                for kind, scale, spec, ref in (
                        ("per tensor", s_t, ops.QSpec(-8, 7), yq_t),
                        ("per channel", torch.from_numpy(s_c).cuda(), ops.QSpec(-8, 7, ch_axis=0), yq_c)):
                    Wf2, bf2, Wq, st = ops.bn_fold(Wd, bd, *bn, eps, scale=scale, zero_point=0, spec=spec,
                                                   want_stats=True)
                    Wq, st = Wq.cpu().numpy(), st.cpu().numpy()
                    if not (bits_equal(Wf2.cpu().numpy(), Wfo) and bits_equal(bf2.cpu().numpy(), bfo)):
                        fails.append(f"{tag} {kind}: W' / b' differ when fused")
                    if not bits_equal(Wq, ref):
                        fails.append(f"{tag} {kind}: Wq {first_mismatch(Wq, ref)}")
                    if not (st[0, 0] == so[0, 0] and st[0, 1] == so[0, 1]):
                        fails.append(f"{tag} {kind}: min/max {st[0, :2]} vs oracle {so[0, :2]}")
                    try:
                        assert_sums_close(st, so)
                    except AssertionError as e:
                        fails.append(f"{tag} {kind}: sums {e}")
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:12])
