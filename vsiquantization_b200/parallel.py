"""Data-parallel plumbing of the QAT path: the two small exchanges the path really has.

QAT shards as pure data parallel (batch shards per rank, replicated weights); fake-quant forward/backward need no
communication.  What must be exchanged (SURVEY.md 8(e)):

  * calibration: every rank sees different batches, so observer extrema are all-reduced -- ONE packed
    all_reduce(MIN) over [min, -max] of all quantisers (exact, so post-calibration scales are bit-identical to a
    single process that saw the union of the batches), plus one all_reduce(SUM) of the LSQ-initialisation statistics;
    scale / zero-point are then recomputed on the device for all observers in one launch (vsiq_qparams_from_minmax).
    The reference has no such step: every rank calibrates on identical un-sharded data (yolov8_qat.py:86-92).
  * training: the LSQ dscale / dzero_point of all layers live in ONE flat buffer per dtype (their .grad are views into
    it) and are reduced with a single all_reduce(SUM) instead of riding in DDP's 25 MB buckets with the weights.

torch.distributed (NCCL over NVLink on the box, gloo in the CPU tests) is the transport.
"""
from __future__ import annotations

from typing import Dict, List, Tuple

import torch
import torch.distributed as dist

from . import ops
from ._lib import HIST_STATE_HEAD, MSE_STATE_WIDTH, STATE_WIDTH


def _world(group=None) -> int:
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def quantization_managers(model) -> List[Tuple[str, torch.nn.Module]]:
    """(qualified name, manager) of every weight_quantizer / activation_quantizer, in module order."""
    out = []
    for name, module in model.named_modules():
        for attr in ("weight_quantizer", "activation_quantizer"):
            if hasattr(module, attr):
                out.append((f"{name}.{attr}" if name else attr, getattr(module, attr)))
    return out


def reduce_observer_states(states: torch.Tensor, group=None) -> torch.Tensor:
    """All-reduce a packed [rows, 8] fp64 observer-state block in place: MIN over run_min, MAX over run_max (as MIN of
    the negation, one collective for both), SUM over the call statistics.  Device-agnostic (CPU/gloo or CUDA/NCCL)."""
    if states.dtype != torch.float64 or states.dim() != 2 or states.shape[1] != STATE_WIDTH:
        raise ValueError("states must be [rows, 8] float64")
    if _world(group) == 1:
        return states
    packed = torch.cat([states[:, 0], -states[:, 1]]).contiguous()
    dist.all_reduce(packed, op=dist.ReduceOp.MIN, group=group)
    n = states.shape[0]
    states[:, 0] = packed[:n]
    states[:, 1] = -packed[n:]
    sums = states[:, 4:8].contiguous()
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    states[:, 4:8] = sums
    return states


def reduce_mse_states(states: torch.Tensor, group=None) -> torch.Tensor:
    """All-reduce a packed [rows, 10] fp64 MSE observer-state block in place: columns 0..7 as reduce_observer_states, the
    clipped means (columns 8, 9) combined as sum_r n_r * m_r / sum_r n_r with n_r the rank's call count, added in rank
    order on every rank (all_gather, then a local sum), so every rank ends with the same bits.  Device-agnostic."""
    if states.dtype != torch.float64 or states.dim() != 2 or states.shape[1] != MSE_STATE_WIDTH:
        raise ValueError("states must be [rows, 10] float64")
    w = _world(group)
    if w == 1:
        return states
    mine = torch.stack([states[:, 4], states[:, 8], states[:, 9]], dim=1).contiguous()
    everyone = [torch.empty_like(mine) for _ in range(w)]
    dist.all_gather(everyone, mine, group=group)
    n = torch.zeros_like(mine[:, 0])
    lo = torch.zeros_like(n)
    hi = torch.zeros_like(n)
    for r in range(w):  # rank order
        n = n + everyone[r][:, 0]
        lo = lo + everyone[r][:, 0] * everyone[r][:, 1]
        hi = hi + everyone[r][:, 0] * everyone[r][:, 2]
    has = n > 0
    base = states[:, :STATE_WIDTH].contiguous()
    reduce_observer_states(base, group)
    states[:, :STATE_WIDTH] = base
    states[:, 8] = torch.where(has, lo / torch.where(has, n, torch.ones_like(n)), states[:, 8])
    states[:, 9] = torch.where(has, hi / torch.where(has, n, torch.ones_like(n)), states[:, 9])
    return states


def _hist_exponent(m: torch.Tensor, log2b: int) -> torch.Tensor:
    """The smallest e >= -149 with m < 2^log2b * 2^e, per entry of a finite float64 m >= 0 (csrc/hist_observer.cu)."""
    _, k = torch.frexp(torch.where(m > 0, m, torch.ones_like(m)))  # m = f * 2^k, f in [0.5, 1)
    e = k.to(torch.int64) - log2b
    return torch.where(m > 0, torch.clamp(e, min=-149), torch.full_like(e, -149))


def reduce_percentile_states(states: torch.Tensor, n_bins: int, group=None) -> torch.Tensor:
    """All-reduce a packed [rows, 12 + 2 * n_bins] fp64 percentile-observer block in place: columns 0..7 as
    reduce_observer_states; per side the bin exponent of the reduced range (and at least every rank's own); each rank's
    counts coarsened to it (old bin i -> new bin i >> delta, exact); the counts summed (exact on integer-valued fp64), so
    every rank ends with the same bits -- the histogram a single process would hold after seeing every rank's calls.
    Columns 2, 3, 8, 9 (the clip) are left to be recomputed (ops.hist_clip).  Device-agnostic."""
    ops._check_hist_args(n_bins, 100.0)
    B = int(n_bins)
    W = HIST_STATE_HEAD + 2 * B
    if states.dtype != torch.float64 or states.dim() != 2 or states.shape[1] != W:
        raise ValueError(f"states must be [rows, {W}] float64")
    if _world(group) == 1:
        return states
    base = states[:, :STATE_WIDTH].contiguous()
    reduce_observer_states(base, group)
    states[:, :STATE_WIDTH] = base
    lo, hi = states[:, 0], states[:, 1]
    e_own = states[:, 10:12].to(torch.int64)
    e = states[:, 10:12].contiguous()
    dist.all_reduce(e, op=dist.ReduceOp.MAX, group=group)
    e = e.to(torch.int64)
    finite = (torch.isfinite(lo) & torch.isfinite(hi)).unsqueeze(1)
    log2b = B.bit_length() - 1
    e_range = torch.stack([_hist_exponent(-lo, log2b), _hist_exponent(hi, log2b)], dim=1)
    e = torch.where(finite, torch.maximum(e, e_range), e)
    counts = states[:, HIST_STATE_HEAD:].reshape(-1, 2, B)
    shift = torch.clamp(e - e_own, 0, 62).unsqueeze(2)
    idx = torch.bitwise_right_shift(torch.arange(B, device=states.device).expand_as(counts), shift)
    merged = torch.zeros_like(counts).scatter_add_(2, idx, counts)
    dist.all_reduce(merged, op=dist.ReduceOp.SUM, group=group)
    states[:, HIST_STATE_HEAD:] = merged.reshape(-1, 2 * B)
    states[:, 10:12] = e.to(torch.float64)
    return states


def reduce_moving_average_states(states: torch.Tensor, group=None) -> torch.Tensor:
    """All-reduce a packed [rows, 8] fp64 moving-average observer block in place: the running min / max AVERAGED over
    the ranks that have observed something (n_calls > 0; a rank without data carries no information) and rounded to fp32
    like the running update, the call statistics summed.  Scale / zero-point are left to be recomputed.
    Device-agnostic."""
    if _world(group) == 1:
        return states
    has = (states[:, 4:5] > 0).to(states.dtype)
    packed = torch.cat([states[:, 0:2] * has, has, states[:, 4:8]], dim=1).contiguous()
    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    n = torch.clamp(packed[:, 2:3], min=1.0)
    states[:, 0:2] = (packed[:, 0:2] / n).to(torch.float32).to(states.dtype)
    states[:, 4:8] = packed[:, 3:7]
    return states


def sync_observers(model, group=None) -> int:
    """Make every rank's observers agree after sharded calibration; returns the number of observer rows synchronised.

    Observers with equal ``sync_key()`` share one arena: their states are concatenated, merged over the ranks by their
    class's ``merge_states`` (the collectives above, then what can be recomputed on the whole arena), copied back, and
    each observer finishes with ``after_merge()``.  Groups run in module order, which every rank shares."""
    groups: Dict[tuple, list] = {}
    for _, m in quantization_managers(model):
        if m.observer.state is not None:
            groups.setdefault(m.observer.sync_key(), []).append(m.observer)
    rows = 0
    for observers in groups.values():
        arena = torch.cat([o.state for o in observers]).contiguous()
        observers[0].merge_states(arena, observers, group)
        at = 0
        for o in observers:
            k = o.state.shape[0]
            o.state.copy_(arena[at:at + k])
            o.after_merge()
            at += k
        rows += at
    return rows


class QParamGradBucket:
    """Flat gradient buffers for the learnable quantisation parameters (…quantizer.scale / …quantizer.zero_point).

    ``p.grad`` of every such parameter becomes a view into one flat tensor per dtype (autograd then accumulates in
    place), ``all_reduce()`` reduces each flat tensor with ONE collective, and ``ddp_ignore()`` keeps DDP from
    reducing the same parameters a second time.  Use ``zero()`` instead of ``optimizer.zero_grad(set_to_none=True)``.
    ``average=True`` divides by the world size (DDP's convention; the reference then multiplies the loss by the world
    size, yolov8_qat.py:235-236)."""

    SUFFIXES = ("quantizer.scale", "quantizer.zero_point")

    def __init__(self, model, group=None, average: bool = True):
        self.group, self.average = group, average
        self.names: List[str] = []
        self.params: List[torch.nn.Parameter] = []
        for name, p in model.named_parameters():
            if name.endswith(self.SUFFIXES) and p.requires_grad:
                self.names.append(name)
                self.params.append(p)
        self.flat: Dict[Tuple[torch.dtype, torch.device], torch.Tensor] = {}
        by_key: Dict[Tuple[torch.dtype, torch.device], List[torch.nn.Parameter]] = {}
        for p in self.params:
            by_key.setdefault((p.dtype, p.device), []).append(p)
        for key, ps in by_key.items():
            flat = torch.zeros(sum(p.numel() for p in ps), dtype=key[0], device=key[1])
            off = 0
            for p in ps:
                p.grad = flat[off:off + p.numel()].view(p.shape)
                off += p.numel()
            self.flat[key] = flat

    def __len__(self):
        return len(self.params)

    def numel(self) -> int:
        return sum(f.numel() for f in self.flat.values())

    def zero(self) -> None:
        for f in self.flat.values():
            f.zero_()

    def all_reduce(self) -> None:
        w = _world(self.group)
        if w == 1:
            return
        for f in self.flat.values():
            dist.all_reduce(f, op=dist.ReduceOp.SUM, group=self.group)
            if self.average:
                f.div_(w)

    def ddp_ignore(self, model) -> None:
        """Tell DistributedDataParallel (call BEFORE wrapping) not to reduce these parameters itself."""
        from torch.nn.parallel import DistributedDataParallel as DDP
        DDP._set_params_and_buffers_to_ignore_for_model(model, list(self.names))


class PeerExchange:
    """The per-layer exchange of BN re-estimation as ONE kernel over NVLink peer memory (vsiq_bn_moments_exchange,
    csrc/peer_exchange.cu) instead of combine kernel -> NCCL all_reduce -> moments kernel.

    One process per GPU on one node, at most 8 ranks.  Every rank allocates an exchange buffer, the cudaIpc handles go
    round once through torch.distributed, and from then on the ranks talk through peer pointers only: publish the shard's
    sums, signal, wait, add all shards in rank order (every rank gets the same bits), finish the moments.  ``local_buffers``
    (tests): run several "ranks" inside one process on buffers of one GPU -- the same kernel and protocol, no IPC."""

    def __init__(self, group=None, device=None, local_buffers=None, rank: int = 0, timeout_s: float = 30.0):
        import ctypes

        from ._lib import check, lib
        self._lib, self._check, self._ct = lib, check, ctypes
        self.timeout_s = float(timeout_s)
        self.group = group
        self._opened: List[int] = []
        self._own = None
        if local_buffers is not None:
            self.rank, self.world = int(rank), len(local_buffers)
            self.device = torch.device(device if device is not None else "cuda")
            self._ptrs = [int(p) for p in local_buffers]
        else:
            if not (dist.is_available() and dist.is_initialized()):
                raise RuntimeError("PeerExchange needs an initialised torch.distributed process group")
            self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
            self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
            if self.world > lib.vsiq_peer_max_world():
                raise RuntimeError(f"PeerExchange handles at most {lib.vsiq_peer_max_world()} ranks of one node")
            import socket
            handle = ctypes.create_string_buffer(64)
            buf = ctypes.c_void_p()
            with torch.cuda.device(self.device):
                rc0 = lib.vsiq_peer_alloc(ctypes.byref(buf), handle)
            self._own = buf.value if rc0 == 0 else None
            # from here to the all-reduced verdict every rank walks the same collectives, whatever failed locally
            mine = (socket.gethostname(), self.device.index, bytes(handle.raw) if rc0 == 0 else None)
            everyone = [None] * self.world
            dist.all_gather_object(everyone, mine, group=group)
            self._ptrs = []
            ok = len({h for h, _, _ in everyone}) == 1 and all(hnd is not None for _, _, hnd in everyone)  # one node
            for r, (_, _, hnd) in enumerate(everyone):
                if r == self.rank:
                    self._ptrs.append(self._own or 0)
                    continue
                p = ctypes.c_void_p()
                rc = -1
                if ok:
                    with torch.cuda.device(self.device):
                        rc = lib.vsiq_peer_open(hnd, ctypes.byref(p))
                if rc != 0:
                    ok = False
                    self._ptrs.append(0)
                else:
                    self._opened.append(p.value)
                    self._ptrs.append(p.value)
            flag = torch.tensor([1.0 if ok else 0.0], device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)  # everybody or nobody
            if float(flag.item()) != 1.0:
                self.close()
                raise RuntimeError("peer memory is not available between all ranks (cudaIpc open failed or several nodes)")
        self._arr = (ctypes.c_void_p * self.world)(*self._ptrs)

    def bn_moments(self, stats: torch.Tensor, weight: float, global_count: float, mean_sum=None, var_sum=None):
        """(batch mean, biased batch variance, unbiased batch variance) over ALL ranks' shards from this rank's [C,5]
        statistics block (ops.observe(x, ch_axis=1)); running sums updated like ops.bn_moments_finalize."""
        from . import _lib
        from .ops import _stream_ptr
        C = stats.shape[0]
        if stats.dtype != torch.float64 or not stats.is_cuda or not stats.is_contiguous() or stats.shape[1] != _lib.STATS_WIDTH:
            raise ValueError("stats must be a contiguous CUDA float64 [channels, 5] block")
        dev = stats.device
        with torch.cuda.device(dev):
            m = torch.empty(C, dtype=torch.float32, device=dev)
            vb = torch.empty(C, dtype=torch.float32, device=dev)
            vu = torch.empty(C, dtype=torch.float32, device=dev)
            self._check(self._lib.vsiq_bn_moments_exchange(
                stats.data_ptr(), float(weight), float(global_count), C, self._arr, self.rank, self.world, self.timeout_s,
                m.data_ptr(), vb.data_ptr(), vu.data_ptr(), mean_sum.data_ptr() if mean_sum is not None else None,
                var_sum.data_ptr() if var_sum is not None else None, _stream_ptr()), "vsiq_bn_moments_exchange")
            _lib.launch_count += 1
        return m, vb, vu

    def status(self) -> Tuple[int, int]:
        """(exchanges completed, sequence number of a timed-out exchange or 0).  Synchronises."""
        ct = self._ct
        seq, bad = ct.c_uint64(), ct.c_uint64()
        self._check(self._lib.vsiq_peer_status(self._ptrs[self.rank], ct.byref(seq), ct.byref(bad)), "vsiq_peer_status")
        return int(seq.value), int(bad.value)

    def close(self) -> None:
        for p in self._opened:
            self._lib.vsiq_peer_close(p)
        self._opened = []
        if self._own is not None:
            self._lib.vsiq_peer_free(self._own)
            self._own = None


_peer_exchanges: Dict[object, object] = {}


def _group_key(group):
    """The process-group OBJECT (a re-initialised default group is a new object: its ranks need new buffers)."""
    if group is not None:
        return group
    return dist.group.WORLD if dist.is_available() and dist.is_initialized() else "world"


def peer_exchange_for(group=None):
    """The process group's PeerExchange, created on first use; None when peer memory cannot be used (gloo / CPU tests,
    more than 8 ranks, several nodes, VSIQ_PEER_EXCHANGE=0) -- callers then keep their NCCL collective."""
    import os
    if os.environ.get("VSIQ_PEER_EXCHANGE", "1") == "0" or not (dist.is_available() and dist.is_initialized()):
        return None
    key = _group_key(group)
    if key not in _peer_exchanges:
        px = None
        try:
            if dist.get_backend(group) == "nccl" and torch.cuda.is_available() and dist.get_world_size(group) > 1:
                px = PeerExchange(group)
        except Exception:  # no peer access between some pair of ranks: every rank raises (all-reduced flag) and falls back
            px = None
        _peer_exchanges[key] = px
    return _peer_exchanges[key]


def drop_peer_exchange(group=None) -> None:
    """Forget the group's PeerExchange after a failed exchange: peer_exchange_for() then answers None (NCCL fallback)."""
    key = _group_key(group)
    px = _peer_exchanges.get(key)
    if px is not None:
        px.close()
    _peer_exchanges[key] = None
