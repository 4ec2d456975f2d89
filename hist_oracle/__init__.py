"""CPU oracle of the percentile observer -- TEST INFRASTRUCTURE ONLY.

Pure NumPy, int64 counts: the semantics of observers/percentile.py (include/vsiq.h, vsiq_hist_observe) restated plainly.
Only tests/ and tools/percentile_bench.py use it, as the checker; nothing under vsiquantization_b200/ imports it.

State of one observer: [C, 12 + 2 * B] float64, laid out as on the device --
  0..7   running min / max, scale, zero-point, n_calls, sum mean|x|, sum mean x, sum std (the min/max observer's rule)
  8, 9   clipped lo / hi;  10, 11  bin exponents e_neg / e_pos (bin width 2^e)
  12..   B counts of x < 0 (bin i: |x| in [i 2^e_neg, (i+1) 2^e_neg)), B counts of x >= 0 (-0.0 included)
"""
from __future__ import annotations

from typing import Optional

import numpy as np

HEAD = 12
MIN_EXP = -149


def layout(shape, ch_axis: Optional[int]):
    """(outer, C, inner) of a contiguous tensor quantised along ``ch_axis`` (None = per tensor)."""
    n = int(np.prod(shape, dtype=np.int64)) if len(shape) else 1
    if ch_axis is None:
        return 1, 1, n
    outer = int(np.prod(shape[:ch_axis], dtype=np.int64)) if ch_axis > 0 else 1
    C = int(shape[ch_axis])
    return outer, C, n // (outer * C)


def new_state(channels: int, n_bins: int = 2048) -> np.ndarray:
    st = np.zeros((channels, HEAD + 2 * n_bins), dtype=np.float64)
    st[:, 2] = 1.0
    st[:, 10:12] = MIN_EXP
    return st


def exponent(m: float, n_bins: int) -> int:
    """The smallest integer e >= -149 with m < n_bins * 2^e (m >= 0, finite)."""
    e = MIN_EXP
    while not m < n_bins * 2.0 ** e:
        e += 1
    return e


def qparams(mn: float, mx: float, bits: int, symmetric: bool, eps: float = 1e-8):
    """observers/minmax.py:67-74 in Python doubles."""
    with np.errstate(all="ignore"):  # a range that is not finite gives inf / NaN qparams, as on the device
        if symmetric:
            return max(abs(mn), abs(mx)) / ((2 ** (bits - 1) - 1) + eps), 0.0
        s = (mx - mn) / ((2 ** bits - 1) + eps)
        return s, float(np.rint(-mn / (s + eps)))


def bins(v: np.ndarray, e: int) -> np.ndarray:
    """floor(|v| / 2^e), exactly (the scaling by a power of two is exact in float64 over this range)."""
    return np.floor(np.ldexp(np.abs(v.astype(np.float64)), -e)).astype(np.int64)


def coarsen(counts: np.ndarray, d: int) -> np.ndarray:
    """Counts at exponent e moved to exponent e + d: old bin i goes into new bin i >> d."""
    out = np.zeros_like(counts)
    np.add.at(out, np.arange(counts.size, dtype=np.int64) >> min(d, 62), counts)
    return out


def clip(st: np.ndarray, n_bins: int, percentile: float, bits: int, symmetric: bool, eps: float = 1e-8) -> None:
    """Columns 8, 9 and 2, 3 of every channel from its counts, in place."""
    B = n_bins
    for c in range(st.shape[0]):
        run_min, run_max = st[c, 0], st[c, 1]
        lo, hi = run_min, run_max
        if np.isfinite(run_min) and np.isfinite(run_max):
            neg = st[c, HEAD:HEAD + B].astype(np.int64)
            pos = st[c, HEAD + B:HEAD + 2 * B].astype(np.int64)
            N = int(neg.sum() + pos.sum())
            T = np.floor((1.0 - percentile / 100.0) * float(N))

            def top(cnt):  # the smallest j with sum_{i > j} cnt[i] <= T
                above = np.concatenate([np.cumsum(cnt[::-1])[::-1][1:], [0]])
                return int(np.argmax(above <= T))

            hi = min(run_max, (top(pos) + 1) * 2.0 ** int(st[c, 11]))
            lo = max(run_min, -(top(neg) + 1) * 2.0 ** int(st[c, 10]))
        st[c, 8], st[c, 9] = lo, hi
        st[c, 2], st[c, 3] = qparams(lo, hi, bits, symmetric, eps)


def observe(x, ch_axis, st: np.ndarray, n_bins: int = 2048, percentile: float = 99.99, bits: int = 8,
            symmetric: bool = True, eps: float = 1e-8) -> None:
    """One PercentileObserver.observe(x) call on the logical (NCHW / OIHW) array x: updates ``st`` in place."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    outer, C, inner = layout(x.shape, ch_axis)
    B = n_bins
    if st.shape != (C, HEAD + 2 * B) or st.dtype != np.float64:
        raise ValueError(f"state must be a float64 [{C}, {HEAD + 2 * B}] array")
    xr = x.reshape(outer, C, inner)
    n = outer * inner
    for c in range(C):
        v = xr[:, c, :].reshape(-1)
        mn, mx = float(np.min(v)), float(np.max(v))  # NaN if the channel holds one, like torch.min / max
        run_min, run_max = st[c, 0], st[c, 1]
        lo = mn if mn < run_min else run_min  # a NaN extremum never updates
        hi = mx if mx > run_max else run_max
        if not (np.isnan(mn) or np.isnan(mx)) and np.isfinite(lo) and np.isfinite(hi):
            for side, m, sel in ((0, -lo, v < 0), (1, hi, v >= 0)):
                e_old = int(st[c, 10 + side])
                e = max(e_old, exponent(m, B))
                cols = slice(HEAD + side * B, HEAD + (side + 1) * B)
                counts = coarsen(st[c, cols].astype(np.int64), e - e_old)
                counts += np.bincount(bins(v[sel], e), minlength=B)
                st[c, cols] = counts
                st[c, 10 + side] = e
        # the min/max observer's running state (csrc/common.cuh observer_state_update)
        vd = v.astype(np.float64)
        with np.errstate(all="ignore"):
            sa, s1, s2 = float(np.sum(np.abs(vd))), float(np.sum(vd)), float(np.sum(vd * vd))
            mean = np.float64(s1) / n
            var = (np.float64(s2) - n * mean * mean) / np.float64(n - 1.0)
        st[c, 0], st[c, 1] = lo, hi
        st[c, 4] += 1.0
        st[c, 5] += sa / n
        st[c, 6] += mean
        st[c, 7] += np.sqrt(var if var > 0.0 else 0.0)
    clip(st, B, percentile, bits, symmetric, eps)


def entropy_fold(st_row: np.ndarray, n_bins: int):
    """(H, e): both sides of one channel's counts coarsened to e = max(e_neg, e_pos) and added, then H[0] = H[1] (the
    search's working copy; the state is not modified)."""
    B = n_bins
    e_neg, e_pos = int(st_row[10]), int(st_row[11])
    e = max(e_neg, e_pos)
    H = (coarsen(st_row[HEAD:HEAD + B].astype(np.int64), e - e_neg)
         + coarsen(st_row[HEAD + B:HEAD + 2 * B].astype(np.int64), e - e_pos))
    H[0] = H[1]
    return H, e


def entropy_levels(run_min: float, bits: int, symmetric: bool) -> int:
    """nq: 2^bits for an asymmetric grid over [0, hi], else 2^(bits - 1)."""
    return 2 ** bits if (not symmetric and run_min >= 0.0) else 2 ** (bits - 1)


def kl_divergence(H: np.ndarray, i: int, nq: int) -> float:
    """D_i = KL(P || Q) of threshold i over the magnitude histogram H, as plain direct sums in fp64."""
    P = H[:i].astype(np.float64)
    P[i - 1] += float(H[i:].sum())  # the outliers into the last bin
    Hi = H[:i].astype(np.float64)
    k = (np.arange(i, dtype=np.int64) * nq) // i  # chunk of bin j: floor(j nq / i)
    nonzero = Hi != 0
    mass = np.bincount(k, weights=Hi, minlength=nq)  # chunk sums, bin by bin
    count = np.bincount(k, weights=nonzero.astype(np.float64), minlength=nq)
    Q = np.where(nonzero, mass[k] / np.maximum(count[k], 1.0), 0.0)
    if np.any((P > 0) & (Q == 0)):
        return np.inf
    p = P / P.sum()
    q = Q / Q.sum()
    m = p > 0
    return float(np.sum(p[m] * np.log(p[m] / q[m])))


def entropy_clip(st: np.ndarray, n_bins: int, start_bin: int, bits: int, symmetric: bool, eps: float = 1e-8):
    """The entropy observer's search (include/vsiq.h, vsiq_hist_entropy_clip): columns 8, 9 and 2, 3 of every channel
    from its counts, in place.  Returns the divergences [C, n_bins + 1] (NaN where i is no candidate)."""
    B = n_bins
    div = np.full((st.shape[0], B + 1), np.nan)
    for c in range(st.shape[0]):
        run_min, run_max = st[c, 0], st[c, 1]
        lo, hi = run_min, run_max
        if np.isfinite(run_min) and np.isfinite(run_max):
            H, e = entropy_fold(st[c], B)
            nz = np.flatnonzero(H)
            n_used = int(nz[-1]) + 1 if nz.size else 0
            nq = entropy_levels(run_min, bits, symmetric)
            best, best_i = np.inf, -1
            for i in range(max(start_bin, nq), n_used + 1):
                d = kl_divergence(H, i, nq)
                div[c, i] = d
                if np.isnan(d):
                    d = np.inf
                if d <= best:  # increasing i: ties go to the larger threshold
                    best, best_i = d, i
            if best_i >= 0:
                amax = best_i * 2.0 ** e
                if -amax > lo:
                    lo = -amax
                if amax < hi:
                    hi = amax
        st[c, 8], st[c, 9] = lo, hi
        st[c, 2], st[c, 3] = qparams(lo, hi, bits, symmetric, eps)
    return div
