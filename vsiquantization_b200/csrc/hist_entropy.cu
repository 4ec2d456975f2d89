// hist_entropy.cu -- the entropy observer (observers/entropy.py): the KL-divergence clip searched over the exact-bin
// histograms that hist_observer.cu keeps (TensorRT's entropy calibration, pytorch-quantization's
// _compute_amax_entropy), per channel, on the device.
//
// Per channel (include/vsiq.h, vsiq_hist_entropy_clip, states the rule): both sides are folded into one magnitude
// histogram H at the larger exponent, H[0] takes H[1] (the exact zeros of a ReLU output must not dominate), and every
// candidate threshold i in [max(start_bin, nq), n_used] is scored with KL(P || Q), P the histogram below i with the
// outlier mass added into bin i - 1, Q the same bins quantised into nq chunks (chunk mass spread evenly over the chunk's
// non-zero bins).  With exclusive prefix sums S (counts), Z (non-zero bins) and L (c ln c) of H, one candidate costs
// O(nq) and nq logarithms:
//     D_i = ( sum_k [L'_k - M'_k ln(M_k / nz_k)] + (S_i - h) ln(S_i / N) ) / N  +  last-bin term
// where M_k, nz_k are chunk k's mass and non-zero count, the primes leave out bin i - 1 (mass h), and the last-bin term
// is p ln(p / q) with p = (h + outliers) / N, q = (M_{nq-1} / nz_{nq-1}) / S_i (+inf when h = 0 < outliers).
//   * entropy_score_kernel: kc CTAs per channel.  Each folds H into shared memory, scans it (fixed order) and scores its
//     share of the candidates, one candidate per thread at a time, then writes one (D, i) record: its argmin, ties to
//     the larger i, NaN as +inf.  The records do not depend on kc: every D_i is one thread's sequential sum.
//   * entropy_finalize_kernel (a programmatic dependent, one thread per channel): the argmin over the channel's records
//     in order, the clip i* 2^e capped by the running range, its scale / zero-point.
#include <math.h>

#include "common.cuh"

namespace vsiq {

constexpr int kEntHead = VSIQ_HIST_STATE_HEAD;
constexpr int kEntThreads = 128;   // candidates in flight per scoring CTA
constexpr int kEntWarps = kEntThreads / 32;
constexpr int kEntMaxBins = 4096;

static inline bool ent_bins_ok(int B) { return B >= 256 && B <= kEntMaxBins && (B & (B - 1)) == 0; }
// CTAs that cover the candidate indices 0..B of one channel once (the most a channel is ever given)
static inline int ent_max_kc(int B) { return (B + 1 + kEntThreads - 1) / kEntThreads; }

struct EntGeom {
    int bins, width, start_bin, bits, symmetric;
    uint32_t kc;  // scoring CTAs per channel
    double eps;
};

struct EntRecord {  // one scoring CTA's argmin; i = -1: no candidate there
    double d;
    int i;
    int pad;
};

// the number of quantisation bins: an asymmetric grid over [0, hi] has all 2^bits levels on the one side
__device__ __forceinline__ int ent_levels(const double* st, const EntGeom& g) {
    return (!g.symmetric && st[0] >= 0.0) ? (1 << g.bits) : (1 << (g.bits - 1));
}

// Exclusive prefix of v over the CTA in thread order, and the CTA total (fixed order: the same bits every run).
template <class T>
__device__ __forceinline__ T ent_exclusive_scan(T v, T* s_w, T* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += y;
    }
    T exc = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) exc = T(0);
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    T off = T(0), tot = T(0);
#pragma unroll
    for (int w = 0; w < kEntWarps; ++w) {
        if (w < warp) off += s_w[w];
        tot += s_w[w];
    }
    __syncthreads();
    *total = tot;
    return off + exc;
}

// D_i from the prefix arrays (see the file comment); N = S[B] > 0, nq <= i <= n_used.
__device__ __forceinline__ double ent_divergence(int i, int nq, const double* __restrict__ S,
                                                 const double* __restrict__ L, const int* __restrict__ Z, double N) {
    const double Si = S[i];
    const double h = Si - S[i - 1];  // H[i - 1] (exact: integer counts)
    const double out = N - Si;       // the outlier mass above the threshold
    double acc = 0.0, lm_last = 0.0;
    int j0 = 0;
    for (int k = 0; k < nq; ++k) {
        const int j1 = ((k + 1) * i + nq - 1) / nq;  // chunk k: bins j with floor(j nq / i) == k
        const int nz = Z[j1] - Z[j0];
        if (nz > 0) {
            const double M = S[j1] - S[j0];
            const double lm = log(M / (double)nz);
            if (k == nq - 1) {  // j1 == i: bin i - 1 is scored on its own below
                acc += (L[i - 1] - L[j0]) - (M - h) * lm;
                lm_last = lm;
            } else {
                acc += (L[j1] - L[j0]) - M * lm;
            }
        }
        j0 = j1;
    }
    double d = (acc + (Si - h) * log(Si / N)) / N;
    const double pm = h + out;  // P's last bin, unnormalised
    if (pm > 0.0) {
        if (h == 0.0) return INFINITY;  // P > 0 where Q = 0
        d += (pm / N) * (log(pm) - log(N) - lm_last + log(Si));
    }
    return d;
}

__global__ void __launch_bounds__(kEntThreads)
    entropy_score_kernel(EntGeom g, const double* __restrict__ state, double* __restrict__ div,
                         EntRecord* __restrict__ rec) {
    extern __shared__ double s_ent[];  // S[B + 1], L[B + 1], then int Z[B + 1]
    __shared__ double s_wd[kEntWarps];
    __shared__ int s_wi[kEntWarps];
    __shared__ int s_top;
    __shared__ EntRecord s_rec[kEntWarps];
    pdl_launch_dependents();
    const int t = threadIdx.x, B = g.bins;
    const int64_t c = blockIdx.x / g.kc;
    const uint32_t part = blockIdx.x - (uint32_t)c * g.kc;
    const double* st = state + c * g.width;
    double* S = s_ent;
    double* L = S + (B + 1);
    int* Z = (int*)(L + (B + 1));
    const double run_min = st[0], run_max = st[1];
    const bool finite = isfinite(run_min) && isfinite(run_max);
    const int e_neg = (int)st[10], e_pos = (int)st[11];
    const int e = max(e_neg, e_pos);
    const int nq = ent_levels(st, g);
    // 1. fold: H[j] = the counts of both sides coarsened to e (old bin i -> i >> delta, exact), staged in S
    if (t == 0) s_top = -1;
    const int per = B / kEntThreads, b0 = t * per;
    {
        const int dn = min(e - e_neg, 40), dp = min(e - e_pos, 40);
        const double* neg = st + kEntHead;
        const double* pos = st + kEntHead + B;
        for (int q = 0; q < per; ++q) {
            const int j = b0 + q;
            double h = 0.0;
            const int64_t an = (int64_t)j << dn, ap = (int64_t)j << dp;
            for (int64_t x = an; x < B && x < an + ((int64_t)1 << dn); ++x) h += neg[x];
            for (int64_t x = ap; x < B && x < ap + ((int64_t)1 << dp); ++x) h += pos[x];
            S[j] = h;
        }
    }
    __syncthreads();
    if (t == 0) S[0] = S[1];  // the working copy only: the stored counts are never modified
    __syncthreads();
    // 2. the highest non-zero bin, and the three prefix sums over the thread's own bins, then across the CTA
    double ls = 0.0, ll = 0.0;
    int lz = 0, top = -1;
    for (int q = 0; q < per; ++q) {
        const double h = S[b0 + q];
        if (h != 0.0) {
            top = b0 + q;
            ls += h;
            ll += h * log(h);
            ++lz;
        }
    }
    if (top >= 0) atomicMax(&s_top, top);  // integer: the same result in any order
    double tot_s, tot_l;
    int tot_z;
    double rs = ent_exclusive_scan(ls, s_wd, &tot_s);
    double rl = ent_exclusive_scan(ll, s_wd, &tot_l);
    int rz = ent_exclusive_scan(lz, s_wi, &tot_z);
    for (int q = 0; q < per; ++q) {  // in place: S[j] becomes sum_{m < j} H[m]
        const int j = b0 + q;
        const double h = S[j];
        S[j] = rs;
        L[j] = rl;
        Z[j] = rz;
        if (h != 0.0) {
            rs += h;
            rl += h * log(h);
            ++rz;
        }
    }
    if (t == kEntThreads - 1) {
        S[B] = rs;
        L[B] = rl;
        Z[B] = rz;
    }
    __syncthreads();
    const int n_used = s_top + 1;
    const double N = S[B];
    const int c_lo = max(g.start_bin, nq), c_hi = finite ? n_used : -1;
    // 3. this CTA's candidates, one per thread at a time, in increasing i: "<=" keeps the larger i on a tie
    double bd = INFINITY;
    int bi = -1;
    double* drow = div ? div + c * (B + 1) : nullptr;
    for (int i = (int)part * kEntThreads + t; i <= B; i += (int)g.kc * kEntThreads) {
        double d = __longlong_as_double(0x7ff8000000000000ll);  // NaN: not a candidate
        if (i >= c_lo && i <= c_hi) {
            d = ent_divergence(i, nq, S, L, Z, N);
            const double dk = isnan(d) ? INFINITY : d;
            if (dk <= bd) {
                bd = dk;
                bi = i;
            }
        }
        if (drow) drow[i] = d;
    }
    // 4. the CTA's argmin: a total order on (d, i), so the result does not depend on the reduction's shape
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_down_sync(0xffffffffu, bd, o);
        const int oi = __shfl_down_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || od < bd || (od == bd && oi > bi))) {
            bd = od;
            bi = oi;
        }
    }
    if ((t & 31) == 0) s_rec[t >> 5] = EntRecord{bd, bi, 0};
    __syncthreads();
    if (t == 0) {
        EntRecord r = s_rec[0];
        for (int w = 1; w < kEntWarps; ++w) {
            const EntRecord o = s_rec[w];
            if (o.i >= 0 && (r.i < 0 || o.d < r.d || (o.d == r.d && o.i > r.i))) r = o;
        }
        rec[blockIdx.x] = r;
    }
}

__global__ void __launch_bounds__(kEntThreads)
    entropy_finalize_kernel(EntGeom g, int64_t channels, double* __restrict__ state,
                            const EntRecord* __restrict__ rec) {
    pdl_wait();
    const int64_t c = (int64_t)blockIdx.x * kEntThreads + threadIdx.x;
    if (c >= channels) return;
    EntRecord r = {INFINITY, -1, 0};
    for (uint32_t k = 0; k < g.kc; ++k) {  // in order
        const EntRecord o = rec[c * g.kc + k];
        if (o.i >= 0 && (r.i < 0 || o.d < r.d || (o.d == r.d && o.i > r.i))) r = o;
    }
    double* st = state + c * g.width;
    double lo = st[0], hi = st[1];
    if (r.i >= 0) {  // only a finite running range has candidates
        const double amax = ldexp((double)r.i, max((int)st[10], (int)st[11]));
        if (-amax > lo) lo = -amax;
        if (amax < hi) hi = amax;
    }
    double s, z;
    qparams_from_minmax(lo, hi, g.bits, g.symmetric, g.eps, &s, &z);
    st[2] = s;
    st[3] = z;
    st[8] = lo;
    st[9] = hi;
}

static size_t ent_records_bytes(int64_t channels, int B) {
    return (size_t)channels * ent_max_kc(B) * sizeof(EntRecord);
}

static size_t ent_smem_bytes(int B) { return (size_t)(B + 1) * (2 * sizeof(double) + sizeof(int)); }

}  // namespace vsiq

using namespace vsiq;

extern "C" size_t vsiq_hist_entropy_workspace_bytes(int64_t channels, int n_bins) {
    if (channels < 1 || channels >= (int64_t(1) << 31) || !ent_bins_ok(n_bins)) return 0;
    return kWsHeader + ent_records_bytes(channels, n_bins);
}

extern "C" int vsiq_hist_entropy_clip(double* state, int64_t channels, int n_bins, int start_bin, int bits,
                                      int symmetric, double eps, double* divergences, void* workspace,
                                      size_t workspace_bytes, vsiq_stream_t stream) {
    if (!state || channels < 1 || channels >= (int64_t(1) << 31) || !ent_bins_ok(n_bins) || start_bin < 1 ||
        start_bin > n_bins || bits < 2 || bits > 8)
        return VSIQ_ERR_INVALID_ARG;
    if (!workspace || workspace_bytes < kWsHeader + ent_records_bytes(channels, n_bins)) return VSIQ_ERR_WORKSPACE;
    EntGeom g;
    g.bins = n_bins;
    g.width = kEntHead + 2 * n_bins;
    g.start_bin = start_bin;
    g.bits = bits;
    g.symmetric = symmetric ? 1 : 0;
    g.eps = eps;
    // about two CTAs per SM over the whole call, at most one candidate per thread
    DeviceProps dp;
    int sms = 148;
    if (get_device_props(&dp) == 0) sms = dp.sm_count;
    int64_t kc = ((int64_t)sms * 2 + channels - 1) / channels;
    if (kc > ent_max_kc(n_bins)) kc = ent_max_kc(n_bins);
    if (kc < 1) kc = 1;
    if (channels * kc >= (int64_t(1) << 31)) return VSIQ_ERR_INVALID_ARG;
    g.kc = (uint32_t)kc;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return VSIQ_ERR_NO_DEVICE;
    if (cudaError_t e = set_smem_once<entropy_score_kernel>(dev, (int)ent_smem_bytes(kEntMaxBins))) return (int)e;
    cudaStream_t st = (cudaStream_t)stream;
    EntRecord* rec = (EntRecord*)((char*)workspace + kWsHeader);
    entropy_score_kernel<<<(unsigned)(channels * kc), kEntThreads, ent_smem_bytes(n_bins), st>>>(g, state, divergences,
                                                                                               rec);
    if (cudaError_t e = cudaGetLastError()) return (int)e;
    return (int)launch_pdl(entropy_finalize_kernel, dim3((unsigned)((channels + kEntThreads - 1) / kEntThreads)),
                           dim3(kEntThreads), 0, st, g, channels, state, (const EntRecord*)rec);
}
