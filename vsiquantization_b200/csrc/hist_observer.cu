// hist_observer.cu -- the percentile observer (observers/percentile.py): exact-bin histograms of everything a channel
// has seen, and the clipped range at a percentile of them.
//
// Per channel two one-sided histograms anchored at 0 (the running range always contains 0: the state starts there and is
// never reset), B bins each, bin width 2^e.  The exponent of a side is the smallest e >= -149 with m < B * 2^e for its
// extent m (run_max, or -run_min).  With integer counts and power-of-two widths, coarsening a side to a larger exponent
// (old bin i -> new bin i >> delta) is exact, so the histogram depends only on the multiset of values observed: not on
// the order of the calls, nor on how they were split, nor on how batches were sharded over ranks.
//   * hist_kernel: one read of x.  A CTA owns a channel group (one channel, or four adjacent channels of a
//     channels_last [rows, C] tensor read as one 16-byte vector per row) and a strided share of its units, and counts
//     into a privatised shared-memory histogram of u32; positive bin 0 (the exact zeros of a ReLU output) is counted in
//     a register.  Non-zero bins are flushed with integer red.global.add into the workspace: the sums do not depend on
//     scheduling.
//   * hist_finalize_kernel (a programmatic dependent, one CTA per channel): coarsens the stored counts, adds the call's,
//     applies observer_state_update, scans both tails from the top and writes the clip and its scale / zero-point.
// Both kernels take the exponents from hist_plan, so the bins the first one counts into are the bins the second expects.
#include "common.cuh"

namespace vsiq {

constexpr int kHistHead = VSIQ_HIST_STATE_HEAD;  // state columns before the counts
constexpr int kHistMinExp = -149;                // 2^-149: the smallest fp32 denormal
constexpr int kHistMaxBins = 4096;
constexpr int kHistUnit1 = 8192;  // elements per unit, one channel per CTA
constexpr int kHistUnit4 = 2048;  // rows per unit, four channels per CTA

static inline bool hist_bins_ok(int B) { return B >= 256 && B <= kHistMaxBins && (B & (B - 1)) == 0; }
static inline int hist_log2(int B) {
    int l = 0;
    while ((1 << l) < B) ++l;
    return l;
}

struct HistGeom {
    int64_t outer, channels, inner;  // channels_last groups: outer = rows, inner = 1
    int64_t n;                       // elements per channel
    uint32_t chunks;                 // units per row (one channel per CTA)
    uint32_t units;                  // units per channel group
    uint32_t kc;                     // CTAs per channel group
    int bins, log2b, width;
    int bits, symmetric;
    double eps, percentile;
};

// e(m): the smallest e >= -149 with m < B * 2^e, for a finite m >= 0
__device__ __forceinline__ int hist_exponent(double m, int log2b) {
    if (!(m > 0.0)) return kHistMinExp;
    int k;
    frexp(m, &k);  // m = f * 2^k, f in [0.5, 1): m < 2^j  <=>  j >= k
    return max(k - log2b, kHistMinExp);
}

struct HistPlan {
    double lo, hi;     // running range after this call (observer_state_update's rule)
    int e_neg, e_pos;  // bin exponents after this call
    bool add;          // this call's values are counted: its extrema are not NaN and the running range is finite
    bool finite;       // the running range is finite: the clip comes from the histogram, else it is the range
};

// The one exponent decision: old state + this call's stats (NULL: no call, the clip recompute) -> range and exponents.
__device__ __forceinline__ HistPlan hist_plan(const double* st, const double* stats, int log2b) {
    HistPlan p;
    double lo = st[0], hi = st[1];
    bool nan_call = false;
    if (stats) {
        const double mn = stats[0], mx = stats[1];
        nan_call = isnan(mn) || isnan(mx);
        if (mn < lo) lo = mn;  // NaN compares false: never updates
        if (mx > hi) hi = mx;
    }
    p.lo = lo;
    p.hi = hi;
    p.finite = isfinite(lo) && isfinite(hi);
    p.add = stats != nullptr && !nan_call && p.finite;
    p.e_neg = (int)st[10];
    p.e_pos = (int)st[11];
    if (p.add) {
        p.e_neg = max(p.e_neg, hist_exponent(-lo, log2b));
        p.e_pos = max(p.e_pos, hist_exponent(hi, log2b));
    }
    return p;
}

struct HistSide {
    int e_neg, e_pos;
    bool add;
};

// One value into the CTA's histogram of its channel: key floor(|v| / 2^e) by an integer shift of the fp32 significand
// (exact; |v| < B * 2^e keeps it below B), x < 0 into [0, B), x >= 0 (-0.0 included) into [B, 2B).
__device__ __forceinline__ void hist_add(float v, const HistSide& h, int B, uint32_t* s_h, uint32_t& zeros) {
    const uint32_t u = __float_as_uint(v), a = u & 0x7fffffffu;
    const bool neg = (u >> 31) && a != 0;
    const uint32_t E = a >> 23;
    const uint32_t M = E ? ((a & 0x7fffffu) | 0x800000u) : a;
    const int p = E ? (int)E - 150 : kHistMinExp;  // |v| = M * 2^p
    const int sh = min(max((neg ? h.e_neg : h.e_pos) - p, 0), 31);
    const uint32_t bin = min(M >> sh, (uint32_t)B - 1u);
    if (!neg && bin == 0)
        ++zeros;  // half of a ReLU output: never through one shared-memory word
    else
        atomicAdd(s_h + (neg ? 0 : B) + bin, 1u);
}

__device__ __forceinline__ float4 ld_stream4(const float* p) {
    float4 v;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// `len` consecutive elements of one channel from p: scalar head up to 16-byte alignment, four 16-byte loads in flight
// per thread, scalar tail.
__device__ __forceinline__ void hist_span(const float* p, int len, const HistSide& h, int B, uint32_t* s_h,
                                          uint32_t& zeros) {
    const int t = threadIdx.x;
    const int head = min((int)(((16u - ((uint32_t)(uintptr_t)p & 15u)) & 15u) >> 2), len);
    if (t < head) hist_add(ld_stream1(p + t), h, B, s_h, zeros);
    const float* pv = p + head;
    const int nv = (len - head) >> 2;
    for (int v = t; v < nv; v += 4 * kThreads) {
        float4 r[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (v + q * kThreads < nv) r[q] = ld_stream4(pv + 4 * (v + q * kThreads));
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (v + q * kThreads < nv) {
                hist_add(r[q].x, h, B, s_h, zeros);
                hist_add(r[q].y, h, B, s_h, zeros);
                hist_add(r[q].z, h, B, s_h, zeros);
                hist_add(r[q].w, h, B, s_h, zeros);
            }
        }
    }
    const int i = head + nv * 4 + t;
    if (i < len) hist_add(ld_stream1(p + i), h, B, s_h, zeros);
}

template <int G>
__global__ void __launch_bounds__(kThreads)
    hist_kernel(const float* __restrict__ x, HistGeom geo, const double* __restrict__ stats,
                const double* __restrict__ state, uint32_t* __restrict__ counts) {
    extern __shared__ uint32_t s_h[];  // [G][2][B]
    pdl_launch_dependents();
    const int t = threadIdx.x, B = geo.bins;
    const uint32_t group = blockIdx.x / geo.kc, j = blockIdx.x - group * geo.kc;
    const int64_t c0 = (int64_t)group * G;
    HistSide hs[G];
    bool any = false;
#pragma unroll
    for (int q = 0; q < G; ++q) {
        const HistPlan p = hist_plan(state + (c0 + q) * geo.width, stats + (c0 + q) * VSIQ_STATS_WIDTH, geo.log2b);
        hs[q].e_neg = p.e_neg;
        hs[q].e_pos = p.e_pos;
        hs[q].add = p.add;
        any |= p.add;
    }
    if (!any) return;  // uniform over the CTA
    for (int i = t; i < G * 2 * B; i += kThreads) s_h[i] = 0;
    __syncthreads();
    uint32_t zeros[G];
#pragma unroll
    for (int q = 0; q < G; ++q) zeros[q] = 0;
    if (G == 1) {
        const int64_t C = geo.channels, inner = geo.inner;
        for (uint32_t u = j; u < geo.units; u += geo.kc) {
            const int64_t o = u / geo.chunks, k = u - o * geo.chunks;
            const int64_t start = k * kHistUnit1;
            const int len = (int)((inner - start) < kHistUnit1 ? (inner - start) : kHistUnit1);
            hist_span(x + (o * C + c0) * inner + start, len, hs[0], B, s_h, zeros[0]);
        }
    } else {  // channels_last [rows, C]: row r holds the group's four channels at r * C + c0
        const int64_t C = geo.channels, rows = geo.outer;
        for (uint32_t u = j; u < geo.units; u += geo.kc) {
            const int64_t r0 = (int64_t)u * kHistUnit4;
            const int len = (int)((rows - r0) < kHistUnit4 ? (rows - r0) : kHistUnit4);
            for (int i = t; i < len; i += 4 * kThreads) {
                float4 r[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (i + q * kThreads < len) r[q] = ld_stream4(x + (r0 + i + q * kThreads) * C + c0);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (i + q * kThreads < len) {
                        const float v[4] = {r[q].x, r[q].y, r[q].z, r[q].w};
#pragma unroll
                        for (int g = 0; g < G; ++g)
                            if (hs[g].add) hist_add(v[g], hs[g], B, s_h + g * 2 * B, zeros[g]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < G; ++q) {
        uint32_t z = zeros[q];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) z += __shfl_down_sync(0xffffffffu, z, d);
        if ((t & 31) == 0 && z) atomicAdd(s_h + q * 2 * B + B, z);
    }
    __syncthreads();
    uint32_t* dst = counts + c0 * 2 * B;  // the group's [G][2][B] block of the [C][2][B] count area
    for (int i = t; i < G * 2 * B; i += kThreads) {
        const uint32_t v = s_h[i];
        if (v) asm volatile("red.global.add.u32 [%0], %1;" ::"l"(dst + i), "r"(v) : "memory");
    }
}

// Sum of v over the threads after this one, and over all threads (exact: integer counts below 2^53, any order).
__device__ __forceinline__ double block_suffix(double v, double* s_w, double* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double y = __shfl_down_sync(0xffffffffu, inc, d);
        if (lane + d < 32) inc += y;
    }
    if (lane == 0) s_w[warp] = inc;
    __syncthreads();
    double after = inc - v, tot = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        if (w > warp) after += s_w[w];
        tot += s_w[w];
    }
    __syncthreads();
    *total = tot;
    return after;
}

__device__ __forceinline__ int block_min(int v, int* s_w) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = min(v, __shfl_down_sync(0xffffffffu, v, d));
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    int m = s_w[0];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) m = min(m, s_w[w]);
    __syncthreads();
    return m;
}

// One CTA per channel.  stats == NULL: no new call, only the clip and its qparams are recomputed (vsiq_hist_clip).
__global__ void __launch_bounds__(kThreads)
    hist_finalize_kernel(HistGeom geo, const double* __restrict__ stats, double* __restrict__ state,
                         const uint32_t* __restrict__ counts) {
    __shared__ unsigned long long s_new[kHistMaxBins];
    __shared__ double s_w[kWarps];
    __shared__ int s_i[kWarps];
    pdl_wait();
    const int t = threadIdx.x, B = geo.bins;
    const int64_t c = blockIdx.x;
    double* st = state + c * geo.width;
    const double* sc = stats ? stats + c * VSIQ_STATS_WIDTH : nullptr;
    const HistPlan p = hist_plan(st, sc, geo.log2b);
    const int e_old[2] = {(int)st[10], (int)st[11]};
    if (p.add) {  // 1. stored counts coarsened to the new exponents, plus this call's counts
        for (int side = 0; side < 2; ++side) {
            double* h = st + kHistHead + side * B;
            const uint32_t* cc = counts + ((size_t)c * 2 + side) * B;
            const int d = min((side ? p.e_pos : p.e_neg) - e_old[side], 31);  // B <= 2^12: d >= 12 empties into bin 0
            for (int k = t; k < B; k += kThreads) s_new[k] = __ldcg(cc + k);
            __syncthreads();
            for (int i = t; i < B; i += kThreads) {
                const double v = h[i];
                if (v != 0.0) atomicAdd(s_new + (i >> d), (unsigned long long)v);  // integer atomics: exact, any order
            }
            __syncthreads();
            for (int k = t; k < B; k += kThreads) h[k] = (double)s_new[k];
            __syncthreads();
        }
    }
    // 2. both tails from the top: thread t owns bins [t * per, (t + 1) * per) of each side
    const int per = B / kThreads;
    double part[2], above[2], tot[2];
    for (int side = 0; side < 2; ++side) {
        const double* h = st + kHistHead + side * B + t * per;
        double s = 0.0;
        for (int q = 0; q < per; ++q) s += h[q];
        part[side] = s;
    }
    for (int side = 0; side < 2; ++side) above[side] = block_suffix(part[side], s_w, &tot[side]);
    const double N = tot[0] + tot[1];
    const double T = floor(__dmul_rn(__dsub_rn(1.0, __ddiv_rn(geo.percentile, 100.0)), N));
    int jj[2];
    for (int side = 0; side < 2; ++side) {  // the smallest j with sum_{i > j} count[i] <= T (the sums fall as j grows)
        const double* h = st + kHistHead + side * B + t * per;
        double s = above[side];
        int jl = B;
        for (int q = per - 1; q >= 0; --q) {
            if (s <= T) jl = t * per + q;
            s += h[q];
        }
        jj[side] = block_min(jl, s_i);
    }
    if (t != 0) return;
    double lo = p.lo, hi = p.hi;
    if (p.finite) {
        const double ch = ldexp((double)(jj[1] + 1), p.e_pos), cl = -ldexp((double)(jj[0] + 1), p.e_neg);
        if (ch < hi) hi = ch;
        if (cl > lo) lo = cl;
    }
    if (sc)
        observer_state_update(st, (float)sc[0], (float)sc[1], sc[2], sc[3], sc[4], (double)geo.n, geo.bits,
                              geo.symmetric, geo.eps);
    double s, z;
    qparams_from_minmax(lo, hi, geo.bits, geo.symmetric, geo.eps, &s, &z);
    st[2] = s;
    st[3] = z;
    st[8] = lo;
    st[9] = hi;
    st[10] = (double)p.e_neg;
    st[11] = (double)p.e_pos;
}

// Channels per CTA: four for a channels_last tensor ([rows, C] = layout {rows, C, 1}) with C % 4 == 0 and 16-byte
// aligned x, else one.
static bool hist_ci_eligible(const vsiq_layout* l) { return l->inner == 1 && l->channels % 4 == 0; }

static bool make_hist_geom(const vsiq_layout* l, int B, int G, HistGeom* g) {
    if (check_layout(l) || !hist_bins_ok(B)) return false;
    const int64_t n = l->outer * l->inner;
    if (n <= 0) return false;
    g->outer = l->outer;
    g->channels = l->channels;
    g->inner = l->inner;
    g->n = n;
    g->bins = B;
    g->log2b = hist_log2(B);
    g->width = kHistHead + 2 * B;
    int64_t chunks = 1, units;
    if (G == 1) {
        chunks = (l->inner + kHistUnit1 - 1) / kHistUnit1;
        units = l->outer * chunks;
    } else {
        units = (l->outer + kHistUnit4 - 1) / kHistUnit4;
    }
    if (units >= (int64_t(1) << 31)) return false;
    g->chunks = (uint32_t)chunks;
    g->units = (uint32_t)units;
    DeviceProps dp;
    int sms = 148;
    if (get_device_props(&dp) == 0) sms = dp.sm_count;
    const int64_t smem = (int64_t)G * 2 * B * 4;
    int64_t per_sm = (228 * 1024) / (smem + 1024);  // CTAs an SM holds by shared memory
    if (per_sm > 8) per_sm = 8;
    const int64_t groups = l->channels / G;
    int64_t kc = ((int64_t)sms * per_sm + groups - 1) / groups;  // one wave over the whole call
    if (kc > units) kc = units;
    if (kc < 1) kc = 1;
    if (groups * kc >= (int64_t(1) << 31)) return false;
    g->kc = (uint32_t)kc;
    return true;
}

static size_t hist_counts_bytes(int64_t channels, int B) { return (size_t)channels * 2 * B * sizeof(uint32_t); }

}  // namespace vsiq

using namespace vsiq;

extern "C" size_t vsiq_hist_observe_workspace_bytes(const vsiq_layout* layout, int n_bins) {
    HistGeom g;
    if (!make_hist_geom(layout, n_bins, 1, &g)) return 0;
    return kWsHeader + hist_counts_bytes(layout->channels, n_bins);
}

extern "C" int vsiq_hist_observe(const float* x, const vsiq_layout* layout, const double* stats, double* state,
                                 int n_bins, double percentile, int bits, int symmetric, double eps, void* workspace,
                                 size_t workspace_bytes, vsiq_stream_t stream) {
    if (!x || !stats || !state || bits < 2 || bits > 8 || !(percentile > 0.0 && percentile <= 100.0))
        return VSIQ_ERR_INVALID_ARG;
    if (int e = check_layout(layout)) return e;
    const int G = hist_ci_eligible(layout) && (reinterpret_cast<uintptr_t>(x) & 15u) == 0 ? 4 : 1;
    HistGeom g;
    if (!make_hist_geom(layout, n_bins, G, &g)) return VSIQ_ERR_INVALID_ARG;
    g.bits = bits;
    g.symmetric = symmetric ? 1 : 0;
    g.eps = eps;
    g.percentile = percentile;
    const size_t cbytes = hist_counts_bytes(layout->channels, n_bins);
    if (!workspace || workspace_bytes < kWsHeader + cbytes) return VSIQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* counts = (uint32_t*)((char*)workspace + kWsHeader);
    // the count area is not covered by vsiq_workspace_reset: zero it here, whatever an earlier call left behind
    if (cudaError_t e = cudaMemsetAsync(counts, 0, cbytes, st)) return (int)e;
    const unsigned grid = (unsigned)((layout->channels / G) * g.kc);
    const size_t smem = (size_t)G * 2 * n_bins * sizeof(uint32_t);
    if (G == 4) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return VSIQ_ERR_NO_DEVICE;
        if (cudaError_t e = set_smem_once<hist_kernel<4>>(dev, 4 * 2 * kHistMaxBins * (int)sizeof(uint32_t))) return (int)e;
        hist_kernel<4><<<grid, kThreads, smem, st>>>(x, g, stats, state, counts);
    } else {
        hist_kernel<1><<<grid, kThreads, smem, st>>>(x, g, stats, state, counts);
    }
    if (cudaError_t e = cudaGetLastError()) return (int)e;
    return (int)launch_pdl(hist_finalize_kernel, dim3((unsigned)layout->channels), dim3(kThreads), 0, st, g, stats,
                           state, (const uint32_t*)counts);
}

extern "C" int vsiq_hist_clip(double* state, int64_t channels, int n_bins, double percentile, int bits, int symmetric,
                              double eps, vsiq_stream_t stream) {
    if (!state || channels < 1 || channels >= (int64_t(1) << 31) || !hist_bins_ok(n_bins) || bits < 2 || bits > 8 ||
        !(percentile > 0.0 && percentile <= 100.0))
        return VSIQ_ERR_INVALID_ARG;
    HistGeom g = {};
    g.channels = channels;
    g.bins = n_bins;
    g.log2b = hist_log2(n_bins);
    g.width = kHistHead + 2 * n_bins;
    g.bits = bits;
    g.symmetric = symmetric ? 1 : 0;
    g.eps = eps;
    g.percentile = percentile;
    hist_finalize_kernel<<<(unsigned)channels, kThreads, 0, (cudaStream_t)stream>>>(g, nullptr, state, nullptr);
    return (int)cudaGetLastError();
}
