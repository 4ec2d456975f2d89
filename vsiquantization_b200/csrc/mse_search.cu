// mse_search.cu -- clipping-range search of the MSE observer (observers/mse.py): per channel, K clipped ranges
// (alpha_k * run_min, alpha_k * run_max), alpha_k = k / K, each scored by the squared error of the quantiser that will run
//     E[c,k] = sum_i ((double)fq(x_i; s_k, z_k) - (double)x_i)^2
// and the winner folded into the observer state as a running mean of the clipped extrema.
//
// Unlike every other pass of this library the kernel is compute-bound: each element is scored K times (K = 100 by
// default), so x is read from HBM once into a shared-memory tile and every candidate is evaluated from there.
//   * a CTA owns a channel group (one channel, or four adjacent channels of a channels_last [rows, C] tensor read as one
//     16-byte vector per row) and a strided share of that group's tiles;
//   * each thread owns one (channel, candidate) pair and, when there are fewer pairs than threads, a slice of the tile's
//     8-element vectors; its fp64 sum stays in a register across all of the CTA's tiles;
//   * the per-element arithmetic is common.cuh's forward (elem_fast under the per-vector FastGuard, elem_slow otherwise):
//     the measured error is that of the kernels that will fake-quantise with the chosen qparams;
//   * one record of P = G * K fp64 sums per CTA (slices added in a fixed order), combined per channel in CTA order by the
//     finalize kernel (a programmatic dependent): no float atomics, the result does not depend on scheduling.
#include "common.cuh"

namespace vsiq {

constexpr int kMseMaxCandidates = 256;
constexpr int kMseTile1 = 2048;  // elements per tile, one channel per CTA
constexpr int kMseTile4 = 512;   // rows per tile, four channels per CTA (2048 elements)

struct MseGeom {
    int64_t outer, channels, inner;
    int64_t n;        // elements per channel (outer * inner)
    int K;            // candidates
    int P;            // (channel, candidate) pairs of a group: G * K
    int S;            // slices: threads sharing one pair (P <= kThreads), else 1
    uint32_t kc;      // CTAs per channel group
    uint32_t tiles;   // tiles per channel group
    int bits, symmetric;
    double eps;
};

// The running range after this call (the rule of observer_state_update), without writing it.
__device__ __forceinline__ void mse_run_range(const double* st, const double* stats, double* lo, double* hi) {
    double a = st[0], b = st[1];
    const double mn = stats[0], mx = stats[1];
    if (mn < a) a = mn;
    if (mx > b) b = mx;
    *lo = a;
    *hi = b;
}

__device__ __forceinline__ QP mse_candidate_qp(const QPDev& d, double lo, double hi, int k, const MseGeom& g) {
    const double alpha = (double)k / (double)g.K;
    double s, z;  // explicit products: a contraction into qparams_from_minmax's (max - min) would change the range
    qparams_from_minmax(__dmul_rn(alpha, lo), __dmul_rn(alpha, hi), g.bits, g.symmetric, g.eps, &s, &z);
    QP q;
    q.lo = d.lo;
    q.hi = d.hi;
    q.tlo = d.tlo;
    q.thi = d.thi;
    q.s = (float)s;  // the fp64 state is rounded to fp32 before use, as in load_qp
    q.zf = (float)z;
    q.z = q.zf;
    q.r = __frcp_rn(q.s);
    q.zero_dx = 0.0f;
    const float as = fabsf(q.s);
    q.fast = (as >= 9.094947017729282e-13f) && (as <= 1.099511627776e12f);
    return q;
}

template <bool FAST>
__device__ __forceinline__ double mse_term(float x, double xd, const QP& q) {
    const Elem e = FAST ? elem_fast(x, q) : elem_slow(x, q);
    const double d = __dsub_rn((double)dequant(e.q, q), xd);
    return __dmul_rn(d, d);
}

// Squared error of the first `len` (<= 8) elements of one vector.
template <bool FULL>
__device__ __forceinline__ double mse_vector(const float* xs, const double* xds, bool ok, const QP& q, int len, double acc) {
    if (ok) {
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (FULL || e < len) acc = __dadd_rn(acc, mse_term<true>(xs[e], xds[e], q));
    } else {
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (FULL || e < len) acc = __dadd_rn(acc, mse_term<false>(xs[e], xds[e], q));
    }
    return acc;
}

template <int G>
__global__ void __launch_bounds__(kThreads)
    mse_search_kernel(const float* __restrict__ x, MseGeom geo, const double* __restrict__ stats,
                      const double* __restrict__ state, QPDev qd, double* __restrict__ records) {
    constexpr int T = G == 1 ? kMseTile1 : kMseTile4;  // elements per channel per tile
    __shared__ __align__(16) float s_x[G * T];
    __shared__ __align__(16) double s_xd[G * T];
    __shared__ unsigned char s_ok[G * T / 8];
    __shared__ double s_red[kThreads];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const uint32_t group = blockIdx.x / geo.kc, j = blockIdx.x - group * geo.kc;
    const int64_t c0 = (int64_t)group * G;

    // this thread's pairs: rounds > 1 only when G * K > kThreads (then one slice)
    constexpr int R = G;
    const int rounds = geo.S > 1 ? 1 : (geo.P + kThreads - 1) / kThreads;
    const int slice = geo.S > 1 ? t / geo.P : 0;
    bool act[R];
    int gch[R];
    QP qp[R];
    double acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int p = geo.S > 1 ? t % geo.P : t + r * kThreads;
        act[r] = r < rounds && p < geo.P && slice < geo.S;
        gch[r] = act[r] ? p / geo.K : 0;
        acc[r] = 0.0;
        if (act[r]) {
            const int64_t c = c0 + gch[r];
            double lo, hi;
            mse_run_range(state + c * VSIQ_MSE_STATE_WIDTH, stats + c * VSIQ_STATS_WIDTH, &lo, &hi);
            qp[r] = mse_candidate_qp(qd, lo, hi, p % geo.K + 1, geo);
        }
    }

    for (uint32_t tile = j; tile < geo.tiles; tile += geo.kc) {
        const int64_t i0 = (int64_t)tile * T;
        const int len = (int)((geo.n - i0) < T ? (geo.n - i0) : T);
        // ---- stage: one read of this tile of the group's channels
        if (G == 1) {
            const int64_t C = geo.channels, inner = geo.inner;
            for (int i = t; i < len; i += kThreads) {
                const int64_t idx = i0 + i;
                const int64_t addr = geo.outer == 1 ? c0 * inner + idx : ((idx / inner) * C + c0) * inner + idx % inner;
                const float v = ld_stream1(x + addr);
                s_x[i] = v;
                s_xd[i] = (double)v;
            }
        } else {  // channels_last [rows, C]: row r holds the group's four channels at r * C + c0
            for (int i = t; i < len; i += kThreads) {
                float4 v;
                asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                    : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                    : "l"(x + (i0 + i) * geo.channels + c0));
                s_x[0 * T + i] = v.x;
                s_x[1 * T + i] = v.y;
                s_x[2 * T + i] = v.z;
                s_x[3 * T + i] = v.w;
                s_xd[0 * T + i] = (double)v.x;
                s_xd[1 * T + i] = (double)v.y;
                s_xd[2 * T + i] = (double)v.z;
                s_xd[3 * T + i] = (double)v.w;
            }
        }
        __syncthreads();
        const int nvec = (len + 7) / 8, nfull = len / 8;
        for (int v = t; v < G * nvec; v += kThreads) {  // the vector's admissibility for the fast division
            const int g = v / nvec, w = v - g * nvec;
            FastGuard fg;
            guard_reset(fg);
            for (int e = 0; e < 8 && w * 8 + e < len; ++e) guard_note(fg, s_x[g * T + w * 8 + e]);
            s_ok[g * (T / 8) + w] = guard_bad(fg) ? 0 : 1;
        }
        __syncthreads();
        // ---- score: every candidate of this thread over its slice of the tile
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (!act[r]) continue;
            const float* xs = s_x + gch[r] * T;
            const double* xds = s_xd + gch[r] * T;
            const unsigned char* oks = s_ok + gch[r] * (T / 8);
            const QP q = qp[r];
            double a = acc[r];
#pragma unroll 1
            for (int w = slice; w < nfull; w += geo.S) {
                const float4 f0 = *(const float4*)&xs[w * 8], f1 = *(const float4*)&xs[w * 8 + 4];
                const double2 d0 = *(const double2*)&xds[w * 8], d1 = *(const double2*)&xds[w * 8 + 2];
                const double2 d2 = *(const double2*)&xds[w * 8 + 4], d3 = *(const double2*)&xds[w * 8 + 6];
                const float xv[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
                const double xdv[8] = {d0.x, d0.y, d1.x, d1.y, d2.x, d2.y, d3.x, d3.y};
                a = mse_vector<true>(xv, xdv, oks[w] && q.fast, q, 8, a);
            }
            if (nfull < nvec && (nfull % geo.S) == slice)
                a = mse_vector<false>(xs + nfull * 8, xds + nfull * 8, oks[nfull] && q.fast, q, len - nfull * 8, a);
            acc[r] = a;
        }
        __syncthreads();
    }

    // ---- one record per CTA: P sums, slices added in slice order
    double* rec = records + (size_t)blockIdx.x * geo.P;
    if (geo.S > 1) {
        s_red[t] = act[0] ? acc[0] : 0.0;
        __syncthreads();
        if (t < geo.P) {
            double s = s_red[t];
            for (int k = 1; k < geo.S; ++k) s = __dadd_rn(s, s_red[k * geo.P + t]);
            rec[t] = s;
        }
    } else {
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (act[r]) rec[t + r * kThreads] = acc[r];
    }
}

// One warp per channel: E[c,k] from the group's records in CTA order, argmin (ties to the larger alpha; any non-finite
// E or range: alpha = 1), then the observer state: running range and call statistics exactly as vsiq_observe's, the
// running means of the clipped extrema, scale / zero-point from those means.
__global__ void __launch_bounds__(kThreads)
    mse_finalize_kernel(MseGeom geo, int G, const double* __restrict__ records, const double* __restrict__ stats,
                        double* __restrict__ state, double* __restrict__ err, double* __restrict__ alpha_out) {
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t c = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (c >= geo.channels) return;
    const int64_t group = c / G, g = c - group * G;
    const double* base = records + (size_t)group * geo.kc * geo.P + g * geo.K;
    double best = INFINITY;
    int best_k = 0;
    bool bad = false;
    for (int k = lane; k < geo.K; k += 32) {
        double e = 0.0;
        for (uint32_t jj = 0; jj < geo.kc; ++jj) e = __dadd_rn(e, __ldcg(base + (size_t)jj * geo.P + k));
        if (err) err[c * geo.K + k] = e;
        if (!isfinite(e)) bad = true;
        else if (best_k == 0 || e <= best) {
            best = e;
            best_k = k + 1;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const double ob = __shfl_down_sync(0xffffffffu, best, d);
        const int ok = __shfl_down_sync(0xffffffffu, best_k, d);
        if (ok != 0 && (best_k == 0 || ob < best || (ob == best && ok > best_k))) {
            best = ob;
            best_k = ok;
        }
    }
    bad = __any_sync(0xffffffffu, bad);
    if (lane != 0) return;
    const double* sc = stats + c * VSIQ_STATS_WIDTH;
    double* st = state + c * VSIQ_MSE_STATE_WIDTH;
    observer_state_update(st, (float)sc[0], (float)sc[1], sc[2], sc[3], sc[4], (double)geo.n, geo.bits, geo.symmetric,
                          geo.eps);
    const double lo = st[0], hi = st[1];
    const bool finite = isfinite(lo) && isfinite(hi) && !bad && best_k > 0;
    const double a = finite ? (double)best_k / (double)geo.K : 1.0;
    const double n = st[4];  // m += (v - m) / n, every operation rounded on its own (no FMA contraction)
    st[8] = __dadd_rn(st[8], __ddiv_rn(__dsub_rn(__dmul_rn(a, lo), st[8]), n));
    st[9] = __dadd_rn(st[9], __ddiv_rn(__dsub_rn(__dmul_rn(a, hi), st[9]), n));
    double s, z;
    qparams_from_minmax(st[8], st[9], geo.bits, geo.symmetric, geo.eps, &s, &z);
    st[2] = s;
    st[3] = z;
    if (alpha_out) alpha_out[c] = a;
}

// Channels per CTA: four for a channels_last tensor ([rows, C] = layout {rows, C, 1}) with C % 4 == 0 and 16-byte
// aligned x (one 16-byte load per row and group), else one.
static bool mse_ci_eligible(const vsiq_layout* l) { return l->inner == 1 && l->channels % 4 == 0; }

// geometry of a call with G channels per CTA; false for arguments the search does not take
static bool make_mse_geom(const vsiq_layout* l, int K, int G, int bits, int symmetric, double eps, MseGeom* g) {
    if (check_layout(l) || K < 1 || K > kMseMaxCandidates) return false;
    const int64_t n = l->outer * l->inner;
    if (n <= 0 || l->channels <= 0) return false;
    const int T = G == 4 ? kMseTile4 : kMseTile1;
    g->outer = l->outer;
    g->channels = l->channels;
    g->inner = l->inner;
    g->n = n;
    g->K = K;
    g->P = G * K;
    g->S = g->P <= kThreads ? kThreads / g->P : 1;
    const int64_t tiles = (n + T - 1) / T;
    if (tiles >= (int64_t(1) << 31)) return false;
    g->tiles = (uint32_t)tiles;
    DeviceProps dp;
    int sms = 148;
    if (get_device_props(&dp) == 0) sms = dp.sm_count;
    const int64_t groups = l->channels / G;
    int64_t kc = ((int64_t)sms * 8 + groups - 1) / groups;  // about eight CTAs per SM over the whole call
    if (kc > tiles) kc = tiles;
    if (kc < 1) kc = 1;
    if (groups * kc >= (int64_t(1) << 31)) return false;
    g->kc = (uint32_t)kc;
    g->bits = bits;
    g->symmetric = symmetric;
    g->eps = eps;
    return true;
}

static size_t mse_records_bytes(const vsiq_layout* l, const MseGeom& g, int G) {
    return (size_t)(l->channels / G) * g.kc * g.P * sizeof(double);
}

}  // namespace vsiq

using namespace vsiq;

extern "C" size_t vsiq_mse_search_workspace_bytes(const vsiq_layout* layout, int n_candidates) {
    MseGeom g;
    if (!make_mse_geom(layout, n_candidates, 1, 8, 1, 0.0, &g)) return 0;
    size_t bytes = mse_records_bytes(layout, g, 1);
    if (mse_ci_eligible(layout) && make_mse_geom(layout, n_candidates, 4, 8, 1, 0.0, &g)) {
        const size_t b4 = mse_records_bytes(layout, g, 4);
        bytes = b4 > bytes ? b4 : bytes;
    }
    return kWsHeader + bytes;
}

extern "C" int vsiq_mse_search(const float* x, const vsiq_layout* layout, const double* stats, double* state, int bits,
                               int symmetric, double eps, int n_candidates, double* err, double* alpha,
                               void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    if (!x || !stats || !state || bits < 2 || bits > 8) return VSIQ_ERR_INVALID_ARG;
    if (int e = check_layout(layout)) return e;
    MseGeom g;
    const int G = mse_ci_eligible(layout) && (reinterpret_cast<uintptr_t>(x) & 15u) == 0 ? 4 : 1;
    if (!make_mse_geom(layout, n_candidates, G, bits, symmetric ? 1 : 0, eps, &g)) return VSIQ_ERR_INVALID_ARG;
    const size_t need = kWsHeader + mse_records_bytes(layout, g, G);
    if (!workspace || workspace_bytes < need) return VSIQ_ERR_WORKSPACE;
    vsiq_qparams q = {};
    q.qmin = symmetric ? -(1 << (bits - 1)) : 0;
    q.qmax = symmetric ? (1 << (bits - 1)) - 1 : (1 << bits) - 1;
    QPDev qd;
    if (int e = fill_qp(&q, &qd)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    double* records = (double*)((char*)workspace + kWsHeader);
    const unsigned grid = (unsigned)((layout->channels / G) * g.kc);
    if (G == 4)
        mse_search_kernel<4><<<grid, kThreads, 0, st>>>(x, g, stats, state, qd, records);
    else
        mse_search_kernel<1><<<grid, kThreads, 0, st>>>(x, g, stats, state, qd, records);
    if (cudaError_t e = cudaGetLastError()) return (int)e;
    const unsigned fgrid = (unsigned)((layout->channels + kWarps - 1) / kWarps);
    return (int)launch_pdl(mse_finalize_kernel, dim3(fgrid), dim3(kThreads), 0, st, g, G, (const double*)records, stats,
                           state, err, alpha);
}
