// observer.cu -- kernels (1), (2) and (6): one-pass min/max + moment reduction with the observer
// state update and scale/zero-point computation folded into its last CTA; batched qparams; LSQ
// step-size initialisation; BN re-estimation finalisers.
//
// Reference semantics:
//   observe           observers/minmax.py:42-47 (x.min()/x.max(): NaN in -> NaN out; NaN never updates the
//                     running state; state starts at 0)
//   extra statistics  quantizers/quantization_manager.py:66-68 (mean|x|, mean x, unbiased std)
//   scale/zero-point  observers/minmax.py:67-74 (Python doubles; banker's round; zp not clamped)
//   LSQ init          quantizers/quantization_manager.py:112
//   BN re-estimation  utils/estimate_bn.py:56-99 (batch mean / UNBIASED batch var, summed, / count)
//
// Roofline: HBM, 4 algorithmic bytes per element (one read of x; the reference makes five passes).
#include "ci_common.cuh"
#include "reduce.cuh"

namespace vsiq {

struct StatsOp : OpBase {
    float mn, mx;        // NaN-propagating extrema (FMNMX.NAN): a NaN input sticks, exactly torch.min / torch.max -- one
                         // instruction each instead of a compare, a predicate merge and a plain min / max
    float fa, f1, f2;    // fp32 partials of the current vector (<= 8 elements)
    double sa, s1, s2;   // fp64 running sums of this thread
    __device__ __forceinline__ void reset() {
        mn = INFINITY;
        mx = -INFINITY;
        fa = f1 = f2 = 0.0f;
        sa = s1 = s2 = 0.0;
    }
    __device__ __forceinline__ void apply(const float (&a)[1], float (&)[1]) {
        const float x = a[0];
        mn = min_nan(mn, x);
        mx = max_nan(mx, x);
        fa += fabsf(x);
        f1 += x;
        f2 = fmaf(x, x, f2);
    }
    __device__ __forceinline__ void apply_slow(const float (&a)[1], float (&o)[1]) { apply(a, o); }
    __device__ __forceinline__ void vec_done() {
        sa += (double)fa;
        s1 += (double)f1;
        s2 += (double)f2;
        fa = f1 = f2 = 0.0f;
    }
    __device__ __forceinline__ StatsRec rec() const { return {mn, mx, sa, s1, s2}; }
};

// One record per tile; combined by the last CTA (small launches) or by finalize_kernel (large ones).
template <int GROUP, int V>
__global__ void __launch_bounds__(kThreads)
    observe_kernel(const float* __restrict__ x, Tiles tiles, int64_t outer, void* ws, ObserveOut o, int use_ticket) {
    __shared__ StatsRec s_red[kWarps];
    pdl_launch_dependents();
    const float* const in[1] = {x};
    float* const out[1] = {nullptr};
    double* partials = ws_partials(ws);
    const bool leader = GROUP == 32 ? (threadIdx.x & 31) == 0 : threadIdx.x == 0;

    StatsOp op;
    for (uint32_t t = group_index<GROUP>(); t < tiles.n_tiles; t += group_count<GROUP>()) {
        const TileCursor<GROUP> c = tile_at<GROUP>(tiles, t);
        op.reset();
        span_apply<GROUP, V, 1, 0>(in, out, c.offset, c.len, op);
        const StatsRec rec = block_record<GROUP>(op.rec(), s_red);
        if (leader) rec.store(partials + (size_t)t * StatsRec::kSlot);
    }
    if (!use_ticket) return;
    if (!last_cta_ticket((unsigned int*)ws, leader)) return;
    combine_in_last_cta(partials, tiles, outer, o, s_red);
}

// Per-tensor observer (rows == 1): persistent CTAs on the look-ahead tile queue, statistics carried in registers,
// one record per CTA (see lsq_bwd_pt_kernel).
template <int V>
__global__ void __launch_bounds__(kThreads)
    observe_pt_kernel(const float* __restrict__ x, Tiles tiles, void* ws, ObserveOut o) {
    __shared__ StatsRec s_red[kWarps];
    __shared__ uint32_t s_tile[2];
    const float* const in[1] = {x};
    float* const out[1] = {nullptr};
    double* partials = ws_partials(ws);
    unsigned int* counter = (unsigned int*)ws + 1;
    StatsOp op;
    op.reset();
    TileQueue tq;
    tq_init(tq, counter, tiles.n_tiles, s_tile);
    for (uint32_t t = tq_current(tq, s_tile); t < tiles.n_tiles; tq_advance(tq, s_tile), t = tq_current(tq, s_tile)) {
        const TileCursor<kThreads> c = tile_at<kThreads>(tiles, t);
        span_apply<kThreads, V, 1, 0>(in, out, c.offset, c.len, op);
    }
    const StatsRec rec = block_record<kThreads>(op.rec(), s_red);
    if (threadIdx.x == 0) rec.store(partials + (size_t)blockIdx.x * StatsRec::kSlot);
    if (!last_cta_ticket((unsigned int*)ws, threadIdx.x == 0)) return;
    if (threadIdx.x == 0) *counter = 0;
    combine_channel<kThreads>(partials, cta_records(gridDim.x), 1, 0, o, s_red);
}

// Per-channel observer on [outer, C, inner] with the channel-item schedule (PcGeom): one record per CTA.  This is the
// kernel behind BN re-estimation's per-batch moments (utils/estimate_bn.py:82) and per-channel calibration.
template <int GROUP, int V>
__global__ void __launch_bounds__(kThreads)
    observe_pc_kernel(const float* __restrict__ x, PcGeom geo, void* ws, ObserveOut o, int use_ticket) {
    __shared__ StatsRec s_red[kWarps];
    pdl_launch_dependents();
    const float* const in[1] = {x};
    float* const out[1] = {nullptr};
    double* partials = ws_partials(ws);
    const int warp = threadIdx.x >> 5;
    const uint32_t C = (uint32_t)geo.channels;
    const uint32_t c = blockIdx.x % C, j = blockIdx.x / C;
    StatsOp op;
    op.reset();
    const uint32_t first = GROUP == 32 ? j + (uint32_t)warp * geo.k : j;
    const uint32_t step = GROUP == 32 ? geo.k * kWarps : geo.k;
    for (uint32_t u = first; u < geo.units; u += step) {
        const uint32_t n = u / geo.chunks, ch = u - n * geo.chunks;
        const int64_t start = (int64_t)ch * geo.chunk;
        const int64_t rem = geo.inner - start;
        const int len = rem < geo.chunk ? (int)rem : geo.chunk;
        span_apply<GROUP, V, 1, 0>(in, out, ((int64_t)n * C + c) * geo.inner + start, len, op);
    }
    // whole CTA -> one record (warps hold different units of channel c)
    const StatsRec rec = block_record<kThreads>(op.rec(), s_red);
    if (threadIdx.x == 0) rec.store(partials + ((size_t)c * geo.k + j) * StatsRec::kSlot);
    if (!use_ticket) return;
    if (!last_cta_ticket((unsigned int*)ws, threadIdx.x == 0)) return;
    combine_in_last_cta(partials, item_records(geo), 1, o, s_red);
}

// ---------------------------------------------------------------------------------------------------------------
// Per-channel statistics of a CHANNEL-INNERMOST tensor ([rows = N*H*W][C], torch.channels_last): the observer pass of
// BN re-estimation (utils/estimate_bn.py:82) and of per-channel activation calibration without converting the conv
// output back to NCHW first (a conversion costs a read and a write of the tensor, this pass one read).  Same mapping as
// channels_inner.cu: thread t owns channel group t % G for the whole kernel, persistent CTAs steal tiles from the
// look-ahead queue, one record [5][C] per CTA, records combined per channel in a fixed order by ci_observe_finalize.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kCiObsFields = 5;  // min, max, sum|x|, sum x, sum x^2   (a NaN in the channel turns min and max into NaN)

__global__ void __launch_bounds__(kThreads, 3)
    ci_observe_kernel(const float* __restrict__ x, CiGeom geo, void* ws) {
    __shared__ double s_acc[kCiObsFields * kCiVec][kThreads];  // [field * 4 + e][thread]: conflict-free columns
    double* records = ws_partials(ws);
    const int t = threadIdx.x;
    const bool active = t < geo.threads;
    pdl_launch_dependents();
    float mn[kCiVec], mx[kCiVec];  // NaN-propagating (FMNMX.NAN): a NaN in the channel sticks, like torch.min / torch.max
    // the fp64 running sums live in this thread's column of shared memory (touched once per 16 vectors; keeps the kernel
    // at 80 registers = 3 CTAs per SM without spilling)
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        mn[e] = INFINITY;
        mx[e] = -INFINITY;
        s_acc[2 * kCiVec + e][t] = 0.0;
        s_acc[3 * kCiVec + e][t] = 0.0;
        s_acc[4 * kCiVec + e][t] = 0.0;
    }
    __shared__ uint32_t s_tile[2];
    CiSched sc;
    CiRange r = ci_sched_first(geo, sc, ws, s_tile, t);
    constexpr int kU = 2 * kCiUnroll;  // one input: twice the loads in flight
    const int64_t stride = (int64_t)geo.threads * kCiVec;
    for (;;) {
        if (active) {
            float fa[kCiVec], f1[kCiVec], f2[kCiVec];  // fp32 partials of 16 vectors (16 elements per channel per thread)
#pragma unroll
            for (int e = 0; e < kCiVec; ++e) fa[e] = f1[e] = f2[e] = 0.0f;
            int it = 0;
            const float* xp = x + ((int64_t)r.s0 * geo.threads + t) * kCiVec;
#pragma unroll 1
            for (uint32_t s = r.s0; s < r.s1; s += kU, xp += kU * stride) {
                Vec4 vin[kU];
#pragma unroll
                for (int j = 0; j < kU; ++j)
                    if (s + j < r.s1) vin[j] = ld4(xp + j * stride);
#pragma unroll
                for (int j = 0; j < kU; ++j) {
                    if (s + j >= r.s1) continue;
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        const float xv = vin[j].v[e];
                        mn[e] = min_nan(mn[e], xv);
                        mx[e] = max_nan(mx[e], xv);
                        fa[e] += fabsf(xv);
                        f1[e] += xv;
                        f2[e] = fmaf(xv, xv, f2[e]);
                    }
                }
                if ((++it & 1) == 0 || s + kU >= r.s1) {
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        s_acc[2 * kCiVec + e][t] += (double)fa[e];
                        s_acc[3 * kCiVec + e][t] += (double)f1[e];
                        s_acc[4 * kCiVec + e][t] += (double)f2[e];
                        fa[e] = f1[e] = f2[e] = 0.0f;
                    }
                }
            }
        }
        if (!ci_sched_next(geo, sc, s_tile, t, r)) break;
    }
    // ---- one record per CTA: fixed-order reduction over the threads that share a channel group
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        s_acc[0 * kCiVec + e][t] = active ? (double)mn[e] : (double)INFINITY;
        s_acc[1 * kCiVec + e][t] = active ? (double)mx[e] : (double)-INFINITY;  // sums: already in place
    }
    __syncthreads();
    const int C = geo.channels;
    const int reps = geo.threads / geo.groups;
    double* rec = records + (size_t)blockIdx.x * kCiObsFields * C;
    for (int idx = t; idx < kCiObsFields * C; idx += kThreads) {
        const int field = idx / C, c = idx - field * C;
        const double* col = s_acc[field * kCiVec + (c % kCiVec)];
        const int g0 = c / kCiVec;
        double v = col[g0];
        for (int k = 1; k < reps; ++k) {
            const double u = col[k * geo.groups + g0];
            if (field == 0) v = (v != v) ? v : ((u != u) ? u : (u < v ? u : v));
            else if (field == 1) v = (v != v) ? v : ((u != u) ? u : (u > v ? u : v));
            else v += u;
        }
        rec[idx] = v;
    }
    if (geo.sched == kCiDynamic && threadIdx.x == 0) {  // the last CTA to leave resets the ticket and the tile counter
        unsigned int* counter = (unsigned int*)ws + 1;
        unsigned int tk = atomicAdd((unsigned int*)ws, 1u);
        if (tk == gridDim.x - 1) {
            *(unsigned int*)ws = 0;
            *counter = 0;
        }
    }
}

// One CTA per 8 channels (a programmatic dependent of ci_observe_kernel, parked in griddepcontrol.wait until the records
// are complete): lane & 7 selects the channel, the 32 (warp, lane >> 3) phases walk the per-CTA records 32 apart (each
// load instruction of a warp reads four 64-byte segments), then a fixed-order shuffle + shared-memory reduction.
__global__ void __launch_bounds__(kThreads)
    ci_observe_finalize_kernel(const void* ws, int C, uint32_t n_rec, ObserveOut o) {
    __shared__ double s_red[kWarps][kCombineEntries][kCiObsFields];
    const double* records = (const double*)((const char*)ws + kWsHeader);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * kCombineEntries + (lane & 7);
    const uint32_t phase = (uint32_t)warp * 4u + (uint32_t)(lane >> 3);
    if (o.state && warp == 0 && lane < kCombineEntries && c < C)  // pull the running state towards L2 while waiting
        asm volatile("prefetch.global.L2 [%0];" ::"l"(o.state + (size_t)c * VSIQ_STATE_WIDTH));
    pdl_wait();
    float mn = INFINITY, mx = -INFINITY;
    double sa = 0.0, s1 = 0.0, s2 = 0.0;
    constexpr int kDepth = 7;  // records per pass: 35 independent loads in flight per thread, then the folds
    for (uint32_t r0 = phase; r0 < n_rec; r0 += 32u * kDepth) {
        double v[kDepth][kCiObsFields];
#pragma unroll
        for (int k = 0; k < kDepth; ++k) {
            const uint32_t r = r0 + 32u * (uint32_t)k;
            const bool ok = c < C && r < n_rec;
            const double* rec = records + (size_t)r * kCiObsFields * C + c;
            v[k][0] = ok ? __ldcg(rec) : (double)INFINITY;
            v[k][1] = ok ? __ldcg(rec + C) : (double)-INFINITY;
            v[k][2] = ok ? __ldcg(rec + 2 * C) : 0.0;
            v[k][3] = ok ? __ldcg(rec + 3 * C) : 0.0;
            v[k][4] = ok ? __ldcg(rec + 4 * C) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < kDepth; ++k) {
            mn = nanmin(mn, (float)v[k][0]);
            mx = nanmax(mx, (float)v[k][1]);
            sa += v[k][2];
            s1 += v[k][3];
            s2 += v[k][4];
        }
    }
#pragma unroll
    for (int d = 8; d <= 16; d <<= 1) {
        mn = nanmin(mn, __shfl_xor_sync(0xffffffffu, mn, d));
        mx = nanmax(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        sa += __longlong_as_double(__shfl_xor_sync(0xffffffffu, __double_as_longlong(sa), d));
        s1 += __longlong_as_double(__shfl_xor_sync(0xffffffffu, __double_as_longlong(s1), d));
        s2 += __longlong_as_double(__shfl_xor_sync(0xffffffffu, __double_as_longlong(s2), d));
    }
    if (lane < kCombineEntries) {
        s_red[warp][lane][0] = (double)mn;
        s_red[warp][lane][1] = (double)mx;
        s_red[warp][lane][2] = sa;
        s_red[warp][lane][3] = s1;
        s_red[warp][lane][4] = s2;
    }
    __syncthreads();
    if (warp == 0 && lane < kCombineEntries && c < C) {
        float a = (float)s_red[0][lane][0], bq = (float)s_red[0][lane][1];
        double x2 = s_red[0][lane][2], x3 = s_red[0][lane][3], x4 = s_red[0][lane][4];
#pragma unroll
        for (int w = 1; w < kWarps; ++w) {
            a = nanmin(a, (float)s_red[w][lane][0]);
            bq = nanmax(bq, (float)s_red[w][lane][1]);
            x2 += s_red[w][lane][2];
            x3 += s_red[w][lane][3];
            x4 += s_red[w][lane][4];
        }
        o.store(c, StatsRec{a, bq, x2, x3, x4});
    }
}

// Calibration epilogue of a fused layer on channels_last memory: y = act(pre(x)) written AND observed in the same pass
// (per-tensor observer of the layer's output: running min / max, scale / zero-point, the LSQ-init statistics).
//   PRE 0: y = act(x)
//   PRE 1: y = act(x + bias[c])                the BN-folded layer's conv bias (modules/fused.py:124-130)
//   PRE 2: y = act(x * a[c] + b[c])            inference-mode BatchNorm of a layer that kept its BN (fused.py:131-134),
//                                              a = gamma / sqrt(var + eps), b = beta - mean * a  (as ci_affine_kernel)
// then quantize_activation -> collect_qparameter -> observer.observe(y) (quantization_manager.py:55-71,
// observers/minmax.py:32-47).  ATen + a separate observer launch move 8 + 8 + 4 (bias form: relu pass; BN form:
// batch_norm + relu) or, with vsiq_ci_bn_normalize, 8 + 4 bytes per element; this kernel moves 8.  The values of y are
// those of the separate passes bit for bit, min / max are exact, the three sums are fp64 sums of 8-element fp32
// partials like every other observer kernel here (a different summation order, same error class).
template <int PRE, int ACT>
__global__ void __launch_bounds__(kThreads, 3)
    ci_epilogue_observe_kernel(const float* __restrict__ x, const float* __restrict__ p0, const float* __restrict__ var,
                               const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                               float* __restrict__ y, CiGeom geo, void* ws, ObserveOut o) {
    __shared__ StatsRec s_red[kWarps];
    __shared__ uint32_t s_tile[2];
    const int t = threadIdx.x;
    const bool active = t < geo.threads;
    const int c0 = (t % geo.groups) * kCiVec;
    constexpr int kU = 2 * kCiUnroll;
    CiSched sc;
    CiRange r = ci_sched_first(geo, sc, ws, s_tile, t);
    float a[kCiVec], b[kCiVec];
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        const int c = active ? c0 + e : 0;
        a[e] = 1.0f;
        b[e] = 0.0f;
        if (PRE == 1) b[e] = __ldg(p0 + c);
        if (PRE == 2) {
            const float g = gamma ? __ldg(gamma + c) : 1.0f;
            a[e] = __fdiv_rn(g, __fsqrt_rn(__fadd_rn(__ldg(var + c), eps)));
            b[e] = __fsub_rn(beta ? __ldg(beta + c) : 0.0f, __fmul_rn(__ldg(p0 + c), a[e]));
        }
    }
    StatsOp op;
    op.reset();
    const int64_t stride = (int64_t)geo.threads * kCiVec;
    const int64_t dy = y - x;
    for (;;) {
        if (active) {
            const float* xp = x + ((int64_t)r.s0 * geo.threads + t) * kCiVec;
#pragma unroll 1
            for (uint32_t s = r.s0; s < r.s1; s += kU, xp += kU * stride) {
                Vec4 vin[kU];
#pragma unroll
                for (int j = 0; j < kU; ++j)
                    if (s + j < r.s1) vin[j] = ld4(xp + j * stride);
#pragma unroll
                for (int j = 0; j < kU; ++j) {
                    if (s + j < r.s1) {
                        Vec4 out;
#pragma unroll
                        for (int e = 0; e < kCiVec; ++e) {
                            float v = vin[j].v[e];
                            if (PRE == 1) v = __fadd_rn(v, b[e]);
                            if (PRE == 2) v = __fmaf_rn(v, a[e], b[e]);
                            v = act_fwd<ACT>(v);
                            out.v[e] = v;
                            op.mn = min_nan(op.mn, v);
                            op.mx = max_nan(op.mx, v);
                            op.fa += fabsf(v);
                            op.f1 += v;
                            op.f2 = fmaf(v, v, op.f2);
                        }
                        st4(const_cast<float*>(xp) + j * stride + dy, out);
                    }
                    if (j & 1) op.vec_done();  // fp32 partials of 8 elements, then fp64
                }
            }
        }
        if (!ci_sched_next(geo, sc, s_tile, t, r)) break;
    }
    const StatsRec rec = block_record<kThreads>(op.rec(), s_red);
    double* partials = ws_partials(ws);
    if (threadIdx.x == 0) rec.store(partials + (size_t)blockIdx.x * StatsRec::kSlot);
    if (!last_cta_ticket((unsigned int*)ws, threadIdx.x == 0)) return;
    if (threadIdx.x == 0) *((unsigned int*)ws + 1) = 0;  // tile counter of the dynamic schedule
    combine_channel<kThreads>(partials, cta_records(gridDim.x), 1, 0, o, s_red);
}

__global__ void qparams_kernel(double* state, int64_t n, const int32_t* __restrict__ bits,
                               const int32_t* __restrict__ symmetric, double eps) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double* st = state + i * VSIQ_STATE_WIDTH;
    double sc, zp;
    qparams_from_minmax(st[0], st[1], bits[i], symmetric[i], eps, &sc, &zp);
    st[2] = sc;
    st[3] = zp;
}

__global__ void lsq_init_kernel(const double* __restrict__ state, int64_t C, int bits, void* out, int out_f64) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double* st = state + c * VSIQ_STATE_WIDTH;
    // quantization_manager.py:112: 2 * np.mean(mean_abs_x) / np.sqrt(2 ** (bits - 1) - 1)
    double s0 = 2.0 * (st[5] / st[4]) / sqrt((double)((1 << (bits - 1)) - 1));
    // a channel that only ever saw zeros (dead ReLU channel) would get step size 0 and turn 0/0 into NaN; torch's
    // own observers floor the scale at fp32 epsilon, so do that (never binding for the reference's per-tensor case)
    if (!(s0 >= 1.1920928955078125e-07)) s0 = (s0 != s0) ? s0 : 1.1920928955078125e-07;
    if (out_f64)
        ((double*)out)[c] = s0;
    else
        ((float*)out)[c] = (float)s0;
}

__global__ void bn_moments_finalize_kernel(const double* __restrict__ stats, double count, int64_t C,
                                           float* batch_mean, float* batch_var_biased, float* batch_var_unbiased,
                                           float* mean_sum, float* var_sum) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double s1 = stats[c * VSIQ_STATS_WIDTH + 3], s2 = stats[c * VSIQ_STATS_WIDTH + 4];
    const double mean = s1 / count;
    double var_b = s2 / count - mean * mean;
    var_b = var_b > 0.0 ? var_b : 0.0;
    const double var_u = var_b * (count / (count - 1.0));
    const float m32 = (float)mean, vu32 = (float)var_u;
    if (batch_mean) batch_mean[c] = m32;
    if (batch_var_biased) batch_var_biased[c] = (float)var_b;
    if (batch_var_unbiased) batch_var_unbiased[c] = vu32;
    if (mean_sum) mean_sum[c] = __fadd_rn(mean_sum[c], m32);   // estimate_bn.py:86
    if (var_sum) var_sum[c] = __fadd_rn(var_sum[c], vu32);      // estimate_bn.py:87
}

__global__ void bn_reestimate_finish_kernel(const float* __restrict__ mean_sum, const float* __restrict__ var_sum,
                                            float k, float* running_mean, float* running_var, int64_t C) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    running_mean[c] = __fdiv_rn(mean_sum[c], k);  // estimate_bn.py:96
    running_var[c] = __fdiv_rn(var_sum[c], k);    // estimate_bn.py:97
}

}  // namespace vsiq

using namespace vsiq;

extern "C" size_t vsiq_observe_workspace_bytes(const vsiq_layout* layout) {
    return reduce_workspace_bytes(layout, StatsRec::kSlot);
}

extern "C" int vsiq_observe(const float* x, const vsiq_layout* layout, double* stats, double* state, int bits,
                            int symmetric, double eps, void* workspace, size_t workspace_bytes,
                            vsiq_stream_t stream) {
    if (!x || (!stats && !state)) return VSIQ_ERR_INVALID_ARG;
    if (int e = check_layout(layout)) return e;
    if (state && (bits < 2 || bits > 8)) return VSIQ_ERR_INVALID_ARG;
    if (layout->outer * layout->channels * layout->inner == 0) return VSIQ_ERR_INVALID_ARG;  // min() of nothing
    if (!workspace || workspace_bytes < vsiq_observe_workspace_bytes(layout)) return VSIQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const bool warp_group = layout->inner < kWarpGroupMaxInner;
    const bool vec8 = aligned32(x);
    ObserveOut oo;
    oo.stats = stats;
    oo.state = state;
    oo.bits = bits;
    oo.symmetric = symmetric;
    oo.eps = eps;
    oo.count = (double)layout->outer * (double)layout->inner;
    DeviceProps dprops;
    if (int e = get_device_props(&dprops)) return e;
    PcGeom pc;
    if (layout->channels > 1 &&
        make_pc_geom(layout->outer, layout->channels, layout->inner, warp_group, dprops.sm_count, &pc) &&
        (size_t)pc.channels * pc.k * StatsRec::kSlot * sizeof(double) + kWsHeader <= workspace_bytes) {
        const int grid = (int)(pc.channels * pc.k);
        const int use_ticket = grid <= dprops.sm_count * 4 ? 1 : 0;  // else: combine kernel as a programmatic dependent
        if (warp_group) {
            if (vec8) observe_pc_kernel<32, 8><<<grid, kThreads, 0, st>>>(x, pc, workspace, oo, use_ticket);
            else observe_pc_kernel<32, 1><<<grid, kThreads, 0, st>>>(x, pc, workspace, oo, use_ticket);
        } else {
            if (vec8) observe_pc_kernel<kThreads, 8><<<grid, kThreads, 0, st>>>(x, pc, workspace, oo, use_ticket);
            else observe_pc_kernel<kThreads, 1><<<grid, kThreads, 0, st>>>(x, pc, workspace, oo, use_ticket);
        }
        if (!use_ticket) launch_finalize<StatsRec>(item_records(pc), 1, false, workspace, oo, st);
        return (int)cudaGetLastError();
    }
    Tiles tiles;
    if (layout->outer == 1 && layout->channels == 1 && !warp_group) {  // per tensor: persistent CTAs
        if (!make_tiles<kThreads>(1, 1, layout->inner, &tiles)) return VSIQ_ERR_INVALID_ARG;
        const uint32_t cap = (uint32_t)dprops.sm_count * 4u;
        const int grid = (int)(tiles.n_tiles < cap ? tiles.n_tiles : cap);
        if (vec8)
            observe_pt_kernel<8><<<grid, kThreads, 0, st>>>(x, tiles, workspace, oo);
        else
            observe_pt_kernel<1><<<grid, kThreads, 0, st>>>(x, tiles, workspace, oo);
        return (int)cudaGetLastError();
    }
#define CALL(G, V)                                                                                              \
    {                                                                                                           \
        const int mult = reduce_tile_mult<G>(layout->outer, layout->channels, layout->inner);                  \
        if (!make_tiles<G>(layout->outer, layout->channels, layout->inner, &tiles, mult))                       \
            return VSIQ_ERR_INVALID_ARG;                                                                        \
        uint32_t want = G == kThreads ? tiles.n_tiles : (tiles.n_tiles + kWarps - 1) / kWarps;                  \
        int grid = launch_grid(want);                                                                           \
        if (grid < 0) return -grid;                                                                             \
        const int use_ticket = (grid <= dprops.sm_count * 4 && tiles.n_tiles <= kTicketMaxRecords) ? 1 : 0;    \
        observe_kernel<G, V><<<grid, kThreads, 0, st>>>(x, tiles, layout->outer, workspace, oo, use_ticket);    \
        if (!use_ticket) launch_finalize<StatsRec>(tiles, layout->outer, true, workspace, oo, st);             \
    }
    if (warp_group) {
        if (vec8) CALL(32, 8) else CALL(32, 1)
    } else {
        if (vec8) CALL(kThreads, 8) else CALL(kThreads, 1)
    }
#undef CALL
    return (int)cudaGetLastError();
}

extern "C" size_t vsiq_ci_observe_workspace_bytes(int64_t rows, int64_t channels) {
    (void)rows;
    DeviceProps dp;
    int sms = 148;
    if (get_device_props(&dp) == 0) sms = dp.sm_count;
    return kWsHeader + (size_t)sms * 3 * (size_t)(kCiObsFields * channels) * sizeof(double);
}

extern "C" int vsiq_ci_observe(const float* x, int64_t rows, int64_t channels, double* stats, double* state, int bits,
                               int symmetric, double eps, void* workspace, size_t workspace_bytes,
                               vsiq_stream_t stream) {
    if (!x || (!stats && !state) || rows <= 0) return VSIQ_ERR_INVALID_ARG;
    if (state && (bits < 2 || bits > 8)) return VSIQ_ERR_INVALID_ARG;
    CiGeom geo;
    if (!make_ci_geom(rows, channels, &geo)) return VSIQ_ERR_UNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(x) & 15u) return VSIQ_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < vsiq_ci_observe_workspace_bytes(rows, channels)) return VSIQ_ERR_WORKSPACE;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    const uint32_t grid = (uint32_t)ci_pick_grid(&geo, dp.sm_count, 3, 2 * kCiUnroll);
    cudaStream_t st = (cudaStream_t)stream;
    ObserveOut oo;
    oo.stats = stats;
    oo.state = state;
    oo.bits = bits;
    oo.symmetric = symmetric;
    oo.eps = eps;
    oo.count = (double)rows;
    ci_observe_kernel<<<grid, kThreads, 0, st>>>(x, geo, workspace);
    if (cudaError_t err = cudaGetLastError()) return (int)err;
    const int fgrid = (int)((channels + kCombineEntries - 1) / kCombineEntries);
    return (int)launch_pdl(ci_observe_finalize_kernel, dim3(fgrid), dim3(kThreads), 0, st, (const void*)workspace,
                           (int)channels, grid, oo);
}

extern "C" int vsiq_ci_epilogue_observe(const float* x, const float* bias, const float* mean, const float* var,
                                        const float* gamma, const float* beta, float bn_eps, int act, float* y,
                                        int64_t rows, int64_t channels, double* stats, double* state, int bits,
                                        int symmetric, double eps, void* workspace, size_t workspace_bytes,
                                        vsiq_stream_t stream) {
    if (!x || !y || (!stats && !state) || rows <= 0) return VSIQ_ERR_INVALID_ARG;
    if (state && (bits < 2 || bits > 8)) return VSIQ_ERR_INVALID_ARG;
    if (bias && (mean || var)) return VSIQ_ERR_INVALID_ARG;  // one pre-op: bias add OR BatchNorm
    if ((mean == nullptr) != (var == nullptr)) return VSIQ_ERR_INVALID_ARG;
    if (act != VSIQ_PRE_NONE && act != VSIQ_PRE_RELU && act != VSIQ_PRE_SILU) return VSIQ_ERR_INVALID_ARG;
    CiGeom geo;
    if (!make_ci_geom(rows, channels, &geo)) return VSIQ_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) return VSIQ_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < vsiq_ci_observe_workspace_bytes(rows, channels)) return VSIQ_ERR_WORKSPACE;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    const uint32_t grid = (uint32_t)ci_pick_grid(&geo, dp.sm_count, 3, 2 * kCiUnroll);
    cudaStream_t st = (cudaStream_t)stream;
    ObserveOut oo;
    oo.stats = stats;
    oo.state = state;
    oo.bits = bits;
    oo.symmetric = symmetric;
    oo.eps = eps;
    oo.count = (double)rows * (double)channels;  // per-tensor statistics
    const int pre = mean ? 2 : (bias ? 1 : 0);
    const float* p0 = mean ? mean : bias;
#define K(P, A) ci_epilogue_observe_kernel<P, A><<<grid, kThreads, 0, st>>>(x, p0, var, gamma, beta, bn_eps, y, geo, workspace, oo)
#define KA(P) { if (act == VSIQ_PRE_RELU) K(P, kActRelu); else if (act == VSIQ_PRE_SILU) K(P, kActSilu); else K(P, kActNone); }
    if (pre == 2) KA(2) else if (pre == 1) KA(1) else KA(0)
#undef KA
#undef K
    return (int)cudaGetLastError();
}

extern "C" int vsiq_qparams_from_minmax(double* state, int64_t n, const int32_t* bits, const int32_t* symmetric,
                                        double eps, vsiq_stream_t stream) {
    if (!state || !bits || !symmetric || n < 0) return VSIQ_ERR_INVALID_ARG;
    if (n == 0) return VSIQ_OK;
    qparams_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(state, n, bits, symmetric, eps);
    return (int)cudaGetLastError();
}

extern "C" int vsiq_lsq_init_scale(const double* state, int64_t channels, int bits, void* scale_out, int scale_dtype,
                                   vsiq_stream_t stream) {
    if (!state || !scale_out || channels <= 0 || bits < 2 || bits > 8) return VSIQ_ERR_INVALID_ARG;
    if (scale_dtype != VSIQ_F32 && scale_dtype != VSIQ_F64) return VSIQ_ERR_INVALID_ARG;
    lsq_init_kernel<<<(unsigned)((channels + 127) / 128), 128, 0, (cudaStream_t)stream>>>(state, channels, bits,
                                                                                          scale_out, scale_dtype);
    return (int)cudaGetLastError();
}

extern "C" int vsiq_bn_moments_finalize(const double* stats, double count, int64_t channels, float* batch_mean,
                                        float* batch_var_biased, float* batch_var_unbiased, float* mean_sum,
                                        float* var_sum, vsiq_stream_t stream) {
    if (!stats || channels <= 0 || !(count > 1.0)) return VSIQ_ERR_INVALID_ARG;
    bn_moments_finalize_kernel<<<(unsigned)((channels + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        stats, count, channels, batch_mean, batch_var_biased, batch_var_unbiased, mean_sum, var_sum);
    return (int)cudaGetLastError();
}

extern "C" int vsiq_bn_reestimate_finish(const float* mean_sum, const float* var_sum, int64_t batch_count,
                                         float* running_mean, float* running_var, int64_t channels,
                                         vsiq_stream_t stream) {
    if (!mean_sum || !var_sum || !running_mean || !running_var || channels <= 0 || batch_count <= 0)
        return VSIQ_ERR_INVALID_ARG;
    bn_reestimate_finish_kernel<<<(unsigned)((channels + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        mean_sum, var_sum, (float)batch_count, running_mean, running_var, channels);
    return (int)cudaGetLastError();
}
