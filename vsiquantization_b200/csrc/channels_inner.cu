// channels_inner.cu -- the fake-quant epilogue for CHANNEL-INNERMOST tensors (NHWC / torch.channels_last, cuDNN's
// native layout on sm_100): [rows = N*H*W][C] with the channel fastest.
//
//   forward : y  = fq(act(x + bias[c]))                       act = relu or identity, qparams per tensor or per channel
//   backward: dx = STE/LSQ gradient w.r.t. x (act mask included), dscale / dzero_point (per tensor or per channel),
//             dbias[c] = sum over rows of dx                  -- the conv's bias gradient, for free in the same pass
//
// Same arithmetic as fake_quant.cu (reference: quantizers/uniform.py:47-55,95,242-271; lsq_module.py:147-173,254-274,
// 317-358); the bias add is the fused layer's conv bias (modules/fused.py:124-130) moved into this epilogue so that its
// gradient (ATen: a separate full-tensor reduction per layer) rides along with dx.
//
// Mapping (ci_common.cuh): C % 4 == 0 and C <= 1024.  A 128-bit vector holds 4 consecutive channels; with G = C/4 vector
// groups per row only T = (256 / G) * G threads of a CTA are active, so thread t ALWAYS owns channel group t % G: its four
// channels' qparams, bias and gradient accumulators live in registers for the whole kernel.  CTAs are persistent and own
// a range of steps (static equal split by default, 16-step tiles from an atomic queue as the alternative); accumulators
// are carried in fp64 and flushed ONCE per CTA; records are combined in a fixed order (deterministic) by the last CTA
// (narrow records) or by ci_finalize_kernel, launched as a programmatic dependent of the streaming kernel.
//
// Roofline: HBM; 8 B/element forward, 12 B/element backward, as for the NCHW kernels.
#include <stdlib.h>

#include "ci_common.cuh"

namespace vsiq {

struct CiOut {
    void* dscale;
    void* dzp;
    float* dbias;
    int ds_f64, dz_f64;
    double gs_host;
    const float* gs_dev;
};

// Record layout per CTA (doubles): [E: nq][B: nq][DB: C]   with nq = C (per-channel qparams) or 1 (per tensor)
// What an entry's store needs besides the combined sum: the gradient scale and, for a zero-point entry, its channel's
// step size and range test.  Loaded separately so that the combine kernel can fetch it BEFORE it waits for the
// streaming grid (these values do not depend on it).
struct CiEntryParams {
    double gs;
    float s;
    bool cz;
};
__device__ __forceinline__ CiEntryParams ci_entry_params(const CiOut& o, const QPDev& qpd, bool pcq, int C, int idx) {
    const int nq = pcq ? C : 1;
    CiEntryParams e;
    e.gs = o.gs_host * (o.gs_dev ? (double)__ldg(o.gs_dev) : 1.0);
    e.s = 0.0f;
    e.cz = true;
    if (idx >= nq && idx < 2 * nq && o.dzp) {
        const QP p = load_qp(qpd, idx - nq);
        const float zr = rintf(p.zf);
        e.s = p.s;
        e.cz = qpd.zp_learned ? ((zr >= p.lo) && (zr <= p.hi)) : true;
    }
    return e;
}
__device__ __forceinline__ void ci_store(const CiOut& o, const CiEntryParams& e, bool pcq, bool bias, int C, int idx, double v) {
    // idx addresses the record: [0,nq) E, [nq,2nq) B, [2nq, 2nq+C) DB
    const int nq = pcq ? C : 1;
    if (idx < nq) {
        if (o.dscale) {
            const double ds = e.gs * v;
            if (o.ds_f64) ((double*)o.dscale)[idx] = ds; else ((float*)o.dscale)[idx] = (float)ds;
        }
    } else if (idx < 2 * nq) {
        if (o.dzp) {
            const int c = idx - nq;
            const double dz = e.cz ? -e.gs * (double)e.s * v : 0.0;  // sum (g*s)*(m-1) = -s * sum over clamped g
            if (o.dz_f64) ((double*)o.dzp)[c] = dz; else ((float*)o.dzp)[c] = (float)dz;
        }
    } else if (bias && o.dbias) {
        o.dbias[idx - 2 * nq] = (float)v;
    }
}
__device__ __forceinline__ void ci_store(const CiOut& o, const QPDev& qpd, bool pcq, bool bias, int C, int idx, double v) {
    ci_store(o, ci_entry_params(o, qpd, pcq, C, idx), pcq, bias, C, idx, v);
}

// CTA-wide barrier over the first kThreads threads: plain __syncthreads() for 256-thread CTAs, named barrier 1 when a
// producer warp rides along (ci_bwd_tma_kernel) and must not take part.
template <bool NAMED>
__device__ __forceinline__ void ci_sync() {
    if (NAMED)
        asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
    else
        __syncthreads();
}

// Combine 32 consecutive record entries [base, base+32) over n_rec per-CTA records (last-CTA path, narrow records): warp
// w sums records w, w+8, ... (each read is one coalesced 256-byte row segment, four independent chains per thread), then
// the eight slices are added in a fixed order.  Deterministic.  s_part: [kWarps][32] doubles of shared memory.
template <bool NAMED = false>
__device__ __forceinline__ void ci_combine_chunk(const double* records, int width, uint32_t n_rec, int base,
                                                 double (*s_part)[32], const CiOut& o, const QPDev& qpd, bool pcq,
                                                 bool bias, int C) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int idx = base + lane;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    if (idx < width) {
        uint32_t r = warp;
        for (; r + 3 * kWarps < n_rec; r += 4 * kWarps) {
            a0 += __ldcg(records + (size_t)r * width + idx);
            a1 += __ldcg(records + (size_t)(r + kWarps) * width + idx);
            a2 += __ldcg(records + (size_t)(r + 2 * kWarps) * width + idx);
            a3 += __ldcg(records + (size_t)(r + 3 * kWarps) * width + idx);
        }
        for (; r < n_rec; r += kWarps) a0 += __ldcg(records + (size_t)r * width + idx);
    }
    ci_sync<NAMED>();
    s_part[warp][lane] = (a0 + a1) + (a2 + a3);
    ci_sync<NAMED>();
    if (warp == 0 && idx < width) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) v += s_part[w][lane];
        ci_store(o, qpd, pcq, bias, C, idx, v);
    }
}

// Wide records: one CTA per 8 record entries (ci_combine8_sum), resident early as a programmatic dependent of the
// streaming kernel.
__global__ void __launch_bounds__(kThreads)
    ci_finalize_kernel(const void* ws, int width, uint32_t n_rec, CiOut o, QPDev qpd, int pcq, int bias, int C) {
    __shared__ double s_part[kWarps][kCombineEntries];
    const double* records = (const double*)((const char*)ws + kWsHeader);
    const int idx = blockIdx.x * kCombineEntries + (threadIdx.x & 7);
    CiEntryParams ep = {};
    if (threadIdx.x < kCombineEntries && idx < width) ep = ci_entry_params(o, qpd, pcq != 0, C, idx);  // before the wait
    pdl_wait();  // the streaming grid has completed and its records are visible
    const double v = ci_combine8_sum(records, (size_t)width, n_rec, (size_t)idx, idx < width, s_part);
    if (threadIdx.x < kCombineEntries && idx < width) ci_store(o, ep, pcq != 0, bias != 0, C, idx, v);
}

// The last CTA to leave resets the ticket (and the tile counter of the dynamic schedule) for the next launch.
__device__ __forceinline__ void ci_leave(void* ws) {
    if (threadIdx.x == 0) {
        unsigned int* counter = (unsigned int*)ws + 1;
        unsigned int tk = atomicAdd((unsigned int*)ws, 1u);
        if (tk == gridDim.x - 1) {
            *(unsigned int*)ws = 0;
            *counter = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------------- forward
template <bool PCQ, bool BIAS, int ACT, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads, 3)  // 80 registers, 3 CTAs per SM: measured 5.84 -> 6.39 TB/s on [64,32,320,320]
    ci_fwd_kernel(const float* __restrict__ x, const float* __restrict__ bias, float* __restrict__ y, CiGeom geo,
                  QPDev qpd, void* ws) {
    const int t = threadIdx.x;
    const bool active = t < geo.threads;
    const int c0 = (t % geo.groups) * kCiVec;
    constexpr int kU = 2 * kCiUnroll;  // forward: one input, so twice the loads in flight
    __shared__ uint32_t s_tile[2];
    CiSched sc;
    CiRange r = ci_sched_first(geo, sc, ws, s_tile, t);
    QP p[kCiVec];
    float bv[kCiVec];
    bool all_fast = true;
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        p[e] = load_qp(qpd, PCQ ? c0 + e : 0);
        all_fast = all_fast && p[e].fast;
        bv[e] = (BIAS && active) ? __ldg(bias + c0 + e) : 0.0f;
    }
    const uint32_t seed = guard_seed(all_fast);
    const int64_t stride = (int64_t)geo.threads * kCiVec;  // floats between a thread's consecutive vectors
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
                    if (s + j >= r.s1) continue;
                    Vec4 out;
                    FastGuard guard;
                    guard_reset(guard, seed);
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        const float xe = act_fwd<ACT>(BIAS ? __fadd_rn(vin[j].v[e], bv[e]) : vin[j].v[e]);
                        guard_note(guard, xe);
                        out.v[e] = dequant(elem_fast<GRID>(xe, p[e]).q, p[e]);
                    }
                    if (guard_bad(guard)) {
#pragma unroll
                        for (int e = 0; e < kCiVec; ++e) {
                            const float xe = act_fwd<ACT>(BIAS ? __fadd_rn(vin[j].v[e], bv[e]) : vin[j].v[e]);
                            out.v[e] = dequant(elem_slow<GRID>(xe, p[e]).q, p[e]);
                        }
                    }
                    st4(const_cast<float*>(xp) + j * stride + dy, out);
                }
            }
        }
        if (!ci_sched_next(geo, sc, s_tile, t, r)) break;
    }
    if (geo.sched == kCiDynamic) ci_leave(ws);
}

// Two outputs from one pass: y = fq1(act(x + bias[c])) (this layer's quantised output) and y2 = fq2(y), the SAME tensor
// as the next layer's `quantize_inp` step would produce from y with ITS activation quantiser (fake_quantize.py:44-45:
// `if self.quantize_inp: x = self.quantize_activation(x)`).  The second stage quantises the value that is about to be
// stored, so it is bit-identical to a separate fake-quant launch over y, for 4 more bytes per element instead of 8
// and one launch less.  Two CTAs per SM: the second set of qparams lives in registers next to the first.
template <bool PCQ, bool BIAS, int ACT, bool PCQ2>
__global__ void __launch_bounds__(kThreads, 2)
    ci_fwd2_kernel(const float* __restrict__ x, const float* __restrict__ bias, float* __restrict__ y,
                   float* __restrict__ y2, CiGeom geo, QPDev qpd, QPDev qpd2, void* ws) {
    const int t = threadIdx.x;
    const bool active = t < geo.threads;
    const int c0 = (t % geo.groups) * kCiVec;
    constexpr int kU = 2 * kCiUnroll;
    __shared__ uint32_t s_tile[2];
    CiSched sc;
    CiRange r = ci_sched_first(geo, sc, ws, s_tile, t);
    QP p[kCiVec], p2[kCiVec];
    float bv[kCiVec];
    bool all_fast = true, all_fast2 = true;
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        p[e] = load_qp(qpd, PCQ ? c0 + e : 0);
        p2[e] = load_qp(qpd2, PCQ2 ? c0 + e : 0);
        all_fast = all_fast && p[e].fast;
        all_fast2 = all_fast2 && p2[e].fast;
        bv[e] = (BIAS && active) ? __ldg(bias + c0 + e) : 0.0f;
    }
    const uint32_t seed = guard_seed(all_fast), seed2 = guard_seed(all_fast2);
    const int64_t stride = (int64_t)geo.threads * kCiVec;
    const int64_t dy = y - x, dy2 = y2 - x;
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
                    if (s + j >= r.s1) continue;
                    Vec4 out, out2;
                    FastGuard guard, guard2;
                    guard_reset(guard, seed);
                    guard_reset(guard2, seed2);
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        const float xe = act_fwd<ACT>(BIAS ? __fadd_rn(vin[j].v[e], bv[e]) : vin[j].v[e]);
                        guard_note(guard, xe);
                        out.v[e] = dequant(elem_fast(xe, p[e]).q, p[e]);
                    }
                    if (guard_bad(guard)) {
#pragma unroll
                        for (int e = 0; e < kCiVec; ++e) {
                            const float xe = act_fwd<ACT>(BIAS ? __fadd_rn(vin[j].v[e], bv[e]) : vin[j].v[e]);
                            out.v[e] = dequant(elem_slow(xe, p[e]).q, p[e]);
                        }
                    }
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        guard_note(guard2, out.v[e]);
                        out2.v[e] = dequant(elem_fast(out.v[e], p2[e]).q, p2[e]);
                    }
                    if (guard_bad(guard2)) {
#pragma unroll
                        for (int e = 0; e < kCiVec; ++e) out2.v[e] = dequant(elem_slow(out.v[e], p2[e]).q, p2[e]);
                    }
                    st4(const_cast<float*>(xp) + j * stride + dy, out);
                    st4(const_cast<float*>(xp) + j * stride + dy2, out2);
                }
            }
        }
        if (!ci_sched_next(geo, sc, s_tile, t, r)) break;
    }
    if (geo.sched == kCiDynamic) ci_leave(ws);
}

// ------------------------------------------------------------------------------ BatchNorm normalise (+ ReLU)
// y = act(x * a[c] + b[c]),  a = gamma / sqrt(var + eps),  b = beta - mean * a: what training-mode BatchNorm computes for
// a layer that kept its BN (is_fuse_bn=False) once the batch moments are known -- the second half of every layer of
// reestimate_BN_stats (utils/estimate_bn.py:79-91: bn in training mode, then modules/fused.py:131-134 applies the ReLU).
// One read and one write instead of ATen's batch_norm pass plus a separate ReLU pass.
template <bool RELU>
__global__ void __launch_bounds__(kThreads, 3)
    ci_affine_kernel(const float* __restrict__ x, const float* __restrict__ mean, const float* __restrict__ var,
                     const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float* __restrict__ y,
                     CiGeom geo, void* ws) {
    const int t = threadIdx.x;
    const bool active = t < geo.threads;
    const int c0 = (t % geo.groups) * kCiVec;
    constexpr int kU = 2 * kCiUnroll;
    __shared__ uint32_t s_tile[2];
    CiSched sc;
    CiRange r = ci_sched_first(geo, sc, ws, s_tile, t);
    float a[kCiVec], b[kCiVec];
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        const int c = active ? c0 + e : 0;
        const float g = gamma ? __ldg(gamma + c) : 1.0f;
        a[e] = __fdiv_rn(g, __fsqrt_rn(__fadd_rn(__ldg(var + c), eps)));
        b[e] = __fsub_rn(beta ? __ldg(beta + c) : 0.0f, __fmul_rn(__ldg(mean + c), a[e]));
    }
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
                    if (s + j >= r.s1) continue;
                    Vec4 out;
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        const float v = __fmaf_rn(vin[j].v[e], a[e], b[e]);
                        out.v[e] = RELU ? max_nan(v, 0.0f) : v;
                    }
                    st4(const_cast<float*>(xp) + j * stride + dy, out);
                }
            }
        }
        if (!ci_sched_next(geo, sc, s_tile, t, r)) break;
    }
    if (geo.sched == kCiDynamic) ci_leave(ws);
}

// --------------------------------------------------------------------------------------------- backward
// The element arithmetic of one vector (four channels): dx, and the LSQ terms when WANT_DS.
template <bool BIAS, int ACT, bool WANT_DS, int GRID = kGridInt>
__device__ __forceinline__ void ci_bwd_vec(const Vec4& vx, const Vec4& vg, const QP (&p)[kCiVec], const float (&bv)[kCiVec],
                                           uint32_t seed, Vec4& out, float (&te)[kCiVec], float (&tb)[kCiVec],
                                           float (&tdb)[kCiVec]) {
    float ve[kCiVec], vbz[kCiVec];
    FastGuard guard;
    guard_reset(guard, seed);
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        const float xb = BIAS ? __fadd_rn(vx.v[e], bv[e]) : vx.v[e];
        const float xe = act_fwd<ACT>(xb);
        const float ge = vg.v[e];
        guard_note(guard, xe);
        guard_note(guard, ge);
        const Elem el = elem_fast<GRID>(xe, p[e]);
        out.v[e] = act_bwd<ACT>(xb, dx_fast(ge, el.m, p[e]));
        if (WANT_DS) {
            // g * ((q - z) - m * v): v is finite on this path, so the masked product is a predicated subtraction
            float dd = __fsub_rn(el.q, p[e].z);
            if (el.m) dd = __fsub_rn(dd, el.v);
            ve[e] = __fmul_rn(ge, dd);
            vbz[e] = el.m ? 0.0f : ge;
        }
    }
    if (guard_bad(guard)) {  // rare: IEEE sequences for the whole vector
#pragma unroll
        for (int e = 0; e < kCiVec; ++e) {
            const float xb = BIAS ? __fadd_rn(vx.v[e], bv[e]) : vx.v[e];
            const float xe = act_fwd<ACT>(xb);
            const float ge = vg.v[e];
            const Elem el = elem_slow<GRID>(xe, p[e]);
            out.v[e] = act_bwd<ACT>(xb, dx_slow(ge, el.m, p[e]));
            if (WANT_DS) {
                const float dd = __fsub_rn(el.q, p[e].z);
                const float mv = __fmul_rn(el.v, el.m ? 1.0f : 0.0f);
                ve[e] = ge * (dd - mv);
                vbz[e] = el.m ? 0.0f : ge;
            }
        }
    }
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        if (WANT_DS) {
            te[e] += ve[e];
            tb[e] += vbz[e];
        }
        if (BIAS) tdb[e] += out.v[e];
    }
}

// One flush per CTA: fixed-order reduction over the threads that share a channel group, record write, and (narrow
// records) ticket + combine by the last CTA.  Runs in the first kThreads threads; s_acc is [kThreads][12] doubles.
template <bool PCQ, bool BIAS, bool WANT_DS, bool NAMED>
__device__ __forceinline__ void ci_bwd_flush(const double (&acc_e)[kCiVec], const double (&acc_b)[kCiVec],
                                             const double (&acc_db)[kCiVec], double (*s_acc)[3 * kCiVec],
                                             const CiGeom& geo, const QPDev& qpd, void* ws, const CiOut& o,
                                             int use_ticket, int t, bool active) {
    double* records = ws_partials(ws);
    const int C = geo.channels;
    const uint32_t n_ctas = gridDim.x, cta = blockIdx.x;
    if (!WANT_DS && !BIAS) {  // plain STE: nothing to reduce
        if (geo.sched == kCiDynamic) ci_leave(ws);
        return;
    }
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        s_acc[t][e] = active ? acc_e[e] : 0.0;
        s_acc[t][kCiVec + e] = active ? acc_b[e] : 0.0;
        s_acc[t][2 * kCiVec + e] = active ? acc_db[e] : 0.0;
    }
    __shared__ double s_pt[2];
    if (WANT_DS && !PCQ) {  // per-tensor sums: warp shuffle, then the eight warps in order
        __shared__ double s_w[kWarps][2];
        double e = 0.0, b = 0.0;
        if (active) {
            e = (acc_e[0] + acc_e[1]) + (acc_e[2] + acc_e[3]);
            b = (acc_b[0] + acc_b[1]) + (acc_b[2] + acc_b[3]);
        }
        e = warp_sum(e);
        b = warp_sum(b);
        if ((t & 31) == 0) {
            s_w[t >> 5][0] = e;
            s_w[t >> 5][1] = b;
        }
        ci_sync<NAMED>();
        if (t == 0) {
            double es = 0.0, bs = 0.0;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) {
                es += s_w[w][0];
                bs += s_w[w][1];
            }
            s_pt[0] = es;
            s_pt[1] = bs;
        }
    }
    ci_sync<NAMED>();
    const int nq = PCQ ? C : 1;
    const int width = 2 * nq + (BIAS ? C : 0);
    double* rec = records + (size_t)cta * width;
    const int reps = geo.threads / geo.groups;
    for (int idx = t; idx < width; idx += kThreads) {
        double s = 0.0;
        if (idx < 2 * nq) {
            const int which = idx < nq ? 0 : 1;
            if (WANT_DS) {
                if (PCQ) {
                    const int c = idx - which * nq;
                    for (int k = 0; k < reps; ++k) s += s_acc[k * geo.groups + c / kCiVec][which * kCiVec + (c % kCiVec)];
                } else {
                    s = s_pt[which];
                }
            }
        } else {
            const int c = idx - 2 * nq;
            for (int k = 0; k < reps; ++k) s += s_acc[k * geo.groups + c / kCiVec][2 * kCiVec + (c % kCiVec)];
        }
        rec[idx] = s;
    }
    // wide records under the static schedule: nothing else to do -- ci_finalize_kernel (a programmatic dependent of this
    // grid) sees the records once the grid has completed
    if (!use_ticket && geo.sched != kCiDynamic) return;
    __shared__ int s_last;
    __threadfence();
    ci_sync<NAMED>();
    if (threadIdx.x == 0) {
        unsigned int* counter = (unsigned int*)ws + 1;
        unsigned int tk = atomicAdd((unsigned int*)ws, 1u);
        s_last = (tk == n_ctas - 1);
        if (s_last) {
            *(unsigned int*)ws = 0;
            *counter = 0;
        }
    }
    ci_sync<NAMED>();
    if (!s_last || !use_ticket) return;
    __threadfence();
    double(*s_part)[32] = reinterpret_cast<double(*)[32]>(&s_acc[0][0]);  // s_acc is free again
    for (int base = 0; base < width; base += 32)
        ci_combine_chunk<NAMED>(records, width, n_ctas, base, s_part, o, qpd, PCQ, BIAS, C);
}

// Direct-load backward: used when grad_output is pitched (a channel slice of a wider NHWC tensor, which is what the
// backward of torch.cat hands out: row r of g starts at g + r * g_pitch) or when VSIQ_CI_TMA=0.
template <bool PCQ, bool BIAS, int ACT, bool WANT_DS, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads, 2)
    ci_bwd_kernel(const float* __restrict__ x, const float* __restrict__ bias, const float* __restrict__ g,
                  float* __restrict__ dx, CiGeom geo, QPDev qpd, void* ws, CiOut o, int use_ticket, int64_t g_pitch) {
    __shared__ double s_acc[kThreads][3 * kCiVec];  // per thread: e[4], b[4], db[4]
    const int t = threadIdx.x;
    const bool active = t < geo.threads;
    const int c0 = (t % geo.groups) * kCiVec;
    pdl_launch_dependents();
    __shared__ uint32_t s_tile[2];
    CiSched sc;
    CiRange r = ci_sched_first(geo, sc, ws, s_tile, t);
    QP p[kCiVec];
    float bv[kCiVec];
    bool all_fast = true;
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        p[e] = load_qp(qpd, PCQ ? c0 + e : 0);
        all_fast = all_fast && p[e].fast;
        bv[e] = (BIAS && active) ? __ldg(bias + c0 + e) : 0.0f;
    }
    const uint32_t seed = guard_seed(all_fast);
    double acc_e[kCiVec], acc_b[kCiVec], acc_db[kCiVec];
    float te[kCiVec], tb[kCiVec], tdb[kCiVec];  // fp32 partials, folded into the fp64 sums every 16 vectors
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        acc_e[e] = acc_b[e] = acc_db[e] = 0.0;
        te[e] = tb[e] = tdb[e] = 0.0f;
    }
    // thread t's vector of step s sits in row s * (T/G) + t/G: x / dx advance by T vectors per step, g by T/G pitched rows
    const int rows_per_step = geo.threads / geo.groups;
    const int64_t stride = (int64_t)geo.threads * kCiVec;
    const int64_t gstride = (int64_t)rows_per_step * g_pitch;
    const int64_t ddx = dx - x;
    for (;;) {
        if (active) {
            const float* xp = x + ((int64_t)r.s0 * geo.threads + t) * kCiVec;
            const float* gp = g + ((int64_t)r.s0 * rows_per_step + t / geo.groups) * g_pitch + c0;
            int it = 0;
#pragma unroll 1
            for (uint32_t s = r.s0; s < r.s1; s += kCiUnroll, xp += kCiUnroll * stride, gp += kCiUnroll * gstride) {
                Vec4 vx[kCiUnroll], vg[kCiUnroll];
#pragma unroll
                for (int j = 0; j < kCiUnroll; ++j) {
                    if (s + j < r.s1) {
                        vx[j] = ld4(xp + j * stride);
                        vg[j] = ld4(gp + j * gstride);
                    }
                }
#pragma unroll
                for (int j = 0; j < kCiUnroll; ++j) {
                    if (s + j >= r.s1) continue;
                    Vec4 out;
                    ci_bwd_vec<BIAS, ACT, WANT_DS, GRID>(vx[j], vg[j], p, bv, seed, out, te, tb, tdb);
                    st4(const_cast<float*>(xp) + j * stride + ddx, out);
                }
                if ((++it & (kCiBatches - 1)) == 0 || s + kCiUnroll >= r.s1) {
#pragma unroll
                    for (int e = 0; e < kCiVec; ++e) {
                        if (WANT_DS) {
                            acc_e[e] += (double)te[e];
                            acc_b[e] += (double)tb[e];
                        }
                        if (BIAS) acc_db[e] += (double)tdb[e];
                        te[e] = tb[e] = tdb[e] = 0.0f;
                    }
                }
            }
        }
        if (!ci_sched_next(geo, sc, s_tile, t, r)) break;
    }
    ci_bwd_flush<PCQ, BIAS, WANT_DS, false>(acc_e, acc_b, acc_db, s_acc, geo, qpd, ws, o, use_ticket, t, active);
}

// ---------------------------------------------------------------------------------------------------------------
// Backward with TMA-staged inputs (dense grad_output).  ncu on the direct-load kernel: the warps wait on global loads
// ("long scoreboard" is the top stall, issue slots 58 % used) while 128 registers per thread cap the CTA count at two, so
// neither more warps nor more loads per thread are available.  Here a producer warp streams x and g through a ring of
// kCiStages shared-memory stages with bulk asynchronous copies (cp.async.bulk -> mbarrier complete_tx), the eight
// consumer warps read 128-bit vectors from shared memory: bytes in flight per SM no longer cost registers, and the
// consumers never touch a global load.  One stage = one unit of up to kCiUnroll steps (T * kCiUnroll vectors, <= 16 KB per
// input); the producer walks the CTA's step range (static split) or claims 16-step tiles from the atomic queue.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kCiStages = 3;
constexpr int kCiMinPitchedRowBytes = 512;  // measured: 2 KB rows 42 vs 52 us, 512 B rows 132 vs 138, 256 B rows 93 vs 79
constexpr uint32_t kCiDone = 0xffffffffu;
constexpr uint32_t kCiTileEnd = 0x80000000u;  // the consumers fold their fp32 partials at tile ends (deterministic sums)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ Vec4 lds4(const float* p) {
    Vec4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3])
                 : "r"(smem_u32(p)));
    return r;
}

struct CiRing {
    uint64_t full[kCiStages];
    uint64_t empty[kCiStages];
    uint32_t nvec[kCiStages];  // vectors of the unit parked in the stage | kCiTileEnd on the last unit of a tile
                               // (kCiDone: no more work)
    int64_t vec0[kCiStages];   // its first vector
};

template <bool PCQ, bool BIAS, int ACT, bool WANT_DS, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads + 32, 2)
    ci_bwd_tma_kernel(const float* __restrict__ x, const float* __restrict__ bias, const float* __restrict__ g,
                      float* __restrict__ dx, CiGeom geo, QPDev qpd, void* ws, CiOut o, int use_ticket, int64_t g_pitch) {
    extern __shared__ __align__(128) unsigned char ci_smem[];  // kCiStages x [x unit | g unit]; later the flush scratch
    __shared__ CiRing ring;
    const int t = threadIdx.x;
    const int unit_vecs = geo.threads * kCiUnroll;          // vectors per full unit (per input)
    const uint32_t unit_bytes = (uint32_t)unit_vecs * 16u;  // <= 16 KB
    if (t == 0) {
#pragma unroll
        for (int s = 0; s < kCiStages; ++s) {
            mbar_init(&ring.full[s], 1);        // the producer's arrive (+ the bytes of its two copies)
            mbar_init(&ring.empty[s], kWarps);  // one arrive per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (t >= kThreads) {  // ---------------------------------------------------------------- producer warp
        // Lane 0 claims the work and owns the barriers; all 32 lanes issue copies when grad_output is pitched (one bulk
        // copy per row of g: a channel slice of a wider NHWC tensor is contiguous only within a row).  Control flow is
        // warp-uniform: the range comes from lane 0 by shuffle.
        const int lane = t - kThreads;
        const bool pitched = g_pitch != geo.channels;
        const uint32_t row_bytes = (uint32_t)geo.channels * 4u;
        if (lane == 0) pdl_launch_dependents();
        unsigned int* counter = (unsigned int*)ws + 1;
        int stage = 0;
        uint32_t phase = 0;
        uint32_t s0 = 0, s1 = 0, tile = blockIdx.x;
        if (geo.sched == kCiStatic) {
            const uint64_t S = (uint64_t)geo.steps;
            s0 = (uint32_t)(S * blockIdx.x / gridDim.x);
            s1 = (uint32_t)(S * (blockIdx.x + 1) / gridDim.x);
        }
        for (;;) {
            if (geo.sched != kCiStatic) {
                if (geo.sched == kCiDynamic) {
                    if (lane == 0) tile = atomicAdd(counter, 1u);
                    tile = __shfl_sync(0xffffffffu, tile, 0);
                }
                if (tile >= geo.n_tiles) break;
                s0 = tile * (uint32_t)geo.tile_steps;
                s1 = s0 + geo.tile_steps < (uint32_t)geo.steps ? s0 + geo.tile_steps : (uint32_t)geo.steps;
                tile += gridDim.x;  // interleaved: the next tile of this CTA
            }
            for (uint32_t s = s0; s < s1; s += kCiUnroll) {
                const int64_t v0 = (int64_t)s * geo.threads;
                int64_t nv = (int64_t)((s + kCiUnroll < s1 ? s + kCiUnroll : s1) - s) * geo.threads;
                if (v0 + nv > geo.n_vec) nv = geo.n_vec - v0;
                const uint32_t bytes = (uint32_t)nv * 16u;
                unsigned char* xs = ci_smem + (size_t)stage * 2 * unit_bytes;
                if (lane == 0) {
                    mbar_wait(&ring.empty[stage], phase ^ 1u);  // the consumers have drained this stage
                    ring.vec0[stage] = v0;
                    ring.nvec[stage] = (uint32_t)nv | (s + kCiUnroll >= s1 ? kCiTileEnd : 0u);
                    mbar_arrive_expect_tx(&ring.full[stage], 2 * bytes);
                    bulk_load(xs, x + v0 * kCiVec, bytes, &ring.full[stage]);
                    if (!pitched) bulk_load(xs + unit_bytes, g + v0 * kCiVec, bytes, &ring.full[stage]);
                }
                if (pitched) {
                    __syncwarp();  // the stage is free and its transaction count is armed
                    const int64_t row0 = v0 / geo.groups;
                    const int rows = (int)(nv / geo.groups);
                    for (int r = lane; r < rows; r += 32)
                        bulk_load(xs + unit_bytes + (size_t)r * row_bytes, g + (row0 + r) * g_pitch, row_bytes,
                                  &ring.full[stage]);
                }
                if (++stage == kCiStages) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
            if (geo.sched == kCiStatic) break;
        }
        if (lane == 0) {
            mbar_wait(&ring.empty[stage], phase ^ 1u);
            ring.nvec[stage] = kCiDone;
            mbar_arrive(&ring.full[stage]);
        }
        return;  // the producer warp takes no part in the flush (named barrier over the consumer threads)
    }

    // -------------------------------------------------------------------------------------- consumer warps
    const bool active = t < geo.threads;
    const int c0 = (t % geo.groups) * kCiVec;
    QP p[kCiVec];
    float bv[kCiVec];
    bool all_fast = true;
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        p[e] = load_qp(qpd, PCQ ? c0 + e : 0);
        all_fast = all_fast && p[e].fast;
        bv[e] = (BIAS && active) ? __ldg(bias + c0 + e) : 0.0f;
    }
    const uint32_t seed = guard_seed(all_fast);
    double acc_e[kCiVec], acc_b[kCiVec], acc_db[kCiVec];
    float te[kCiVec], tb[kCiVec], tdb[kCiVec];  // fp32 partials, folded into the fp64 sums every kCiBatches units
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        acc_e[e] = acc_b[e] = acc_db[e] = 0.0;
        te[e] = tb[e] = tdb[e] = 0.0f;
    }
    int stage = 0, it = 0;
    uint32_t phase = 0;
    for (;;) {
        mbar_wait(&ring.full[stage], phase);  // the unit's bytes have landed (or there is nothing left)
        const uint32_t tag = ring.nvec[stage];
        if (tag == kCiDone) break;
        const uint32_t nv = tag & ~kCiTileEnd;
        const int64_t v0 = ring.vec0[stage];
        const float* xs = (const float*)(ci_smem + (size_t)stage * 2 * unit_bytes);
        const float* gs = (const float*)(ci_smem + (size_t)stage * 2 * unit_bytes + unit_bytes);
        if (active) {
#pragma unroll
            for (int j = 0; j < kCiUnroll; ++j) {
                const uint32_t u = (uint32_t)(j * geo.threads + t);
                if (u >= nv) continue;
                const Vec4 vx = lds4(xs + (size_t)u * kCiVec);
                const Vec4 vg = lds4(gs + (size_t)u * kCiVec);
                Vec4 out;
                ci_bwd_vec<BIAS, ACT, WANT_DS, GRID>(vx, vg, p, bv, seed, out, te, tb, tdb);
                st4(dx + (v0 + u) * kCiVec, out);
            }
        }
        __syncwarp();
        if ((t & 31) == 0) mbar_arrive(&ring.empty[stage]);  // this warp has read everything it needs from the stage
        if ((++it & (kCiBatches - 1)) == 0 || (tag & kCiTileEnd)) {  // fold the fp32 partials into the fp64 running sums
            it = 0;
#pragma unroll
            for (int e = 0; e < kCiVec; ++e) {
                if (WANT_DS) {
                    acc_e[e] += (double)te[e];
                    acc_b[e] += (double)tb[e];
                }
                if (BIAS) acc_db[e] += (double)tdb[e];
                te[e] = tb[e] = tdb[e] = 0.0f;
            }
        }
        if (++stage == kCiStages) {
            stage = 0;
            phase ^= 1u;
        }
    }
#pragma unroll
    for (int e = 0; e < kCiVec; ++e) {
        if (WANT_DS) {
            acc_e[e] += (double)te[e];
            acc_b[e] += (double)tb[e];
        }
        if (BIAS) acc_db[e] += (double)tdb[e];
    }
    // every copy has landed and been consumed: the ring's memory is free for the flush scratch
    ci_sync<true>();
    ci_bwd_flush<PCQ, BIAS, WANT_DS, true>(acc_e, acc_b, acc_db, reinterpret_cast<double(*)[3 * kCiVec]>(ci_smem), geo, qpd,
                                           ws, o, use_ticket, t, active);
}

}  // namespace vsiq

using namespace vsiq;

extern "C" size_t vsiq_ci_workspace_bytes(int64_t rows, int64_t channels) {
    CiGeom g;
    if (!make_ci_geom(rows, channels, &g)) return 0;
    DeviceProps dp;
    int sms = get_device_props(&dp) ? 256 : dp.sm_count;
    return kWsHeader + (size_t)sms * 2 * (size_t)(3 * channels) * sizeof(double);
}

// The launch bodies of the integer entry points and their FP8 siblings (GRID: common.cuh)
template <int GRID>
static int ci_fwd_impl(const float* x, const float* bias, float* y, int64_t rows, int64_t channels, const vsiq_qparams* qp,
                       int64_t qp_channels, void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    QPDev qpd;
    if (int e = GRID == kGridInt ? fill_qp(qp, &qpd) : fill_qp_fp8(qp, GRID, &qpd)) return e;
    if (rows == 0) return VSIQ_OK;
    if (!x || !y) return VSIQ_ERR_INVALID_ARG;
    if (qp_channels != 1 && qp_channels != channels) return VSIQ_ERR_INVALID_ARG;
    CiGeom geo;
    if (!make_ci_geom(rows, channels, &geo)) return VSIQ_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) return VSIQ_ERR_UNSUPPORTED;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    const int grid = ci_pick_grid(&geo, dp.sm_count, 3, 2 * kCiUnroll);
    if (geo.sched == kCiDynamic && (!workspace || workspace_bytes < kWsHeader)) return VSIQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const bool pcq = qp_channels == channels && channels > 1, hb = bias != nullptr;
    const int act = qp->pre_op;  // VSIQ_PRE_* == kAct*
#define F(P, B, A) ci_fwd_kernel<P, B, A, GRID><<<grid, kThreads, 0, st>>>(x, bias, y, geo, qpd, workspace)
#define F2(P, B) { if (act == kActRelu) F(P, B, kActRelu); else if (act == kActSilu) F(P, B, kActSilu); else F(P, B, kActNone); }
    if (pcq) { if (hb) F2(true, true) else F2(true, false) } else { if (hb) F2(false, true) else F2(false, false) }
#undef F2
#undef F
    return (int)cudaGetLastError();
}

extern "C" int vsiq_ci_fake_quant_fwd(const float* x, const float* bias, float* y, int64_t rows, int64_t channels,
                                      const vsiq_qparams* qp, int64_t qp_channels, void* workspace,
                                      size_t workspace_bytes, vsiq_stream_t stream) {
    return ci_fwd_impl<kGridInt>(x, bias, y, rows, channels, qp, qp_channels, workspace, workspace_bytes, stream);
}

extern "C" int vsiq_ci_fp8_fake_quant_fwd(const float* x, const float* bias, float* y, int64_t rows, int64_t channels,
                                          const vsiq_qparams* qp, int64_t qp_channels, int fp8_format, void* workspace,
                                          size_t workspace_bytes, vsiq_stream_t stream) {
    if (fp8_format == VSIQ_FP8_E4M3)
        return ci_fwd_impl<VSIQ_FP8_E4M3>(x, bias, y, rows, channels, qp, qp_channels, workspace, workspace_bytes, stream);
    if (fp8_format == VSIQ_FP8_E5M2)
        return ci_fwd_impl<VSIQ_FP8_E5M2>(x, bias, y, rows, channels, qp, qp_channels, workspace, workspace_bytes, stream);
    return VSIQ_ERR_INVALID_ARG;
}

extern "C" int vsiq_ci_fake_quant_fwd2(const float* x, const float* bias, float* y, float* y2, int64_t rows,
                                       int64_t channels, const vsiq_qparams* qp, int64_t qp_channels,
                                       const vsiq_qparams* qp2, int64_t qp2_channels, void* workspace,
                                       size_t workspace_bytes, vsiq_stream_t stream) {
    QPDev qpd, qpd2;
    if (int e = fill_qp(qp, &qpd)) return e;
    if (int e = fill_qp(qp2, &qpd2)) return e;
    if (qp2->pre_op != VSIQ_PRE_NONE) return VSIQ_ERR_INVALID_ARG;  // the second stage quantises y as it is
    if (rows == 0) return VSIQ_OK;
    if (!x || !y || !y2 || y == y2) return VSIQ_ERR_INVALID_ARG;
    if (qp_channels != 1 && qp_channels != channels) return VSIQ_ERR_INVALID_ARG;
    if (qp2_channels != 1 && qp2_channels != channels) return VSIQ_ERR_INVALID_ARG;
    CiGeom geo;
    if (!make_ci_geom(rows, channels, &geo)) return VSIQ_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(y2)) & 15u)
        return VSIQ_ERR_UNSUPPORTED;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    const int grid = ci_pick_grid(&geo, dp.sm_count, 2, 2 * kCiUnroll);
    if (geo.sched == kCiDynamic && (!workspace || workspace_bytes < kWsHeader)) return VSIQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const bool pcq = qp_channels == channels && channels > 1, pcq2 = qp2_channels == channels && channels > 1;
    const bool hb = bias != nullptr;
    const int act = qp->pre_op;
#define F(P, B, A, Q) ci_fwd2_kernel<P, B, A, Q><<<grid, kThreads, 0, st>>>(x, bias, y, y2, geo, qpd, qpd2, workspace)
#define F1(P, B, A) { if (pcq2) F(P, B, A, true); else F(P, B, A, false); }
#define F2(P, B) { if (act == kActRelu) F1(P, B, kActRelu) else if (act == kActSilu) F1(P, B, kActSilu) else F1(P, B, kActNone) }
    if (pcq) { if (hb) F2(true, true) else F2(true, false) } else { if (hb) F2(false, true) else F2(false, false) }
#undef F2
#undef F1
#undef F
    return (int)cudaGetLastError();
}

extern "C" int vsiq_ci_bn_normalize(const float* x, const float* mean, const float* var, const float* gamma,
                                    const float* beta, float eps, float* y, int64_t rows, int64_t channels, int relu,
                                    void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    if (rows == 0) return VSIQ_OK;
    if (!x || !y || !mean || !var) return VSIQ_ERR_INVALID_ARG;
    CiGeom geo;
    if (!make_ci_geom(rows, channels, &geo)) return VSIQ_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) return VSIQ_ERR_UNSUPPORTED;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    const int grid = ci_pick_grid(&geo, dp.sm_count, 3, 2 * kCiUnroll);
    if (geo.sched == kCiDynamic && (!workspace || workspace_bytes < kWsHeader)) return VSIQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    if (relu)
        ci_affine_kernel<true><<<grid, kThreads, 0, st>>>(x, mean, var, gamma, beta, eps, y, geo, workspace);
    else
        ci_affine_kernel<false><<<grid, kThreads, 0, st>>>(x, mean, var, gamma, beta, eps, y, geo, workspace);
    return (int)cudaGetLastError();
}

template <int GRID>
static int ci_lsq_bwd_impl(const float* x, const float* bias, const float* g, float* dx, void* dscale, int dscale_dtype,
                           void* dzp, int dzp_dtype, float* dbias, int64_t rows, int64_t channels, const vsiq_qparams* qp,
                           int64_t qp_channels, double grad_scale_host, const float* grad_scale_dev, int64_t g_row_pitch,
                           void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    QPDev qpd;
    if (int e = GRID == kGridInt ? fill_qp(qp, &qpd) : fill_qp_fp8(qp, GRID, &qpd)) return e;
    if (qp_channels != 1 && qp_channels != channels) return VSIQ_ERR_INVALID_ARG;
    if (dzp && !dscale) return VSIQ_ERR_INVALID_ARG;
    if (g_row_pitch == 0) g_row_pitch = channels;
    if (g_row_pitch < channels || (g_row_pitch & 3)) return VSIQ_ERR_UNSUPPORTED;
    if (dbias && !bias) return VSIQ_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (rows == 0) {
        cudaError_t ce = cudaSuccess;
        if (dscale) ce = cudaMemsetAsync(dscale, 0, (size_t)qp_channels * (dscale_dtype ? 8 : 4), st);
        if (ce == cudaSuccess && dzp) ce = cudaMemsetAsync(dzp, 0, (size_t)qp_channels * (dzp_dtype ? 8 : 4), st);
        if (ce == cudaSuccess && dbias) ce = cudaMemsetAsync(dbias, 0, (size_t)channels * 4, st);
        return (int)ce;
    }
    if (!x || !g || !dx) return VSIQ_ERR_INVALID_ARG;
    CiGeom geo;
    if (!make_ci_geom(rows, channels, &geo)) return VSIQ_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(dx)) & 15u)
        return VSIQ_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < vsiq_ci_workspace_bytes(rows, channels)) return VSIQ_ERR_WORKSPACE;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    const int grid = ci_pick_grid(&geo, dp.sm_count, 2, kCiUnroll);
    const bool pcq = qp_channels == channels && channels > 1, hb = bias != nullptr;
    const int act = qp->pre_op;  // VSIQ_PRE_* == kAct*
    const bool want_ds = dscale != nullptr;
    CiOut o;
    o.dscale = dscale;
    o.dzp = dzp;
    o.dbias = dbias;
    o.ds_f64 = dscale_dtype == VSIQ_F64;
    o.dz_f64 = dzp_dtype == VSIQ_F64;
    o.gs_host = grad_scale_host;
    o.gs_dev = grad_scale_dev;
    const int width = 2 * (pcq ? (int)channels : 1) + (hb ? (int)channels : 0);
    const int use_ticket = width <= 64 ? 1 : 0;  // wider records: ci_finalize_kernel, one CTA per 8 entries
    // inputs staged through shared memory by bulk asynchronous copies (ci_bwd_tma_kernel); a pitched grad_output (channel
    // slice of a wider NHWC tensor) is fetched row by row, rows of >= kCiMinPitchedRowBytes only (below that the copies
    // are too small to pay and the direct-load kernel runs).  VSIQ_CI_TMA=0 forces the direct kernel, =2 the staged one.
    static const int tma_mode = []() { const char* e = getenv("VSIQ_CI_TMA"); return e ? atoi(e) : 1; }();
    const bool use_tma = tma_mode != 0 && (g_row_pitch == channels || tma_mode == 2 || channels * 4 >= kCiMinPitchedRowBytes);
    int cur_dev = 0;
    if (use_tma && cudaGetDevice(&cur_dev) != cudaSuccess) return VSIQ_ERR_NO_DEVICE;
    const size_t ring_bytes = (size_t)kCiStages * 2 * (size_t)geo.threads * kCiUnroll * 16;
    const size_t flush_bytes = sizeof(double) * kThreads * 3 * kCiVec;
    const size_t dyn_smem = ring_bytes > flush_bytes ? ring_bytes : flush_bytes;
#define B(P, H, R, D)                                                                                                      \
    {                                                                                                                      \
        if (use_tma) {                                                                                                     \
            if (cudaError_t ae = set_smem_once<ci_bwd_tma_kernel<P, H, R, D, GRID>>(cur_dev, 3 * 2 * 16384))             \
                return (int)ae;                                                                                            \
            ci_bwd_tma_kernel<P, H, R, D, GRID><<<grid, kThreads + 32, dyn_smem, st>>>(x, bias, g, dx, geo, qpd, workspace, \
                                                                                o,                                         \
                                                                                use_ticket, g_row_pitch);                 \
        } else {                                                                                                           \
            ci_bwd_kernel<P, H, R, D, GRID><<<grid, kThreads, 0, st>>>(x, bias, g, dx, geo, qpd, workspace, o, use_ticket,  \
                                                                 g_row_pitch);                                            \
        }                                                                                                                  \
    }
#define B3(P, H, R) { if (want_ds) B(P, H, R, true) else B(P, H, R, false) }
#define B2(P, H) { if (act == kActRelu) B3(P, H, kActRelu) else if (act == kActSilu) B3(P, H, kActSilu) else B3(P, H, kActNone) }
    if (pcq) { if (hb) B2(true, true) else B2(true, false) } else { if (hb) B2(false, true) else B2(false, false) }
#undef B2
#undef B3
#undef B
    if (cudaError_t le = cudaGetLastError()) return (int)le;
    if ((want_ds || hb) && !use_ticket) {
        const int fgrid = (width + kCombineEntries - 1) / kCombineEntries;
        if (cudaError_t fe = launch_pdl(ci_finalize_kernel, dim3(fgrid), dim3(kThreads), 0, st, (const void*)workspace, width,
                                        (uint32_t)grid, o, qpd, pcq ? 1 : 0, hb ? 1 : 0, (int)channels))
            return (int)fe;
    }
    return (int)cudaGetLastError();
}

extern "C" int vsiq_ci_lsq_bwd(const float* x, const float* bias, const float* g, float* dx, void* dscale,
                               int dscale_dtype, void* dzp, int dzp_dtype, float* dbias, int64_t rows, int64_t channels,
                               const vsiq_qparams* qp, int64_t qp_channels, double grad_scale_host,
                               const float* grad_scale_dev, int64_t g_row_pitch, void* workspace,
                               size_t workspace_bytes, vsiq_stream_t stream) {
    return ci_lsq_bwd_impl<kGridInt>(x, bias, g, dx, dscale, dscale_dtype, dzp, dzp_dtype, dbias, rows, channels, qp,
                                     qp_channels, grad_scale_host, grad_scale_dev, g_row_pitch, workspace, workspace_bytes,
                                     stream);
}

extern "C" int vsiq_ci_fp8_lsq_bwd(const float* x, const float* bias, const float* g, float* dx, void* dscale,
                                   int dscale_dtype, void* dzp, int dzp_dtype, float* dbias, int64_t rows, int64_t channels,
                                   const vsiq_qparams* qp, int64_t qp_channels, int fp8_format, double grad_scale_host,
                                   const float* grad_scale_dev, int64_t g_row_pitch, void* workspace,
                                   size_t workspace_bytes, vsiq_stream_t stream) {
    if (fp8_format != VSIQ_FP8_E4M3 && fp8_format != VSIQ_FP8_E5M2) return VSIQ_ERR_INVALID_ARG;
    if (dzp) return VSIQ_ERR_UNSUPPORTED;  // symmetric: no zero-point gradient
    return fp8_format == VSIQ_FP8_E4M3
               ? ci_lsq_bwd_impl<VSIQ_FP8_E4M3>(x, bias, g, dx, dscale, dscale_dtype, nullptr, dzp_dtype, dbias, rows,
                                                channels, qp, qp_channels, grad_scale_host, grad_scale_dev, g_row_pitch,
                                                workspace, workspace_bytes, stream)
               : ci_lsq_bwd_impl<VSIQ_FP8_E5M2>(x, bias, g, dx, dscale, dscale_dtype, nullptr, dzp_dtype, dbias, rows,
                                                channels, qp, qp_channels, grad_scale_host, grad_scale_dev, g_row_pitch,
                                                workspace, workspace_bytes, stream);
}
