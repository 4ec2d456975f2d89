// common.cuh -- device-side building blocks shared by every kernel of libvsiq.so (sm_100a).
//
// All kernels on this path are HBM-bound streaming passes over fp32 tensors, so the whole design is
// about keeping enough 256-bit requests in flight per SM and never touching a byte twice:
//   * a tensor is walked as [rows = outer*channels][inner]; a "tile" is a contiguous chunk of ONE row,
//     so the quantisation parameters are uniform over a tile and the inner loop has no index math;
//   * a tile is owned by a thread GROUP: a whole CTA (256 threads, 8192-element tiles) for long rows,
//     or one warp (1024-element tiles) for short rows (20x20 feature maps, small filters), so short
//     rows still keep every SM's load queue full;
//   * inside a tile every thread issues UNROLL 256-bit loads per input (LDG.E.256, sm_100+) before any
//     arithmetic, computes, then issues 256-bit stores; ragged heads/tails and unaligned rows fall to
//     a scalar peel, fully unaligned tensors to the V=1 instantiation;
//   * grids launch one CTA per tile (or per 8 warp-tiles) and let the hardware scheduler balance the SMs:
//     measured on B200 this reaches the copy roofline where a static persistent grid stalls at ~85 %.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "../../include/vsiq.h"

namespace vsiq {

constexpr int kThreads = 256;  // threads per CTA
constexpr int kWarps = kThreads / 32;
constexpr int kVec = 8;        // fp32 lanes per 256-bit access
#ifndef VSIQ_UNROLL
#define VSIQ_UNROLL 2
#endif
#ifndef VSIQ_BATCHES
#define VSIQ_BATCHES 2
#endif
constexpr int kUnroll = VSIQ_UNROLL;            // vectors in flight per thread per input array
constexpr int kBatchesPerTile = VSIQ_BATCHES;   // batches per tile

template <int GROUP>
struct TileGeom {
    static constexpr int kBatch = GROUP * kVec * kUnroll;     // elements one group moves per batch
    static constexpr int kTile = kBatch * kBatchesPerTile;    // elements per tile
};
constexpr int kCtaTile = TileGeom<kThreads>::kTile;   // 8192
constexpr int kWarpTile = TileGeom<32>::kTile;        // 1024
constexpr int64_t kWarpGroupMaxInner = 2048;          // rows shorter than this are walked warp-per-tile

// ---------------------------------------------------------------------------------------------
// 256-bit / 32-bit streaming global accesses.  Inputs are read exactly once: bypass L1 allocation.
// ---------------------------------------------------------------------------------------------
template <int V>
struct Vec {
    float v[V];
};

__device__ __forceinline__ Vec<8> ld_stream(const float* p, Vec<8>*) {
    Vec<8> r;
#ifdef VSIQ_LOAD_EVICT_FIRST
    asm("ld.global.nc.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#else
    asm("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#endif
        : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]),
          "=f"(r.v[7])
        : "l"(p));
    return r;
}
__device__ __forceinline__ Vec<1> ld_stream(const float* p, Vec<1>*) {
    Vec<1> r;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r.v[0]) : "l"(p));
    return r;
}
__device__ __forceinline__ float ld_stream1(const float* p) {
    float r;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(float* p, const Vec<8>& r) {
#ifdef VSIQ_STORE_CS
    asm volatile("st.global.cs.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
#elif defined(VSIQ_STORE_NA)
    asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
#else
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
#endif
                 "f"(r.v[2]), "f"(r.v[3]), "f"(r.v[4]), "f"(r.v[5]), "f"(r.v[6]), "f"(r.v[7])
                 : "memory");
}
__device__ __forceinline__ void st_stream(float* p, const Vec<1>& r) { *p = r.v[0]; }

// ---------------------------------------------------------------------------------------------
// Quantisation parameters and the element arithmetic
// ---------------------------------------------------------------------------------------------
struct QPDev {  // kernel-argument mirror of vsiq_qparams
    const void* scale;
    const void* zp;
    int scale_f64;
    int zp_f64;
    float scale_host;
    float zp_host;
    int zp_learned;
    float lo;   // (float)qmin
    float hi;   // (float)qmax
    float tlo;  // smallest t with rint(t) >= qmin   (qmin - 0.5 if qmin is even, else the next float up)
    float thi;  // largest  t with rint(t) <= qmax   (qmax + 0.5 if qmax is even, else the next float down)
};

struct QP {  // per-tile (uniform) values
    float s;        // scale rounded to fp32 (ATen rounds the fp64 0-dim Parameter the same way)
    float r;        // RN(1/s), hoisted out of the element loop
    float z;        // effective zero-point used by the forward
    float zf;       // raw (float) zero-point parameter
    float lo, hi;   // integer range as floats
    float tlo, thi; // pre-rounding clamp thresholds (see QPDev)
    float zero_dx;  // (+0) / s : what a clamped-out element's dx is
    bool fast;      // |s| in [2^-40, 2^40]: the reciprocal-based exact division below is valid
};

// torch.clamp semantics: NaN propagates, -0.0 survives a 0 lower bound (fminf/fmaxf would lose both).
__device__ __forceinline__ float clamp_torch(float r, float lo, float hi) {
    r = (r < lo) ? lo : r;
    r = (r > hi) ? hi : r;
    return r;
}
// NaN-propagating min / max in one instruction each (FMNMX.NAN)
__device__ __forceinline__ float max_nan(float a, float b) {
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ float min_nan(float a, float b) {
    float d;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}

__device__ __forceinline__ QP load_qp(const QPDev& d, int64_t c) {
    QP q;
    q.lo = d.lo;
    q.hi = d.hi;
    q.tlo = d.tlo;
    q.thi = d.thi;
    if (d.scale)
        q.s = d.scale_f64 ? (float)__ldg((const double*)d.scale + c) : __ldg((const float*)d.scale + c);
    else
        q.s = d.scale_host;
    if (d.zp)
        q.zf = d.zp_f64 ? (float)__ldg((const double*)d.zp + c) : __ldg((const float*)d.zp + c);
    else
        q.zf = d.zp_host;
    q.z = d.zp_learned ? clamp_torch(rintf(q.zf), q.lo, q.hi) : q.zf;
    q.r = __frcp_rn(q.s);
    q.zero_dx = __fdiv_rn(0.0f, q.s);
    const float as = fabsf(q.s);
    q.fast = (as >= 9.094947017729282e-13f) && (as <= 1.099511627776e12f);  // 2^-40 .. 2^40
    return q;
}

// ---- exact arithmetic, IEEE instruction sequences (the "slow" path; also the definition) -----------
// Reference forward, one element (quantizers/uniform.py:54-55,95), every op individually rounded:
//   v = x / s;  t = v + z;  r = rint(t);  q = clamp(r, qmin, qmax);  y = (q - z) * s
// Reference backward (autograd): m = [qmin <= r <= qmax];  dx = where(m, g*s, 0) / s
struct Elem {
    float v;  // x / s
    float t;  // v + z
    float q;  // clamp(rint(t))
    bool m;   // rint(t) within [qmin, qmax]
};
// clamp(rint(t), lo, hi) == rint(clamp_t(t)) for every t, NaN and signed zeros included: below tlo the
// value is replaced by lo itself (rint(tlo) would be -0.0 for lo == 0 where torch gives +0.0), above thi
// by thi (rint(thi) == hi); inside, rint keeps the sign of a negative zero exactly like torch.
__device__ __forceinline__ float clamp_t(float t, const QP& p) { return min_nan(t < p.tlo ? p.lo : t, p.thi); }
__device__ __forceinline__ float quantize_t(float t, const QP& p) { return rintf(clamp_t(t, p)); }
__device__ __forceinline__ float dequant(float q, const QP& p) { return __fmul_rn(__fsub_rn(q, p.z), p.s); }

// ---- value grids ----------------------------------------------------------------------------------------------------
// GRID selects what the rounding step maps onto: kGridInt = the integers (rint), VSIQ_FP8_E4M3 / VSIQ_FP8_E5M2 = the
// finite values of that FP8 format (round to nearest, ties to an even mantissa).  An FP8 grid has no zero-point
// (t = v, so a -0.0 quotient keeps its sign) and its QP carries lo = tlo = -F, hi = thi = F: clamp_t is then
// torch.clamp(v, -F, F) and m = (clamp == v) its backward mask, inclusive at +-F and false for NaN.
constexpr int kGridInt = 0;
__host__ __device__ constexpr float fp8_max(int grid) { return grid == VSIQ_FP8_E4M3 ? 448.0f : 57344.0f; }

// Two floats (|v| <= F or NaN, i.e. already clamped) to two FP8 codes in one F2FP: `lo` in the low byte.  satfinite only
// matters for NaN (which stays NaN); the clamp has already kept every finite value inside the format's range.
template <int GRID>
__device__ __forceinline__ uint16_t fp8_pack2(float lo, float hi) {
    uint16_t p;
    if (GRID == VSIQ_FP8_E4M3)
        asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(p) : "f"(hi), "f"(lo));
    else
        asm("cvt.rn.satfinite.e5m2x2.f32 %0, %1, %2;" : "=h"(p) : "f"(hi), "f"(lo));
    return p;
}
// ... and their values back (exact: every FP8 value is an fp16 value is an fp32 value)
template <int GRID>
__device__ __forceinline__ void fp8_unpack2(uint16_t p, float& lo, float& hi) {
    uint32_t h;
    if (GRID == VSIQ_FP8_E4M3)
        asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h) : "h"(p));
    else
        asm("cvt.rn.f16x2.e5m2x2 %0, %1;" : "=r"(h) : "h"(p));
    asm("{.reg .f16 l, u; mov.b32 {l, u}, %2; cvt.f32.f16 %0, l; cvt.f32.f16 %1, u;}" : "=f"(lo), "=f"(hi) : "r"(h));
}
// the rounding step of the element functions: t is already clamp_t'ed
template <int GRID>
__device__ __forceinline__ float grid_round(float t) {
    if (GRID == kGridInt) return rintf(t);
    float q, unused;
    fp8_unpack2<GRID>(fp8_pack2<GRID>(t, 0.0f), q, unused);
    return q;
}

// The IEEE division is the only out-of-line piece: scalar in, scalar out, so the call passes everything in registers and
// no caller ever has to park its QP (or the op that holds it) in local memory for the sake of this rare path.
static __device__ __noinline__ float div_ieee(float a, float b) { return __fdiv_rn(a, b); }
template <int GRID = kGridInt>
__device__ __forceinline__ Elem elem_slow(float x, const QP& p) {
    Elem e;
    e.v = div_ieee(x, p.s);
    e.t = GRID == kGridInt ? __fadd_rn(e.v, p.z) : e.v;
    e.q = grid_round<GRID>(clamp_t(e.t, p));
    e.m = (e.t >= p.tlo) && (e.t <= p.thi);
    return e;
}
__device__ __forceinline__ float dx_slow(float g, bool m, const QP& p) {
    return div_ieee(m ? __fmul_rn(g, p.s) : 0.0f, p.s);
}

// ---- the same results without a per-element MUFU.RCP + FCHK + branch ------------------------------
// x / s by the hoisted r = RN(1/s) and exact-residual FMAs (the XU pipe issues only 16 lanes/clk/SM and
// would bound these kernels before HBM does):
//     q0 = RN(x*r); q1 = RN(q0 + (x - q0*s)*r)   -> faithful (relative error < 2^-46 before rounding)
//     q2 = RN(q1 + (x - q1*s)*r)                 -> correctly rounded (Markstein's theorem)
// The residuals are exact as long as nothing under/overflows: guaranteed for 2^-60 <= |x| < 2^61 and
// 2^-40 <= |s| <= 2^40.  x == 0 gives a zero whose sign is taken from q0 (= sign(x) xor sign(s)).
// Anything else (denormal, huge, inf, NaN, odd scale) fails the vector's FastGuard (below); the caller then recomputes
// the whole vector with the IEEE sequence above, so the branch is per 4-8 elements and almost never taken.
// dx = RN(RN(g*s) / s): g itself is a faithful quotient, so ONE correction step is exact:
//     gd = RN(g*s);  rho = gd - g*s (exact FMA);  dx = RN(g + rho*r), sign taken from g.
// tests/test_gpu_kernels.py::test_division_* check both against the IEEE division over ALL 2^32 inputs.
constexpr float kFastLo = 8.673617379884035e-19f;  // 2^-60
constexpr float kFastHi = 2.305843009213694e18f;   // 2^61

// The admissibility test is per VECTOR, not per element (three compares and a predicate merge per value made up a quarter
// of the backward's instructions and all of them issue on the ALU pipe, the busiest one):
//   hi = sum |v_i|          (FADD, FMA pipe)   hi < 2^61 implies every |v_i| < 2^61; NaN / inf make the test fail
//   lo = min (2*bits_i - 1) (unsigned)         zero maps to 0xffffffff, 0 < |v| < 2^-60 to a key below kTinyKey
// so "guard_ok" still guarantees 2^-60 <= |v| < 2^61 or v == 0 for every value noted -- the condition under which
// div_fast / dx_fast are proven exact -- and only errs towards the slow path (values within 16x of 2^61).
struct FastGuard {
    float hi;
    uint32_t lo;
};
constexpr uint32_t kTinyKey = 0x42ffffffu;  // 2 * bits(2^-60) - 1
__device__ __forceinline__ void guard_reset(FastGuard& g, uint32_t lo0 = 0xffffffffu) {
    g.hi = 0.0f;
    g.lo = lo0;  // 0 here poisons the guard: the way an out-of-range SCALE forces the IEEE path without a second test
}
// loop-invariant seed for guard_reset: all-ones when every scale of this thread admits the fast arithmetic
__device__ __forceinline__ uint32_t guard_seed(bool all_fast) { return all_fast ? 0xffffffffu : 0u; }
__device__ __forceinline__ void guard_note(FastGuard& g, float v) {
    g.hi = __fadd_rn(g.hi, fabsf(v));
    g.lo = min(g.lo, 2u * __float_as_uint(v) - 1u);
}
__device__ __forceinline__ bool guard_bad(const FastGuard& g) { return !(g.hi < kFastHi) || (g.lo < kTinyKey); }

__device__ __forceinline__ float div_fast(float x, const QP& p) {
    const float q0 = __fmul_rn(x, p.r);
    const float e0 = __fmaf_rn(-q0, p.s, x);
    const float q1 = __fmaf_rn(e0, p.r, q0);
    const float e1 = __fmaf_rn(-q1, p.s, x);
    const float q2 = __fmaf_rn(e1, p.r, q1);
    return copysignf(q2, q0);
}
template <int GRID = kGridInt>
__device__ __forceinline__ Elem elem_fast(float x, const QP& p) {
    Elem e;
    e.v = div_fast(x, p);
    e.t = GRID == kGridInt ? __fadd_rn(e.v, p.z) : e.v;
    const float tc = clamp_t(e.t, p);
    e.q = grid_round<GRID>(tc);
    e.m = (tc == e.t);  // clamped value unchanged <=> in range (false for NaN)
    return e;
}
__device__ __forceinline__ float dx_fast(float g, bool m, const QP& p) {
    const float gd = __fmul_rn(g, p.s);
    const float rho = __fmaf_rn(-g, p.s, gd);
    const float q = copysignf(__fmaf_rn(rho, p.r, g), g);
    return m ? q : p.zero_dx;
}

// Ops plug into span_apply through this protocol (one vector = up to 8 consecutive elements):
//   vec_begin()            reset per-vector state
//   apply(in, out)         one element, fast arithmetic; may raise the op's `bad` flag
//   vec_bad()              true -> span_apply calls vec_begin() and apply_slow() for the whole vector
//   vec_done()             commit per-vector partial sums
struct OpBase {
    __device__ __forceinline__ void vec_begin() {}
    __device__ __forceinline__ bool vec_bad() const { return false; }
    __device__ __forceinline__ void vec_done() {}
};

// observers/minmax.py:67-74 in IEEE doubles
__device__ __forceinline__ void qparams_from_minmax(double mn, double mx, int bits, int symmetric, double eps,
                                                    double* scale, double* zp) {
    if (symmetric) {
        const double a = fabs(mn), b = fabs(mx);
        const double max_abs = (b > a) ? b : a;  // Python max(a, b)
        *scale = max_abs / ((double)((1 << (bits - 1)) - 1) + eps);
        *zp = 0.0;
    } else {
        const double s = (mx - mn) / ((double)((1 << bits) - 1) + eps);
        *scale = s;
        *zp = rint(-mn / (s + eps));
    }
}

// The running-state rule of every min/max observer (observers/minmax.py:44-47, quantization_manager.py:66-68): one call's
// extrema and sums (count elements per channel) folded into st[0..7], scale / zero-point from the running extrema.
__device__ __forceinline__ void observer_state_update(double* st, float mn, float mx, double sa, double s1, double s2,
                                                      double count, int bits, int symmetric, double eps) {
    double run_min = st[0], run_max = st[1];
    if ((double)mn < run_min) run_min = (double)mn;  // NaN compares false: never updates (minmax.py:44-47)
    if ((double)mx > run_max) run_max = (double)mx;
    double sc, zp;
    qparams_from_minmax(run_min, run_max, bits, symmetric, eps, &sc, &zp);
    const double mean = s1 / count;
    const double var = (s2 - count * mean * mean) / (count - 1.0);  // torch.std: unbiased
    st[0] = run_min;
    st[1] = run_max;
    st[2] = sc;
    st[3] = zp;
    st[4] += 1.0;
    st[5] += sa / count;
    st[6] += mean;
    st[7] += sqrt(var > 0.0 ? var : 0.0);
}

// ---------------------------------------------------------------------------------------------
// Tile schedule
// ---------------------------------------------------------------------------------------------
struct Tiles {
    int64_t rows;       // outer * channels
    int64_t channels;
    int64_t inner;
    uint32_t chunks;    // tiles per row
    uint32_t n_tiles;   // rows * chunks  (< 2^31)
    int tile;           // elements per tile: TileGeom<GROUP>::kTile x tile_mult
};

template <int GROUP>
__host__ __device__ inline bool make_tiles(int64_t outer, int64_t channels, int64_t inner, Tiles* t,
                                           int tile_mult = 1) {
    t->rows = outer * channels;
    t->channels = channels;
    t->inner = inner;
    const int64_t max_tile = (int64_t)TileGeom<GROUP>::kTile * tile_mult;
    int64_t chunks = (inner + max_tile - 1) / max_tile;
    if (chunks <= 0) return false;
    // even out the chunks of a row: the smallest multiple of one batch that still covers the row in `chunks` tiles
    const int64_t batch = TileGeom<GROUP>::kBatch;
    int64_t tile = ((inner + chunks - 1) / chunks + batch - 1) / batch * batch;
    if (tile > max_tile) tile = max_tile;
    chunks = (inner + tile - 1) / tile;
    t->tile = (int)tile;
    int64_t n = t->rows * chunks;
    if (chunks <= 0 || n <= 0 || n >= (int64_t(1) << 31)) return false;
    t->chunks = (uint32_t)chunks;
    t->n_tiles = (uint32_t)n;
    return true;
}

template <int GROUP>
struct TileCursor {  // which tile this thread's group owns right now
    int64_t offset;  // element offset of the tile in the tensor
    int len;         // elements in the tile
    int64_t row;
    int64_t channel;
};

template <int GROUP>
__device__ __forceinline__ uint32_t group_index() {
    return GROUP == kThreads ? blockIdx.x : blockIdx.x * kWarps + (threadIdx.x >> 5);
}
template <int GROUP>
__device__ __forceinline__ uint32_t group_count() {
    return GROUP == kThreads ? gridDim.x : gridDim.x * kWarps;
}
template <int GROUP>
__device__ __forceinline__ int group_tid() {
    return GROUP == kThreads ? threadIdx.x : (threadIdx.x & 31);
}

template <int GROUP>
__device__ __forceinline__ TileCursor<GROUP> tile_at(const Tiles& t, uint32_t idx) {
    TileCursor<GROUP> c;
    uint32_t row = idx / t.chunks;
    uint32_t chunk = idx - row * t.chunks;
    int64_t start = (int64_t)chunk * t.tile;
    int64_t rem = t.inner - start;
    c.len = rem < t.tile ? (int)rem : t.tile;
    c.row = row;
    c.channel = t.channels == 1 ? 0 : (int64_t)(row % (uint32_t)t.channels);
    c.offset = (int64_t)row * t.inner + start;
    return c;
}

// ---------------------------------------------------------------------------------------------
// span_apply: run Op over `len` consecutive elements starting at element `off`, cooperatively by a
// GROUP of threads through the OpBase protocol above (apply per element, vec_begin / vec_bad / vec_done
// per vector of <= 8 elements, apply_slow when a vector needs the IEEE sequences).
// Base pointers are 32-byte aligned when V == 8 (checked on the host); the row offset need not be.
// ---------------------------------------------------------------------------------------------
template <int GROUP, int V, int NIN, int NOUT, class Op>
__device__ __forceinline__ void span_apply(const float* const (&in)[NIN],
                                           float* const (&out)[NOUT > 0 ? NOUT : 1], int64_t off,
                                           int len, Op& op) {
    const int tid = group_tid<GROUP>();
    int head = 0;
    if (V > 1) {
        head = (int)((V - (off & (V - 1))) & (V - 1));
        head = head < len ? head : len;
        if (tid < head) {
            float a[NIN], o[NOUT > 0 ? NOUT : 1];
#pragma unroll
            for (int k = 0; k < NIN; ++k) a[k] = ld_stream1(in[k] + off + tid);
            op.vec_begin();
            op.apply(a, o);
            if (op.vec_bad()) {
                op.vec_begin();
                op.apply_slow(a, o);
            }
            op.vec_done();
#pragma unroll
            for (int k = 0; k < NOUT; ++k) out[k][off + tid] = o[k];
        }
    }
    const int nvec = (len - head) / V;
    const int64_t vbase = off + head;
    for (int b = 0; b < nvec; b += GROUP * kUnroll) {
        Vec<V> vin[NIN][kUnroll];
        bool ok[kUnroll];
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const int vi = b + j * GROUP + tid;
            ok[j] = vi < nvec;
            if (ok[j]) {
#pragma unroll
                for (int k = 0; k < NIN; ++k)
                    vin[k][j] = ld_stream(in[k] + vbase + (int64_t)vi * V, (Vec<V>*)nullptr);
            }
        }
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            if (ok[j]) {
                const int vi = b + j * GROUP + tid;
                Vec<V> vout[NOUT > 0 ? NOUT : 1];
                op.vec_begin();
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    float a[NIN], o[NOUT > 0 ? NOUT : 1];
#pragma unroll
                    for (int k = 0; k < NIN; ++k) a[k] = vin[k][j].v[e];
                    op.apply(a, o);
#pragma unroll
                    for (int k = 0; k < NOUT; ++k) vout[k].v[e] = o[k];
                }
                if (op.vec_bad()) {  // rare: redo the vector with the IEEE sequences
                    op.vec_begin();
#pragma unroll
                    for (int e = 0; e < V; ++e) {
                        float a[NIN], o[NOUT > 0 ? NOUT : 1];
#pragma unroll
                        for (int k = 0; k < NIN; ++k) a[k] = vin[k][j].v[e];
                        op.apply_slow(a, o);
#pragma unroll
                        for (int k = 0; k < NOUT; ++k) vout[k].v[e] = o[k];
                    }
                }
                op.vec_done();
#pragma unroll
                for (int k = 0; k < NOUT; ++k) st_stream(out[k] + vbase + (int64_t)vi * V, vout[k]);
            }
        }
    }
    if (V > 1) {
        const int done = head + nvec * V;
        const int i = done + tid;
        if (i < len) {
            float a[NIN], o[NOUT > 0 ? NOUT : 1];
#pragma unroll
            for (int k = 0; k < NIN; ++k) a[k] = ld_stream1(in[k] + off + i);
            op.vec_begin();
            op.apply(a, o);
            if (op.vec_bad()) {
                op.vec_begin();
                op.apply_slow(a, o);
            }
            op.vec_done();
#pragma unroll
            for (int k = 0; k < NOUT; ++k) out[k][off + i] = o[k];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Reductions.  Within a warp: shuffles.  Across the warps of a CTA: shared memory, fixed order.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double shfl_down_d(double v, int d) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_down_sync(0xffffffffu, lo, d);
    hi = __shfl_down_sync(0xffffffffu, hi, d);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += shfl_down_d(v, d);
    return v;  // valid in lane 0
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    return v;
}
// NaN-propagating min / max (torch.min / torch.max semantics)
__device__ __forceinline__ float nanmin(float a, float b) { return (a != a) ? a : ((b != b) ? b : (b < a ? b : a)); }
__device__ __forceinline__ float nanmax(float a, float b) { return (a != a) ? a : ((b != b) ? b : (b > a ? b : a)); }
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = nanmin(v, __shfl_down_sync(0xffffffffu, v, d));
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = nanmax(v, __shfl_down_sync(0xffffffffu, v, d));
    return v;
}

// "last CTA finishes" ticket: returns true in every thread of the CTA that arrives last.  The partial
// records written by this CTA before the call are visible to the last CTA after it: only the threads that
// wrote a record fence (a fence in every thread would make each CTA wait for all of its streaming stores).
__device__ __forceinline__ bool last_cta_ticket(unsigned int* counter, bool wrote_record) {
    __shared__ int s_last;
    if (wrote_record) __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = atomicAdd(counter, 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) *counter = 0;  // leave the workspace ready for the next launch
    }
    __syncthreads();
    const bool last = s_last != 0;
    if (last) __threadfence();
    return last;
}

// Workspace layout shared by the reducing kernels: a 256-byte header (ticket) then fp64 partials.
constexpr size_t kWsHeader = 256;
__device__ __forceinline__ double* ws_partials(void* ws) { return (double*)((char*)ws + kWsHeader); }

// workspace header: [0] ticket, [1] tile counter (both left zero), records after kWsHeader.
// Dynamic tile scheduler with a one-tile look-ahead: thread 0 claims tile i+1 (atomicAdd) BEFORE the CTA works on
// tile i and publishes it afterwards, so the ~1 us round trip of the atomic hides behind a tile's worth of traffic
// and the CTA pays one __syncthreads per tile.
struct TileQueue {
    unsigned int* counter;
    uint32_t n_tiles;
    uint32_t ahead;  // thread 0 only: the tile claimed for the next iteration
    int buf;
};
__device__ __forceinline__ void tq_init(TileQueue& q, unsigned int* counter, uint32_t n_tiles, uint32_t* s_tile) {
    q.counter = counter;
    q.n_tiles = n_tiles;
    q.buf = 0;
    q.ahead = 0;
    if (threadIdx.x == 0) s_tile[0] = atomicAdd(counter, 1u);
    __syncthreads();
}
// returns the current tile (>= n_tiles: done) and starts claiming the next one
__device__ __forceinline__ uint32_t tq_current(TileQueue& q, const uint32_t* s_tile) {
    const uint32_t tile = s_tile[q.buf];
    if (threadIdx.x == 0 && tile < q.n_tiles) q.ahead = atomicAdd(q.counter, 1u);
    return tile;
}
__device__ __forceinline__ void tq_advance(TileQueue& q, uint32_t* s_tile) {
    if (threadIdx.x == 0) s_tile[q.buf ^ 1] = q.ahead;
    __syncthreads();
    q.buf ^= 1;
}

// Per-channel reductions over NCHW-like [outer, C, inner] tensors: "channel items".  All (row n, chunk) units of channel
// c are dealt round-robin to k CTAs, so a CTA only ever sees ONE channel: qparams are loaded once, the sums stay in
// registers across units and are flushed once (k records per channel) instead of once per tile.  GROUP = 256: the CTA
// cooperates on each unit (rows >= 2048 elements, 16384-element chunks); GROUP = 32: every warp takes its own units
// (short rows, one unit per row).
struct PcGeom {
    int64_t outer, channels, inner;
    uint32_t chunks;  // units per row
    uint32_t units;   // outer * chunks: units per channel
    uint32_t k;       // CTAs per channel
    int chunk;        // elements per unit
};
int pc_chunk_override();  // VSIQ_PC_CHUNK (abi.cu)
inline bool make_pc_geom(int64_t outer, int64_t channels, int64_t inner, bool warp_group, int sm_count, PcGeom* g) {
    if (outer <= 0 || channels <= 1 || inner <= 0) return false;
    g->outer = outer;
    g->channels = channels;
    g->inner = inner;
    // 16384-element units; halved (down to 4096) while the whole problem is only a wave or two of CTAs, so that mid-size
    // tensors (2^22 .. 2^24 elements) are not dealt out as 2.3 waves of fat CTAs with an idle tail
    int64_t chunk = warp_group ? inner : 16384;
    if (!warp_group) {
        const int64_t ov = pc_chunk_override();
        if (ov > 0)
            chunk = ov;
        else
            while (chunk > 4096 && channels * outer * ((inner + chunk - 1) / chunk) < (int64_t)sm_count * 3 * 6) chunk >>= 1;
    }
    const int64_t chunks = (inner + chunk - 1) / chunk;
    const int64_t units = outer * chunks;
    if (units >= (int64_t(1) << 31) || chunk >= (int64_t(1) << 31)) return false;
    g->chunk = (int)chunk;
    g->chunks = (uint32_t)chunks;
    g->units = (uint32_t)units;
    const int64_t per_cta = warp_group ? kWarps : 1;  // units a CTA works on concurrently
    // thousands of short rows with fewer units per channel than a CTA has warps ([4096, 1024] weights): a CTA per channel
    // would leave 7 of 8 warps idle -- the warp-per-tile schedule (one warp per row, eight rows per CTA) is the right one
    if (warp_group && units < kWarps) return false;
    int64_t k = ((int64_t)sm_count * 8 + channels - 1) / channels;
    const int64_t kmax = (units + per_cta - 1) / per_cta;
    if (k > kmax || kmax <= 4) k = kmax;  // a handful of units per channel: one CTA each (k < kmax would pair them unevenly)
    if (k < 1) k = 1;
    g->k = (uint32_t)k;
    if (channels * k >= (int64_t(1) << 31)) return false;
    return channels * k >= (int64_t)sm_count * 2;  // else too few CTAs: the per-tile schedule is the better one
}

// Record index of (channel c, item i) where a channel owns outer * chunks records: tile index is
// (o * C + c) * chunks + k.  32-bit math (n_tiles < 2^31); outer == 1 needs no division.
__device__ __forceinline__ uint32_t record_slot(const Tiles& t, uint32_t outer, uint32_t c, uint32_t i) {
    if (outer == 1) return c * t.chunks + i;
    const uint32_t o = i / t.chunks, k = i - o * t.chunks;
    return (o * (uint32_t)t.channels + c) * t.chunks + k;
}
constexpr uint32_t kTicketMaxRecords = 8192;     // above this the combine step gets its own multi-CTA launch
constexpr uint32_t kThreadCombineMaxItems = 32;  // <= this many records per channel: one thread per channel

// ---------------------------------------------------------------------------------------------
// Host-side helpers (abi)
// ---------------------------------------------------------------------------------------------
struct DeviceProps {
    int sm_count;
    int cc_major, cc_minor;
};
int get_device_props(DeviceProps* out);         // cached per device
int launch_grid(uint32_t n_ctas_wanted);   // one CTA per tile group unless VSIQ_GRID_WAVES caps it (tuning knob)
int single_wave_ctas();                    // CTAs that are co-resident for sure (SM count x 4)
// Reducing kernels pay a block reduction + a partial record per tile: pick the largest tile multiplier that
// still leaves >= 8 tiles per SM for the hardware scheduler to balance (1 for small problems).
template <int GROUP>
inline int reduce_tile_mult(int64_t outer, int64_t channels, int64_t inner) {
    const int64_t want = (int64_t)single_wave_ctas() * 2 * (GROUP == kThreads ? 1 : kWarps);
    for (int m = 8; m > 1; m >>= 1) {
        Tiles t;
        if (make_tiles<GROUP>(outer, channels, inner, &t, m) && (int64_t)t.n_tiles >= want) return m;
    }
    return 1;
}
bool aligned32(const void* p);
bool pdl_enabled();         // programmatic dependent launch for the combine kernels (VSIQ_PDL=0 disables; A/B knob)
int ci_sched_override();    // VSIQ_CI_SCHED=static|dynamic|interleaved -> 0 | 1 | 2, else -1 (automatic)
int ci_tile_override();     // VSIQ_CI_TILE=<steps per tile>, else 0 (automatic)
int pc_chunk_override();    // VSIQ_PC_CHUNK=<elements per unit of the NCHW per-channel schedule>, else 0 (automatic)
int check_layout(const vsiq_layout* l);
int fill_qp(const vsiq_qparams* in, QPDev* out);
int fill_qp_fp8(const vsiq_qparams* in, int fp8_format, QPDev* out);  // FP8 grid: qmin == qmax == 0, no zero-point

// opt in to > 48 KB of dynamic shared memory once per kernel instantiation and device (thread-safe)
template <auto Kernel>  // a non-type parameter: every instantiation of the kernel gets its own flags
static cudaError_t set_smem_once(int device, int bytes) {
    static std::mutex mu;
    static bool done[64];
    std::lock_guard<std::mutex> lk(mu);
    if (device < 0 || device >= 64) return cudaErrorInvalidDevice;
    if (done[device]) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done[device] = true;
    return e;
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL)
// ---------------------------------------------------------------------------------------------
// A reducing kernel that leaves wide per-CTA records is followed by a small combine kernel on the same stream.  The
// combine kernel is launched with cudaLaunchAttributeProgrammaticStreamSerialization: its CTAs become resident while the
// streaming kernel is still running (the streaming kernel signals launch_dependents in its prologue) and park in
// griddepcontrol.wait, which returns once the streaming grid has completed and its writes are visible.  The ~5 us
// launch-and-drain bubble of a plain back-to-back launch shrinks to the wake-up latency.  Both instructions are no-ops
// when the kernel was launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaError_t err = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
    if (err == cudaErrorInvalidValue && cfg.numAttrs) {  // attribute refused (driver / stream kind): launch without it
        (void)cudaGetLastError();
        cfg.numAttrs = 0;
        err = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
    }
    return err;
}

}  // namespace vsiq
