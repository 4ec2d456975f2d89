// fake_quant.cu -- kernels (3) and (4): uniform fake-quant forward, STE backward, LSQ backward with
// the per-channel step-size / zero-point gradients in the same pass, and the fused fwd+bwd sweep.
//
// Reference semantics reproduced here (bit-exact for y, codes and dx; fp64-accumulated sums):
//   forward   quantizers/uniform.py:54-55, :95          per channel: quantizers/lsq_module.py:254-274
//   backward  autograd of the above through RoundStraightThrough (uniform.py:258-271), torch.clamp and
//             ScaleGradient (uniform.py:242-255); grad-scale uniform.py:69-71 / lsq_module.py:327-340
//   FunLSQ    quantizers/uniform.py:144-150 (mask_mode 1)
//
// Roofline: HBM.  Algorithmic bytes per element: fwd 8 (read x, write y), bwd 12 (read g, read x,
// write dx; the mask is recomputed from x, per-channel outputs are O(C)), fused fwd+bwd 16.
#include "common.cuh"
#include "quant_ops.cuh"
#include "reduce.cuh"

namespace vsiq {

// -------------------------------------------------------------------------------------- kernels
template <int GROUP, int V, class Op, int NIN, int NOUT>
__device__ __forceinline__ void run_elementwise(const float* const (&in)[NIN], float* const (&out)[NOUT],
                                                const Tiles& tiles, const QPDev& qpd) {
    Op op;
    int64_t cur_channel = -1;
    for (uint32_t t = group_index<GROUP>(); t < tiles.n_tiles; t += group_count<GROUP>()) {
        const TileCursor<GROUP> c = tile_at<GROUP>(tiles, t);
        if (c.channel != cur_channel) {
            op.p = load_qp(qpd, c.channel);
            cur_channel = c.channel;
        }
        span_apply<GROUP, V, NIN, NOUT>(in, out, c.offset, c.len, op);
    }
}

template <int GROUP, int V, bool RELU, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads) fq_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                          Tiles tiles, QPDev qpd) {
    const float* const in[1] = {x};
    float* const out[1] = {y};
    run_elementwise<GROUP, V, FwdOp<RELU, GRID>, 1, 1>(in, out, tiles, qpd);
}

template <int GROUP, int V, bool RELU, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads) fq_bwd_ste_kernel(const float* __restrict__ x,
                                                              const float* __restrict__ g,
                                                              float* __restrict__ dx, Tiles tiles, QPDev qpd) {
    const float* const in[2] = {x, g};
    float* const out[1] = {dx};
    run_elementwise<GROUP, V, SteBwdOp<RELU, GRID>, 2, 1>(in, out, tiles, qpd);
}

template <int GROUP, int V>
__global__ void __launch_bounds__(kThreads) fq_fwd_bwd_kernel(const float* __restrict__ x,
                                                              const float* __restrict__ g, float* __restrict__ y,
                                                              float* __restrict__ dx, Tiles tiles, QPDev qpd) {
    const float* const in[2] = {x, g};
    float* const out[2] = {y, dx};
    run_elementwise<GROUP, V, FwdBwdOp, 2, 2>(in, out, tiles, qpd);
}

// Integer-code export (the deployment / ONNX path: the reference only ever holds the codes as floats, uniform.py:54).
// Same tiles as the forward; a thread turns one 256-bit load into 8 codes and stores them as ONE word: 8 x int4 in 32 bits
// (low nibble = even element), 8 x int8 in 64 bits, 8 x int16 in 128 bits; the fake-quantised values ride along as a
// 256-bit store when wanted.  Ragged heads / tails go element by element (byte by byte for int4: rows hold an even number
// of elements, so a byte never straddles two channels).  Roofline: HBM, 4.5 / 5 / 6 B per element (+4 with y).
template <int BITS>
struct CodePack;
template <>
struct CodePack<4> {
    __device__ static __forceinline__ void store8(void* codes, int64_t i, const int (&q)[8]) {
        uint32_t w = 0;
#pragma unroll
        for (int e = 0; e < 8; ++e) w |= ((uint32_t)q[e] & 0xfu) << (4 * e);
        *reinterpret_cast<uint32_t*>((uint8_t*)codes + (i >> 1)) = w;
    }
};
template <>
struct CodePack<8> {
    __device__ static __forceinline__ void store8(void* codes, int64_t i, const int (&q)[8]) {
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            lo |= ((uint32_t)q[e] & 0xffu) << (8 * e);
            hi |= ((uint32_t)q[e + 4] & 0xffu) << (8 * e);
        }
        *reinterpret_cast<uint2*>((uint8_t*)codes + i) = make_uint2(lo, hi);
    }
};
template <>
struct CodePack<16> {
    __device__ static __forceinline__ void store8(void* codes, int64_t i, const int (&q)[8]) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) w[e] = ((uint32_t)q[2 * e] & 0xffffu) | (((uint32_t)q[2 * e + 1] & 0xffffu) << 16);
        *reinterpret_cast<uint4*>((uint16_t*)codes + i) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};
__device__ __forceinline__ int code_of(float q) { return (q == q) ? (int)q : 0; }  // NaN has no code: emit 0

template <int BITS>
__device__ __forceinline__ void code_store1(void* codes, int64_t i, int q) {
    if (BITS == 8) ((uint8_t*)codes)[i] = (uint8_t)(q & 0xff);
    if (BITS == 16) ((uint16_t*)codes)[i] = (uint16_t)(q & 0xffff);
}

// One 256-bit vector -> 8 codes.  On the fast path (every |x| in [2^-60, 2^61) or 0, |s| in [2^-40, 2^40]: no NaN can
// appear) the pre-rounding clamp leaves t in [qmin - 0.5, qmax + 0.5], so ONE add of 1.5 * 2^23 both rounds to nearest
// even and leaves the two's-complement code in the low mantissa bits: no F2I on the conversion pipe.
constexpr float kCodeMagic = 12582912.0f;  // 0x4B400000: low 22 bits of (t + magic) == rint(t) mod 2^22
template <int BITS, bool WANT_Y>
__device__ __forceinline__ void codes_vec(const Vec<kVec>& in, int64_t i, const QP& p, uint32_t seed, float* y,
                                          void* codes) {
    FastGuard guard;
    guard_reset(guard, seed);
    float t[kVec];
#pragma unroll
    for (int e = 0; e < kVec; ++e) {
        guard_note(guard, in.v[e]);
        t[e] = clamp_t(__fadd_rn(div_fast(in.v[e], p), p.z), p);
    }
    int qi[kVec];
    Vec<kVec> vy;
    if (guard_bad(guard)) {
#pragma unroll
        for (int e = 0; e < kVec; ++e) {
            const float q = elem_slow(in.v[e], p).q;
            qi[e] = code_of(q);
            if (WANT_Y) vy.v[e] = dequant(q, p);
        }
    } else {
#pragma unroll
        for (int e = 0; e < kVec; ++e) {
            if (WANT_Y) {
                const float q = rintf(t[e]);  // keeps the sign of a negative zero for y
                vy.v[e] = dequant(q, p);
                qi[e] = __float_as_int(__fadd_rn(q, kCodeMagic));
            } else {
                qi[e] = __float_as_int(__fadd_rn(t[e], kCodeMagic));
            }
        }
    }
    CodePack<BITS>::store8(codes, i, qi);
    if (WANT_Y) st_stream(y + i, vy);
}

// Tiles are up to 8 batches long for large tensors (reduce_tile_mult): the kernel moves only 4.5-5 bytes per element, so
// with one 8192-element batch per CTA the launch / drain of a CTA is not covered by its own traffic.  Measured on B200 at
// 2^28 elements (profiles/r02_ab_code_export.log): int8 236 -> 205 us, packed int4 256 -> 205 us; a register
// double buffer (loads of batch k+1 issued before batch k is converted) and 5 CTAs/SM were measured too and add nothing.
template <int BITS, bool WANT_Y>
__global__ void __launch_bounds__(kThreads, 4)
    fq_codes_kernel(const float* __restrict__ x, float* __restrict__ y, void* __restrict__ codes, Tiles tiles, QPDev qpd) {
    const int tid = threadIdx.x;
    int64_t cur_channel = -1;
    QP p;
    uint32_t seed = 0;
    constexpr int kCodeUnroll = 4;
    for (uint32_t t = blockIdx.x; t < tiles.n_tiles; t += gridDim.x) {
        const TileCursor<kThreads> c = tile_at<kThreads>(tiles, t);
        if (c.channel != cur_channel) {
            p = load_qp(qpd, c.channel);
            seed = guard_seed(p.fast);
            cur_channel = c.channel;
        }
        const int64_t off = c.offset;
        int head = (int)((kVec - (off & (kVec - 1))) & (kVec - 1));
        head = head < c.len ? head : c.len;
        const int nvec = (c.len - head) / kVec;
        const int tail0 = head + nvec * kVec;
        const float* xb = x + off + head;
        // ---- ragged head and tail: IEEE sequence, one element (int4: one byte = two elements) per thread
        const int ragged = head + (c.len - tail0);
        const int per = BITS == 4 ? 2 : 1;
        for (int k = tid * per; k < ragged; k += kThreads * per) {
            const int i0 = k < head ? k : tail0 + (k - head);
            int q2[2] = {0, 0};
#pragma unroll
            for (int u = 0; u < per; ++u) {
                const float q = elem_slow(ld_stream1(x + off + i0 + u), p).q;
                if (WANT_Y) y[off + i0 + u] = dequant(q, p);
                q2[u] = code_of(q);
            }
            if (BITS == 4)
                ((uint8_t*)codes)[(off + i0) >> 1] = (uint8_t)((q2[0] & 0xf) | ((q2[1] & 0xf) << 4));
            else
                code_store1<BITS>(codes, off + i0, q2[0]);
        }
        // ---- vector body: kCodeUnroll 256-bit loads in flight per thread before any arithmetic
        for (int v0 = tid; v0 < nvec; v0 += kThreads * kCodeUnroll) {
            Vec<kVec> vin[kCodeUnroll];
#pragma unroll
            for (int j = 0; j < kCodeUnroll; ++j) {
                const int v = v0 + j * kThreads;
                if (v < nvec) vin[j] = ld_stream(xb + (int64_t)v * kVec, (Vec<kVec>*)nullptr);
            }
#pragma unroll
            for (int j = 0; j < kCodeUnroll; ++j) {
                const int v = v0 + j * kThreads;
                if (v < nvec) codes_vec<BITS, WANT_Y>(vin[j], off + head + (int64_t)v * kVec, p, seed, y, codes);
            }
        }
    }
}

// FP8 code export: the byte the F2FP conversion produces IS the deployable float8 value, so one 256-bit load becomes four
// packed conversions and one 64-bit store; y (optional) is unpacked from the same bytes.  Same tiles and alignment rules as
// the integer export.  Roofline: HBM, 5 B per element (+4 with y).
template <int GRID, bool WANT_Y>
__global__ void __launch_bounds__(kThreads, 4)
    fq_fp8_codes_kernel(const float* __restrict__ x, float* __restrict__ y, uint8_t* __restrict__ codes, Tiles tiles,
                        QPDev qpd) {
    const int tid = threadIdx.x;
    int64_t cur_channel = -1;
    QP p;
    uint32_t seed = 0;
    constexpr int kCodeUnroll = 4;
    for (uint32_t t = blockIdx.x; t < tiles.n_tiles; t += gridDim.x) {
        const TileCursor<kThreads> c = tile_at<kThreads>(tiles, t);
        if (c.channel != cur_channel) {
            p = load_qp(qpd, c.channel);
            seed = guard_seed(p.fast);
            cur_channel = c.channel;
        }
        const int64_t off = c.offset;
        int head = (int)((kVec - (off & (kVec - 1))) & (kVec - 1));
        head = head < c.len ? head : c.len;
        const int nvec = (c.len - head) / kVec;
        const int tail0 = head + nvec * kVec;
        const float* xb = x + off + head;
        // ---- ragged head and tail: IEEE division, one element per thread
        const int ragged = head + (c.len - tail0);
        for (int k = tid; k < ragged; k += kThreads) {
            const int64_t i = off + (k < head ? k : tail0 + (k - head));
            const uint16_t pk = fp8_pack2<GRID>(clamp_t(div_ieee(ld_stream1(x + i), p.s), p), 0.0f);
            codes[i] = (uint8_t)(pk & 0xffu);
            if (WANT_Y) {
                float q, unused;
                fp8_unpack2<GRID>(pk, q, unused);
                y[i] = dequant(q, p);
            }
        }
        // ---- vector body
        for (int v0 = tid; v0 < nvec; v0 += kThreads * kCodeUnroll) {
            Vec<kVec> vin[kCodeUnroll];
#pragma unroll
            for (int j = 0; j < kCodeUnroll; ++j) {
                const int v = v0 + j * kThreads;
                if (v < nvec) vin[j] = ld_stream(xb + (int64_t)v * kVec, (Vec<kVec>*)nullptr);
            }
#pragma unroll
            for (int j = 0; j < kCodeUnroll; ++j) {
                const int v = v0 + j * kThreads;
                if (v >= nvec) continue;
                FastGuard guard;
                guard_reset(guard, seed);
                float tc[kVec];
#pragma unroll
                for (int e = 0; e < kVec; ++e) {
                    guard_note(guard, vin[j].v[e]);
                    tc[e] = clamp_t(div_fast(vin[j].v[e], p), p);
                }
                if (guard_bad(guard)) {
#pragma unroll
                    for (int e = 0; e < kVec; ++e) tc[e] = clamp_t(div_ieee(vin[j].v[e], p.s), p);
                }
                uint32_t w[2];
                Vec<kVec> vy;
#pragma unroll
                for (int k = 0; k < kVec / 2; ++k) {
                    const uint16_t pk = fp8_pack2<GRID>(tc[2 * k], tc[2 * k + 1]);
                    if (k & 1)
                        w[k >> 1] |= (uint32_t)pk << 16;
                    else
                        w[k >> 1] = pk;
                    if (WANT_Y) {
                        float q0, q1;
                        fp8_unpack2<GRID>(pk, q0, q1);
                        vy.v[2 * k] = dequant(q0, p);
                        vy.v[2 * k + 1] = dequant(q1, p);
                    }
                }
                const int64_t i = off + head + (int64_t)v * kVec;
                *reinterpret_cast<uint2*>(codes + i) = make_uint2(w[0], w[1]);
                if (WANT_Y) st_stream(y + i, vy);
            }
        }
    }
}

// FP8 scale of each channel from an observer's chosen range: amax / F with amax = max(|lo|, |hi|); 1.0 when amax is zero
// or not finite, so an all-zero channel stays exactly zero.  lo / hi are strided fp64 columns of the observer state.
__global__ void fp8_scale_from_range_kernel(const double* lo, const double* hi, int64_t stride, int64_t channels, double F,
                                            double* scale) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= channels) return;
    const double a = fabs(lo[c * stride]), b = fabs(hi[c * stride]);
    const double amax = b > a ? b : a;
    scale[c] = (amax > 0.0 && amax <= 1.7976931348623157e308) ? amax / F : 1.0;
}

// LSQ backward.  Every tile emits one partial record {E, B} (fp32 inside a warp, fp64 across warps);
// the records of a channel are then combined in a fixed order in fp64 and scaled by the grad-scale (reduce.cuh):
//   * small launches (a single wave of CTAs): by the last CTA to finish, in the same launch;
//   * large launches: by finalize_kernel on the same stream, so the streaming CTAs retire without a
//     fence or an atomic (a per-CTA __threadfence would expose the store latency of every tile).
// Tile index = (o * C + c) * chunks + k, so channel c owns `outer * chunks` records.
struct LsqOut {
    QPDev qpd;
    void* dscale;
    void* dzp;
    int ds_f64, dz_f64;
    double gs_host;
    const float* gs_dev;
    int want_dz;
    __device__ __forceinline__ void store(int64_t c, const LsqRec& r) const {
        const double gs = gs_host * (gs_dev ? (double)__ldg(gs_dev) : 1.0);
        double ds, dz;
        lsq_channel_grads(gs, r.e, r.b, qpd, c, &ds, &dz);
        if (ds_f64)
            ((double*)dscale)[c] = ds;
        else
            ((float*)dscale)[c] = (float)ds;
        if (want_dz) {
            if (dz_f64)
                ((double*)dzp)[c] = dz;
            else
                ((float*)dzp)[c] = (float)dz;
        }
    }
};

template <int GROUP, int V, int MASK_MODE, bool WANT_DZ, bool RELU, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads, 3)  // <= 85 registers: three CTAs per SM (the RELU variants drifted to 95-110)
    lsq_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, float* __restrict__ dx, Tiles tiles,
                   void* ws, LsqOut o, int64_t outer, int use_ticket) {
    __shared__ LsqRec s_red[kWarps];
    pdl_launch_dependents();
    const float* const in[2] = {x, g};
    float* const out[1] = {dx};
    double* partials = ws_partials(ws);
    const bool leader = GROUP == 32 ? (threadIdx.x & 31) == 0 : threadIdx.x == 0;

    LsqBwdOp<MASK_MODE, WANT_DZ, RELU, GRID> op;
    int64_t cur_channel = -1;
    for (uint32_t t = group_index<GROUP>(); t < tiles.n_tiles; t += group_count<GROUP>()) {
        const TileCursor<GROUP> c = tile_at<GROUP>(tiles, t);
        if (c.channel != cur_channel) {
            op.p = load_qp(o.qpd, c.channel);
            cur_channel = c.channel;
        }
        op.e_acc = 0.0f;
        op.b_acc = 0.0f;
        span_apply<GROUP, V, 2, 1>(in, out, c.offset, c.len, op);
        const LsqRec rec = block_record<GROUP>(LsqSums<float, WANT_DZ>{op.e_acc, op.b_acc}, s_red);
        if (leader) rec.store(partials + (size_t)t * LsqRec::kSlot);
    }
    if (!use_ticket) return;
    if (!last_cta_ticket((unsigned int*)ws, leader)) return;
    combine_in_last_cta(partials, tiles, outer, o, s_red);
}

// Per-tensor LSQ backward (rows == 1): no tile ever needs its own record, so CTAs are persistent, steal 8192-element
// tiles from the look-ahead queue, carry the two sums in registers (fp32 per tile, fp64 across tiles) and flush ONCE.
// Keeps the hardware-like balance of the per-tile grid without a block reduction per tile: mid-size activations
// (2^22..2^26 elements) no longer pay for the reduction epilogue.
template <int V, int MASK_MODE, bool WANT_DZ, bool RELU, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads, 3)  // <= 85 registers: three CTAs per SM (the RELU variants drifted to 95-110)
    lsq_bwd_pt_kernel(const float* __restrict__ x, const float* __restrict__ g, float* __restrict__ dx, Tiles tiles,
                      void* ws, LsqOut o) {
    __shared__ LsqRec s_red[kWarps];
    __shared__ uint32_t s_tile[2];
    const float* const in[2] = {x, g};
    float* const out[1] = {dx};
    double* partials = ws_partials(ws);
    unsigned int* counter = (unsigned int*)ws + 1;
    LsqBwdOp<MASK_MODE, WANT_DZ, RELU, GRID> op;
    op.p = load_qp(o.qpd, 0);
    double e_run = 0.0, b_run = 0.0;
    TileQueue tq;
    tq_init(tq, counter, tiles.n_tiles, s_tile);
    for (uint32_t t = tq_current(tq, s_tile); t < tiles.n_tiles; tq_advance(tq, s_tile), t = tq_current(tq, s_tile)) {
        const TileCursor<kThreads> c = tile_at<kThreads>(tiles, t);
        op.e_acc = 0.0f;
        op.b_acc = 0.0f;
        span_apply<kThreads, V, 2, 1>(in, out, c.offset, c.len, op);
        e_run += (double)op.e_acc;
        if (WANT_DZ) b_run += (double)op.b_acc;
    }
    const LsqRec rec = block_record<kThreads>(LsqSums<double, WANT_DZ>{e_run, b_run}, s_red);
    if (threadIdx.x == 0) rec.store(partials + (size_t)blockIdx.x * LsqRec::kSlot);
    if (!last_cta_ticket((unsigned int*)ws, threadIdx.x == 0)) return;
    if (threadIdx.x == 0) *counter = 0;  // every other CTA has left its tile loop
    combine_channel<kThreads>(partials, cta_records(gridDim.x), 1, 0, o, s_red);
}

// Per-channel LSQ backward on [outer, C, inner] with the channel-item schedule (see PcGeom): one flush per CTA.
template <int GROUP, int V, bool WANT_DZ, bool RELU, int GRID = kGridInt>
__global__ void __launch_bounds__(kThreads, 3)  // <= 85 registers: three CTAs per SM (the RELU variants drifted to 95-110)
    lsq_bwd_pc_kernel(const float* __restrict__ x, const float* __restrict__ g, float* __restrict__ dx, PcGeom geo,
                      void* ws, LsqOut o, int use_ticket) {
    __shared__ LsqRec s_red[kWarps];
    pdl_launch_dependents();
    const float* const in[2] = {x, g};
    float* const out[1] = {dx};
    double* partials = ws_partials(ws);
    const int warp = threadIdx.x >> 5;
    const uint32_t C = (uint32_t)geo.channels;
    const uint32_t c = blockIdx.x % C, j = blockIdx.x / C;
    LsqBwdOp<VSIQ_MASK_ROUNDED, WANT_DZ, RELU, GRID> op;
    op.p = load_qp(o.qpd, c);
    double e_run = 0.0, b_run = 0.0;
    const uint32_t first = GROUP == 32 ? j + (uint32_t)warp * geo.k : j;
    const uint32_t step = GROUP == 32 ? geo.k * kWarps : geo.k;
    for (uint32_t u = first; u < geo.units; u += step) {
        const uint32_t n = u / geo.chunks, ch = u - n * geo.chunks;
        const int64_t start = (int64_t)ch * geo.chunk;
        const int64_t rem = geo.inner - start;
        const int len = rem < geo.chunk ? (int)rem : geo.chunk;
        const int64_t off = ((int64_t)n * C + c) * geo.inner + start;
        op.e_acc = 0.0f;
        op.b_acc = 0.0f;
        span_apply<GROUP, V, 2, 1>(in, out, off, len, op);
        e_run += (double)op.e_acc;
        if (WANT_DZ) b_run += (double)op.b_acc;
    }
    const LsqRec rec = block_record<kThreads>(LsqSums<double, WANT_DZ>{e_run, b_run}, s_red);
    if (threadIdx.x == 0) rec.store(partials + ((size_t)c * geo.k + j) * LsqRec::kSlot);
    if (!use_ticket) return;
    if (!last_cta_ticket((unsigned int*)ws, threadIdx.x == 0)) return;
    combine_in_last_cta(partials, item_records(geo), 1, o, s_red);
}

// ------------------------------------------------------------------------------------ launchers
template <int GROUP>
static uint32_t ctas_for_tiles(uint32_t n_tiles) {
    return GROUP == kThreads ? n_tiles : (n_tiles + kWarps - 1) / kWarps;
}

#define VSIQ_DISPATCH_GROUP_VEC(warp_group, vec8, CALL) \
    do {                                                \
        if (warp_group) {                               \
            if (vec8) {                                 \
                CALL(32, 8);                            \
            } else {                                    \
                CALL(32, 1);                            \
            }                                           \
        } else {                                        \
            if (vec8) {                                 \
                CALL(kThreads, 8);                      \
            } else {                                    \
                CALL(kThreads, 1);                      \
            }                                           \
        }                                               \
    } while (0)

// The launch bodies shared by the integer entry points and their FP8 siblings (GRID: common.cuh)
template <int GRID>
static int fq_fwd_launch(const float* x, float* y, const vsiq_layout* layout, const QPDev& qpd, bool relu,
                         cudaStream_t st) {
    const bool warp_group = layout->inner < kWarpGroupMaxInner;
    const bool vec8 = aligned32(x) && aligned32(y);
    Tiles tiles;
#define CALL(G, V)                                                                          \
    {                                                                                       \
        if (!make_tiles<G>(layout->outer, layout->channels, layout->inner, &tiles))         \
            return VSIQ_ERR_INVALID_ARG;                                                    \
        int grid = launch_grid(ctas_for_tiles<G>(tiles.n_tiles));                           \
        if (grid < 0) return -grid;                                                         \
        if (relu)                                                                           \
            fq_fwd_kernel<G, V, true, GRID><<<grid, kThreads, 0, st>>>(x, y, tiles, qpd);   \
        else                                                                                \
            fq_fwd_kernel<G, V, false, GRID><<<grid, kThreads, 0, st>>>(x, y, tiles, qpd);  \
    }
    VSIQ_DISPATCH_GROUP_VEC(warp_group, vec8, CALL);
#undef CALL
    return (int)cudaGetLastError();
}

template <int GRID>
static int fq_bwd_ste_launch(const float* x, const float* g, float* dx, const vsiq_layout* layout, const QPDev& qpd,
                             bool relu, cudaStream_t st) {
    const bool warp_group = layout->inner < kWarpGroupMaxInner;
    const bool vec8 = aligned32(x) && aligned32(g) && aligned32(dx);
    Tiles tiles;
#define CALL(G, V)                                                                                  \
    {                                                                                               \
        if (!make_tiles<G>(layout->outer, layout->channels, layout->inner, &tiles))                 \
            return VSIQ_ERR_INVALID_ARG;                                                            \
        int grid = launch_grid(ctas_for_tiles<G>(tiles.n_tiles));                                   \
        if (grid < 0) return -grid;                                                                 \
        if (relu)                                                                                   \
            fq_bwd_ste_kernel<G, V, true, GRID><<<grid, kThreads, 0, st>>>(x, g, dx, tiles, qpd);   \
        else                                                                                        \
            fq_bwd_ste_kernel<G, V, false, GRID><<<grid, kThreads, 0, st>>>(x, g, dx, tiles, qpd);  \
    }
    VSIQ_DISPATCH_GROUP_VEC(warp_group, vec8, CALL);
#undef CALL
    return (int)cudaGetLastError();
}

}  // namespace vsiq

using namespace vsiq;

extern "C" int vsiq_fake_quant_fwd(const float* x, float* y, void* codes, const vsiq_layout* layout,
                                   const vsiq_qparams* qp, vsiq_stream_t stream) {
    if (int e = check_layout(layout)) return e;
    QPDev qpd;
    if (int e = fill_qp(qp, &qpd)) return e;
    const int64_t n = layout->outer * layout->channels * layout->inner;
    if (n == 0) return VSIQ_OK;
    if (!x || (!y && !codes)) return VSIQ_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (qp->pre_op == VSIQ_PRE_SILU) return VSIQ_ERR_UNSUPPORTED;  // SiLU: channel-innermost entry points only
    if (codes)  // int8 (qmin < 0) / uint8 codes: the 8-bit form of vsiq_quantize_codes
        return vsiq_quantize_codes(x, y, codes, 8, layout, qp, stream);
    return fq_fwd_launch<kGridInt>(x, y, layout, qpd, qp->pre_op == VSIQ_PRE_RELU, st);
}

extern "C" int vsiq_quantize_codes(const float* x, float* y, void* codes, int code_bits, const vsiq_layout* layout,
                                   const vsiq_qparams* qp, vsiq_stream_t stream) {
    if (int e = check_layout(layout)) return e;
    QPDev qpd;
    if (int e = fill_qp(qp, &qpd)) return e;
    if (code_bits != 4 && code_bits != 8 && code_bits != 16) return VSIQ_ERR_INVALID_ARG;
    const int64_t n = layout->outer * layout->channels * layout->inner;
    if (n == 0) return VSIQ_OK;
    if (!x || !codes) return VSIQ_ERR_INVALID_ARG;
    if (qp->pre_op != VSIQ_PRE_NONE) return VSIQ_ERR_UNSUPPORTED;
    // the integer range must fit the code width: two's complement when qmin < 0, unsigned otherwise
    const int64_t lo = qp->qmin < 0 ? -(int64_t(1) << (code_bits - 1)) : 0;
    const int64_t hi = qp->qmin < 0 ? (int64_t(1) << (code_bits - 1)) - 1 : (int64_t(1) << code_bits) - 1;
    if (qp->qmin < lo || qp->qmax > hi) return VSIQ_ERR_UNSUPPORTED;
    if (code_bits == 4 && (layout->inner & 1)) return VSIQ_ERR_UNSUPPORTED;  // a byte must not straddle two rows
    // 256-bit loads of x need a 32-byte aligned base; the packed stores then are aligned as well when codes (and y) are
    const uintptr_t amask = reinterpret_cast<uintptr_t>(x) | (y ? reinterpret_cast<uintptr_t>(y) : 0);
    if ((amask & 31u) || (reinterpret_cast<uintptr_t>(codes) & 15u)) return VSIQ_ERR_UNSUPPORTED;
    Tiles tiles;
    const int mult = reduce_tile_mult<kThreads>(layout->outer, layout->channels, layout->inner);
    if (!make_tiles<kThreads>(layout->outer, layout->channels, layout->inner, &tiles, mult)) return VSIQ_ERR_INVALID_ARG;
    const int grid = launch_grid(tiles.n_tiles);
    if (grid < 0) return -grid;
    cudaStream_t st = (cudaStream_t)stream;
#define C(B)                                                                                   \
    {                                                                                          \
        if (y) fq_codes_kernel<B, true><<<grid, kThreads, 0, st>>>(x, y, codes, tiles, qpd);    \
        else fq_codes_kernel<B, false><<<grid, kThreads, 0, st>>>(x, y, codes, tiles, qpd);     \
    }
    if (code_bits == 4) C(4) else if (code_bits == 8) C(8) else C(16)
#undef C
    return (int)cudaGetLastError();
}

extern "C" int vsiq_fake_quant_bwd_ste(const float* x, const float* g, float* dx, const vsiq_layout* layout,
                                       const vsiq_qparams* qp, vsiq_stream_t stream) {
    if (int e = check_layout(layout)) return e;
    QPDev qpd;
    if (int e = fill_qp(qp, &qpd)) return e;
    if (qp->pre_op == VSIQ_PRE_SILU) return VSIQ_ERR_UNSUPPORTED;
    if (layout->outer * layout->channels * layout->inner == 0) return VSIQ_OK;
    if (!x || !g || !dx) return VSIQ_ERR_INVALID_ARG;
    return fq_bwd_ste_launch<kGridInt>(x, g, dx, layout, qpd, qp->pre_op == VSIQ_PRE_RELU, (cudaStream_t)stream);
}

extern "C" int vsiq_fake_quant_fwd_bwd(const float* x, const float* g, float* y, float* dx,
                                       const vsiq_layout* layout, const vsiq_qparams* qp, vsiq_stream_t stream) {
    if (int e = check_layout(layout)) return e;
    QPDev qpd;
    if (int e = fill_qp(qp, &qpd)) return e;
    if (layout->outer * layout->channels * layout->inner == 0) return VSIQ_OK;
    if (!x || !g || !y || !dx) return VSIQ_ERR_INVALID_ARG;
    if (qp->pre_op != VSIQ_PRE_NONE) return VSIQ_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const bool warp_group = layout->inner < kWarpGroupMaxInner;
    const bool vec8 = aligned32(x) && aligned32(g) && aligned32(y) && aligned32(dx);
    Tiles tiles;
#define CALL(G, V)                                                                            \
    {                                                                                         \
        if (!make_tiles<G>(layout->outer, layout->channels, layout->inner, &tiles))           \
            return VSIQ_ERR_INVALID_ARG;                                                      \
        int grid = launch_grid(ctas_for_tiles<G>(tiles.n_tiles)); \
        if (grid < 0) return -grid;                                                           \
        fq_fwd_bwd_kernel<G, V><<<grid, kThreads, 0, st>>>(x, g, y, dx, tiles, qpd);          \
    }
    VSIQ_DISPATCH_GROUP_VEC(warp_group, vec8, CALL);
#undef CALL
    return (int)cudaGetLastError();
}

extern "C" size_t vsiq_lsq_bwd_workspace_bytes(const vsiq_layout* layout) {
    return reduce_workspace_bytes(layout, LsqRec::kSlot);
}

// vsiq_lsq_bwd for the integer grid, vsiq_fp8_lsq_bwd for the FP8 ones (which has already refused FunLSQ and dzp: the
// FunLSQ / dzp instantiations below collapse onto the rounded, dzp-free one for them and are never reached)
template <int GRID>
static int lsq_bwd_impl(const float* x, const float* g, float* dx, void* dscale, int dscale_dtype, void* dzp,
                        int dzp_dtype, const vsiq_layout* layout, const vsiq_qparams* qp, double grad_scale_host,
                        const float* grad_scale_dev, int mask_mode, void* workspace, size_t workspace_bytes,
                        vsiq_stream_t stream) {
    constexpr int kFunlsq = GRID == kGridInt ? VSIQ_MASK_FUNLSQ : VSIQ_MASK_ROUNDED;
    constexpr bool kDz = GRID == kGridInt;
    if (!dscale) return VSIQ_ERR_INVALID_ARG;
    if (int e = check_layout(layout)) return e;
    if (mask_mode != VSIQ_MASK_ROUNDED && mask_mode != VSIQ_MASK_FUNLSQ) return VSIQ_ERR_INVALID_ARG;
    if (mask_mode == VSIQ_MASK_FUNLSQ && (dzp || (qp && qp->pre_op != VSIQ_PRE_NONE))) return VSIQ_ERR_UNSUPPORTED;
    if ((dscale_dtype != VSIQ_F32 && dscale_dtype != VSIQ_F64) || (dzp && dzp_dtype != VSIQ_F32 && dzp_dtype != VSIQ_F64))
        return VSIQ_ERR_INVALID_ARG;
    LsqOut lo;
    if (int e = GRID == kGridInt ? fill_qp(qp, &lo.qpd) : fill_qp_fp8(qp, GRID, &lo.qpd)) return e;
    if (qp->pre_op == VSIQ_PRE_SILU) return VSIQ_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < vsiq_lsq_bwd_workspace_bytes(layout)) return VSIQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    if (layout->outer * layout->channels * layout->inner == 0) {
        // empty tensor: gradients are zero
        cudaError_t ce = cudaMemsetAsync(dscale, 0, (size_t)layout->channels * (dscale_dtype ? 8 : 4), st);
        if (ce == cudaSuccess && dzp) ce = cudaMemsetAsync(dzp, 0, (size_t)layout->channels * (dzp_dtype ? 8 : 4), st);
        return (int)ce;
    }
    if (!x || !g || !dx) return VSIQ_ERR_INVALID_ARG;
    const bool warp_group = layout->inner < kWarpGroupMaxInner;
    const bool vec8 = aligned32(x) && aligned32(g) && aligned32(dx);
    const bool relu = qp->pre_op == VSIQ_PRE_RELU;
    lo.dscale = dscale;
    lo.dzp = dzp;
    lo.ds_f64 = dscale_dtype == VSIQ_F64;
    lo.dz_f64 = dzp_dtype == VSIQ_F64;
    lo.gs_host = grad_scale_host;
    lo.gs_dev = grad_scale_dev;
    lo.want_dz = dzp != nullptr;
    DeviceProps dprops;
    if (int e = get_device_props(&dprops)) return e;
    PcGeom pc;
    if (mask_mode == VSIQ_MASK_ROUNDED && layout->channels > 1 &&
        make_pc_geom(layout->outer, layout->channels, layout->inner, warp_group, dprops.sm_count, &pc) &&
        (size_t)pc.channels * pc.k * LsqRec::kSlot * sizeof(double) + kWsHeader <= workspace_bytes) {
        const int grid = (int)(pc.channels * pc.k);
        // one partial wave: the last CTA combines; more: no ticket, no fence -- the combine kernel is a programmatic dependent
        const int use_ticket = grid <= dprops.sm_count * 4 ? 1 : 0;
#define PC(G, V, Z, R) lsq_bwd_pc_kernel<G, V, Z, R, GRID><<<grid, kThreads, 0, st>>>(x, g, dx, pc, workspace, lo, use_ticket)
#define PC2(G, V, Z) { if (relu) PC(G, V, Z, true); else PC(G, V, Z, false); }
#define PC1(G, V) { if (dzp) PC2(G, V, kDz) else PC2(G, V, false) }
        if (warp_group) { if (vec8) PC1(32, 8) else PC1(32, 1) } else { if (vec8) PC1(kThreads, 8) else PC1(kThreads, 1) }
#undef PC1
#undef PC2
#undef PC
        if (!use_ticket) launch_finalize<LsqRec>(item_records(pc), 1, false, workspace, lo, st);
        return (int)cudaGetLastError();
    }
    Tiles tiles;
    if (layout->outer == 1 && layout->channels == 1 && !warp_group) {  // per tensor: persistent CTAs
        if (!make_tiles<kThreads>(1, 1, layout->inner, &tiles)) return VSIQ_ERR_INVALID_ARG;
        const uint32_t cap = (uint32_t)dprops.sm_count * 3u;
        const int grid = (int)(tiles.n_tiles < cap ? tiles.n_tiles : cap);
#define PT(V, M, Z, R) lsq_bwd_pt_kernel<V, M, Z, R, GRID><<<grid, kThreads, 0, st>>>(x, g, dx, tiles, workspace, lo)
#define PT2(V, M, Z) { if (relu) PT(V, M, Z, true); else PT(V, M, Z, false); }
#define PT1(V) { if (mask_mode == VSIQ_MASK_FUNLSQ) PT(V, kFunlsq, false, false); else if (dzp) PT2(V, VSIQ_MASK_ROUNDED, kDz) else PT2(V, VSIQ_MASK_ROUNDED, false) }
        if (vec8) PT1(8) else PT1(1)
#undef PT1
#undef PT2
#undef PT
        return (int)cudaGetLastError();
    }
#define LAUNCH(G, V, M, Z)                                                                                     \
    {                                                                                                          \
        if (relu) {                                                                                            \
            LAUNCH_R(G, V, M, Z, true);                                                                        \
        } else {                                                                                               \
            LAUNCH_R(G, V, M, Z, false);                                                                       \
        }                                                                                                      \
    }
#define LAUNCH_R(G, V, M, Z, R)                                                                                \
    {                                                                                                          \
        const int mult = reduce_tile_mult<G>(layout->outer, layout->channels, layout->inner);                 \
        if (!make_tiles<G>(layout->outer, layout->channels, layout->inner, &tiles, mult))                      \
            return VSIQ_ERR_INVALID_ARG;                                                                       \
        int grid = launch_grid(ctas_for_tiles<G>(tiles.n_tiles));                                              \
        if (grid < 0) return -grid;                                                                            \
        const int use_ticket = (grid <= dprops.sm_count * 4 && tiles.n_tiles <= kTicketMaxRecords) ? 1 : 0;   \
        lsq_bwd_kernel<G, V, M, Z, R, GRID><<<grid, kThreads, 0, st>>>(x, g, dx, tiles, workspace, lo,        \
                                                                    layout->outer, use_ticket);                                     \
        if (!use_ticket) launch_finalize<LsqRec>(tiles, layout->outer, true, workspace, lo, st);               \
    }
#define CALL(G, V)                                   \
    {                                                \
        if (mask_mode == VSIQ_MASK_FUNLSQ) {         \
            LAUNCH(G, V, kFunlsq, false);            \
        } else if (dzp) {                            \
            LAUNCH(G, V, VSIQ_MASK_ROUNDED, kDz);    \
        } else {                                     \
            LAUNCH(G, V, VSIQ_MASK_ROUNDED, false);  \
        }                                            \
    }
    VSIQ_DISPATCH_GROUP_VEC(warp_group, vec8, CALL);
#undef CALL
#undef LAUNCH
#undef LAUNCH_R
    return (int)cudaGetLastError();
}

extern "C" int vsiq_lsq_bwd(const float* x, const float* g, float* dx, void* dscale, int dscale_dtype, void* dzp,
                            int dzp_dtype, const vsiq_layout* layout, const vsiq_qparams* qp, double grad_scale_host,
                            const float* grad_scale_dev, int mask_mode, void* workspace, size_t workspace_bytes,
                            vsiq_stream_t stream) {
    return lsq_bwd_impl<kGridInt>(x, g, dx, dscale, dscale_dtype, dzp, dzp_dtype, layout, qp, grad_scale_host,
                                  grad_scale_dev, mask_mode, workspace, workspace_bytes, stream);
}

// ------------------------------------------------------------------------------------ FP8 entry points
extern "C" int vsiq_fp8_fake_quant_fwd(const float* x, float* y, void* codes, const vsiq_layout* layout,
                                       const vsiq_qparams* qp, int fp8_format, vsiq_stream_t stream) {
    if (int e = check_layout(layout)) return e;
    QPDev qpd;
    if (int e = fill_qp_fp8(qp, fp8_format, &qpd)) return e;
    if (qp->pre_op == VSIQ_PRE_SILU) return VSIQ_ERR_UNSUPPORTED;
    const int64_t n = layout->outer * layout->channels * layout->inner;
    if (n == 0) return VSIQ_OK;
    if (!x || (!y && !codes)) return VSIQ_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (!codes) {
        const bool relu = qp->pre_op == VSIQ_PRE_RELU;
        return fp8_format == VSIQ_FP8_E4M3 ? fq_fwd_launch<VSIQ_FP8_E4M3>(x, y, layout, qpd, relu, st)
                                           : fq_fwd_launch<VSIQ_FP8_E5M2>(x, y, layout, qpd, relu, st);
    }
    if (qp->pre_op != VSIQ_PRE_NONE) return VSIQ_ERR_UNSUPPORTED;
    const uintptr_t amask = reinterpret_cast<uintptr_t>(x) | (y ? reinterpret_cast<uintptr_t>(y) : 0);
    if ((amask & 31u) || (reinterpret_cast<uintptr_t>(codes) & 15u)) return VSIQ_ERR_UNSUPPORTED;
    Tiles tiles;
    const int mult = reduce_tile_mult<kThreads>(layout->outer, layout->channels, layout->inner);
    if (!make_tiles<kThreads>(layout->outer, layout->channels, layout->inner, &tiles, mult)) return VSIQ_ERR_INVALID_ARG;
    const int grid = launch_grid(tiles.n_tiles);
    if (grid < 0) return -grid;
    uint8_t* c8 = (uint8_t*)codes;
#define C(F)                                                                                       \
    {                                                                                              \
        if (y) fq_fp8_codes_kernel<F, true><<<grid, kThreads, 0, st>>>(x, y, c8, tiles, qpd);      \
        else fq_fp8_codes_kernel<F, false><<<grid, kThreads, 0, st>>>(x, y, c8, tiles, qpd);       \
    }
    if (fp8_format == VSIQ_FP8_E4M3) C(VSIQ_FP8_E4M3) else C(VSIQ_FP8_E5M2)
#undef C
    return (int)cudaGetLastError();
}

extern "C" int vsiq_fp8_fake_quant_bwd_ste(const float* x, const float* g, float* dx, const vsiq_layout* layout,
                                           const vsiq_qparams* qp, int fp8_format, vsiq_stream_t stream) {
    if (int e = check_layout(layout)) return e;
    QPDev qpd;
    if (int e = fill_qp_fp8(qp, fp8_format, &qpd)) return e;
    if (qp->pre_op == VSIQ_PRE_SILU) return VSIQ_ERR_UNSUPPORTED;
    if (layout->outer * layout->channels * layout->inner == 0) return VSIQ_OK;
    if (!x || !g || !dx) return VSIQ_ERR_INVALID_ARG;
    const bool relu = qp->pre_op == VSIQ_PRE_RELU;
    cudaStream_t st = (cudaStream_t)stream;
    return fp8_format == VSIQ_FP8_E4M3 ? fq_bwd_ste_launch<VSIQ_FP8_E4M3>(x, g, dx, layout, qpd, relu, st)
                                       : fq_bwd_ste_launch<VSIQ_FP8_E5M2>(x, g, dx, layout, qpd, relu, st);
}

extern "C" int vsiq_fp8_lsq_bwd(const float* x, const float* g, float* dx, void* dscale, int dscale_dtype, void* dzp,
                                int dzp_dtype, const vsiq_layout* layout, const vsiq_qparams* qp, int fp8_format,
                                double grad_scale_host, const float* grad_scale_dev, int mask_mode, void* workspace,
                                size_t workspace_bytes, vsiq_stream_t stream) {
    if (fp8_format != VSIQ_FP8_E4M3 && fp8_format != VSIQ_FP8_E5M2) return VSIQ_ERR_INVALID_ARG;
    if (mask_mode != VSIQ_MASK_ROUNDED && mask_mode != VSIQ_MASK_FUNLSQ) return VSIQ_ERR_INVALID_ARG;
    if (mask_mode != VSIQ_MASK_ROUNDED || dzp) return VSIQ_ERR_UNSUPPORTED;  // symmetric, autograd-mask semantics only
    return fp8_format == VSIQ_FP8_E4M3
               ? lsq_bwd_impl<VSIQ_FP8_E4M3>(x, g, dx, dscale, dscale_dtype, nullptr, dzp_dtype, layout, qp,
                                             grad_scale_host, grad_scale_dev, mask_mode, workspace, workspace_bytes, stream)
               : lsq_bwd_impl<VSIQ_FP8_E5M2>(x, g, dx, dscale, dscale_dtype, nullptr, dzp_dtype, layout, qp,
                                             grad_scale_host, grad_scale_dev, mask_mode, workspace, workspace_bytes, stream);
}

extern "C" int vsiq_fp8_scale_from_range(const double* lo, const double* hi, int64_t stride, int64_t channels,
                                         int fp8_format, double* scale, vsiq_stream_t stream) {
    if (fp8_format != VSIQ_FP8_E4M3 && fp8_format != VSIQ_FP8_E5M2) return VSIQ_ERR_INVALID_ARG;
    if (channels < 0 || stride < 1) return VSIQ_ERR_INVALID_ARG;
    if (channels == 0) return VSIQ_OK;
    if (!lo || !hi || !scale) return VSIQ_ERR_INVALID_ARG;
    const int threads = 128;
    fp8_scale_from_range_kernel<<<(unsigned)((channels + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        lo, hi, stride, channels, (double)fp8_max(fp8_format), scale);
    return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------ self-test
// Counts the input bit patterns (all 2^32 of them) for which the fast arithmetic differs from the IEEE
// sequences, for one divisor s.  mode 0: x / s (div_fast, with the vector-level fallback the kernels
// use).  mode 1: RN(RN(g*s) / s) (dx_fast).  NaN results compare equal to NaN.
namespace vsiq {
__global__ void __launch_bounds__(kThreads) division_selftest_kernel(float s, int mode, unsigned long long* mismatches) {
    QP p;
    p.s = s;
    p.r = __frcp_rn(s);
    p.z = 0.0f;
    p.zf = 0.0f;
    p.lo = -128.0f;
    p.hi = 127.0f;
    p.tlo = -128.5f;
    p.thi = 127.49999f;
    p.zero_dx = __fdiv_rn(0.0f, s);
    const float as = fabsf(s);
    p.fast = (as >= 9.094947017729282e-13f) && (as <= 1.099511627776e12f);
    unsigned int wrong = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const float x = __uint_as_float((uint32_t)i);
        FastGuard guard;
        guard_reset(guard);
        guard_note(guard, x);
        float a, b;
        if (mode == 0) {
            a = div_fast(x, p);
            b = __fdiv_rn(x, s);
        } else {
            a = dx_fast(x, true, p);
            b = __fdiv_rn(__fmul_rn(x, s), s);
        }
        if (!p.fast || guard_bad(guard)) a = b;  // the kernels redo such vectors with the IEEE sequence
        const bool same = (__float_as_uint(a) == __float_as_uint(b)) || ((a != a) && (b != b));
        wrong += same ? 0u : 1u;
    }
    wrong = __reduce_add_sync(0xffffffffu, wrong);
    if ((threadIdx.x & 31) == 0 && wrong) atomicAdd(mismatches, (unsigned long long)wrong);
}
}  // namespace vsiq

extern "C" int vsiq_selftest_division(float s, int mode, unsigned long long* mismatches_dev, vsiq_stream_t stream) {
    if (!mismatches_dev || (mode != 0 && mode != 1)) return VSIQ_ERR_INVALID_ARG;
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return e;
    division_selftest_kernel<<<dp.sm_count * 8, kThreads, 0, (cudaStream_t)stream>>>(s, mode, mismatches_dev);
    return (int)cudaGetLastError();
}
