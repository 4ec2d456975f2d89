// quant_ops.cuh -- the per-element operators of the fake-quant kernels (forward, STE backward, fused forward +
// backward, LSQ backward), shared by fake_quant.cu (one tensor per launch) and multi_tensor.cu (all weight tensors of
// a step per launch).  They plug into span_apply (common.cuh) through the OpBase protocol.
#pragma once

#include "common.cuh"

namespace vsiq {

// ------------------------------------------------------------------------------------------ ops
struct QuantOpBase : OpBase {
    QP p;
    FastGuard guard;  // admissibility of the current vector for the division-free arithmetic (common.cuh)
    __device__ __forceinline__ void vec_begin() { guard_reset(guard, guard_seed(p.fast)); }
    __device__ __forceinline__ bool vec_bad() const { return guard_bad(guard); }
};

// RELU = true fuses the preceding activation into the quantiser: the kernels see the conv output x, quantise
// relu(x) = max(x, 0) (NaN propagates like torch.relu) and, in the backward, also apply relu's mask [x > 0]
// (threshold_backward) -- one pass instead of relu + fake-quant (fused.py:133 then fake_quantize.py:49-50).
template <bool RELU>
__device__ __forceinline__ float pre_act(float x) { return RELU ? max_nan(x, 0.0f) : x; }

// GRID (common.cuh): kGridInt, or an FP8 grid (no zero-point; dequant's q - 0 is exact, -0.0 and NaN included)
template <bool RELU, int GRID = kGridInt>
struct FwdOp : QuantOpBase {
    __device__ __forceinline__ void apply(const float (&a)[1], float (&o)[1]) {
        const float x = pre_act<RELU>(a[0]);
        guard_note(guard, x);
        o[0] = dequant(elem_fast<GRID>(x, p).q, p);
    }
    __device__ __forceinline__ void apply_slow(const float (&a)[1], float (&o)[1]) {
        o[0] = dequant(elem_slow<GRID>(pre_act<RELU>(a[0]), p).q, p);
    }
};

template <bool RELU, int GRID = kGridInt>
struct SteBwdOp : QuantOpBase {
    __device__ __forceinline__ void apply(const float (&a)[2], float (&o)[1]) {
        const float x = pre_act<RELU>(a[0]);
        guard_note(guard, x);
        guard_note(guard, a[1]);
        const Elem e = elem_fast<GRID>(x, p);
        const float dx = dx_fast(a[1], e.m, p);
        o[0] = (!RELU || a[0] > 0.0f) ? dx : 0.0f;
    }
    __device__ __forceinline__ void apply_slow(const float (&a)[2], float (&o)[1]) {
        const float dx = dx_slow(a[1], elem_slow<GRID>(pre_act<RELU>(a[0]), p).m, p);
        o[0] = (!RELU || a[0] > 0.0f) ? dx : 0.0f;
    }
};

struct FwdBwdOp : QuantOpBase {
    __device__ __forceinline__ void apply(const float (&a)[2], float (&o)[2]) {
        guard_note(guard, a[0]);
        guard_note(guard, a[1]);
        const Elem e = elem_fast(a[0], p);
        o[0] = dequant(e.q, p);
        o[1] = dx_fast(a[1], e.m, p);
    }
    __device__ __forceinline__ void apply_slow(const float (&a)[2], float (&o)[2]) {
        const Elem e = elem_slow(a[0], p);
        o[0] = dequant(e.q, p);
        o[1] = dx_slow(a[1], e.m, p);
    }
};

// FP8 grids: MASK_MODE = VSIQ_MASK_ROUNDED and WANT_DZ = false only (z = 0, so the sum is g * (q - m * x/s))
template <int MASK_MODE, bool WANT_DZ, bool RELU, int GRID = kGridInt>
struct LsqBwdOp : QuantOpBase {
    float e_acc;  // sum g * ((q - z) - m * x/s)   over this thread's elements of the current tile
    float b_acc;  // sum g over clamped-out elements
    float e_vec, b_vec;  // the current vector's share (committed by vec_done, discarded on a redo)
    __device__ __forceinline__ void vec_begin() {
        guard_reset(guard, guard_seed(p.fast));
        e_vec = 0.0f;
        b_vec = 0.0f;
    }
    __device__ __forceinline__ void vec_done() {
        e_acc += e_vec;
        if (WANT_DZ) b_acc += b_vec;
    }
    __device__ __forceinline__ void accumulate(float g, const Elem& e, float (&o)[1]) {
        if (MASK_MODE == VSIQ_MASK_ROUNDED) {
            // reference: g*(q-z) from mul-backward minus where(m, g*s, 0) * ((x/s)/s) from div-backward;
            // v * 0 keeps the reference's NaN for infinite inputs.
            const float d = __fsub_rn(e.q, p.z);
            const float mv = __fmul_rn(e.v, e.m ? 1.0f : 0.0f);
            e_vec = fmaf(g, d - mv, e_vec);
            if (WANT_DZ) b_vec += e.m ? 0.0f : g;
        } else {
            // FunLSQ (quantizers/uniform.py:144-150): strict masks on the unrounded v, z ignored
            const float small = e.v < p.lo ? 1.0f : 0.0f;
            const float big = e.v > p.hi ? 1.0f : 0.0f;
            const float mid = 1.0f - small - big;
            const float term = small * p.lo + big * p.hi + mid * (rintf(e.v) - e.v);
            e_vec = fmaf(term, g, e_vec);
            o[0] = __fmul_rn(mid, g);
        }
    }
    __device__ __forceinline__ void apply(const float (&a)[2], float (&o)[1]) {
        const float x = pre_act<RELU>(a[0]);
        guard_note(guard, x);
        guard_note(guard, a[1]);
        const Elem e = elem_fast<GRID>(x, p);
        if (MASK_MODE == VSIQ_MASK_ROUNDED) o[0] = dx_fast(a[1], e.m, p);
        accumulate(a[1], e, o);
        if (RELU) o[0] = a[0] > 0.0f ? o[0] : 0.0f;
    }
    __device__ __forceinline__ void apply_slow(const float (&a)[2], float (&o)[1]) {
        const Elem e = elem_slow<GRID>(pre_act<RELU>(a[0]), p);
        if (MASK_MODE == VSIQ_MASK_ROUNDED) o[0] = dx_slow(a[1], e.m, p);
        accumulate(a[1], e, o);
        if (RELU) o[0] = a[0] > 0.0f ? o[0] : 0.0f;
    }
};

// dscale and dzero_point of channel c from its combined LsqBwdOp sums E and B and the grad-scale gs
__device__ __forceinline__ void lsq_channel_grads(double gs, double e, double b, const QPDev& qpd, int64_t c, double* ds,
                                                  double* dz) {
    const QP p = load_qp(qpd, c);
    *ds = gs * e;
    const float zr = rintf(p.zf);
    const bool cz = qpd.zp_learned ? ((zr >= p.lo) && (zr <= p.hi)) : true;
    *dz = cz ? -gs * (double)p.s * b : 0.0;  // sum (g*s)*(m-1) = -s * sum_{clamped} g
}

}  // namespace vsiq
