/*
 * vsiq.h -- C ABI of libvsiq.so: the B200 (sm_100a) fake-quantization hot path.
 *
 * The reference (tranngocduvnvp/VSIQuantization) is pure Python/PyTorch and has
 * no FFI of its own; its boundary for this path is the duck-typed plugin
 * registry (utils/registry.py:5-27) whose plugins call ATen.  These entry
 * points are what a binding for that path binds instead of the ATen op chains:
 * each declaration cites the reference code it replaces.  The Python host side
 * (vsiquantization_b200/) loads this library with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every tensor pointer is DEVICE memory
 *     (fp32 unless stated) owned by the caller, except in the *_host entry.
 *   - every call is asynchronous on the given stream (a cudaStream_t passed as
 *     void*), allocates nothing (scratch comes in as `workspace`; the exceptions say so: the host pipeline's
 *     handle and vsiq_peer_alloc, whose buffer must be cudaMalloc memory to be exported to other processes), keeps no
 *     global mutable state (beyond mutex-guarded, write-once per-device caches of
 *     device attributes and kernel attributes) and is re-entrant across streams and devices.
 *     Workspaces must not be shared by calls running concurrently on
 *     different streams.  A workspace must be zero-filled once when it is
 *     allocated; every call leaves it zero-filled where it needs it to be.
 *   - return value: 0 on success, a positive cudaError_t, or a negative
 *     VSIQ_ERR_* code.  Nothing throws; there is no CPU fallback.
 *   - outputs must not alias inputs.
 *   - layout: a contiguous tensor is described as [outer, channels, inner];
 *     the channel of flat index i is (i / inner) % channels.
 *       per tensor             outer = 1, channels = 1,        inner = numel
 *       per channel, ch_axis 0 outer = 1, channels = shape[0], inner = numel / shape[0]   (OIHW weights)
 *       per channel, ch_axis 1 outer = N, channels = shape[1], inner = H*W                (NCHW activations)
 *   - arithmetic: fp32, every operation individually rounded (IEEE division,
 *     no FMA contraction, round-half-even) so results are bit-identical to the
 *     reference's ATen-on-CPU composition; sums are accumulated in fp64.
 */
#ifndef VSIQ_H_
#define VSIQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSIQ_VERSION 100 /* major*1000 + minor*100 + patch */

typedef void *vsiq_stream_t; /* cudaStream_t */

enum {
    VSIQ_OK = 0,
    VSIQ_ERR_INVALID_ARG = -1, /* null pointer, negative size, bits outside 2..8, qmin >= qmax ... */
    VSIQ_ERR_WORKSPACE = -2,   /* workspace missing or smaller than *_workspace_bytes() */
    VSIQ_ERR_UNSUPPORTED = -3, /* combination not implemented (reported, never silently ignored) */
    VSIQ_ERR_NO_DEVICE = -4    /* no sm_100 device / driver */
};

enum { VSIQ_F32 = 0, VSIQ_F64 = 1 };

/* activation fused in front of the quantiser (fwd, STE bwd, LSQ bwd): the fused layer's F.relu (modules/fused.py:133)
 * followed by quantize_activation (quantizers/fake_quantize.py:49-50) becomes one pass over the conv output */
enum {
    VSIQ_PRE_NONE = 0,
    VSIQ_PRE_RELU = 1,
    /* SiLU, x / (1 + exp(-x)) and its derivative in ATen-CUDA's operation order: the channel-innermost entry points only
     * (vsiq_ci_fake_quant_fwd / vsiq_ci_lsq_bwd); everything else returns VSIQ_ERR_UNSUPPORTED for it. */
    VSIQ_PRE_SILU = 2
};

/* mask semantics of the LSQ backward */
enum {
    VSIQ_MASK_ROUNDED = 0, /* reference autograd: qmin <= rint(x/s+z) <= qmax, inclusive (uniform.py:54,95) */
    VSIQ_MASK_FUNLSQ = 1   /* reference dead code FunLSQ: strict bounds on the unrounded x/s (uniform.py:144-150) */
};

/* FP8 value grids of the vsiq_fp8_* entry points (F = the largest finite value) */
enum {
    VSIQ_FP8_E4M3 = 1, /* float8_e4m3fn, F = 448 */
    VSIQ_FP8_E5M2 = 2  /* float8_e5m2,   F = 57344 */
};

typedef struct vsiq_layout {
    int64_t outer;
    int64_t channels;
    int64_t inner;
} vsiq_layout;

/* Quantisation parameters: `channels` entries each (1 for per tensor).
 * scale / zero_point are DEVICE pointers of the stated dtype (the reference's learned scale is a
 * 0-dim float64 Parameter, quantization_manager.py:99; it is rounded to fp32 before use exactly as
 * ATen does).  A NULL pointer selects the host scalar instead (the reference's Python float / int
 * qparams of the non-learning mode, quantization_manager.py:69-71).
 * zp_learned = 1: zero_point holds the float parameter z_f and the forward uses
 * clamp(rint(z_f), qmin, qmax) (uniform.py:98-102, lsq_module.py:354-358). */
typedef struct vsiq_qparams {
    const void *scale;
    const void *zero_point;
    int32_t scale_dtype;
    int32_t zp_dtype;
    float scale_host;
    float zp_host;
    int32_t zp_learned;
    int32_t qmin;
    int32_t qmax;
    int32_t pre_op; /* VSIQ_PRE_NONE, or VSIQ_PRE_RELU / VSIQ_PRE_SILU: quantise act(x) and chain act's derivative in the backward */
} vsiq_qparams;

/* ---- library ---------------------------------------------------------------------------- */
int vsiq_version(void);
const char *vsiq_error_string(int code);
/* SM count and compute capability of the current device (VSIQ_ERR_NO_DEVICE without one). */
int vsiq_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* Workspaces.  The reducing entry points (observer, LSQ backward, NHWC kernels, multi-tensor backward) take a caller-owned
 * scratch buffer.  Its first 256 bytes hold a ticket and a tile counter that must be ZERO when a call starts; every call
 * leaves them zero when its kernels complete (zero-fill the buffer once after allocating it).  If a call is abandoned --
 * the library returned an error, the stream was destroyed, a capture was invalidated -- clear the header before the
 * buffer is used again: vsiq_workspace_reset enqueues that (asynchronous, 256 bytes) on `stream`.  A non-zero header
 * makes the next launch skip work silently; the Python host side resets on every reported error and offers
 * VSIQ_WS_PARANOID=1 (reset before every use) for debugging. */
int vsiq_workspace_reset(void *workspace, size_t workspace_bytes, vsiq_stream_t stream);

/* ---- (3) fake-quant forward ---------------------------------------------------------------
 * y = (clamp(rint(x / s + z), qmin, qmax) - z) * s
 * replaces UniformQuantizer.quantize / discreate_tensor (quantizers/uniform.py:54-55, :95) and
 * LSQFakeQuantize.fake_quantize_per_{tensor,channel}_affine (quantizers/lsq_module.py:220-274).
 * codes (optional, may be NULL): the integer codes as int8 (qmin < 0) or uint8 (qmin >= 0) bytes;
 * the reference only ever holds them as floats (uniform.py:54). */
int vsiq_fake_quant_fwd(const float *x, float *y, void *codes, const vsiq_layout *layout,
                        const vsiq_qparams *qp, vsiq_stream_t stream);

/* ---- integer-code export ------------------------------------------------------------------
 * codes[i] = clamp(rint(x / s + z), qmin, qmax) as integers -- what the reference computes as `x_int` and only ever keeps
 * as a float tensor (quantizers/uniform.py:54,95); the on-wire format of a deployed / exported model (utils/util.py:356-374
 * exports the fake-quantised floats).  code_bits: 16 (int16 / uint16), 8 (int8 / uint8) or 4 (two codes per byte, element
 * 2k in the low nibble; needs an even `inner`); two's complement when qmin < 0, unsigned otherwise; [qmin, qmax] must fit.
 * y (optional): the fake-quantised values from the same pass.  x (and y) 32-byte aligned, codes 16-byte aligned, else
 * VSIQ_ERR_UNSUPPORTED.  NaN inputs get code 0.  Algorithmic traffic: 4 + code_bits/8 bytes per element (+4 with y). */
int vsiq_quantize_codes(const float *x, float *y, void *codes, int code_bits, const vsiq_layout *layout,
                        const vsiq_qparams *qp, vsiq_stream_t stream);

/* ---- (3) STE backward ---------------------------------------------------------------------
 * dx = ((g * s) * m) / s,  m = [qmin <= rint(x/s+z) <= qmax]  -- the autograd graph of the forward
 * through RoundStraightThrough (quantizers/uniform.py:258-271) and torch.clamp; no qparam grads. */
int vsiq_fake_quant_bwd_ste(const float *x, const float *g, float *dx, const vsiq_layout *layout,
                            const vsiq_qparams *qp, vsiq_stream_t stream);

/* ---- (4) LSQ backward ---------------------------------------------------------------------
 * One pass over (x, g): dx as above plus the per-channel step-size and zero-point gradients
 *   dscale[c] = gs * sum g * ((q - z) - m * x/s)
 *   dzp[c]    = gs * [qmin <= rint(z_f) <= qmax] * sum (g*s) * (m - 1)         (dzp may be NULL)
 * replacing autograd over quantizers/uniform.py:47-55 + ScaleGradient (:242-255) and
 * quantizers/lsq_module.py:147-173, :317-340.  gs = grad_scale_host * (grad_scale_dev ? *grad_scale_dev : 1)
 * (the caller computes (qmax * numel / channels) ** -0.5 [* calib_grad_scale, * 5000]).
 * dscale / dzp: `channels` entries of the stated dtype, OVERWRITTEN (not accumulated).
 * Deterministic: fixed-order fp64 combination of per-tile partials (no floating-point atomics). */
size_t vsiq_lsq_bwd_workspace_bytes(const vsiq_layout *layout);
int vsiq_lsq_bwd(const float *x, const float *g, float *dx, void *dscale, int dscale_dtype, void *dzp,
                 int dzp_dtype, const vsiq_layout *layout, const vsiq_qparams *qp, double grad_scale_host,
                 const float *grad_scale_dev, int mask_mode, void *workspace, size_t workspace_bytes,
                 vsiq_stream_t stream);

/* ---- FP8 fake-quant (E4M3 / E5M2) ---------------------------------------------------------
 * The same layouts, qparams and rules as the integer entry points above, with the rounding step on the FP8 value set
 * named by fp8_format (VSIQ_FP8_E4M3: F = 448, VSIQ_FP8_E5M2: F = 57344) instead of the integers.  Per element:
 *   v = x / s;  c = clamp(v, -F, F);  q = value of fp8_rne(c);  y = q * s            (each op rounded once, fp32)
 *   m = (c == v)   inclusive at +-F, false for NaN;  dx = (g * s) * m / s           (as vsiq_fake_quant_bwd_ste)
 *   dscale[c] = gs * sum g * (q - m * v)                                             (as vsiq_lsq_bwd with z = 0)
 * fp8_rne rounds to the nearest FP8 value, ties to an even mantissa; -0.0 stays -0.0 and NaN stays NaN.  The caller's gs
 * is (F * numel / channels) ** -0.5 [* calib_grad_scale].  Symmetric only: qp->qmin == qp->qmax == 0 (else
 * VSIQ_ERR_INVALID_ARG); qp->zero_point NULL, qp->zp_host 0 and qp->zp_learned 0 (else VSIQ_ERR_UNSUPPORTED).  An unknown
 * fp8_format is VSIQ_ERR_INVALID_ARG.  pre_op VSIQ_PRE_RELU is fused as in the integer entry points; VSIQ_PRE_SILU is
 * VSIQ_ERR_UNSUPPORTED here and fused by the channels_last entry points vsiq_ci_fp8_*. */
/* y (optional when codes is given) and codes (optional): one byte per element, the float8_e4m3fn / float8_e5m2 encoding of
 * q.  With codes: pre_op VSIQ_PRE_NONE, x (and y) 32-byte aligned, codes 16-byte aligned, else VSIQ_ERR_UNSUPPORTED. */
int vsiq_fp8_fake_quant_fwd(const float *x, float *y, void *codes, const vsiq_layout *layout, const vsiq_qparams *qp,
                            int fp8_format, vsiq_stream_t stream);
int vsiq_fp8_fake_quant_bwd_ste(const float *x, const float *g, float *dx, const vsiq_layout *layout,
                                const vsiq_qparams *qp, int fp8_format, vsiq_stream_t stream);
/* Workspace: vsiq_lsq_bwd_workspace_bytes.  dzp must be NULL and mask_mode VSIQ_MASK_ROUNDED (else VSIQ_ERR_UNSUPPORTED).
 * Deterministic like vsiq_lsq_bwd. */
int vsiq_fp8_lsq_bwd(const float *x, const float *g, float *dx, void *dscale, int dscale_dtype, void *dzp, int dzp_dtype,
                     const vsiq_layout *layout, const vsiq_qparams *qp, int fp8_format, double grad_scale_host,
                     const float *grad_scale_dev, int mask_mode, void *workspace, size_t workspace_bytes,
                     vsiq_stream_t stream);
/* The channels_last epilogue on the FP8 grids: vsiq_ci_fake_quant_fwd / vsiq_ci_lsq_bwd (below) with the element arithmetic
 * of the FP8 entry points above applied to act(x + bias[c]) (SiLU included); the same layout, alignment, workspace
 * (vsiq_ci_workspace_bytes) and determinism rules.  dzp must be NULL (VSIQ_ERR_UNSUPPORTED); dscale and dbias come from
 * the one backward pass. */
int vsiq_ci_fp8_fake_quant_fwd(const float *x, const float *bias, float *y, int64_t rows, int64_t channels,
                               const vsiq_qparams *qp, int64_t qp_channels, int fp8_format, void *workspace,
                               size_t workspace_bytes, vsiq_stream_t stream);
int vsiq_ci_fp8_lsq_bwd(const float *x, const float *bias, const float *g, float *dx, void *dscale, int dscale_dtype,
                        void *dzp, int dzp_dtype, float *dbias, int64_t rows, int64_t channels, const vsiq_qparams *qp,
                        int64_t qp_channels, int fp8_format, double grad_scale_host, const float *grad_scale_dev,
                        int64_t g_row_pitch, void *workspace, size_t workspace_bytes, vsiq_stream_t stream);
/* The FP8 scale of each channel from an observer's chosen range: scale[c] = max(|lo[c]|, |hi[c]|) / F, or 1.0 when that
 * maximum is zero or not finite.  lo / hi: device fp64 arrays read at c * stride; scale: `channels` device fp64 values,
 * overwritten in place.  No host synchronisation. */
int vsiq_fp8_scale_from_range(const double *lo, const double *hi, int64_t stride, int64_t channels, int fp8_format,
                              double *scale, vsiq_stream_t stream);

/* ---- (1)+(2) observer ---------------------------------------------------------------------
 * One pass over x producing, per channel, {min, max, sum|x|, sum x, sum x^2} (fp64; min/max are the
 * exact fp32 extrema, NaN if the channel holds a NaN, like torch.min/max) -- replaces
 * MinMaxObserver.observe (observers/minmax.py:42-43) and the three extra reductions of
 * QuantizationManager.collect_qparameter (quantizers/quantization_manager.py:66-68): five passes
 * and five host syncs become one pass and none.
 *
 * stats (optional): [channels][VSIQ_STATS_WIDTH] fp64, this call only.
 * state (optional): [channels][VSIQ_STATE_WIDTH] fp64 running observer state, updated in the same
 *   launch: running min/max with the reference's rule (a NaN call extremum never updates,
 *   minmax.py:44-47; the state starts at 0, :28-29), then scale / zero-point from the running
 *   extrema exactly as get_scale_zero_point computes them in Python doubles (minmax.py:67-74), and
 *   the per-call means the LSQ initialisation needs (quantization_manager.py:66,112). */
#define VSIQ_STATS_WIDTH 5 /* min, max, sum|x|, sum x, sum x^2 */
#define VSIQ_STATE_WIDTH 8 /* run_min, run_max, scale, zero_point, n_calls, sum mean|x|, sum mean x, sum std */
size_t vsiq_observe_workspace_bytes(const vsiq_layout *layout);
int vsiq_observe(const float *x, const vsiq_layout *layout, double *stats, double *state, int bits,
                 int symmetric, double eps, void *workspace, size_t workspace_bytes, vsiq_stream_t stream);

/* Calibration epilogue of a fused layer on a channel-innermost tensor: y = act(pre(x)) written AND observed (per tensor)
 * in one pass -- the fused layer's bias add / inference-mode BatchNorm + ReLU / SiLU (modules/fused.py:124-134) followed by
 * quantize_activation -> collect_qparameter -> observer.observe(y) (quantizers/quantization_manager.py:55-71,
 * observers/minmax.py:32-47).  pre: `bias` (x + bias[c]) or `mean`/`var`/`gamma`/`beta`/`bn_eps`
 * (x * a[c] + b[c], a = gamma / sqrt(var + eps), b = beta - mean * a, as vsiq_ci_bn_normalize), or neither; never both.
 * act: VSIQ_PRE_NONE / _RELU / _SILU.  stats / state / bits / symmetric / eps as vsiq_observe with a per-tensor layout.
 * 8 bytes per element instead of 8 + 4 (or ATen's 8 + 8 + 4).  Workspace: vsiq_ci_observe_workspace_bytes(). */
int vsiq_ci_epilogue_observe(const float *x, const float *bias, const float *mean, const float *var, const float *gamma,
                             const float *beta, float bn_eps, int act, float *y, int64_t rows, int64_t channels,
                             double *stats, double *state, int bits, int symmetric, double eps, void *workspace,
                             size_t workspace_bytes, vsiq_stream_t stream);

/* scale / zero-point for n observers at once from their running extrema (after an all-reduce MIN/MAX
 * of the packed state, see parallel.py): state is [n][VSIQ_STATE_WIDTH]; columns 2,3 are rewritten.
 * bits / symmetric: one entry per observer (device int32 arrays) -- observers/minmax.py:67-74. */
int vsiq_qparams_from_minmax(double *state, int64_t n, const int32_t *bits, const int32_t *symmetric,
                             double eps, vsiq_stream_t stream);

/* LSQ step-size initialisation 2 * mean(mean|x|) / sqrt(2^(bits-1) - 1) from the running state
 * (quantizers/quantization_manager.py:112), written to scale_out[channels] of the stated dtype. */
int vsiq_lsq_init_scale(const double *state, int64_t channels, int bits, void *scale_out, int scale_dtype,
                        vsiq_stream_t stream);

/* ---- MSE observer: clipping-range search --------------------------------------------------------------------------
 * One calibration call of observers/mse.py's MSEObserver after vsiq_observe / vsiq_ci_observe has produced this call's
 * per-channel stats (state NULL).  For k = 1..K, alpha_k = k / K (fp64), candidate k clips the running range to
 * (alpha_k * run_min, alpha_k * run_max) and takes (s_k, z_k) from the vsiq_qparams_from_minmax formula at `bits` /
 * `symmetric`; its error is
 *     E[c,k] = sum_i ((double)fq(x_i; s_k, z_k) - (double)x_i)^2      (fq: the fake-quant forward with s_k rounded to fp32,
 *                                                                      integer range of a `bits`-bit quantiser)
 * summed in fp64.  k* = argmin_k E[c,k], ties to the larger alpha; a channel whose range or any E is not finite takes
 * alpha = 1.  The state is [channels][VSIQ_MSE_STATE_WIDTH]: columns 0..7 follow vsiq_observe's rule exactly (running
 * range, call statistics), columns 8, 9 are running means m += (alpha* x run_min - m) / n_calls (and run_max), and columns
 * 2, 3 become scale / zero-point of the mean clipped range.
 * layout: [outer, channels, inner] as everywhere (per tensor, ch_axis 0, NCHW ch_axis 1), or a channels_last [rows, C]
 * tensor as {rows, C, 1} (read in place, four channels per 16-byte load when C % 4 == 0 and x is 16-byte aligned).
 * x is read once; all K candidates are scored from shared memory.  n_candidates: 1..256.
 * err (optional): [channels][n_candidates] fp64, E of this call.  alpha (optional): [channels] fp64, the chosen alpha.
 * Deterministic (fixed-order fp64 combination).  Two launches (search + finalize). */
#define VSIQ_MSE_STATE_WIDTH 10 /* VSIQ_STATE_WIDTH columns, mean clipped min, mean clipped max */
size_t vsiq_mse_search_workspace_bytes(const vsiq_layout *layout, int n_candidates);
int vsiq_mse_search(const float *x, const vsiq_layout *layout, const double *stats, double *state, int bits,
                    int symmetric, double eps, int n_candidates, double *err, double *alpha, void *workspace,
                    size_t workspace_bytes, vsiq_stream_t stream);

/* ---- percentile observer: exact-bin histograms and the clip at a percentile ---------------------------------------
 * One calibration call of observers/percentile.py's PercentileObserver after vsiq_observe / vsiq_ci_observe has produced
 * this call's per-channel stats (state NULL).  B = n_bins bins per side, a power of two in 256..4096.  The state is
 * [channels][VSIQ_HIST_STATE_HEAD + 2 * B] fp64:
 *   0..7   vsiq_observe's running range and call statistics, exactly its rule (columns 2, 3 are then overwritten below)
 *   8, 9   the clipped lo / hi
 *   10, 11 bin exponents e_neg, e_pos: the bin width of a side is 2^e, e the smallest integer >= -149 with
 *          m < B * 2^e for the side's extent m (-run_min, run_max)
 *   12 ..  B counts of x < 0 (bin i: |x| in [i 2^e_neg, (i+1) 2^e_neg)), then B counts of x >= 0, -0.0 included
 * A fresh state is zero except scale = 1 and e_neg = e_pos = -149.  A call first takes the new running range, coarsens
 * the stored counts of a side whose exponent grows (old bin i -> new bin i >> delta, exact), then adds its values.  A
 * channel whose call extrema are NaN keeps its counts; once its running range is not finite the counts are frozen and the
 * clip is the running range.  The clip, from all counts so far: N = total count, T = floor((1 - percentile / 100) * N)
 * (fp64, each operation rounded), hi = min(run_max, (j + 1) 2^e_pos) with j the smallest index whose counts above it sum
 * to <= T, lo = max(run_min, -(j' + 1) 2^e_neg) likewise; columns 2, 3 = scale / zero-point of (lo, hi) with the
 * vsiq_qparams_from_minmax formula.  percentile = 100 gives the min/max result bit for bit.  The counts depend only on the
 * multiset of values observed (integer counts, power-of-two bins), not on call order or on how calls were split.
 * layout: as vsiq_mse_search (channels_last [rows, C] read in place as {rows, C, 1}).  x is read once.  Workspace: the
 * 256-byte header (left untouched) and a count area the call zero-fills itself.  Two launches (histogram + finalize).
 * vsiq_hist_clip recomputes columns 2, 3, 8, 9 from the stored counts at another percentile, with no new data. */
#define VSIQ_HIST_STATE_HEAD 12
size_t vsiq_hist_observe_workspace_bytes(const vsiq_layout *layout, int n_bins); /* 0 for an invalid layout / n_bins */
int vsiq_hist_observe(const float *x, const vsiq_layout *layout, const double *stats, double *state, int n_bins,
                      double percentile, int bits, int symmetric, double eps, void *workspace, size_t workspace_bytes,
                      vsiq_stream_t stream);
int vsiq_hist_clip(double *state, int64_t channels, int n_bins, double percentile, int bits, int symmetric, double eps,
                   vsiq_stream_t stream);

/* ---- entropy observer: the KL-divergence clip searched over the percentile observer's histograms ----------------
 * Recomputes columns 2, 3, 8, 9 of a [channels][VSIQ_HIST_STATE_HEAD + 2 * B] state (vsiq_hist_observe's layout, counts
 * and exponents read only) as observers/entropy.py's EntropyObserver does after every call.  Per channel whose running
 * range (columns 0, 1) is finite:
 *   1. e = max(e_neg, e_pos); both sides coarsened to e (old bin i -> i >> (e - e_side)) and added into one magnitude
 *      histogram H[0..B); then H[0] = H[1] in the search's working copy (the exact zeros of a ReLU output).
 *   2. nq = 2^bits when asymmetric and run_min >= 0, else 2^(bits - 1).
 *   3. candidates i in [max(start_bin, nq), n_used], n_used = 1 + the highest non-zero bin of H; none: the clip is the
 *      running range.
 *   4. D_i = KL(P || Q) in fp64: P = H[0..i) plus the outlier mass sum H[i..B) in bin i - 1; Q = H[0..i) without the
 *      outliers, bin j in chunk floor(j nq / i), each chunk's mass spread evenly over its non-zero bins; both normalised;
 *      D_i = sum_{p_j > 0} p_j ln(p_j / q_j), +inf when some p_j > 0 has q_j = 0.
 *   5. i* = argmin D_i, ties to the largest i, NaN as +inf; amax = i* 2^e, lo = max(run_min, -amax),
 *      hi = min(run_max, amax).
 *   6. columns 8, 9 = (lo, hi); 2, 3 = their vsiq_qparams_from_minmax scale / zero-point.
 * A channel whose running range is not finite keeps it.  start_bin = n_bins gives the min/max result bit for bit.
 * n_bins: a power of two in 256..4096; start_bin: 1..n_bins; bits: 2..8.  divergences (optional, NULL: none):
 * [channels][n_bins + 1] fp64, entry i = D_i, NaN where i is no candidate.  Workspace: the 256-byte header (left zero)
 * and one record per scoring CTA.  Deterministic (every D_i one thread's sequential sum, a total-order argmin), no host
 * synchronisation, graph-capturable.  Two launches (score + finalize). */
size_t vsiq_hist_entropy_workspace_bytes(int64_t channels, int n_bins); /* 0 for invalid channels / n_bins */
int vsiq_hist_entropy_clip(double *state, int64_t channels, int n_bins, int start_bin, int bits, int symmetric,
                           double eps, double *divergences, void *workspace, size_t workspace_bytes,
                           vsiq_stream_t stream);

/* ---- BN re-estimation under data parallelism: the per-layer exchange as ONE kernel over NVLink peer memory -------
 * reestimate_BN_stats (utils/estimate_bn.py:56-99) with the batch sharded over ranks needs sum x / sum x^2 of every rank
 * before a layer's output can be normalised (SURVEY.md 8e).  Instead of combine kernel -> ncclAllReduce -> moments kernel,
 * every rank launches vsiq_bn_moments_exchange: it publishes weight * (sum x, sum x^2) of its shard in its exchange buffer,
 * signals its peers, waits for theirs (release / acquire flag words, system scope), adds all shards in rank order through
 * the peer pointers -- bit-identical sums on every rank -- and finishes like vsiq_bn_moments_finalize (global_count =
 * elements per channel over all ranks).  One process per GPU, one node, world <= vsiq_peer_max_world(), channels <=
 * vsiq_peer_max_channels().  Buffers: vsiq_peer_alloc() (cudaMalloc, zeroed, 64-byte cudaIpc handle to hand to the other
 * ranks), vsiq_peer_open() on their handles, peer_buffers[r] = rank r's buffer as seen from this process (own buffer at
 * [rank]).  Every rank must issue the same sequence of exchanges.  A peer that does not arrive within timeout_s (<= 0:
 * 10 s) makes the kernel give up: outputs untouched, vsiq_peer_status() reports the failed sequence number. */
size_t vsiq_peer_buffer_bytes(void);
int vsiq_peer_max_world(void);
int vsiq_peer_max_channels(void);
int vsiq_peer_alloc(void **buffer, unsigned char *handle64);
int vsiq_peer_open(const unsigned char *handle64, void **buffer);
int vsiq_peer_close(void *buffer);
int vsiq_peer_free(void *buffer);
int vsiq_peer_status(const void *own_buffer, uint64_t *sequence, uint64_t *failed_sequence);
int vsiq_bn_moments_exchange(const double *stats, double weight, double global_count, int64_t channels,
                             void *const *peer_buffers, int rank, int world, double timeout_s, float *batch_mean,
                             float *batch_var_biased, float *batch_var_unbiased, float *mean_sum, float *var_sum,
                             vsiq_stream_t stream);

/* ---- (5) Conv/Linear + BN fold (+ weight fake-quant) ---------------------------------------
 * t = gamma / sqrt(var + eps);  W' = W * t[c];  b' = beta + (b - mean) * t   (b = 0 if bias NULL)
 * replaces ConvBnReLU.__init__ modules/fused.py:98-108 and LinearBnReLU.__init__ :292-300.
 * W is [channels, inner].  b_out may be NULL.
 * Wq_out (optional): the fake-quantised folded weight in the same pass; qp must be non-NULL when Wq_out
 * is, with qp_channels = 1 (per tensor) or = channels (per channel, ch_axis 0) entries.
 * stats (optional, needs workspace): per-tensor {min,max,sum|x|,sum x,sum x^2} of W' from the same
 * pass, to seed the weight observer without re-reading W'. */
size_t vsiq_bn_fold_workspace_bytes(int64_t channels, int64_t inner);
int vsiq_bn_fold(const float *W, const float *bias, const float *gamma, const float *beta, const float *mean,
                 const float *var, float eps, int64_t channels, int64_t inner, float *W_out, float *b_out,
                 float *Wq_out, const vsiq_qparams *qp, int64_t qp_channels, double *stats, void *workspace,
                 size_t workspace_bytes, vsiq_stream_t stream);

/* ---- (6) BN statistics re-estimation ------------------------------------------------------
 * utils/estimate_bn.py:56-99.  The per-batch moments of a conv output [N, C, H*W] come from
 * vsiq_observe(per channel, ch_axis 1): stats[c] = {.., sum x, sum x^2}.  Optionally all-reduce(SUM)
 * the stats over ranks (SyncBN-style), then:
 *   bn_moments_finalize: mean = sum/n, var_b = max(sumsq/n - mean^2, 0), var_u = var_b * n/(n-1)
 *       batch_mean / batch_var_biased / batch_var_unbiased (each optional) <- this batch
 *       mean_sum += mean; var_sum += var_u                  (estimate_bn.py:86-87; optional)
 *   bn_reestimate_finish: running_mean = mean_sum / k; running_var = var_sum / k   (:96-97) */
int vsiq_bn_moments_finalize(const double *stats, double count, int64_t channels, float *batch_mean,
                             float *batch_var_biased, float *batch_var_unbiased, float *mean_sum,
                             float *var_sum, vsiq_stream_t stream);
int vsiq_bn_reestimate_finish(const float *mean_sum, const float *var_sum, int64_t batch_count,
                              float *running_mean, float *running_var, int64_t channels,
                              vsiq_stream_t stream);

/* ---- host-buffer pipeline (end-to-end entry) ----------------------------------------------
 * Forward + STE backward of one per-tensor quantiser over HOST buffers: x, g -> y, dx.  The range is
 * cut into chunks that flow H2D -> fused kernel -> D2H through `n_slots` sets of device staging buffers on
 * three event-linked streams (one per engine), so the two copy directions and the kernel overlap.  Host buffers should be page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory);
 * pageable memory works but serialises.  The handle owns its device staging buffers and streams
 * (these and vsiq_peer_alloc are the only entry points that allocate).  fwd_bwd returns after everything has landed in y / dx. */
typedef struct vsiq_host_pipeline vsiq_host_pipeline;
int vsiq_host_pipeline_create(vsiq_host_pipeline **out, int64_t chunk_elems, int n_slots);
int vsiq_host_pipeline_destroy(vsiq_host_pipeline *p);
int vsiq_host_pipeline_fwd_bwd(vsiq_host_pipeline *p, const float *x_host, const float *g_host, float *y_host,
                               float *dx_host, int64_t n, float scale, float zero_point, int qmin, int qmax);
/* number of kernels the last fwd_bwd call launched (for launch accounting) */
int64_t vsiq_host_pipeline_last_launches(const vsiq_host_pipeline *p);
/* host time (ns) the last vsiq_host_pipeline_fwd_bwd call spent submitting its copies and launches, before waiting */
int64_t vsiq_host_pipeline_last_enqueue_ns(const vsiq_host_pipeline *p);

/* fused forward + STE backward on DEVICE buffers (what the pipeline launches per chunk):
 * one read of x and g, one write of y and dx -- 16 B/element instead of 20. */
int vsiq_fake_quant_fwd_bwd(const float *x, const float *g, float *y, float *dx, const vsiq_layout *layout,
                            const vsiq_qparams *qp, vsiq_stream_t stream);

/* ---- channel-innermost tensors (NHWC / torch.channels_last: cuDNN's native layout on sm_100) ----------
 * The tensor is [rows, channels] with the channel fastest (rows = N*H*W).  channels % 4 == 0 and <= 1024, 16-byte
 * aligned pointers; anything else returns VSIQ_ERR_UNSUPPORTED (the caller converts to NCHW).
 *   forward : y  = fq(act(x + bias[c]))     bias may be NULL; act from qp->pre_op; qp_channels = 1 or channels
 *   backward: dx (act mask included), dscale / dzp (qp_channels entries; dscale NULL = plain STE),
 *             dbias[c] = sum_rows dx (NULL allowed) -- the fused layer's conv-bias gradient (modules/fused.py:124-130;
 *             ATen computes it with a separate full-tensor reduction) comes out of the same pass.
 *             g_row_pitch: elements between consecutive rows of g (0 or `channels` = dense; larger when g is a channel
 *             slice of a wider NHWC tensor, which is what the backward of torch.cat produces; multiple of 4).
 * Same arithmetic, bit-identical values, as vsiq_fake_quant_fwd / vsiq_lsq_bwd on the NCHW-permuted tensor. */
size_t vsiq_ci_workspace_bytes(int64_t rows, int64_t channels);
int vsiq_ci_fake_quant_fwd(const float *x, const float *bias, float *y, int64_t rows, int64_t channels,
                           const vsiq_qparams *qp, int64_t qp_channels, void *workspace, size_t workspace_bytes,
                           vsiq_stream_t stream);
/* Two outputs from one pass over the conv output: y = fq(act(x + bias[c])) with qp, and y2 = fq2(y) with qp2 -- the
 * tensor the NEXT layer's `quantize_inp` step (quantizers/fake_quantize.py:44-45: x = self.quantize_activation(x))
 * would compute from y with its own activation quantiser.  y2 is bit-identical to vsiq_fake_quant_fwd(y, qp2); the pass
 * costs 12 bytes per element instead of 8 + 8 for the two launches it replaces.  qp2->pre_op must be VSIQ_PRE_NONE;
 * qp2_channels = 1 or channels.  The backward is the composition of the existing entry points (vsiq_lsq_bwd /
 * vsiq_fake_quant_bwd_ste at y for the second quantiser, vsiq_ci_lsq_bwd at x for the first). */
int vsiq_ci_fake_quant_fwd2(const float *x, const float *bias, float *y, float *y2, int64_t rows, int64_t channels,
                            const vsiq_qparams *qp, int64_t qp_channels, const vsiq_qparams *qp2,
                            int64_t qp2_channels, void *workspace, size_t workspace_bytes, vsiq_stream_t stream);
int vsiq_ci_lsq_bwd(const float *x, const float *bias, const float *g, float *dx, void *dscale, int dscale_dtype,
                    void *dzp, int dzp_dtype, float *dbias, int64_t rows, int64_t channels, const vsiq_qparams *qp,
                    int64_t qp_channels, double grad_scale_host, const float *grad_scale_dev, int64_t g_row_pitch,
                    void *workspace, size_t workspace_bytes, vsiq_stream_t stream);

/* BatchNorm normalisation of a channel-innermost tensor with GIVEN moments, optionally followed by ReLU:
 *   y = act((x - mean[c]) / sqrt(var[c] + eps) * gamma[c] + beta[c])      (computed as x * a[c] + b[c], one FMA)
 * the second half of each layer of reestimate_BN_stats (utils/estimate_bn.py:79-91 runs the BN in training mode, i.e. with
 * the batch mean and the BIASED batch variance; modules/fused.py:131-134 then applies the ReLU) once vsiq_ci_observe +
 * vsiq_bn_moments_finalize have produced the moments: one read and one write instead of ATen's batch_norm and relu
 * passes.  gamma / beta may be NULL (1 / 0).  Within 2 ulp of ATen's op order (same bar as north_star's BN tolerance). */
int vsiq_ci_bn_normalize(const float *x, const float *mean, const float *var, const float *gamma, const float *beta,
                         float eps, float *y, int64_t rows, int64_t channels, int relu, void *workspace,
                         size_t workspace_bytes, vsiq_stream_t stream);

/* Per-channel observer on a channel-innermost tensor [rows, channels]: the same outputs as vsiq_observe with
 * layout {outer = N, channels, inner = H*W} on the NCHW-permuted tensor (stats[c] / state[c]; min / max exact, sums to
 * summation order), in one read of the NHWC memory -- the moments pass of reestimate_BN_stats
 * (utils/estimate_bn.py:82) and per-channel activation calibration under torch.channels_last.
 * channels % 4 == 0, <= 1024, 16-byte aligned x; else VSIQ_ERR_UNSUPPORTED.  Two launches (stream pass + combine). */
size_t vsiq_ci_observe_workspace_bytes(int64_t rows, int64_t channels);
int vsiq_ci_observe(const float *x, int64_t rows, int64_t channels, double *stats, double *state, int bits,
                    int symmetric, double eps, void *workspace, size_t workspace_bytes, vsiq_stream_t stream);

/* ---- multi-tensor weight path ("weight bank") ---------------------------------------------
 * Every fused layer fake-quantises its (small) weight tensor each step: FakeQuantize.quantize_weights
 * (quantizers/fake_quantize.py:62-63) -> QuantizationManager.quantize (quantization_manager.py:73-90) ->
 * UniformQuantizer.quantize (uniform.py:34-56), i.e. L forward launches and L backward launches per step for
 * L = 57..97 YOLOv8 layers.  These entry points do all L tensors in ONE launch each way (plus one tiny combine
 * launch for the LSQ sums): a table of vsiq_mt_entry describes the tensors, warps take 1024-element tiles across the
 * whole table.  Same arithmetic, bit-identical values, as L calls of vsiq_fake_quant_fwd / vsiq_lsq_bwd.
 *
 * The caller fills one vsiq_mt_entry per tensor, calls vsiq_mt_plan on the HOST array (it fills the fields below the
 * marker), copies the array to the device as plain bytes and passes both copies to the launchers (the host copy gives
 * the launch geometry, the kernels read the device copy).  Pointers inside the table (x, qparams) must stay valid;
 * per-step buffers (y, g, dx, gradient outputs) are launch arguments.  pre_op must be VSIQ_PRE_NONE. */
typedef struct vsiq_mt_entry {
    const float *x;              /* weight [rows, inner] fp32 (any alignment; 32-byte aligned is the fast path); may be NULL
                                    when rows * inner == 0 */
    int64_t rows;                /* output channels */
    int64_t inner;               /* elements per output channel */
    int64_t out_offset;          /* element offset of this tensor inside the flat y (fwd) / dx (bwd) buffer; multiple of 8 */
    int64_t qp_offset;           /* first entry of this tensor inside the flat dscale / dzp outputs */
    int64_t qp_channels;         /* 1 = per tensor, rows = per channel (ch_axis 0) */
    vsiq_qparams qp;
    double grad_scale;           /* LSQ gradient scale, host factor ((qmax * numel / qp_channels) ** -0.5 [* ...]) */
    const float *grad_scale_dev; /* optional device factor (calib_grad_scale), may be NULL */
    int32_t learn;               /* backward: 0 = STE only, 1 = dscale, 2 = dscale and dzero_point */
    /* ---- filled by vsiq_mt_plan ---- */
    uint32_t first_tile;
    uint32_t n_tiles;
    uint32_t chunks;             /* tiles per row */
    int32_t tile;                /* elements per tile */
    float tlo, thi;              /* pre-rounding clamp thresholds derived from qmin / qmax */
} vsiq_mt_entry;

#define VSIQ_MT_MAX_TENSORS 4096
/* Validates the entries and fills their plan fields; *total_tiles receives the tile count of the whole table. */
int vsiq_mt_plan(vsiq_mt_entry *table_host, int n, uint32_t *total_tiles);
/* y_flat[out_offset + i] = fq(x[i]) for every tensor of the table: one launch (none, and y_flat may be NULL, when no
 * tensor of the table has an element; dx_flat likewise below). */
int vsiq_mt_fake_quant_fwd(const vsiq_mt_entry *table_host, const vsiq_mt_entry *table_dev, int n, float *y_flat,
                           vsiq_stream_t stream);
/* dx_flat[out_offset + i], dscale_flat[qp_offset + c] (fp64), dzp_flat[qp_offset + c] (fp32) for every tensor:
 * one streaming launch per 120 tensors plus one combine launch.  g: HOST array of n DEVICE pointers (the upstream
 * gradient of each tensor, same shape as x).  dscale_flat / dzp_flat may be NULL when no entry learns.  The
 * workspace needs no initialisation.  Deterministic (fixed-order fp64 combination). */
size_t vsiq_mt_workspace_bytes(uint32_t total_tiles);
int vsiq_mt_lsq_bwd(const vsiq_mt_entry *table_host, const vsiq_mt_entry *table_dev, int n, const float *const *g,
                    float *dx_flat, double *dscale_flat, float *dzp_flat, void *workspace, size_t workspace_bytes,
                    vsiq_stream_t stream);

/* ---- self-test ---------------------------------------------------------------------------
 * The kernels divide by the (tile-uniform) scale through a hoisted correctly-rounded reciprocal and
 * exact-residual FMA corrections instead of the per-element IEEE division sequence.  This entry
 * counts, over ALL 2^32 bit patterns of the input, how often the fast arithmetic differs from the IEEE
 * sequence (expected: 0).  mode 0: x / s.  mode 1: RN(RN(g*s) / s) (the dx path).
 * *mismatches_dev (device, zero it first) receives the count. */
int vsiq_selftest_division(float s, int mode, unsigned long long *mismatches_dev, vsiq_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VSIQ_H_ */
