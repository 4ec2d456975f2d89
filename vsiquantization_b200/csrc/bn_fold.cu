// bn_fold.cu -- kernel (5): Conv/Linear + BatchNorm fold, optionally fused with the weight fake-quant
// and with the weight observer's statistics, all in one pass over W.
//
// Reference semantics (bit-exact, fp32, this operation order):
//   std = sqrt(running_var + eps); t = gamma / std; W' = W * t[c]; b' = beta + (b - running_mean) * t
//   modules/fused.py:98-108 (ConvBnReLU.__init__), :292-300 (LinearBnReLU.__init__)
//   fake-quant of W': quantizers/uniform.py:54-55,95
//
// Roofline: HBM, 8 algorithmic bytes per element (read W, write W'), +4 when Wq is also written.
#include "reduce.cuh"

namespace vsiq {

template <bool WANT_Q, bool WANT_STATS>
struct FoldOp : OpBase {
    float t;
    QP p;
    // statistics of W' (only with WANT_STATS)
    float mn, mx;
    bool bad;
    float fa, f1, f2;
    double sa, s1, s2;
    __device__ __forceinline__ void reset_stats() {
        mn = INFINITY;
        mx = -INFINITY;
        bad = false;
        fa = f1 = f2 = 0.0f;
        sa = s1 = s2 = 0.0;
    }
    // Folded weights are quantised with the IEEE sequence: W is a few MB at most (launch-bound), and it
    // keeps the statistics free of the redo protocol.
    __device__ __forceinline__ void apply_slow(const float (&a)[1], float (&o)[WANT_Q ? 2 : 1]) { apply(a, o); }
    __device__ __forceinline__ void apply(const float (&a)[1], float (&o)[WANT_Q ? 2 : 1]) {
        const float w = __fmul_rn(a[0], t);
        o[0] = w;
        if (WANT_Q) o[WANT_Q ? 1 : 0] = dequant(elem_slow(w, p).q, p);
        if (WANT_STATS) {
            bad = bad || (w != w);
            mn = fminf(mn, w);
            mx = fmaxf(mx, w);
            fa += fabsf(w);
            f1 += w;
            f2 = fmaf(w, w, f2);
        }
    }
    __device__ __forceinline__ void vec_done() {
        if (WANT_STATS) {
            sa += (double)fa;
            s1 += (double)f1;
            s2 += (double)f2;
            fa = f1 = f2 = 0.0f;
        }
    }
};

template <int GROUP, int V, bool WANT_Q, bool WANT_STATS>
__global__ void __launch_bounds__(kThreads)
    bn_fold_kernel(const float* __restrict__ W, const float* __restrict__ bias, const float* __restrict__ gamma,
                   const float* __restrict__ beta, const float* __restrict__ mean, const float* __restrict__ var,
                   float eps, Tiles tiles, float* __restrict__ W_out, float* __restrict__ b_out,
                   float* __restrict__ Wq_out, QPDev qpd, int qp_per_channel, double* __restrict__ stats, void* ws) {
    __shared__ StatsRec s_red[kWarps];
    constexpr int NOUT = WANT_Q ? 2 : 1;
    const float* const in[1] = {W};
    float* outs[2] = {W_out, Wq_out};
    float* const(&out)[NOUT] = reinterpret_cast<float* const(&)[NOUT]>(outs);
    const bool leader = GROUP == 32 ? (threadIdx.x & 31) == 0 : threadIdx.x == 0;

    FoldOp<WANT_Q, WANT_STATS> op;
    if (WANT_STATS) op.reset_stats();
    for (uint32_t ti = group_index<GROUP>(); ti < tiles.n_tiles; ti += group_count<GROUP>()) {
        const TileCursor<GROUP> c = tile_at<GROUP>(tiles, ti);
        const int64_t ch = c.row;  // W is [channels, inner]: row == output channel
        const float sd = __fsqrt_rn(__fadd_rn(__ldg(var + ch), eps));
        op.t = __fdiv_rn(__ldg(gamma + ch), sd);
        if (WANT_Q) op.p = load_qp(qpd, qp_per_channel ? ch : 0);
        if (b_out && leader && c.offset == ch * tiles.inner) {  // first chunk of the row folds the bias
            const float b = bias ? __ldg(bias + ch) : 0.0f;
            b_out[ch] = __fadd_rn(__ldg(beta + ch), __fmul_rn(__fsub_rn(b, __ldg(mean + ch)), op.t));
        }
        span_apply<GROUP, V, 1, NOUT>(in, out, c.offset, c.len, op);
    }
    if (!WANT_STATS) return;

    // per-tensor statistics of W': one record per group (fminf / fmaxf drop NaN, so a NaN seen turns both into NaN),
    // combined by a warp of the last CTA
    double* partials = ws_partials(ws);
    const StatsRec rec = block_record<GROUP>(
        StatsRec{op.bad ? NAN : op.mn, op.bad ? NAN : op.mx, op.sa, op.s1, op.s2}, s_red);
    if (leader) rec.store(partials + (size_t)group_index<GROUP>() * StatsRec::kSlot);
    if (!last_cta_ticket((unsigned int*)ws, leader)) return;
    ObserveOut o = {};
    o.stats = stats;
    if (threadIdx.x < 32) combine_channel<32>(partials, cta_records(group_count<GROUP>()), 1, 0, o, s_red);
}

// upper bound of groups any launch of this kernel can have (partials are per group)
static size_t fold_max_groups(int64_t channels, int64_t inner) {
    Tiles tc, tw;
    size_t g = 1;
    if (make_tiles<kThreads>(1, channels, inner, &tc)) g = tc.n_tiles;
    if (inner < kWarpGroupMaxInner && make_tiles<32>(1, channels, inner, &tw)) {
        size_t w = ((size_t)tw.n_tiles + kWarps - 1) / kWarps * kWarps;
        g = w > g ? w : g;
    }
    return g;
}

}  // namespace vsiq

using namespace vsiq;

extern "C" size_t vsiq_bn_fold_workspace_bytes(int64_t channels, int64_t inner) {
    if (channels <= 0 || inner <= 0) return 0;
    return kWsHeader + fold_max_groups(channels, inner) * StatsRec::kSlot * sizeof(double);
}

extern "C" int vsiq_bn_fold(const float* W, const float* bias, const float* gamma, const float* beta,
                            const float* mean, const float* var, float eps, int64_t channels, int64_t inner,
                            float* W_out, float* b_out, float* Wq_out, const vsiq_qparams* qp, int64_t qp_channels,
                            double* stats, void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    if (!W || !gamma || !beta || !mean || !var || !W_out || channels <= 0 || inner <= 0) return VSIQ_ERR_INVALID_ARG;
    if (Wq_out && !qp) return VSIQ_ERR_INVALID_ARG;
    if (stats && (!workspace || workspace_bytes < vsiq_bn_fold_workspace_bytes(channels, inner)))
        return VSIQ_ERR_WORKSPACE;
    QPDev qpd = {};
    if (Wq_out)
        if (int e = fill_qp(qp, &qpd)) return e;
    if (Wq_out && qp_channels != 1 && qp_channels != channels) return VSIQ_ERR_INVALID_ARG;
    const int qp_per_channel = (Wq_out && qp_channels == channels && channels > 1) ? 1 : 0;
    cudaStream_t st = (cudaStream_t)stream;
    const bool warp_group = inner < kWarpGroupMaxInner;
    const bool vec8 = aligned32(W) && aligned32(W_out) && (!Wq_out || aligned32(Wq_out));
    Tiles tiles;
#define LAUNCH(G, V, Q, S)                                                                                      \
    {                                                                                                           \
        if (!make_tiles<G>(1, channels, inner, &tiles)) return VSIQ_ERR_INVALID_ARG;                            \
        uint32_t want = G == kThreads ? tiles.n_tiles : (tiles.n_tiles + kWarps - 1) / kWarps;                  \
        int grid = launch_grid(want);                                            \
        if (grid < 0) return -grid;                                                                             \
        bn_fold_kernel<G, V, Q, S><<<grid, kThreads, 0, st>>>(W, bias, gamma, beta, mean, var, eps, tiles, W_out, \
                                                              b_out, Wq_out, qpd, qp_per_channel, stats, workspace); \
    }
#define CALL(G, V)                        \
    {                                     \
        if (Wq_out && stats) {            \
            LAUNCH(G, V, true, true);     \
        } else if (Wq_out) {              \
            LAUNCH(G, V, true, false);    \
        } else if (stats) {               \
            LAUNCH(G, V, false, true);    \
        } else {                          \
            LAUNCH(G, V, false, false);   \
        }                                 \
    }
    if (warp_group) {
        if (vec8) CALL(32, 8) else CALL(32, 1)
    } else {
        if (vec8) CALL(kThreads, 8) else CALL(kThreads, 1)
    }
#undef CALL
#undef LAUNCH
    return (int)cudaGetLastError();
}
