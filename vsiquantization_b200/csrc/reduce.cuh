// reduce.cuh -- the record-and-combine scheme of the reducing kernels (observer, LSQ backward, BN-fold statistics).
//
// A streaming kernel reduces its share of the tensor to one fp64 record per tile, persistent CTA or channel-item CTA and
// writes it into the workspace (after kWsHeader).  The records of each channel are then combined in a fixed order, so
// results are deterministic and need no floating-point atomics:
//   * by the last CTA of the launch (ticket, see last_cta_ticket) when the grid fits one wave: combine_in_last_cta;
//   * otherwise by finalize_kernel, launched as a programmatic dependent of the streaming kernel: launch_finalize.
// A channel's records are combined by one thread, one warp or one CTA (combine_channel<1 / 32 / kThreads>).
//
// A record type Rec provides identity(), fold(), load() from a workspace slot, store() into one, warp_reduce() (result in
// lane 0) and kSlot, its slot width in doubles.  block_record takes any per-thread type whose warp_reduce() yields a Rec,
// which is how a kernel chooses the precision of its warp stage.
#pragma once

#include "common.cuh"

namespace vsiq {

// min / max (NaN-propagating, fp32), sum|x|, sum x, sum x^2 (fp64).  Slot 5 is written as 0 and never read.
struct StatsRec {
    float mn, mx;
    double sa, s1, s2;
    static constexpr int kSlot = 6;
    __device__ __forceinline__ static StatsRec identity() { return {INFINITY, -INFINITY, 0.0, 0.0, 0.0}; }
    __device__ __forceinline__ void fold(const StatsRec& o) {
        mn = nanmin(mn, o.mn);
        mx = nanmax(mx, o.mx);
        sa += o.sa;
        s1 += o.s1;
        s2 += o.s2;
    }
    __device__ __forceinline__ static StatsRec load(const double* p) {
        return {(float)__ldcg(p), (float)__ldcg(p + 1), __ldcg(p + 2), __ldcg(p + 3), __ldcg(p + 4)};
    }
    __device__ __forceinline__ void store(double* p) const {
        p[0] = (double)mn;
        p[1] = (double)mx;
        p[2] = sa;
        p[3] = s1;
        p[4] = s2;
        p[5] = 0.0;
    }
    __device__ __forceinline__ StatsRec warp_reduce() const {
        return {warp_min(mn), warp_max(mx), warp_sum(sa), warp_sum(s1), warp_sum(s2)};
    }
};

// LSQ backward sums: E = sum g * ((q - z) - m * x/s), B = sum g over clamped-out elements (fp64).
struct LsqRec {
    double e, b;
    static constexpr int kSlot = 2;
    __device__ __forceinline__ static LsqRec identity() { return {0.0, 0.0}; }
    __device__ __forceinline__ void fold(const LsqRec& o) {
        e += o.e;
        b += o.b;
    }
    __device__ __forceinline__ static LsqRec load(const double* p) { return {__ldcg(p), __ldcg(p + 1)}; }
    __device__ __forceinline__ void store(double* p) const {
        p[0] = e;
        p[1] = b;
    }
    __device__ __forceinline__ LsqRec warp_reduce() const { return {warp_sum(e), warp_sum(b)}; }
};

// A thread's LSQ sums in T (float: the per-tile records are fp32 warp sums; double: sums carried across tiles);
// B is reduced only when the kernel computes it.
template <class T, bool WANT_B>
struct LsqSums {
    T e, b;
    __device__ __forceinline__ LsqRec warp_reduce() const {
        return {(double)warp_sum(e), WANT_B ? (double)warp_sum(b) : 0.0};
    }
};

// The warps' records (already warp-reduced, lane 0) folded in warp order; valid in thread 0.
template <class Rec>
__device__ __forceinline__ Rec cta_fold(const Rec& warp_rec, Rec* s_red) {
    __syncthreads();  // s_red may still be read by the previous fold
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = warp_rec;
    __syncthreads();
    Rec r = s_red[0];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) r.fold(s_red[w]);
    return r;
}

// One group's per-thread values -> one record, valid in lane 0 (GROUP 32) or thread 0 (GROUP kThreads).
template <int GROUP, class Rec, class Part>
__device__ __forceinline__ Rec block_record(const Part& mine, Rec* s_red) {
    const Rec r = mine.warp_reduce();
    if constexpr (GROUP == 32)
        return r;
    else
        return cta_fold(r, s_red);
}

// Combine the records of channel c (it owns outer * tiles.chunks of them, see record_slot) and hand the result to
// out.store(c, rec): STRIDE threads cooperate (1, 32 = one warp, kThreads = the whole CTA).
template <int STRIDE, class Rec, class Out>
__device__ __forceinline__ void combine_channel(const double* partials, const Tiles& tiles, int64_t outer, int64_t c,
                                                const Out& out, Rec* s_red) {
    const int lane = threadIdx.x & 31;
    const int tid = STRIDE == 1 ? 0 : (STRIDE == 32 ? lane : (int)threadIdx.x);
    const uint32_t items = (uint32_t)outer * tiles.chunks;
    Rec r = Rec::identity();
#pragma unroll 2
    for (uint32_t i = tid; i < items; i += STRIDE)
        r.fold(Rec::load(partials + (size_t)record_slot(tiles, (uint32_t)outer, (uint32_t)c, i) * Rec::kSlot));
    if constexpr (STRIDE == 1) {
        out.store(c, r);
    } else if constexpr (STRIDE == 32) {
        r = r.warp_reduce();
        if (lane == 0) out.store(c, r);
    } else {
        r = cta_fold(r.warp_reduce(), s_red);
        if (threadIdx.x == 0) out.store(c, r);
    }
}

// The last CTA combines every channel: a thread per channel when channels own few records, else the whole CTA per
// channel when there are fewer channels than warps, else a warp per channel.
template <class Rec, class Out>
__device__ __forceinline__ void combine_in_last_cta(const double* partials, const Tiles& tiles, int64_t outer,
                                                    const Out& out, Rec* s_red) {
    if ((uint32_t)outer * tiles.chunks <= kThreadCombineMaxItems) {
        for (int64_t c = threadIdx.x; c < tiles.channels; c += kThreads) combine_channel<1>(partials, tiles, outer, c, out, s_red);
    } else if (tiles.channels < kWarps) {
        for (int64_t c = 0; c < tiles.channels; ++c) combine_channel<kThreads>(partials, tiles, outer, c, out, s_red);
    } else {
        for (int64_t c = threadIdx.x >> 5; c < tiles.channels; c += kWarps) combine_channel<32>(partials, tiles, outer, c, out, s_red);
    }
}

// MODE 0: thread per channel, 1: warp per channel, 2: CTA per channel
template <int MODE, class Rec, class Out>
__global__ void __launch_bounds__(kThreads) finalize_kernel(Tiles tiles, int64_t outer, const void* ws, Out o) {
    __shared__ Rec s_red[kWarps];
    const double* partials = (const double*)((const char*)ws + kWsHeader);
    pdl_wait();  // a programmatic dependent of the streaming kernel: its records are complete from here on
    if (MODE == 0) {
        for (int64_t c = (int64_t)blockIdx.x * kThreads + threadIdx.x; c < tiles.channels; c += (int64_t)gridDim.x * kThreads)
            combine_channel<1>(partials, tiles, outer, c, o, s_red);
    } else if (MODE == 2) {
        for (int64_t c = blockIdx.x; c < tiles.channels; c += gridDim.x) combine_channel<kThreads>(partials, tiles, outer, c, o, s_red);
    } else {
        for (int64_t c = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); c < tiles.channels; c += (int64_t)gridDim.x * kWarps)
            combine_channel<32>(partials, tiles, outer, c, o, s_red);
    }
}

// Records of the channel-item schedule (PcGeom): k consecutive records per channel.
__host__ __device__ inline Tiles item_records(const PcGeom& g) {
    Tiles t;
    t.rows = g.channels;
    t.channels = g.channels;
    t.inner = 0;
    t.chunks = g.k;
    t.n_tiles = (uint32_t)g.channels * g.k;
    t.tile = 0;
    return t;
}

// One record per CTA (or per group) of a single channel: the per-tensor, epilogue and BN-fold kernels.
__host__ __device__ inline Tiles cta_records(uint32_t n) {
    Tiles t;
    t.rows = 1;
    t.channels = 1;
    t.inner = 0;
    t.chunks = n;
    t.n_tiles = n;
    t.tile = 0;
    return t;
}

// The finalize launch for records no ticket combined.  The channel-item schedule (cta_per_channel false) combines with
// a thread or a warp per channel whatever its record count.
template <class Rec, class Out>
inline void launch_finalize(const Tiles& recs, int64_t outer, bool cta_per_channel, void* ws, const Out& o,
                            cudaStream_t st) {
    const int64_t items = outer * (int64_t)recs.chunks;
    const int64_t C = recs.channels;
    if (items <= kThreadCombineMaxItems) {
        const int64_t fg = (C + kThreads - 1) / kThreads;
        launch_pdl(finalize_kernel<0, Rec, Out>, dim3((unsigned)(fg < 4096 ? fg : 4096)), dim3(kThreads), 0, st, recs, outer, ws, o);
    } else if (cta_per_channel && items >= 512) {
        launch_pdl(finalize_kernel<2, Rec, Out>, dim3((unsigned)(C < 1024 ? C : 1024)), dim3(kThreads), 0, st, recs, outer, ws, o);
    } else {
        const int64_t fg = (C + kWarps - 1) / kWarps;
        launch_pdl(finalize_kernel<1, Rec, Out>, dim3((unsigned)(fg < 4096 ? fg : 4096)), dim3(kThreads), 0, st, recs, outer, ws, o);
    }
}

// Workspace of vsiq_observe / vsiq_lsq_bwd: one slot per tile of the larger of the CTA- and warp-tile schedules, so the
// caller need not know the launch geometry; x2: the channel-item schedule may use 4096-element units.
inline size_t reduce_workspace_bytes(const vsiq_layout* layout, int slot_doubles) {
    if (check_layout(layout)) return 0;
    Tiles tc, tw;
    size_t slots = 1;
    if (make_tiles<kThreads>(layout->outer, layout->channels, layout->inner, &tc)) slots = tc.n_tiles;
    if (layout->inner < kWarpGroupMaxInner && make_tiles<32>(layout->outer, layout->channels, layout->inner, &tw))
        slots = tw.n_tiles > slots ? tw.n_tiles : slots;
    return kWsHeader + 2 * slots * slot_doubles * sizeof(double);
}

// What the observer combine produces / updates for one channel.
struct ObserveOut {
    double* stats;  // [C][VSIQ_STATS_WIDTH] or null
    double* state;  // [C][VSIQ_STATE_WIDTH] or null
    int bits;
    int symmetric;
    double eps;
    double count;   // elements per channel
    __device__ __forceinline__ void store(int64_t c, const StatsRec& r) const {
        if (stats) {
            double* d = stats + c * VSIQ_STATS_WIDTH;
            d[0] = (double)r.mn;
            d[1] = (double)r.mx;
            d[2] = r.sa;
            d[3] = r.s1;
            d[4] = r.s2;
        }
        if (state) observer_state_update(state + c * VSIQ_STATE_WIDTH, r.mn, r.mx, r.sa, r.s1, r.s2, count, bits, symmetric, eps);
    }
};

}  // namespace vsiq
