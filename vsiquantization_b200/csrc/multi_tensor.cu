// multi_tensor.cu -- the weight path of a whole QAT step in one launch each way ("weight bank").
//
// A fused layer fake-quantises its weight every step (reference: FakeQuantize.quantize_weights,
// quantizers/fake_quantize.py:62-63 -> quantization_manager.py:73-90 -> uniform.py:34-56): YOLOv8 has 57..97 such
// tensors of 432 .. 2.4 M elements, i.e. 2 L launches of mostly tiny kernels per step.  Here a device-resident table
// (vsiq_mt_entry, include/vsiq.h) describes all of them and every warp of the grid takes 1024-element tiles across
// the whole table: one launch for the forward, one streaming launch (+ one combine launch for the per-channel /
// per-tensor LSQ sums) for the backward.  The element arithmetic is the same code as fake_quant.cu (quant_ops.cuh), so
// values are bit-identical to L single-tensor launches.
//
// Roofline: HBM (8 B/element forward, 12 B/element backward) over the sum of the weight tensors (11 M .. 44 M
// elements for YOLOv8s .. l): tens of microseconds, so what this really removes is launch overhead.
#include "quant_ops.cuh"

namespace vsiq {

constexpr int kMtPack = 120;  // upstream-gradient pointers carried as kernel arguments per backward launch

struct MtGradPack {
    const float* g[kMtPack];
};

// largest e in [lo, hi) with table[e].first_tile <= t  (entries without tiles share their successor's first_tile and are
// never selected)
__device__ __forceinline__ int mt_find_entry(const vsiq_mt_entry* __restrict__ table, int lo, int hi, uint32_t t) {
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(&table[mid].first_tile) <= t)
            lo = mid;
        else
            hi = mid;
    }
    return lo;
}

struct MtTile {
    int64_t offset;  // element offset inside the tensor
    int len;
    int64_t channel;  // qparam index
};

__device__ __forceinline__ MtTile mt_tile_at(const vsiq_mt_entry& e, uint32_t local) {
    // per-channel qparams: rows of `inner` elements; per tensor: the whole tensor is one row
    const bool pc = e.qp_channels > 1;
    const int64_t inner = pc ? e.inner : e.rows * e.inner;
    const uint32_t row = local / e.chunks;
    const uint32_t chunk = local - row * e.chunks;
    const int64_t start = (int64_t)chunk * e.tile;
    const int64_t rem = inner - start;
    MtTile t;
    t.len = rem < e.tile ? (int)rem : e.tile;
    t.offset = (int64_t)row * inner + start;
    t.channel = pc ? row : 0;
    return t;
}

__device__ __forceinline__ QPDev mt_qpdev(const vsiq_mt_entry& e) {
    QPDev d;
    d.scale = e.qp.scale;
    d.zp = e.qp.zero_point;
    d.scale_f64 = e.qp.scale_dtype == VSIQ_F64;
    d.zp_f64 = e.qp.zp_dtype == VSIQ_F64;
    d.scale_host = e.qp.scale_host;
    d.zp_host = e.qp.zp_host;
    d.zp_learned = e.qp.zp_learned ? 1 : 0;
    d.lo = (float)e.qp.qmin;
    d.hi = (float)e.qp.qmax;
    d.tlo = e.tlo;
    d.thi = e.thi;
    return d;
}

__device__ __forceinline__ bool mt_aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

__global__ void __launch_bounds__(kThreads)
    mt_fwd_kernel(const vsiq_mt_entry* __restrict__ table, int n, uint32_t total_tiles, float* __restrict__ y_flat) {
    const uint32_t t = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (t >= total_tiles) return;
    const int ei = mt_find_entry(table, 0, n, t);
    const vsiq_mt_entry e = table[ei];
    const MtTile tl = mt_tile_at(e, t - e.first_tile);
    const QPDev qpd = mt_qpdev(e);
    FwdOp<false> op;
    op.p = load_qp(qpd, tl.channel);
    const float* const in[1] = {e.x};
    float* const out[1] = {y_flat + e.out_offset};
    if (mt_aligned32(e.x) && mt_aligned32(out[0]))
        span_apply<32, kVec, 1, 1>(in, out, tl.offset, tl.len, op);
    else
        span_apply<32, 1, 1, 1>(in, out, tl.offset, tl.len, op);
}

// entries [e_lo, e_hi) of the table, tiles [tile_lo, tile_hi); g.g[i] belongs to entry e_lo + i
__global__ void __launch_bounds__(kThreads)
    mt_bwd_kernel(const vsiq_mt_entry* __restrict__ table, int e_lo, int e_hi, uint32_t tile_lo, uint32_t tile_hi,
                  MtGradPack g, float* __restrict__ dx_flat, double* __restrict__ partials) {
    const uint32_t t = tile_lo + blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (t >= tile_hi) return;
    const int ei = mt_find_entry(table, e_lo, e_hi, t);
    const vsiq_mt_entry e = table[ei];
    const MtTile tl = mt_tile_at(e, t - e.first_tile);
    const QPDev qpd = mt_qpdev(e);
    LsqBwdOp<VSIQ_MASK_ROUNDED, true, false> op;
    op.p = load_qp(qpd, tl.channel);
    op.e_acc = 0.0f;
    op.b_acc = 0.0f;
    const float* gp = g.g[ei - e_lo];
    const float* const in[2] = {e.x, gp};
    float* const out[1] = {dx_flat + e.out_offset};
    if (mt_aligned32(e.x) && mt_aligned32(gp) && mt_aligned32(out[0]))
        span_apply<32, kVec, 2, 1>(in, out, tl.offset, tl.len, op);
    else
        span_apply<32, 1, 2, 1>(in, out, tl.offset, tl.len, op);
    if (e.learn) {  // warp-uniform
        const float es = warp_sum(op.e_acc);
        const float bs = warp_sum(op.b_acc);
        if ((threadIdx.x & 31) == 0) {
            partials[2 * (size_t)t] = (double)es;
            partials[2 * (size_t)t + 1] = (double)bs;
        }
    }
}

// one warp per qparam entry of the flat gradient outputs: fixed-order fp64 sum of that channel's tile records
__global__ void __launch_bounds__(kThreads)
    mt_combine_kernel(const vsiq_mt_entry* __restrict__ table, int n, int64_t total_q, const double* __restrict__ partials,
                      double* __restrict__ dscale_flat, float* __restrict__ dzp_flat) {
    const int lane = threadIdx.x & 31;
    for (int64_t q = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); q < total_q; q += (int64_t)gridDim.x * kWarps) {
        int lo = 0, hi = n;  // largest entry with qp_offset <= q
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(&table[mid].qp_offset) <= q)
                lo = mid;
            else
                hi = mid;
        }
        const vsiq_mt_entry e = table[lo];
        const int64_t c = q - e.qp_offset;
        if (!e.learn || c >= e.qp_channels) continue;
        const bool pc = e.qp_channels > 1;
        const uint32_t first = e.first_tile + (pc ? (uint32_t)c * e.chunks : 0u);
        const uint32_t items = pc ? e.chunks : e.n_tiles;
        double es = 0.0, bs = 0.0;
        for (uint32_t i = lane; i < items; i += 32) {
            es += __ldcg(partials + 2 * (size_t)(first + i));
            bs += __ldcg(partials + 2 * (size_t)(first + i) + 1);
        }
        es = warp_sum(es);
        bs = warp_sum(bs);
        if (lane == 0) {
            const double gs = e.grad_scale * (e.grad_scale_dev ? (double)__ldg(e.grad_scale_dev) : 1.0);
            double ds, dz;
            lsq_channel_grads(gs, es, bs, mt_qpdev(e), c, &ds, &dz);
            if (dscale_flat) dscale_flat[q] = ds;
            if (dzp_flat && e.learn > 1) dzp_flat[q] = (float)dz;
        }
    }
}

}  // namespace vsiq

using namespace vsiq;

extern "C" int vsiq_mt_plan(vsiq_mt_entry* table, int n, uint32_t* total_tiles) {
    if (!table || n < 1 || n > VSIQ_MT_MAX_TENSORS || !total_tiles) return VSIQ_ERR_INVALID_ARG;
    uint64_t tiles = 0;
    for (int i = 0; i < n; ++i) {
        vsiq_mt_entry& e = table[i];
        // an entry without elements is never read: its x may be NULL (torch gives every empty tensor a NULL data_ptr)
        if ((!e.x && e.rows && e.inner) || e.rows < 0 || e.inner < 0 || e.out_offset < 0 || (e.out_offset & 7) || e.qp_offset < 0)
            return VSIQ_ERR_INVALID_ARG;
        if (e.qp_channels != 1 && e.qp_channels != e.rows) return VSIQ_ERR_INVALID_ARG;
        if (e.learn < 0 || e.learn > 2) return VSIQ_ERR_INVALID_ARG;
        if (e.qp.pre_op != VSIQ_PRE_NONE) return VSIQ_ERR_UNSUPPORTED;
        if (i > 0 && e.qp_offset < table[i - 1].qp_offset + table[i - 1].qp_channels) return VSIQ_ERR_INVALID_ARG;
        QPDev d;
        if (int err = fill_qp(&e.qp, &d)) return err;
        e.tlo = d.tlo;
        e.thi = d.thi;
        const bool pc = e.qp_channels > 1;
        const int64_t rows = pc ? e.rows : 1;
        const int64_t inner = pc ? e.inner : e.rows * e.inner;
        e.first_tile = (uint32_t)tiles;
        e.n_tiles = 0;
        e.chunks = 1;
        e.tile = kWarpTile;
        if (rows > 0 && inner > 0) {
            Tiles t;
            if (!make_tiles<32>(1, rows, inner, &t)) return VSIQ_ERR_UNSUPPORTED;
            e.n_tiles = t.n_tiles;
            e.chunks = t.chunks;
            e.tile = t.tile;
        }
        tiles += e.n_tiles;
        if (tiles >= (uint64_t(1) << 31)) return VSIQ_ERR_UNSUPPORTED;
    }
    *total_tiles = (uint32_t)tiles;
    return VSIQ_OK;
}

static uint32_t mt_total_tiles(const vsiq_mt_entry* table, int n) { return table[n - 1].first_tile + table[n - 1].n_tiles; }

extern "C" int vsiq_mt_fake_quant_fwd(const vsiq_mt_entry* table_host, const vsiq_mt_entry* table_dev, int n,
                                      float* y_flat, vsiq_stream_t stream) {
    if (!table_host || !table_dev || n < 1 || n > VSIQ_MT_MAX_TENSORS) return VSIQ_ERR_INVALID_ARG;
    const uint32_t total = mt_total_tiles(table_host, n);
    if (total == 0) return VSIQ_OK;  // nothing to write: y_flat may be NULL (torch's empty buffer)
    if (!y_flat) return VSIQ_ERR_INVALID_ARG;
    const uint32_t grid = (total + kWarps - 1) / kWarps;
    mt_fwd_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(table_dev, n, total, y_flat);
    return (int)cudaGetLastError();
}

extern "C" size_t vsiq_mt_workspace_bytes(uint32_t total_tiles) { return kWsHeader + (size_t)total_tiles * 2 * sizeof(double); }

extern "C" int vsiq_mt_lsq_bwd(const vsiq_mt_entry* table_host, const vsiq_mt_entry* table_dev, int n,
                               const float* const* g, float* dx_flat, double* dscale_flat, float* dzp_flat,
                               void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    if (!table_host || !table_dev || n < 1 || n > VSIQ_MT_MAX_TENSORS || !g) return VSIQ_ERR_INVALID_ARG;
    const uint32_t total = mt_total_tiles(table_host, n);
    if (!dx_flat && total) return VSIQ_ERR_INVALID_ARG;  // a table without tiles writes no dx
    bool learns = false;
    for (int i = 0; i < n; ++i) {
        if (!g[i] && table_host[i].n_tiles) return VSIQ_ERR_INVALID_ARG;
        learns = learns || table_host[i].learn != 0;
        if (table_host[i].learn > 0 && !dscale_flat) return VSIQ_ERR_INVALID_ARG;
        if (table_host[i].learn > 1 && !dzp_flat) return VSIQ_ERR_INVALID_ARG;
    }
    if (learns && (!workspace || workspace_bytes < vsiq_mt_workspace_bytes(total))) return VSIQ_ERR_WORKSPACE;
    double* partials = learns ? (double*)((char*)workspace + kWsHeader) : nullptr;
    for (int e_lo = 0; e_lo < n; e_lo += kMtPack) {
        const int e_hi = e_lo + kMtPack < n ? e_lo + kMtPack : n;
        const uint32_t tile_lo = table_host[e_lo].first_tile;
        const uint32_t tile_hi = table_host[e_hi - 1].first_tile + table_host[e_hi - 1].n_tiles;
        if (tile_hi == tile_lo) continue;
        MtGradPack pack;
        for (int i = 0; i < kMtPack; ++i) pack.g[i] = e_lo + i < e_hi ? g[e_lo + i] : nullptr;
        const uint32_t grid = (tile_hi - tile_lo + kWarps - 1) / kWarps;
        mt_bwd_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(table_dev, e_lo, e_hi, tile_lo, tile_hi, pack, dx_flat,
                                                                  partials);
        if (cudaError_t err = cudaGetLastError()) return (int)err;
    }
    const int64_t total_q = table_host[n - 1].qp_offset + table_host[n - 1].qp_channels;
    if (learns && total_q > 0) {  // learning entries with zero channels (rows == 0, per channel) have nothing to combine
        int64_t grid = (total_q + kWarps - 1) / kWarps;
        if (grid > 1184) grid = 1184;
        mt_combine_kernel<<<(unsigned)grid, kThreads, 0, (cudaStream_t)stream>>>(table_dev, n, total_q, partials,
                                                                                  dscale_flat, dzp_flat);
        if (cudaError_t err = cudaGetLastError()) return (int)err;
    }
    return VSIQ_OK;
}
