// abi.cu -- library-level entry points and the host-side helpers shared by the launchers.
#include <math.h>
#include <stdlib.h>

#include <mutex>

#include "common.cuh"

namespace vsiq {

static std::mutex g_props_mutex;
static DeviceProps g_props[64];
static bool g_props_valid[64];

int get_device_props(DeviceProps* out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 0 || dev >= 64) return (int)cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lk(g_props_mutex);
    if (!g_props_valid[dev]) {
        DeviceProps p;
        if ((e = cudaDeviceGetAttribute(&p.sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
        if ((e = cudaDeviceGetAttribute(&p.cc_major, cudaDevAttrComputeCapabilityMajor, dev)) != cudaSuccess) return (int)e;
        if ((e = cudaDeviceGetAttribute(&p.cc_minor, cudaDevAttrComputeCapabilityMinor, dev)) != cudaSuccess) return (int)e;
        g_props[dev] = p;
        g_props_valid[dev] = true;
    }
    *out = g_props[dev];
    return 0;
}

// Grid policy.  Default: one CTA per tile group, scheduled by the hardware -- the first A/B on B200 showed
// 1.02-1.05x the measured copy bandwidth against 0.85x for a static persistent grid (profiles/README.md).
// VSIQ_GRID_WAVES=k (k >= 1) caps the grid at k x (SM count x 4) CTAs that walk the tiles with a grid
// stride instead (tuning knob for experiments, read once).
static int grid_waves() {
    static int waves = -1;
    if (waves < 0) {
        const char* s = getenv("VSIQ_GRID_WAVES");
        waves = s ? atoi(s) : 0;
        if (waves < 0) waves = 0;
    }
    return waves;
}

int single_wave_ctas() {
    DeviceProps dp;
    if (get_device_props(&dp)) return 1;
    return dp.sm_count * 4;
}

int launch_grid(uint32_t n_ctas_wanted) {
    DeviceProps dp;
    if (int e = get_device_props(&dp)) return -e;
    if (n_ctas_wanted < 1) n_ctas_wanted = 1;
    const int waves = grid_waves();
    if (waves == 0) return (int)(n_ctas_wanted > 0x7fffffffu ? 0x7fffffffu : n_ctas_wanted);
    const uint64_t cap = (uint64_t)dp.sm_count * 4u * (uint64_t)waves;
    return (int)(n_ctas_wanted < cap ? n_ctas_wanted : cap);
}

bool pdl_enabled() {
    static const bool on = []() { const char* e = getenv("VSIQ_PDL"); return !(e && e[0] == '0'); }();
    return on;
}

int ci_sched_override() {
    static const int v = []() {
        const char* e = getenv("VSIQ_CI_SCHED");
        if (!e) return -1;
        if (e[0] == 's') return 0;
        if (e[0] == 'd') return 1;
        if (e[0] == 'i') return 2;
        return -1;
    }();
    return v;
}

int ci_tile_override() {
    static const int v = []() {
        const char* e = getenv("VSIQ_CI_TILE");
        const int n = e ? atoi(e) : 0;
        return n > 0 && n <= 4096 ? n : 0;
    }();
    return v;
}

int pc_chunk_override() {
    static const int v = []() {
        const char* e = getenv("VSIQ_PC_CHUNK");
        const int n = e ? atoi(e) : 0;
        return n >= 2048 && n <= (1 << 20) ? (n / 2048) * 2048 : 0;
    }();
    return v;
}

bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

int check_layout(const vsiq_layout* l) {
    if (!l) return VSIQ_ERR_INVALID_ARG;
    if (l->outer < 0 || l->channels < 1 || l->inner < 0) return VSIQ_ERR_INVALID_ARG;
    if (l->outer > 0 && l->inner > 0) {
        // total element count must fit comfortably in int64 and the tile count in 31 bits
        const long double n = (long double)l->outer * (long double)l->channels * (long double)l->inner;
        if (n >= 9.0e18L) return VSIQ_ERR_INVALID_ARG;
    }
    return VSIQ_OK;
}

int fill_qp(const vsiq_qparams* in, QPDev* out) {
    if (!in) return VSIQ_ERR_INVALID_ARG;
    if (in->qmin >= in->qmax) return VSIQ_ERR_INVALID_ARG;
    if (in->pre_op != VSIQ_PRE_NONE && in->pre_op != VSIQ_PRE_RELU && in->pre_op != VSIQ_PRE_SILU) return VSIQ_ERR_INVALID_ARG;
    if ((in->scale_dtype != VSIQ_F32 && in->scale_dtype != VSIQ_F64) ||
        (in->zp_dtype != VSIQ_F32 && in->zp_dtype != VSIQ_F64))
        return VSIQ_ERR_INVALID_ARG;
    out->scale = in->scale;
    out->zp = in->zero_point;
    out->scale_f64 = in->scale_dtype == VSIQ_F64;
    out->zp_f64 = in->zp_dtype == VSIQ_F64;
    out->scale_host = in->scale_host;
    out->zp_host = in->zp_host;
    out->zp_learned = in->zp_learned ? 1 : 0;
    if (in->qmin < -(1 << 22) || in->qmax > (1 << 22)) return VSIQ_ERR_UNSUPPORTED;  // keeps q +- 0.5 exact in fp32
    out->lo = (float)in->qmin;
    out->hi = (float)in->qmax;
    // rint(t) >= qmin  <=>  t >= qmin - 0.5 when qmin is even (the tie rounds up to qmin), else t > qmin - 0.5
    out->tlo = out->lo - 0.5f;
    if (in->qmin & 1) out->tlo = nextafterf(out->tlo, INFINITY);
    // rint(t) <= qmax  <=>  t <= qmax + 0.5 when qmax is even, else t < qmax + 0.5
    out->thi = out->hi + 0.5f;
    if (in->qmax & 1) out->thi = nextafterf(out->thi, -INFINITY);
    return VSIQ_OK;
}

int fill_qp_fp8(const vsiq_qparams* in, int fp8_format, QPDev* out) {
    if (!in || (fp8_format != VSIQ_FP8_E4M3 && fp8_format != VSIQ_FP8_E5M2)) return VSIQ_ERR_INVALID_ARG;
    if (in->qmin != 0 || in->qmax != 0) return VSIQ_ERR_INVALID_ARG;  // the grid comes from fp8_format
    if (in->pre_op != VSIQ_PRE_NONE && in->pre_op != VSIQ_PRE_RELU && in->pre_op != VSIQ_PRE_SILU) return VSIQ_ERR_INVALID_ARG;
    if (in->scale_dtype != VSIQ_F32 && in->scale_dtype != VSIQ_F64) return VSIQ_ERR_INVALID_ARG;
    // symmetric only: no zero-point tensor, a zero host zero-point, nothing learned
    if (in->zero_point || in->zp_host != 0.0f || in->zp_learned) return VSIQ_ERR_UNSUPPORTED;
    out->scale = in->scale;
    out->zp = nullptr;
    out->scale_f64 = in->scale_dtype == VSIQ_F64;
    out->zp_f64 = 0;
    out->scale_host = in->scale_host;
    out->zp_host = 0.0f;
    out->zp_learned = 0;
    const float F = fp8_max(fp8_format);
    out->lo = out->tlo = -F;
    out->hi = out->thi = F;
    return VSIQ_OK;
}

}  // namespace vsiq

extern "C" int vsiq_version(void) { return VSIQ_VERSION; }

extern "C" int vsiq_workspace_reset(void* workspace, size_t workspace_bytes, vsiq_stream_t stream) {
    if (!workspace || workspace_bytes < vsiq::kWsHeader) return VSIQ_ERR_WORKSPACE;
    return (int)cudaMemsetAsync(workspace, 0, vsiq::kWsHeader, (cudaStream_t)stream);
}

extern "C" const char* vsiq_error_string(int code) {
    switch (code) {
        case VSIQ_OK: return "ok";
        case VSIQ_ERR_INVALID_ARG: return "vsiq: invalid argument";
        case VSIQ_ERR_WORKSPACE: return "vsiq: workspace missing or too small";
        case VSIQ_ERR_UNSUPPORTED: return "vsiq: unsupported combination";
        case VSIQ_ERR_NO_DEVICE: return "vsiq: no usable CUDA device";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "vsiq: unknown error";
}

extern "C" int vsiq_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    vsiq::DeviceProps dp;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1) {
        (void)cudaGetLastError();
        return VSIQ_ERR_NO_DEVICE;
    }
    if (int e = vsiq::get_device_props(&dp)) return e;
    if (sm_count) *sm_count = dp.sm_count;
    if (cc_major) *cc_major = dp.cc_major;
    if (cc_minor) *cc_minor = dp.cc_minor;
    return VSIQ_OK;
}
