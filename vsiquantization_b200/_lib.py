"""ctypes binding of libvsiq.so (the C ABI declared in include/vsiq.h).

There is no CPU fallback anywhere in this package: if the shared library is missing this module
raises at import time, and every op raises when it is handed a tensor it cannot run on the GPU.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VSIQ_LIB") or os.path.join(_HERE, "libvsiq.so")  # VSIQ_LIB: A/B-testing builds

F32, F64 = 0, 1
MASK_ROUNDED, MASK_FUNLSQ = 0, 1
PRE_NONE, PRE_RELU, PRE_SILU = 0, 1, 2
FP8_E4M3, FP8_E5M2 = 1, 2
FP8_MAX = {FP8_E4M3: 448.0, FP8_E5M2: 57344.0}  # largest finite value of each format
STATS_WIDTH, STATE_WIDTH = 5, 8
MSE_STATE_WIDTH = 10
HIST_STATE_HEAD = 12  # percentile observer state: [C, HIST_STATE_HEAD + 2 * n_bins]

c_void_p, c_int, c_int64, c_float, c_double, c_size_t = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double, ctypes.c_size_t)


class Layout(ctypes.Structure):
    _fields_ = [("outer", c_int64), ("channels", c_int64), ("inner", c_int64)]


class QParams(ctypes.Structure):
    _fields_ = [("scale", c_void_p), ("zero_point", c_void_p), ("scale_dtype", ctypes.c_int32),
                ("zp_dtype", ctypes.c_int32), ("scale_host", c_float), ("zp_host", c_float),
                ("zp_learned", ctypes.c_int32), ("qmin", ctypes.c_int32), ("qmax", ctypes.c_int32),
                ("pre_op", ctypes.c_int32)]


class MtEntry(ctypes.Structure):
    """vsiq_mt_entry (include/vsiq.h): one weight tensor of a multi-tensor launch."""
    _fields_ = [("x", c_void_p), ("rows", c_int64), ("inner", c_int64), ("out_offset", c_int64), ("qp_offset", c_int64),
                ("qp_channels", c_int64), ("qp", QParams), ("grad_scale", c_double), ("grad_scale_dev", c_void_p),
                ("learn", ctypes.c_int32), ("first_tile", ctypes.c_uint32), ("n_tiles", ctypes.c_uint32),
                ("chunks", ctypes.c_uint32), ("tile", ctypes.c_int32), ("tlo", c_float), ("thi", c_float)]


MT_PACK = 120  # upstream-gradient pointers per backward launch (multi_tensor.cu kMtPack)


class VsiqError(RuntimeError):
    pass


def build(force: bool = False) -> str:
    """Compile libvsiq.so in-tree with nvcc for sm_100a (works without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))
            if f.endswith((".cu", ".cuh"))] + [os.path.join(os.path.dirname(_HERE), "include", "vsiq.h")]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < newest:
        subprocess.run(["bash", os.path.join(_HERE, "csrc", "build.sh"), LIB_PATH], check=True)
    return LIB_PATH


_SIGNATURES = {
    "vsiq_version": (c_int, []),
    "vsiq_error_string": (ctypes.c_char_p, [c_int]),
    "vsiq_device_info": (c_int, [ctypes.POINTER(c_int)] * 3),
    "vsiq_workspace_reset": (c_int, [c_void_p, c_size_t, c_void_p]),
    "vsiq_fake_quant_fwd": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.POINTER(Layout), ctypes.POINTER(QParams), c_void_p]),
    "vsiq_quantize_codes": (c_int, [c_void_p, c_void_p, c_void_p, c_int, ctypes.POINTER(Layout), ctypes.POINTER(QParams), c_void_p]),
    "vsiq_fake_quant_bwd_ste": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.POINTER(Layout), ctypes.POINTER(QParams), c_void_p]),
    "vsiq_fake_quant_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.POINTER(Layout), ctypes.POINTER(QParams), c_void_p]),
    "vsiq_lsq_bwd_workspace_bytes": (c_size_t, [ctypes.POINTER(Layout)]),
    "vsiq_lsq_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, ctypes.POINTER(Layout),
                             ctypes.POINTER(QParams), c_double, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "vsiq_fp8_fake_quant_fwd": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.POINTER(Layout), ctypes.POINTER(QParams), c_int,
                                        c_void_p]),
    "vsiq_fp8_fake_quant_bwd_ste": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.POINTER(Layout), ctypes.POINTER(QParams),
                                            c_int, c_void_p]),
    "vsiq_fp8_lsq_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, ctypes.POINTER(Layout),
                                 ctypes.POINTER(QParams), c_int, c_double, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "vsiq_ci_fp8_fake_quant_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, ctypes.POINTER(QParams), c_int64,
                                           c_int, c_void_p, c_size_t, c_void_p]),
    "vsiq_ci_fp8_lsq_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                    c_int64, c_int64, ctypes.POINTER(QParams), c_int64, c_int, c_double, c_void_p, c_int64,
                                    c_void_p, c_size_t, c_void_p]),
    "vsiq_fp8_scale_from_range": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "vsiq_observe_workspace_bytes": (c_size_t, [ctypes.POINTER(Layout)]),
    "vsiq_observe": (c_int, [c_void_p, ctypes.POINTER(Layout), c_void_p, c_void_p, c_int, c_int, c_double, c_void_p,
                             c_size_t, c_void_p]),
    "vsiq_qparams_from_minmax": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_double, c_void_p]),
    "vsiq_lsq_init_scale": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p]),
    "vsiq_bn_fold_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "vsiq_bn_fold": (c_int, [c_void_p] * 6 + [c_float, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                             ctypes.POINTER(QParams), c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vsiq_bn_moments_finalize": (c_int, [c_void_p, c_double, c_int64] + [c_void_p] * 5 + [c_void_p]),
    "vsiq_bn_reestimate_finish": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p]),
    "vsiq_host_pipeline_create": (c_int, [ctypes.POINTER(c_void_p), c_int64, c_int]),
    "vsiq_host_pipeline_destroy": (c_int, [c_void_p]),
    "vsiq_host_pipeline_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float,
                                           c_int, c_int]),
    "vsiq_host_pipeline_last_launches": (c_int64, [c_void_p]),
    "vsiq_host_pipeline_last_enqueue_ns": (c_int64, [c_void_p]),
    "vsiq_ci_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "vsiq_ci_fake_quant_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, ctypes.POINTER(QParams), c_int64,
                                       c_void_p, c_size_t, c_void_p]),
    "vsiq_ci_fake_quant_fwd2": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, ctypes.POINTER(QParams),
                                        c_int64, ctypes.POINTER(QParams), c_int64, c_void_p, c_size_t, c_void_p]),
    "vsiq_ci_lsq_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                c_int64, c_int64, ctypes.POINTER(QParams), c_int64, c_double, c_void_p, c_int64, c_void_p,
                                c_size_t, c_void_p]),
    "vsiq_ci_bn_normalize": (c_int, [c_void_p] * 5 + [c_float, c_void_p, c_int64, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "vsiq_ci_observe_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "vsiq_ci_observe": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_size_t,
                                c_void_p]),
    "vsiq_ci_epilogue_observe": (c_int, [c_void_p] * 6 + [c_float, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                         c_int, c_int, c_double, c_void_p, c_size_t, c_void_p]),
    "vsiq_mse_search_workspace_bytes": (c_size_t, [ctypes.POINTER(Layout), c_int]),
    "vsiq_mse_search": (c_int, [c_void_p, ctypes.POINTER(Layout), c_void_p, c_void_p, c_int, c_int, c_double, c_int, c_void_p,
                                c_void_p, c_void_p, c_size_t, c_void_p]),
    "vsiq_hist_observe_workspace_bytes": (c_size_t, [ctypes.POINTER(Layout), c_int]),
    "vsiq_hist_observe": (c_int, [c_void_p, ctypes.POINTER(Layout), c_void_p, c_void_p, c_int, c_double, c_int, c_int,
                                  c_double, c_void_p, c_size_t, c_void_p]),
    "vsiq_hist_clip": (c_int, [c_void_p, c_int64, c_int, c_double, c_int, c_int, c_double, c_void_p]),
    "vsiq_hist_entropy_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "vsiq_hist_entropy_clip": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_double, c_void_p, c_void_p,
                                       c_size_t, c_void_p]),
    "vsiq_peer_buffer_bytes": (c_size_t, []),
    "vsiq_peer_max_world": (c_int, []),
    "vsiq_peer_max_channels": (c_int, []),
    "vsiq_peer_alloc": (c_int, [ctypes.POINTER(c_void_p), ctypes.c_char_p]),
    "vsiq_peer_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_void_p)]),
    "vsiq_peer_close": (c_int, [c_void_p]),
    "vsiq_peer_free": (c_int, [c_void_p]),
    "vsiq_peer_status": (c_int, [c_void_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "vsiq_bn_moments_exchange": (c_int, [c_void_p, c_double, c_double, c_int64, ctypes.POINTER(c_void_p), c_int, c_int,
                                         c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vsiq_selftest_division": (c_int, [c_float, c_int, c_void_p, c_void_p]),
    "vsiq_mt_plan": (c_int, [ctypes.POINTER(MtEntry), c_int, ctypes.POINTER(ctypes.c_uint32)]),
    "vsiq_mt_fake_quant_fwd": (c_int, [ctypes.POINTER(MtEntry), c_void_p, c_int, c_void_p, c_void_p]),
    "vsiq_mt_workspace_bytes": (c_size_t, [ctypes.c_uint32]),
    "vsiq_mt_lsq_bwd": (c_int, [ctypes.POINTER(MtEntry), c_void_p, c_int, ctypes.POINTER(c_void_p), c_void_p, c_void_p,
                                c_void_p, c_void_p, c_size_t, c_void_p]),
}

EXPORTED = tuple(_SIGNATURES)


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or vsiquantization_b200/csrc/build.sh). "
            "vsiquantization_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = stale library; fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.vsiq_version() // 100 != 1:
        raise ImportError(f"libvsiq.so version {lib.vsiq_version()} does not match this package")
    return lib


lib = _load()

# every kernel launch made through this binding is counted (bench.py reports it as gpu_launches)
launch_count = 0


# hook run before a library error is raised (ops.py clears the workspace headers: a failed launch must not leave a ticket
# or tile counter behind for the next one)
on_error = None


def check(code: int, what: str = "") -> None:
    if code != 0:
        if on_error is not None:
            try:
                on_error()
            except Exception:
                pass
        msg = lib.vsiq_error_string(code)
        raise VsiqError(f"{what or 'libvsiq'} failed: {msg.decode() if msg else code} (code {code})")
