"""Cost and quality of the MSE observer's clipping-range search (csrc/mse_search.cu, observers/mse.py).

    python tools/mse_bench.py [--reps 5] [--calib-batches 4] [--skip-quality] > profiles/<name>.log

Sections (one JSON line each):
  card        GPU name, SM count, max SM clock and power limit (every number below was measured on it);
  build       registers / spills of the search kernels (nvcc -Xptxas -v on csrc/mse_search.cu, into a temp directory);
  sass        instructions of the hot loop (fast path, 8 elements x 1 candidate per iteration) from cuobjdump -sass of the
              library, and the issue-rate bound that follows: SMs x clock x 128 thread-instructions / (instructions per
              candidate-evaluation).  The kernel is compute-bound (4 bytes read per element, about K x 17 instructions), so this
              bound, not HBM, is the roofline;
  weights     one observe() per YOLOv8s fused-layer weight (57 tensors, W4 per channel asymmetric, K = 100): time per call
              (CUDA events, median of --reps), total, candidate-evaluations/s;
  activations the five NHWC (channels_last) activation shapes of profiles/r02_ci_bench.log at batch 64, per tensor and per
              channel (ch_axis 1, searched in place), W4, K = 100;
  calibration benchmarks/calibration.py on YOLOv8m (b64@640, --calib-batches batches): MinMax weight observers, then MSE;
  quality     per-layer relative error ||fq(W) - W||^2 / ||W||^2 of the seeded YOLOv8s weights, W2 / W4 / W8 per channel
              asymmetric, min/max (K = 1) against MSE (K = 100), from the CPU oracle (deterministic).
Writes nothing into the tree (nvcc output goes to a temporary directory)."""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = [(64, 32, 320, 320), (64, 64, 160, 160), (64, 128, 80, 80), (64, 256, 40, 40), (64, 512, 20, 20)]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUOBJDUMP = os.path.join(os.path.dirname(NVCC), "cuobjdump")


def emit(section, **kw):
    print(json.dumps({"section": section, **kw}), flush=True)


def card():
    p = torch.cuda.get_device_properties(0)
    info = {"name": p.name, "sms": p.multi_processor_count}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, check=True).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(out[0]), float(out[1])
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi_error"] = str(e)
    return info


def build_stats():
    src = os.path.join(ROOT, "vsiquantization_b200", "csrc", "mse_search.cu")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                            "-c", src, "-o", os.path.join(d, "m.o")], capture_output=True, text=True)
    out, kern = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?(\S+?)'?$", line.strip())
        if m:
            name = m.group(1)
            kern = ("search<1>" if "kernelILi1E" in name else "search<4>" if "kernelILi4E" in name
                    else "finalize" if "finalize" in name else None)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and kern:
            out.setdefault(kern, {})["spill_stores"], out[kern]["spill_loads"] = int(m.group(1)), int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m and kern:
            out.setdefault(kern, {})["registers"] = int(m.group(1))
    return out


def sass_loop(lib_path):
    """Instructions per candidate-evaluation of the fast path of search<1>: the longest branch-free run of the kernel's
    SASS that widens results to fp64 (F2F.F64.F32, one per element and candidate) -- the unrolled 8-element vector of
    the candidate loop -- divided by its number of F2F.F64.F32.  Loop control (a few instructions per 8 evaluations) is
    left out, so the bound derived from it is slightly optimistic."""
    txt = subprocess.run([CUOBJDUMP, "-sass", lib_path], capture_output=True, text=True, check=True).stdout
    start = txt.find("Function : _ZN4vsiq17mse_search_kernelILi1E")
    body = txt[start:txt.find("Function :", start + 10)]
    ops_ = [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s+(.*?);", body)]
    runs, cur = [], []
    for o in ops_:
        if re.search(r"\b(BRA|CALL|EXIT|RET|BSSY|BSYNC|WARPSYNC|BAR)\b", o):
            runs.append(cur)
            cur = []
        else:
            cur.append(o)
    runs.append(cur)
    best = max(runs, key=lambda r: sum("F2F.F64.F32" in o for o in r))
    n_cvt = sum("F2F.F64.F32" in o for o in best)
    if n_cvt == 0:
        return {"error": "fast block not found"}
    kinds = {}
    for o in best:
        op = re.sub(r"^@!?U?P\w+\s+", "", o).split()[0].split(".")[0]
        kinds[op] = kinds.get(op, 0) + 1
    return {"block_instructions": len(best), "evaluations_per_block": n_cvt,
            "instructions_per_evaluation": len(best) / n_cvt, "opcode_mix": dict(sorted(kinds.items()))}


def time_call(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def yolo_s_weights(dev):
    from vsiquantization_b200.modules.fuse import fuse_modules_unified
    from vsiquantization_b200.modules.fuse_config import FuseConfig, create_fuse_config_manager
    from vsiquantization_b200.nets import yolov8
    torch.manual_seed(0)
    model = yolov8.yolo_v8_s(num_classes=80)
    g = torch.Generator().manual_seed(1)
    for mod in model.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    model = fuse_modules_unified(model.to(dev), [["conv", "bn", "relu"]],
                                 config_manager=create_fuse_config_manager(FuseConfig()))
    out = []
    with torch.no_grad():
        for n, m in model.named_modules():
            if hasattr(m, "weight_quantizer"):
                out.append((n, m.get_weight_bias()[0].detach().contiguous()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calib-batches", type=int, default=4)
    ap.add_argument("--skip-quality", action="store_true")
    args = ap.parse_args()
    from vsiquantization_b200 import _lib, ops
    dev = torch.device("cuda")
    info = card()
    emit("card", **info)
    emit("build", kernels=build_stats())
    sass = sass_loop(_lib.LIB_PATH)
    clock_hz = info.get("max_sm_clock_mhz", 0) * 1e6
    if "instructions_per_evaluation" in sass and clock_hz:
        sass["issue_bound_evals_per_s"] = info["sms"] * clock_hz * 128 / sass["instructions_per_evaluation"]
    emit("sass", **sass)
    bound = sass.get("issue_bound_evals_per_s")
    K = 100

    ws = yolo_s_weights(dev)
    per, total_ms, evals = [], 0.0, 0
    for n, w in ws:
        st = ops.new_mse_state(w.shape[0], dev)
        ms = time_call(lambda: ops.mse_search(w, 0, st, 4, False, 1e-8, K), args.reps)
        per.append({"layer": n, "shape": list(w.shape), "ms": round(ms, 4)})
        total_ms += ms
        evals += w.numel() * K
    emit("weights", model="yolov8s", tensors=len(ws), elements=sum(w.numel() for _, w in ws), bits=4, symmetric=False,
         K=K, total_ms=round(total_ms, 3), evals_per_s=evals / (total_ms * 1e-3),
         share_of_issue_bound=(evals / (total_ms * 1e-3) / bound) if bound else None, per_call=per)

    for shape in SHAPES:
        x = torch.randn(shape, device=dev).contiguous(memory_format=torch.channels_last)
        for ch_axis in (None, 1):
            C = 1 if ch_axis is None else shape[1]
            st = ops.new_mse_state(C, dev)
            ops.slow_path_counters(reset=True)
            ms = time_call(lambda: ops.mse_search(x, ch_axis, st, 4, False, 1e-8, K), args.reps)
            obs_ms = time_call(lambda: ops.observe(x, ch_axis, None, 4, False, 1e-8), args.reps)
            ev = x.numel() * K / (ms * 1e-3)
            emit("activations", shape=list(shape), layout="channels_last", ch_axis=ch_axis, K=K, ms=round(ms, 3),
                 of_which_minmax_pass_ms=round(obs_ms, 3), evals_per_s=ev,
                 share_of_issue_bound=(ev / bound) if bound else None,
                 layout_conversion_copies=ops.slow_path_counters()["layout_conversion_copies"])
        del x
        torch.cuda.empty_cache()

    from benchmarks import calibration
    for obs in ("MinMaxObserver", "MSEObserver"):
        res = calibration.run(calibration.parse(["--model", "m", "--batch", "64", "--imgsz", "640", "--batches",
                                                 str(args.calib_batches), "--channels-last", "--observer", obs]))
        emit("calibration", **{k: res[k] for k in ("model", "weight_observer", "batch", "imgsz", "global_batches",
                                                   "calibration_s", "calibration_images_per_s", "weight_scales_sha256")})

    if not args.skip_quality:
        import mse_oracle
        t0 = time.perf_counter()
        rows = []
        for n, w in ws:
            wn = w.cpu().numpy()
            row = {"layer": n, "shape": list(w.shape)}
            for bits in (2, 4, 8):
                row[f"w{bits}_minmax"] = mse_oracle.relative_error(wn, bits, False, 1)
                row[f"w{bits}_mse"] = mse_oracle.relative_error(wn, bits, False, K)
            rows.append(row)
        tot = {}
        for bits in (2, 4, 8):
            for kind in ("minmax", "mse"):
                num = sum(r[f"w{bits}_{kind}"] * float((w.double() ** 2).sum()) for r, (_, w) in zip(rows, ws))
                tot[f"w{bits}_{kind}"] = num / sum(float((w.double() ** 2).sum()) for _, w in ws)
        emit("quality", source="mse_oracle (CPU, deterministic)", granularity="per channel (ch_axis 0), asymmetric",
             K=K, all_layers=tot, per_layer=rows, seconds=round(time.perf_counter() - t0, 1))


if __name__ == "__main__":
    main()
