"""Cost and quality of the histogram observers: percentile (csrc/hist_observer.cu, observers/percentile.py) and entropy
(csrc/hist_entropy.cu, observers/entropy.py).

    python tools/percentile_bench.py [--reps 7] [--calib-batches 4] [--skip-calibration] [--skip-quality] > profiles/<name>.log

Sections (one JSON line each):
  card        GPU name, SM count, max SM clock and power limit (every number below was measured on it);
  build       registers / spills of the kernels (nvcc -Xptxas -v on csrc/hist_observer.cu and csrc/hist_entropy.cu, into a
              temporary directory);
  activations the five NHWC (channels_last) activation shapes at batch 64 of profiles/r03_mse_bench.log, per tensor and
              per channel (ch_axis 1, read in place), Gaussian and ReLU-like (half exact zeros) input, B = 2048, A4:
              the histogram pass by itself (vsiq_hist_observe: histogram kernel + finalize), the whole observe call
              (min/max pass + histogram pass), the min/max pass alone and torch's copy_ of the same tensor -- CUDA events,
              median of --reps, the 126 MB L2 overwritten before every timed call;
  entropy     the same maps, per tensor and per channel, Gaussian and ReLU-like input, B = 2048, start_bin 128, A4 and A8
              (asymmetric): the entropy search by itself (vsiq_hist_entropy_clip over the counts of one call), the whole
              EntropyObserver.observe call, and ops.hist_observe at percentile 100 (the min/max pass plus the histogram
              pass: the part of that call before the search; reported as histogram_pass_ms) -- timed like the
              activations section;
  calibration benchmarks/calibration.py on YOLOv8m (b64@640, channels_last, --calib-batches batches): MinMax activation
              observers, then Percentile, then Entropy;
  quality     per layer of the seeded YOLOv8s on SYNTHETIC batches (uniform random images, not a dataset): the relative A4
              activation error ||fq(a) - a||^2 / ||a||^2 on held-out batches, per-tensor asymmetric qparams calibrated on
              other batches by min/max (percentile 100), by percentiles 99.99 and 99.9 and by the entropy search of the
              same histograms.
Writes nothing into the tree (nvcc output goes to a temporary directory)."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = [(64, 32, 320, 320), (64, 64, 160, 160), (64, 128, 80, 80), (64, 256, 40, 40), (64, 512, 20, 20)]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
B = 2048


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
    stderr = ""
    with tempfile.TemporaryDirectory() as d:
        for f in ("hist_observer.cu", "hist_entropy.cu"):
            src = os.path.join(ROOT, "vsiquantization_b200", "csrc", f)
            stderr += subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas",
                                      "-v", "-c", src, "-o", os.path.join(d, "h.o")], capture_output=True, text=True).stderr
    out, kern = {}, None
    for line in stderr.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?(\S+?)'?$", line.strip())
        if m:
            name = m.group(1)
            kern = ("hist<1>" if "hist_kernelILi1E" in name else "hist<4>" if "hist_kernelILi4E" in name
                    else "entropy_score" if "entropy_score" in name else "entropy_finalize" if "entropy_finalize" in name
                    else "finalize" if "finalize" in name else None)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and kern:
            out.setdefault(kern, {})["spill_stores"], out[kern]["spill_loads"] = int(m.group(1)), int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m and kern:
            out.setdefault(kern, {})["registers"] = int(m.group(1))
    return out


_flush_buf = None


def flush_l2():
    global _flush_buf
    if _flush_buf is None:
        _flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    _flush_buf.fill_(1)


def time_call(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush_l2()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def activations(reps):
    from vsiquantization_b200 import _lib, ops
    dev = torch.device("cuda")
    for shape in SHAPES:
        x = torch.randn(shape, device=dev).contiguous(memory_format=torch.channels_last)
        for kind in ("gaussian", "relu"):
            if kind == "relu":
                x.clamp_(min=0.0)
            y = torch.empty_like(x)
            for ch_axis in (None, 1):
                C = 1 if ch_axis is None else shape[1]
                st = ops.new_percentile_state(C, B, dev)
                ops.slow_path_counters(reset=True)
                whole = time_call(lambda: ops.hist_observe(x, ch_axis, st, B, 99.99, 4, False, 1e-8), reps)
                minmax = time_call(lambda: ops.observe(x, ch_axis, None, 4, False, 1e-8), reps)
                stats = ops.observe(x, ch_axis, None, 4, False, 1e-8)
                N, _, H, W = shape
                lay = _lib.Layout(N * H * W, C, 1) if ch_axis == 1 else _lib.Layout(1, 1, x.numel())
                nbytes = _lib.lib.vsiq_hist_observe_workspace_bytes(ctypes.byref(lay), B)
                ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
                sp = torch.cuda.current_stream().cuda_stream

                def hist_only():
                    _lib.check(_lib.lib.vsiq_hist_observe(x.data_ptr(), ctypes.byref(lay), stats.data_ptr(),
                                                          st.data_ptr(), B, 99.99, 4, 0, 1e-8, ws.data_ptr(), nbytes,
                                                          sp), "vsiq_hist_observe")
                hist = time_call(hist_only, reps)
                copy = time_call(lambda: y.copy_(x), reps)
                emit("activations", shape=list(shape), layout="channels_last", ch_axis=ch_axis, input=kind, n_bins=B,
                     elements=x.numel(), histogram_pass_ms=round(hist, 4), whole_call_ms=round(whole, 4),
                     minmax_pass_ms=round(minmax, 4), copy_ms=round(copy, 4),
                     histogram_over_minmax=round(hist / minmax, 3),
                     histogram_pass_GBps=round(x.numel() * 4 / (hist * 1e-3) / 1e9, 1),
                     layout_conversion_copies=ops.slow_path_counters()["layout_conversion_copies"])
            del y
        del x
        torch.cuda.empty_cache()


def entropy(reps):
    from vsiquantization_b200 import ops
    from vsiquantization_b200.observers.entropy import EntropyObserver
    dev = torch.device("cuda")
    for shape in SHAPES:
        x = torch.randn(shape, device=dev).contiguous(memory_format=torch.channels_last)
        for kind in ("gaussian", "relu"):
            if kind == "relu":
                x.clamp_(min=0.0)
            for ch_axis in (None, 1):
                C = 1 if ch_axis is None else shape[1]
                st = ops.new_percentile_state(C, B, dev)
                hist = time_call(lambda: ops.hist_observe(x, ch_axis, st, B, 100.0, 4, False, 1e-8), reps)
                for bits in (4, 8):
                    st.copy_(ops.new_percentile_state(C, B, dev))
                    ops.hist_observe(x, ch_axis, st, B, 100.0, bits, False, 1e-8)
                    search = time_call(lambda: ops.hist_entropy_clip(st, B, 128, bits, False, 1e-8), reps)
                    obs = EntropyObserver(False, bits, ch_axis=ch_axis, n_bins=B)
                    whole = time_call(lambda: obs.observe(x), reps)
                    nq = 2 ** bits if kind == "relu" else 2 ** (bits - 1)
                    emit("entropy", shape=list(shape), layout="channels_last", ch_axis=ch_axis, input=kind, n_bins=B,
                         start_bin=128, bits=bits, nq=nq, elements=x.numel(), search_ms=round(search, 4),
                         whole_call_ms=round(whole, 4), histogram_pass_ms=round(hist, 4),
                         search_over_histogram=round(search / hist, 3),
                         log_evaluations_at_most=C * (B + 1 - 128) * nq)
        del x
        torch.cuda.empty_cache()


def calibration(batches):
    from benchmarks import calibration as cal
    for obs in ("MinMaxObserver", "PercentileObserver", "EntropyObserver"):
        res = cal.run(cal.parse(["--model", "m", "--batch", "64", "--imgsz", "640", "--batches", str(batches),
                                 "--channels-last", "--act-observer", obs]))
        emit("calibration", activation_observer=obs, **{k: res[k] for k in (
            "model", "batch", "imgsz", "global_batches", "calibration_s", "calibration_images_per_s",
            "activation_scales_sha256")})


def quality(calib_batches=4, held_out=2, batch=8, imgsz=320):
    """Relative A4 error on held-out synthetic batches, per-tensor asymmetric qparams from the same histograms."""
    from vsiquantization_b200 import ops
    from vsiquantization_b200.modules.fuse import fuse_modules_unified
    from vsiquantization_b200.modules.fuse_config import FuseConfig, create_fuse_config_manager
    from vsiquantization_b200.nets import yolov8
    from vsiquantization_b200.utils.quantize_manager import calibrate_qat_model
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = yolov8.yolo_v8_s(num_classes=80)
    g = torch.Generator().manual_seed(1)
    for mod in model.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    cfg = FuseConfig(bits_a=4, a_symmetric=False, observer_a_name="PercentileObserver")
    model = fuse_modules_unified(model.to(dev), [["conv", "bn", "relu"]], config_manager=create_fuse_config_manager(cfg))
    model = model.to(memory_format=torch.channels_last)
    gen = torch.Generator(device=dev).manual_seed(7)
    imgs = [torch.rand(batch, 3, imgsz, imgsz, device=dev, generator=gen).contiguous(memory_format=torch.channels_last)
            for _ in range(calib_batches + held_out)]

    def run(m, loader, d):
        m.eval()
        with torch.no_grad():
            for x in loader:
                m(x)
    calibrate_qat_model(model, imgs[:calib_batches], run, dev)
    mgrs = [(n, m.activation_quantizer) for n, m in model.named_modules() if hasattr(m, "activation_quantizer")]
    percentiles = (100.0, 99.99, 99.9)
    methods = percentiles + ("entropy",)
    qp = {}
    for n, q in mgrs:
        for p in percentiles:
            q.observer.set_percentile(p)
            s, z = q.observer.get_scale_zero_point()
            qp[(n, p)] = (float(s), float(z))
        st = q.observer.state.clone()  # the same histogram, searched by the entropy rule (EntropyObserver's defaults)
        ops.hist_entropy_clip(st, q.observer.n_bins, 128, 4, False, q.observer.eps)
        qp[(n, "entropy")] = (float(st[0, 2]), float(st[0, 3]))
    err = {(n, p): [0.0, 0.0] for n, _ in mgrs for p in methods}
    spec = ops.QSpec(0, 15)
    for n, q in mgrs:
        def measure(a, n=n):
            for p in methods:
                s, z = qp[(n, p)]
                y = ops.fake_quant_forward(a, s, z, spec)
                err[(n, p)][0] += float(((y.double() - a.double()) ** 2).sum())
                err[(n, p)][1] += float((a.double() ** 2).sum())
        q.observer.observe = measure  # the held-out passes only measure: the observers keep their calibration
    run(model, imgs[calib_batches:], dev)
    key = lambda p: p if isinstance(p, str) else f"p{p:g}"  # noqa: E731
    rows = []
    for n, _ in mgrs:
        row = {"layer": n}
        for p in methods:
            num, den = err[(n, p)]
            row[key(p)] = num / den if den else None
        rows.append(row)
    tot = {key(p): sum(err[(n, p)][0] for n, _ in mgrs) / sum(err[(n, p)][1] for n, _ in mgrs) for p in methods}
    better = {key(p): sum(1 for r in rows if r[key(p)] is not None and r[key(p)] < r["p100"]) for p in methods[1:]}
    emit("quality", data="SYNTHETIC: uniform random images, seeded YOLOv8s with seeded BN statistics",
         model="yolov8s", granularity="per tensor, asymmetric, A4", entropy_start_bin=128,
         calibration_batches=calib_batches,
         held_out_batches=held_out, batch=batch, imgsz=imgsz, p100_is="min/max", all_layers_relative_error=tot,
         layers_better_than_minmax=better, layers=len(rows), per_layer=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calib-batches", type=int, default=4)
    ap.add_argument("--skip-calibration", action="store_true")
    ap.add_argument("--skip-quality", action="store_true")
    ap.add_argument("--skip-activations", action="store_true", help="skip the percentile observer's activation rows")
    args = ap.parse_args()
    emit("card", **card())
    emit("build", kernels=build_stats())
    if not args.skip_activations:
        activations(args.reps)
    entropy(args.reps)
    if not args.skip_calibration:
        calibration(args.calib_batches)
    if not args.skip_quality:
        quality()


if __name__ == "__main__":
    main()
