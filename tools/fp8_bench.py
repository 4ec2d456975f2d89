"""FP8 fake-quant kernels against the integer kernels and torch's copy_ on the same tensors, in one run.

For each tensor: copy_ (8 B/element), then forward (8 B), STE backward (12 B) and learned (LSQ) backward (12 B) for the
integer W8A8 grid [-128, 127], E4M3 and E5M2, per tensor and per channel, alternated launch by launch with a 512 MB
buffer rewritten between timed launches so that no input is read from L2.  CUDA events around each launch, median of
``--iters``.  Sizes: flat 2^24 .. 2^30 elements (per channel: [C = 256, n / 256] rows), and the five NHWC activation maps
of the YOLOv8s step at batch 64 (DESIGN.md §4), channels_last, per tensor on the rows kernels (per-tensor qparams walk
NHWC memory in place).  Prints the card (name, SM count, power limit) first;
with ``--log`` the same lines go to that file.

    python tools/fp8_bench.py --log profiles/r06_fp8_bench.log
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vsiquantization_b200 import _lib, ops  # noqa: E402

YOLO_MAPS = [(64, 32, 320, 320), (64, 64, 160, 160), (64, 128, 80, 80), (64, 256, 40, 40), (64, 512, 20, 20)]
GRIDS = (("int8", 0), ("e4m3", _lib.FP8_E4M3), ("e5m2", _lib.FP8_E5M2))


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


def spec_for(fmt, ch_axis):
    return ops.QSpec(0, 0, ch_axis=ch_axis, fp8_format=fmt) if fmt else ops.QSpec(-128, 127, ch_axis=ch_axis)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=15)
    ap.add_argument("--max-log2", type=int, default=30)
    ap.add_argument("--log", default=None)
    args = ap.parse_args()
    logf = open(args.log, "w") if args.log else None

    def emit(**kw):
        line = json.dumps(kw)
        print(line, flush=True)
        if logf:
            logf.write(line + "\n")
            logf.flush()

    emit(section="card", **card())
    flush = torch.empty(1 << 27, device="cuda")  # 512 MB, 4x the L2

    def timed(fn):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        return a, b

    def run(name, shape, ch_axis, memfmt=None):
        torch.manual_seed(0)
        x = torch.randn(shape, device="cuda") * 3
        g = torch.randn(shape, device="cuda")
        if memfmt is not None:
            x, g = x.contiguous(memory_format=memfmt), g.contiguous(memory_format=memfmt)
        n = x.numel()
        C = 1 if ch_axis is None else shape[ch_axis]
        s = (torch.rand(C, device="cuda") * 0.01 + 0.01) if C > 1 else torch.tensor(0.02, device="cuda")
        y, dx, cp = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
        ds = torch.empty(C, device="cuda", dtype=torch.float32)
        ops_ = {"copy": (8, lambda: cp.copy_(x))}
        for gname, fmt in GRIDS:
            sp = spec_for(fmt, ch_axis if C > 1 else None)
            ops_[f"{gname}_fwd"] = (8, lambda sp=sp: ops.fake_quant_forward(x, s, 0, sp, out=y))
            ops_[f"{gname}_ste"] = (12, lambda sp=sp: ops.fake_quant_backward_ste(x, g, s, 0, sp, out=dx))
            ops_[f"{gname}_lsq"] = (12, lambda sp=sp: ops.lsq_backward(x, g, s, 0, sp, 1e-4, ds_out=ds, dx_out=dx))
        for _, fn in ops_.values():  # warm-up: module load, workspace allocation
            fn()
        torch.cuda.synchronize()
        evs = {k: [] for k in ops_}
        for _ in range(args.iters):  # alternate every op launch by launch
            for k, (_, fn) in ops_.items():
                evs[k].append(timed(fn))
        torch.cuda.synchronize()
        res = {}
        for k, (bpe, _) in ops_.items():
            ts = sorted(a.elapsed_time(b) for a, b in evs[k])
            us = ts[len(ts) // 2] * 1e3
            res[k] = {"us": round(us, 2), "gbs": round(bpe * n / (us * 1e-6) / 1e9, 1)}
        emit(section="kernels", tensor=name, shape=list(shape), layout="channels_last" if memfmt else "contiguous",
             qparams="per_channel" if C > 1 else "per_tensor", elements=n, **res)
        del x, g, y, dx, cp

    for log2n in range(24, args.max_log2 + 1, 2):
        n = 1 << log2n
        run(f"2^{log2n}", (n,), None)
        run(f"2^{log2n}", (256, n // 256), 0)
    for shp in YOLO_MAPS:
        run("yolov8s_b64", shp, None, torch.channels_last)
    if logf:
        logf.close()


if __name__ == "__main__":
    main()
