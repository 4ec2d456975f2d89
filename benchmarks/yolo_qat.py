"""YOLOv8 QAT step benchmark (BASELINE.json configs 0/2/3/4): images/s of fwd + bwd + optimizer step through the fused
QAT layers, synthetic data, one process per GPU.

    python -m benchmarks.yolo_qat --model s --batch 64 --imgsz 640 [--w-bits 4 --a-bits 8 --asym --per-channel]
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 -m benchmarks.yolo_qat --model l --batch 16

Every step copies its uint8 image batch from pinned host memory, runs forward / backward / (flat qparam-gradient
all-reduce) / SGD step and reads the loss back to the host: the number is end to end.  Loss = sum over the three
heads of mean(out^2) (the reference's ComputeLoss needs box targets; the detection loss is out of scope, SURVEY 2).
`--quant-impl eager` swaps every quantizer plugin object for the torch-eager restatement of the reference's op sequence
on the SAME GPU after calibration -- the GPU-vs-GPU yardstick of SURVEY 8(d) -- everything else (fused layers, manager,
calibrated parameters, cuDNN convs) unchanged.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def swap_in_eager_quantizers(model) -> int:
    """The GPU-vs-GPU yardstick: same fused layers, same calibrated / initialised parameters, same cuDNN convolutions --
    only the quantizer plugin objects are replaced by the reference's eager composition (oracle/torch_port.EagerQuantizer:
    quantizers/uniform.py:34-56 per tensor, the per-channel form of quantizers/lsq_module.py:147-173 otherwise): six ATen
    kernels forward and ~14 backward per quantiser instead of one each.  Returns the number of quantisers swapped."""
    from oracle.torch_port import EagerQuantizer
    n = 0
    for mod in model.modules():
        for attr in ("weight_quantizer", "activation_quantizer"):
            mgr = getattr(mod, attr, None)
            if mgr is not None and hasattr(mgr, "quantizer"):
                mgr.quantizer = EagerQuantizer.like(mgr.quantizer)
                n += 1
    return n


def kernel_time_profile(step, n_steps: int):
    """Device time of this library's kernels inside the step (CUPTI activity records of `n_steps` extra steps, outside
    the timed region): the measured counterpart of the HBM floor.  `kernel_ms_per_step` is the UNION of the kernels'
    [start, end] intervals -- a combine kernel launched as a programmatic dependent is resident (waiting) while its
    streaming kernel still runs, so the plain sum of durations (`kernel_ms_sum_per_step`) counts that overlap twice."""
    try:
        from torch.autograd import DeviceType
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(n_steps):
                step(i)
            torch.cuda.synchronize()
        total, by, spans = 0.0, {}, []
        for e in prof.events():
            if e.device_type != DeviceType.CUDA:
                continue
            t0, t1 = float(e.time_range.start), float(e.time_range.end)
            total += t1 - t0
            if "vsiq::" in e.name:
                spans.append((t0, t1))
                name = e.name.split("vsiq::")[1].split("<")[0].split("(")[0]
                d = by.setdefault(name, [0.0, 0])
                d[0] += t1 - t0
                d[1] += 1
        spans.sort()
        union, cur0, cur1 = 0.0, None, None
        for t0, t1 in spans:
            if cur1 is None or t0 > cur1:
                if cur1 is not None:
                    union += cur1 - cur0
                cur0, cur1 = t0, t1
            else:
                cur1 = max(cur1, t1)
        if cur1 is not None:
            union += cur1 - cur0
        return {"kernel_ms_per_step": union / n_steps / 1e3,
                "kernel_ms_sum_per_step": sum(v[0] for v in by.values()) / n_steps / 1e3,
                "device_ms_per_step": total / n_steps / 1e3,
                "kernels": {k: {"ms_per_step": round(v[0] / n_steps / 1e3, 4), "launches_per_step": v[1] / n_steps}
                            for k, v in sorted(by.items(), key=lambda kv: -kv[1][0])}}
    except Exception as e:  # CUPTI unavailable (e.g. under ncu): report why, never fail the benchmark
        return {"kernel_ms_per_step": None, "profile_error": f"{type(e).__name__}: {str(e)[:120]}"}


def build_model(args, device):
    from vsiquantization_b200.modules.fuse import fuse_modules_unified
    from vsiquantization_b200.modules.fuse_config import FuseConfig, create_fuse_config_manager
    from vsiquantization_b200.nets import yolov8
    from vsiquantization_b200.utils.quantize_manager import activate_learning_qparam, activate_quantizer, calibrate_qat_model
    torch.manual_seed(0)
    model = getattr(yolov8, f"yolo_v8_{args.model}")(num_classes=20).to(device)
    qname = "LSQQuantizer" if args.lsq else "UniformQuantizer"
    oname = "LSQObserver" if args.lsq else "MinMaxObserver"
    if args.fp8:  # FP8 E4M3 weights and activations (8-bit, symmetric by definition)
        qname = "FP8Quantizer"
    cfg = FuseConfig(observer_w_name=oname, quantizer_w_name=qname, observer_a_name=oname, quantizer_a_name=qname,
                     w_symmetric=not args.asym, a_symmetric=not args.asym, is_fuse_bn=not args.keep_bn,
                     bits_w=args.w_bits, bits_a=args.a_bits,
                     w_ch_axis=0 if args.per_channel else None, a_ch_axis=1 if args.per_channel else None)
    layer_cfgs = {}
    if args.mixed:  # BASELINE configs[4]: backbone LSQ W4, head UniformQuantizer W8
        layer_cfgs = {r"^net\..*conv": FuseConfig(observer_w_name="LSQObserver", quantizer_w_name="LSQQuantizer",
                                                  observer_a_name="LSQObserver", quantizer_a_name="LSQQuantizer",
                                                  bits_w=4, bits_a=8),
                      r"^head\.": FuseConfig(bits_w=8, bits_a=8)}
    model = fuse_modules_unified(model, [["conv", "bn", "relu"]], config_manager=create_fuse_config_manager(cfg, layer_cfgs))
    n_fused = sum(1 for m in model.modules() if hasattr(m, "weight_quantizer"))
    g = torch.Generator().manual_seed(1)
    calib = [(torch.randint(0, 256, (args.calib_batch, 3, args.imgsz, args.imgsz), generator=g, dtype=torch.uint8), None)
             for _ in range(args.calib_batches)]

    def data_calib(m, loader, dev):
        m.eval()
        with torch.no_grad():
            for imgs, _ in loader:
                m(imgs.to(dev, non_blocking=True).float() / 255.0)

    t0 = time.perf_counter()
    calibrate_qat_model(model, calib, data_calib, device)
    torch.cuda.synchronize()
    calib_s = time.perf_counter() - t0
    if dist.is_initialized():
        from vsiquantization_b200.parallel import sync_observers
        sync_observers(model)
    activate_learning_qparam(model, use_init=True)
    activate_quantizer(model)
    model.to(device)
    return model, n_fused, calib_s


def run(args) -> dict:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    torch.backends.cudnn.benchmark = True
    from vsiquantization_b200 import _lib
    model, n_fused, calib_s = build_model(args, device)
    if args.quant_impl == "eager":
        swap_in_eager_quantizers(model)
    model.train()
    if args.channels_last:
        model.to(memory_format=torch.channels_last)
    bank = None
    if args.weight_bank and args.quant_impl == "native":
        from vsiquantization_b200.bank import WeightBank
        # under DDP every layer keeps its own backward node so the gradient all-reduce still overlaps the backward pass
        bank = WeightBank(model, backward="per_layer" if (world > 1 and not args.cuda_graph) else "bank").install()
    bucket = None
    net = model
    if world > 1 and not args.cuda_graph:
        from torch.nn.parallel import DistributedDataParallel as DDP
        if args.quant_impl == "native":
            from vsiquantization_b200.parallel import QParamGradBucket
            bucket = QParamGradBucket(model)
            bucket.ddp_ignore(model)
        net = DDP(model, device_ids=[local])
    opt = torch.optim.SGD(model.parameters(), lr=1e-4, momentum=0.9, nesterov=True)
    g = torch.Generator().manual_seed(100 + rank)
    host = [torch.randint(0, 256, (args.batch, 3, args.imgsz, args.imgsz), generator=g, dtype=torch.uint8).pin_memory()
            for _ in range(2)]

    cl = (lambda t: t.contiguous(memory_format=torch.channels_last)) if args.channels_last else (lambda t: t)

    # Input pipeline: like any prefetching loader, the uint8 batch of step i+1 crosses PCIe (pinned host -> device, on a
    # copy stream) while step i computes.  Every step still copies its own batch inside the timed region; the copy just
    # no longer sits on the critical path (8 ranks share the host's memory bandwidth: 78.6 MB per rank per step).
    class Prefetch:
        def __init__(self):
            self.stream = torch.cuda.Stream()
            self.dev = [torch.empty_like(host[0], device=device) for _ in range(2)]
            self.ready = [torch.cuda.Event() for _ in range(2)]   # copy into dev[k] done
            self.free = [torch.cuda.Event() for _ in range(2)]    # compute stream has consumed dev[k]
            for e in self.free:
                e.record()
            self.next_i = 0   # batches issued
            self.cur = 0      # batches consumed
            self.h2d = []     # (start, end) timing events of the copies issued inside the timed region
            self.timing = False
            self.issue()

        def issue(self):
            k = self.next_i % 2
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(self.free[k])
                if self.timing:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(self.stream)
                self.dev[k].copy_(host[k], non_blocking=True)
                if self.timing:
                    e1.record(self.stream)
                    self.h2d.append((e0, e1))
                self.ready[k].record(self.stream)
            self.next_i += 1

        def get(self):
            k = self.cur % 2
            self.cur += 1
            torch.cuda.current_stream().wait_event(self.ready[k])
            imgs = cl(self.dev[k].float() / 255.0)
            self.free[k].record()
            self.issue()  # start moving the next batch now
            return imgs

    pre = Prefetch() if not args.no_prefetch else None

    def batch_for(i):
        if pre is not None:
            return pre.get()
        return cl(host[i % 2].to(device, non_blocking=True).float() / 255.0)

    def step(i):
        imgs = batch_for(i)
        outs = net(imgs)
        loss = sum((o.float() ** 2).mean() for o in outs)
        if world > 1:
            loss = loss * world  # the reference undoes DDP's averaging the same way (yolov8_qat.py:235-236)
        loss.backward()
        if bucket is not None:
            bucket.all_reduce()
        opt.step()
        if bucket is not None:
            bucket.zero()
            for p in model.parameters():
                if p.grad is not None and p not in bucket_params:
                    p.grad = None
        else:
            opt.zero_grad(set_to_none=True)
        return float(loss.item())  # device -> host read of the step's result

    bucket_params = set(bucket.params) if bucket is not None else set()
    from vsiquantization_b200 import ops as _ops
    _ops.slow_path_counters(reset=True)  # from here on: warm-up / capture / timed steps only
    graphed = None
    if args.cuda_graph:
        # world > 1: no DDP wrapper -- the graphed step all-reduces one flat gradient buffer inside the captured graph
        from vsiquantization_b200.graph import GraphedQATStep
        graphed = GraphedQATStep(model, opt, lambda outs: sum((o.float() ** 2).mean() for o in outs),
                                 cl(host[0].to(device).float() / 255.0))

        def step(i):  # noqa: F811
            return float(graphed(batch_for(i)).item())
    # fake-quant traffic of one step (SURVEY.md 8: 20 algorithmic bytes per quantised element, forward + backward):
    # every weight tensor plus every tensor an activation quantiser sees, counted by hooks during one eager forward
    fq_elems = {"w": 0, "a": 0}
    wrapped = []

    def counting(mgr, kind):
        orig = mgr.quantize

        def quantize(x, *a, **kw):
            y = orig(x, *a, **kw)
            if mgr.is_quantize:
                fq_elems[kind] += y.numel()
            return y
        mgr.quantize = quantize
        wrapped.append(mgr)
    for mod in model.modules():
        if hasattr(mod, "weight_quantizer") and hasattr(mod, "activation_quantizer"):
            counting(mod.weight_quantizer, "w")
            counting(mod.activation_quantizer, "a")
    with torch.no_grad():
        bank_on = bank.enabled if bank is not None else False
        if bank is not None:
            bank.enabled = False
        model(cl(host[0].to(device).float() / 255.0))
        if bank is not None:
            bank.enabled = bank_on
    for mgr in wrapped:
        del mgr.quantize
    for i in range(max(args.warmup, 3)):
        step(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if pre is not None:
        pre.timing = True
    l0 = _lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss = 0.0
    ar_ms = []
    for i in range(args.steps):
        loss = step(i)  # reads the loss back: the device is idle here, the in-graph events of this step are final
        if graphed is not None and graphed.allreduce_ms() is not None:
            ar_ms.append(graphed.allreduce_ms())
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if pre is not None:
        pre.timing = False
    ms = e0.elapsed_time(e1)
    mine = ms
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    spread = None
    if world > 1:
        every = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(every, t)
        spread = [float(v.item()) / args.steps for v in every]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    launches = _lib.launch_count - l0
    h2d_ms = None
    if pre is not None and pre.h2d:
        v = sorted(a.elapsed_time(b) for a, b in pre.h2d)
        h2d_ms = v[len(v) // 2]
    # the gradient all-reduce timed on its own (same buffer size, idle GPU): what the collective costs when nothing
    # competes with it, against its duration inside the step (which includes waiting for the slowest rank)
    ar_alone = None
    if world > 1:
        nbytes = getattr(graphed, "allreduce_bytes", 0) or sum(p.numel() * p.element_size() for p in model.parameters())
        buf = torch.zeros(nbytes // 4, dtype=torch.float32, device=device)
        for _ in range(3):
            dist.all_reduce(buf)
        ts = []
        for _ in range(10):
            dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            dist.all_reduce(buf)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        ar_alone = {"ms": ts[len(ts) // 2], "bytes": int(nbytes)}
        del buf
    fq_prof = kernel_time_profile(step, args.profile_steps) if args.profile_steps > 0 else None
    res = {"model": f"yolov8{args.model}", "fused_layers": n_fused, "batch_per_gpu": args.batch, "imgsz": args.imgsz,
           "n_gpus": world, "steps": args.steps, "ms_per_step": ms / args.steps,
           "images_per_s": args.batch * world * args.steps / (ms * 1e-3), "quant_impl": args.quant_impl,
           "fp8": bool(args.fp8),
           "w_bits": args.w_bits, "a_bits": args.a_bits, "asymmetric": args.asym, "per_channel": args.per_channel,
           "lsq": args.lsq, "mixed": args.mixed, "cuda_graph": args.cuda_graph, "channels_last": args.channels_last,
           "weight_bank": bool(bank is not None and (bank.last_used or args.cuda_graph)), "prefetch": pre is not None,
           "loss": loss, "vsiq_launches_per_step": launches / args.steps,
           "calibration_s": calib_s, "calib_batches": args.calib_batches,
           "h2d_bytes_per_step": args.batch * 3 * args.imgsz * args.imgsz, "d2h_bytes_per_step": 4,
           "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30,
           "h2d_ms": h2d_ms, "allreduce_ms": (sorted(ar_ms)[len(ar_ms) // 2] if ar_ms else None),
           "allreduce_alone": ar_alone, "ms_per_step_by_rank": spread, "ms_per_step_this_rank": mine / args.steps,
           # copies / scalar instantiations the wrappers fell back to while the step was executed eagerly (warm-up, graph
           # capture, and -- without a graph -- the timed steps): all zero means every tensor took a fast path
           "slow_paths": _ops.slow_path_counters()}
    if graphed is not None and getattr(graphed, "_marks", None):
        res["step_timeline_ms"] = graphed.step_timeline_ms()
    peak = 6531.9
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    fq_bytes = 20.0 * (fq_elems["w"] + fq_elems["a"])
    res["fake_quant"] = {"weight_elements": fq_elems["w"], "activation_elements": fq_elems["a"],
                         "algorithmic_gb_per_step_per_gpu": fq_bytes / 1e9, "hbm_peak_gbs": peak,
                         "hbm_floor_ms_per_step": fq_bytes / peak / 1e6,
                         "floor_fraction_of_step": fq_bytes / peak / 1e6 / (ms / args.steps)}
    if fq_prof is not None:
        res["fake_quant"].update(fq_prof)
        if fq_prof.get("kernel_ms_per_step"):
            res["fake_quant"]["fraction_of_hbm_floor"] = res["fake_quant"]["hbm_floor_ms_per_step"] / fq_prof["kernel_ms_per_step"]
    return res


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="n", choices=list("ntsmlx"))
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--imgsz", type=int, default=320)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--w-bits", type=int, default=8)
    ap.add_argument("--a-bits", type=int, default=8)
    ap.add_argument("--asym", action="store_true")
    ap.add_argument("--per-channel", action="store_true")
    ap.add_argument("--lsq", action="store_true")
    ap.add_argument("--fp8", action="store_true", help="FP8 E4M3 weights and activations (FP8Quantizer) instead of integers")
    ap.add_argument("--mixed", action="store_true")
    ap.add_argument("--keep-bn", action="store_true")
    ap.add_argument("--calib-batches", type=int, default=2)
    ap.add_argument("--calib-batch", type=int, default=2)
    ap.add_argument("--quant-impl", default="native", choices=["native", "eager"])
    ap.add_argument("--channels-last", action="store_true", help="NHWC memory format (cuDNN's native layout on sm_100)")
    ap.add_argument("--cuda-graph", action="store_true", help="capture fwd+bwd+optimizer once, replay per step")
    ap.add_argument("--no-prefetch", action="store_true", help="copy each batch on the compute stream (no overlap)")
    ap.add_argument("--weight-bank", action="store_true", help="all weight quantisers in one multi-tensor launch each way")
    ap.add_argument("--profile-steps", type=int, default=0,
                    help="after the timed region, profile this many extra steps (CUPTI) and report the fake-quant kernel time")
    return ap.parse_args(argv)


def main():
    args = parse()
    res = run(args)
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps(res), flush=True)
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
