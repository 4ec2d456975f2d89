"""Calibration-pass benchmark (BASELINE.json configs[3]): calibrate_qat_model + reestimate_BN_stats over `--batches`
synthetic batches on YOLOv8m, calibration batches sharded across ranks, observer statistics all-reduced (MIN/MAX, exact)
and BN moments all-reduced per layer (SyncBN-style).

    python -m benchmarks.calibration --model m --batch 64 --imgsz 640 --batches 50
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 -m benchmarks.calibration ...

Reports seconds and images/s for both phases, the time of the observer synchronisation by itself (`sync_ms`: one packed
all_reduce(MIN) + one all_reduce(SUM) + one qparam kernel), the number of kernel launches the calibration forward passes
made, and digests of the post-calibration scales: MIN/MAX are exact, so the digests are identical at every world size
(the global set of batches is the same at every N) and on every rank (`ranks_agree`, checked with an all_gather)."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="m")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--imgsz", type=int, default=640)
    ap.add_argument("--batches", type=int, default=50, help="GLOBAL number of calibration batches")
    ap.add_argument("--channels-last", action="store_true",
                    help="NHWC weights / activations (cuDNN's native layout on sm_100); observers and the BN moments "
                         "pass walk that memory in place")
    ap.add_argument("--cudnn-benchmark", action="store_true", help="autotuned (non-reproducible) cuDNN algorithms")
    ap.add_argument("--observer", default="MinMaxObserver",
                    help="weight observer by registry name, e.g. MSEObserver (clipping-range search at the weight width)")
    ap.add_argument("--act-observer", default="MinMaxObserver",
                    help="activation observer by registry name, e.g. PercentileObserver (histogram clip at the activation "
                         "width); its histograms are merged exactly by the observer sync, so the digests still agree")
    return ap.parse_args(argv)


def _digest(pairs) -> str:
    h = hashlib.sha256()
    for s, z in pairs:
        h.update(repr((s, z)).encode())
    return h.hexdigest()


def run(args) -> dict:
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    # heuristic, deterministic cuDNN algorithms: a given batch then produces the same bits whichever rank runs it, which is
    # what makes the activation digests comparable across world sizes (cudnn.benchmark picks per process and per run)
    torch.backends.cudnn.benchmark = bool(args.cudnn_benchmark)
    torch.backends.cudnn.deterministic = not args.cudnn_benchmark
    from vsiquantization_b200 import _lib
    from vsiquantization_b200.modules.fuse import fuse_modules_unified
    from vsiquantization_b200.modules.fuse_config import FuseConfig, create_fuse_config_manager
    from vsiquantization_b200.nets import yolov8
    from vsiquantization_b200.parallel import quantization_managers, sync_observers
    from vsiquantization_b200.utils.estimate_bn import reestimate_BN_stats
    from vsiquantization_b200.utils.quantize_manager import calibrate_qat_model

    torch.manual_seed(0)
    model = getattr(yolov8, f"yolo_v8_{args.model}")(num_classes=20).to(dev)
    cfg = create_fuse_config_manager(FuseConfig(is_fuse_bn=False, bits_w=8, bits_a=8,  # BN kept: needed for re-estimation
                                                observer_w_name=args.observer, observer_a_name=args.act_observer))
    model = fuse_modules_unified(model, [["conv", "bn", "relu"]], config_manager=cfg)
    if args.channels_last:
        model.to(memory_format=torch.channels_last)

    # the same GLOBAL set of batches at every world size; rank r takes batches r, r+world, ...  Contents come from the
    # device's Philox generator seeded with the batch index (identical on every B200) and are parked in pinned host memory.
    def batch(i):
        g = torch.Generator(device=dev).manual_seed(1000 + i)
        b = torch.randint(0, 256, (args.batch, 3, args.imgsz, args.imgsz), generator=g, dtype=torch.uint8, device=dev)
        h = torch.empty(b.shape, dtype=torch.uint8, pin_memory=True)
        h.copy_(b)
        return h
    mine = [(batch(i), None) for i in range(rank, args.batches, world)]
    if not mine:
        raise SystemExit("calibration: fewer batches than ranks")

    def data_calib(m, loader, device):
        m.eval()
        with torch.no_grad():
            for imgs, _ in loader:
                m(imgs.to(device, non_blocking=True).float() / 255.0)

    data_calib(model, mine[:1], dev)  # warm-up (cuDNN plans, allocator) outside the timing
    for _, q in quantization_managers(model):  # forget the warm-up observation
        q.observer._state = None
        q._call_stats.clear()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = _lib.launch_count
    t0 = time.perf_counter()
    calibrate_qat_model(model, mine, data_calib, dev)
    torch.cuda.synchronize()
    t_fwd = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    ts = time.perf_counter()
    rows = sync_observers(model) if world > 1 else sum(1 for _ in quantization_managers(model))
    torch.cuda.synchronize()
    sync_ms = (time.perf_counter() - ts) * 1e3 if world > 1 else 0.0
    if world > 1:
        dist.barrier()
    t_cal = time.perf_counter() - t0
    launches_cal = _lib.launch_count - l0
    # post-sync scales: digested HERE -- the re-estimation pass below runs the model in calibration mode again, so (as in
    # the reference, quantization_manager.py:55-71) the observers keep absorbing each rank's local batches afterwards
    mgrs = quantization_managers(model)
    hw = _digest((q.scale, q.zero_point) for n, q in mgrs if n.endswith("weight_quantizer"))
    ha = _digest((q.scale, q.zero_point) for n, q in mgrs if n.endswith("activation_quantizer"))
    px = None
    if world > 1:  # one-off set-up of the peer-memory exchange (buffers + cudaIpc handles), outside the timed pass
        from vsiquantization_b200.parallel import peer_exchange_for
        px = peer_exchange_for(None)
        dist.barrier()
    t0 = time.perf_counter()
    reestimate_BN_stats(model, mine, num_batches=len(mine), sync=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_bn = time.perf_counter() - t0
    bn = [m.bn for m in model.modules() if hasattr(m, "bn")]
    hb = hashlib.sha256(b"".join(b.running_mean.detach().cpu().numpy().tobytes() + b.running_var.detach().cpu().numpy().tobytes()
                                 for b in bn)).hexdigest()
    agree = True
    if world > 1:  # every rank must hold bit-identical post-sync scales and re-estimated BN statistics
        mine_d = torch.tensor([int(h[:15], 16) for h in (hw, ha, hb)], dtype=torch.int64, device=dev)
        every = [torch.zeros_like(mine_d) for _ in range(world)]
        dist.all_gather(every, mine_d)
        agree = all(bool(torch.equal(e, every[0])) for e in every)
        if not agree and rank == 0:
            print("calibration: ranks disagree after the sync:", [e.tolist() for e in every], file=sys.stderr, flush=True)
    t = torch.tensor([t_cal, t_bn, sync_ms, t_fwd], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_cal, t_bn, sync_ms, t_fwd = (float(v) for v in t.tolist())
    n_img = args.batches * args.batch
    return {"model": f"yolov8{args.model}", "weight_observer": args.observer, **(
                {"activation_observer": args.act_observer} if args.act_observer != "MinMaxObserver" else {}),
            "n_gpus": world, "global_batches": args.batches, "batch": args.batch,
            "imgsz": args.imgsz, "channels_last": args.channels_last, "observer_rows_synced": rows,
            "calibration_s": t_cal, "images_per_s": n_img / t_cal, "calibration_images_per_s": n_img / t_cal,
            "calibration_forward_s": t_fwd, "sync_ms": sync_ms,
            "bn_reestimate_s": t_bn, "bn_reestimate_images_per_s": n_img / t_bn,
            "vsiq_launches_calibration": launches_cal, "host_syncs_in_calibration_forward": 0,
            "weight_scales_sha256": hw[:16], "activation_scales_sha256": ha[:16], "bn_stats_sha256": hb[:16],
            "ranks_agree": bool(agree),
            "bn_exchange": ("none (one rank)" if world == 1 else
                            (f"vsiq_bn_moments_exchange over peer memory, {px.status()[0]} exchanges" if px is not None
                             else "NCCL all_reduce per layer")),
            "bn0_running_mean_head": [round(float(v), 6) for v in bn[0].running_mean[:3]]}


def main():
    args = parse()
    res = run(args)
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps(res), flush=True)
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
