"""Cost of synchronised BatchNorm statistics in data-parallel training: the median time of a training step (forward + backward,
GradSync all-reduce included; CUDA events after a barrier) with per-rank BatchNorm statistics and with the MaxViT BatchNorms
converted by nn.SyncBatchNorm.convert_sync_batchnorm, steps of the variants alternating in one run, one process per GPU over
NCCL.  Variants: 'per-rank' (unconverted), 'sync' (converted; DataParallel gives the statistics a dedicated process group) and
'sync, shared group' (converted with process_group = WORLD, so the exchanges queue behind GradSync's gradient all-reduces).
Cases:
  12hr : the 12-hour model (82x67, 25 x 24 inputs, 12 lead times) in 'bf16', 16 samples per GPU;
  c4   : BASELINE configs[4] (512 channels, 32 x 64 heads, MaxViT depth 4) in 'tf32_conv', 12 fields (one sample) per GPU;
  c3   : BASELINE configs[3] (512x512 domain, MaxViT depth 2) in 'bf16', 12 fields (one sample) per GPU.
The card's name and power limit are printed with the numbers.  Writes nothing.
usage: python tools/sync_batchnorm_cost.py [--gpus 2 8] [--reps 20] [--cases 12hr c4 c3]"""
import argparse
import copy
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from oracle import synth

CASES = {
    "12hr": ("12-hour, 16 samples/GPU, bf16", synth.CFG_12HR, 16, "bf16"),
    "c4": ("configs[4], 12 fields/GPU, tf32_conv", synth.GridConfig(dim=512, heads=32, dim_head=64, vit_depth=4), 1, "tf32_conv"),
    "c3": ("configs[3], 12 fields/GPU, bf16", synth.GridConfig(H=512, W=512, vit_depth=2), 1, "bf16"),
}


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def run_case(rank, world, dev, key, reps):
    from vit_grid_model_b200 import DataParallel, MetNet3, focal_r_loss
    label, cfg, B, precision = CASES[key]
    base = MetNet3(**cfg.metnet3_kwargs(), dropout=0.1)
    base.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
    variants = {}
    for name in ("per-rank", "sync", "sync, shared group"):
        m = copy.deepcopy(base)
        if name != "per-rank":
            m = nn.SyncBatchNorm.convert_sync_batchnorm(m)
            if name == "sync, shared group":
                for bn in m.modules():
                    if isinstance(bn, nn.SyncBatchNorm):
                        bn.process_group = dist.group.WORLD
        m = m.to(dev).set_precision(precision).train()
        variants[name] = (m, DataParallel(m))
    del base
    x, ts, target = synth.make_inputs(cfg, B, seed=4321 + rank)
    x, ts, target = x.to(dev), ts.to(dev), target.to(dev)

    def step(name):
        m, net = variants[name]
        for p in m.parameters():
            p.grad = None
        focal_r_loss(net(x, timestamps=ts), target).backward()

    def timed(name):
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(name)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(3):
        for name in variants:
            step(name)
    t = {name: [] for name in variants}
    for _ in range(reps):
        for name in variants:
            t[name].append(timed(name))
    # the step time of the slowest rank
    med = torch.tensor([median(t[name]) for name in variants], device=dev)
    dist.all_reduce(med, op=dist.ReduceOp.MAX)
    if rank == 0:
        a = med[0].item()
        cols = "  ".join(f"{name} {v:.2f} ms ({v - a:+.2f})" for name, v in zip(variants, med.tolist()))
        print(f"{world} GPUs, {label}: {cols}", flush=True)
    del variants
    torch.cuda.empty_cache()


def worker(rank, world, port, cases, reps):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        for key in cases:
            run_case(rank, world, dev, key, reps)
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, nargs="+", default=[2, 8])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cases", nargs="+", default=list(CASES), choices=list(CASES))
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"cards: {len(card)} x {card[0] if card else '?'}   reps={args.reps} (medians; +x: difference to per-rank)", flush=True)
    for world in args.gpus:
        if world > torch.cuda.device_count():
            print(f"{world} GPUs: skipped, {torch.cuda.device_count()} visible")
            continue
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        mp.spawn(worker, args=(world, port, args.cases, args.reps), nprocs=world, join=True)


if __name__ == "__main__":
    main()
