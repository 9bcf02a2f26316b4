"""Cost of the deterministic training backward (torch.use_deterministic_algorithms(True)): the median time of a training step
(forward + backward, CUDA events) with the flag off and on, steps of the two modes alternating in one process, on
  (1) the bench step: the 12-hour geometry (82x67, 25 x 24 inputs, 12 lead times), 16 samples, 'bf16' mixed precision;
  (2) the BASELINE configs[4] shape in 'tf32_conv': n_start_channels 512, 32 x 64 heads, MaxViT depth 4, 12 fields;
  (3) the same 12-hour step in 'fp32', where every reduction of the backward (attention core included) is deterministic.
In (1) and (2) the mixed-precision attention core backward still reduces with atomics (it has no deterministic kernel yet); the
other reductions take the fixed-order path.  The card's name and power limit are printed with the numbers.  Writes nothing.
usage: python tools/deterministic_train_cost.py [reps] [B]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import synth
from vit_grid_model_b200 import MetNet3, focal_r_loss

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
B = int(sys.argv[2]) if len(sys.argv) > 2 else 16
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}   reps={REPS}")


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def measure(label, cfg, batch, precision):
    model = MetNet3(**cfg.metnet3_kwargs(), dropout=0.1)
    model.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
    model = model.to(dev).set_precision(precision).train()
    x, ts, target = synth.make_inputs(cfg, batch, seed=4321)
    x, ts, target = x.to(dev), ts.to(dev), target.to(dev)

    def step(det):
        torch.use_deterministic_algorithms(det)
        try:
            for p in model.parameters():
                p.grad = None
            focal_r_loss(model(x, timestamps=ts), target).backward()
        finally:
            torch.use_deterministic_algorithms(False)

    for _ in range(3):
        step(False), step(True)
    t_off, t_on = [], []
    for _ in range(REPS):
        t_off.append(timed(lambda: step(False)))
        t_on.append(timed(lambda: step(True)))
    a, b = median(t_off), median(t_on)
    print(f"{label}: step {a:.2f} ms (atomics)  {b:.2f} ms (deterministic)  overhead {b - a:+.2f} ms ({100 * (b / a - 1):+.1f} %)")
    del model
    torch.cuda.empty_cache()


measure(f"12-hour, B={B}, bf16", synth.CFG_12HR, B, "bf16")
measure("configs[4], 12 fields, tf32_conv",
        synth.GridConfig(T=25, C=24, H=82, W=67, dim=512, L=12, heads=32, dim_head=64, vit_depth=4), 1, "tf32_conv")
measure(f"12-hour, B={B}, fp32", synth.CFG_12HR, B, "fp32")
