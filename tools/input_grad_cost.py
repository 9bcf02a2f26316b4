"""Cost of input gradients at the 12-hour geometry, 16 samples, mixed precision: (1) the extra time of a training step when
x.requires_grad is on, (2) one eval-mode forward + backward (the frozen-BatchNorm graph), (3) vg_prepare_bwd against the bytes
it must move.  Steps of the compared variants alternate in one process; the card's name and power limit are printed with the
numbers.  Writes nothing.   usage: python tools/input_grad_cost.py [B] [reps]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import synth
from vit_grid_model_b200 import MetNet3, focal_r_loss
from vit_grid_model_b200 import ops, ops_train as ot

cfg = synth.CFG_12HR
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 10
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}   B={B}  reps={REPS}  precision=bf16 (mixed)")

model = MetNet3(**cfg.metnet3_kwargs(), dropout=0.0)
model.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
model = model.to(dev).set_precision("bf16")
x, ts, target = synth.make_inputs(cfg, B, seed=4321)
x, ts, target = x.to(dev), ts.to(dev), target.to(dev)


def step(want_dx):
    for p in model.parameters():
        p.grad = None
    xi = x.detach().requires_grad_(want_dx)
    focal_r_loss(model(xi, timestamps=ts), target).backward()


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


# (1) training step with / without x.requires_grad, alternating
model.train()
for _ in range(2):
    step(False), step(True)
t_off, t_on = [], []
for _ in range(REPS):
    t_off.append(timed(lambda: step(False)))
    t_on.append(timed(lambda: step(True)))
a, b = median(t_off), median(t_on)
print(f"train step: x.requires_grad off {a:.2f} ms, on {b:.2f} ms, extra {b - a:+.2f} ms ({100 * (b - a) / a:+.1f} %)  "
      f"[median of {REPS}; spread off {min(t_off):.2f}..{max(t_off):.2f}, on {min(t_on):.2f}..{max(t_on):.2f}]")

# (2) eval-mode forward + backward with an input that requires grad, next to the no_grad inference call
model.eval()


def infer():
    with torch.no_grad():
        model(x, timestamps=ts)


for _ in range(2):
    step(True), infer()
t_ev, t_inf = [], []
for _ in range(REPS):
    t_ev.append(timed(lambda: step(True)))
    t_inf.append(timed(infer))
print(f"eval forward+backward (x.requires_grad): {median(t_ev):.2f} ms  [no_grad inference of the same batch {median(t_inf):.2f} ms]")

# (3) vg_prepare_bwd alone: reads the frame pixels' first T*C channels of the PG gradient, writes (B,T,C,H,W) fp32
HP, WP = cfg.HP, cfg.WP
cpad = (cfg.T * cfg.C + 63) // 64 * 64
g = torch.randn(ops.pg_pixels(B, HP, WP), cpad, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB: evicts the 126 MB L2 between timed calls
for _ in range(3):
    ot.prepare_bwd(g, B, cfg.T, cfg.C, cfg.H, cfg.W, cfg.pads, HP, WP, cfg.pm25_std)
ts_k = []
for _ in range(max(REPS, 20)):
    flush.zero_()
    ts_k.append(timed(lambda: ot.prepare_bwd(g, B, cfg.T, cfg.C, cfg.H, cfg.W, cfg.pads, HP, WP, cfg.pm25_std)))
nbytes = 2 * B * cfg.T * cfg.C * cfg.H * cfg.W * 4
t = median(ts_k)
print(f"vg_prepare_bwd: {t * 1e3:.1f} us for {nbytes / 1e6:.0f} MB algorithmic (read + write) -> {nbytes / t / 1e6:.0f} GB/s "
      f"({100 * nbytes / t / 1e6 / 7700:.0f} % of the 7.7 TB/s data-sheet HBM bandwidth; L2 flushed, event timing incl. the "
      f"torch.empty of the output)")
