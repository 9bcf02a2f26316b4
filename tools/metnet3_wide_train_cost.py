"""Cost of one 'tf32_conv' training step of MetNet3 on the BASELINE configs[4] shape: n_start_channels 512, 32 x 64 heads, MaxViT
depth 4, the 82x67 grid of the 12-hour model (25 time steps x 24 variables), 12 fields (B = 1, 12 lead times), dropout 0.1.
Prints (1) the step time (forward + backward, CUDA events, median of `reps` steps after three warm-up steps), (2) a CUDA-event
split of the same steps between the MaxViT half (train.maxvit_train_forward / maxvit_train_backward) and the rest, the conv side
(stem, conv blocks, pooling, ConvTranspose, head, embeddings), (3) the row kernels of the wide conv side alone, L2 flushed, with
the bytes they must move and the rate.  The card's name and power limit are read in the same run and printed with the numbers.
Writes nothing.
usage: python tools/metnet3_wide_train_cost.py [reps]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import synth
from vit_grid_model_b200 import MetNet3, focal_r_loss, ops
from vit_grid_model_b200 import ops_train as ot
from vit_grid_model_b200 import train as tr
from vit_grid_model_b200.metnet3 import _pack_conv3x3

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
CFG = synth.GridConfig(T=25, C=24, H=82, W=67, dim=512, L=12, heads=32, dim_head=64, vit_depth=4)
B = 1
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}   MetNet3 n_start_channels={CFG.dim}, {CFG.heads} x {CFG.dim_head} heads, MaxViT depth {CFG.vit_depth}, "
      f"{CFG.H}x{CFG.W}, {B * CFG.L} fields, tf32_conv, reps={REPS}")


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


m = MetNet3(**CFG.metnet3_kwargs(), dropout=0.1)
m.load_state_dict(synth.make_state_dict(synth.metnet3_spec(CFG), seed=0), strict=True)
m = m.to(dev).train().set_precision("tf32_conv")
x, ts, _ = synth.make_inputs(CFG, B, seed=1)
x, ts = x.to(dev), ts.to(dev)
target = torch.rand(B, CFG.L, CFG.H, CFG.W, device=dev, generator=torch.Generator(device=dev).manual_seed(2)) * 40

# events around the MaxViT half of the step (its forward and its backward)
vit_events = []
for name in ("maxvit_train_forward", "maxvit_train_backward"):
    inner = getattr(tr, name)

    def wrapped(*a, _inner=inner, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = _inner(*a, **kw)
        e1.record()
        vit_events.append((e0, e1))
        return r
    setattr(tr, name, wrapped)


def step():
    for p in m.parameters():
        p.grad = None
    focal_r_loss(m(x, timestamps=ts), target).backward()


for _ in range(3):
    step()
t, tv = [], []
for _ in range(REPS):
    vit_events.clear()
    t.append(timed(step))
    tv.append(sum(e0.elapsed_time(e1) for e0, e1 in vit_events))
print(f"training step (forward + backward): {median(t):.1f} ms  [median of {REPS}; spread {min(t):.1f}..{max(t):.1f}]")
print(f"  MaxViT half: {median(tv):.1f} ms   conv side (the rest): {median([a - b for a, b in zip(t, tv)]):.1f} ms  [medians]")

# the wide row kernels alone at this shape (N = 12 fields, 84x70 frame, C = 512), L2 flushed before each call
N, HP, WP, C = B * CFG.L, 84, 70, CFG.dim
Q = ops.pg_pixels(N, HP, WP)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB: evicts the 126 MB L2


def rate(label, fn, nbytes):
    for _ in range(3):
        fn()
    ts_ = []
    for _ in range(max(REPS, 20)):
        flush.zero_()
        ts_.append(timed(fn))
    tt = median(ts_)
    print(f"{label:52s} {tt * 1e3:8.1f} us  {nbytes / 1e6:7.1f} MB  {nbytes / tt / 1e6:6.0f} GB/s "
          f"({100 * nbytes / tt / 1e6 / 7700:.0f} % of the 7.7 TB/s data-sheet HBM bandwidth)")


g = torch.Generator(device=dev).manual_seed(3)
xin = ops.pg_from_nchw(torch.randn(N, C, HP, WP, device=dev, generator=g), torch.float32)
w = torch.randn(C, C, 3, 3, device=dev, generator=g) * (9 * C) ** -0.5
Wt = _pack_conv3x3(w, torch.float32)
bias, lg, lb = torch.zeros(C, device=dev), torch.ones(C, device=dev), torch.zeros(C, device=dev)
film = torch.randn(N, 2 * C, device=dev, generator=g) * 0.1
out = torch.empty_like(xin)
_, saved = ot.conv3x3_ln_train(xin, Wt, bias, lg, lb, 1e-5, film, None, out, N, HP, WP, tf32=True)
xhat, rstd, mask = saved
# the whole training forward of a conv block (tf32 GEMM into the scratch + the row kernel): the bytes counted are those of the
# row kernel (reads the scratch; writes out, xhat, rstd and the mask), so the rate is a lower bound of the row kernel's
rate(f"conv block training forward C={C} (tf32 GEMM + row kernel)",
     lambda: ot.conv3x3_ln_train(xin, Wt, bias, lg, lb, 1e-5, film, None, out, N, HP, WP, tf32=True), Q * C * 4 * 3 + Q * (4 + C // 8))
dY = torch.randn(Q, C, device=dev, generator=g)
rate(f"Block backward C={C} (dconv + per-field sums)",
     lambda: ot.conv_ln_bwd(dY, saved, lg, film, 1e-5, N, HP, WP, torch.float32), Q * C * 4 * 3 + Q * (4 + C // 8))
h1, res = torch.empty_like(xin), torch.empty_like(xin)
Bp = ops.pg_pixels(B, HP, WP)
raw3, rawres = torch.randn(Bp, C, device=dev, generator=g), torch.randn(Bp, C, device=dev, generator=g)
tt_, tres = torch.randn(N, 9, C, device=dev, generator=g), torch.randn(N, C, device=dev, generator=g)
rate(f"stem finish, training C={C} (12 leads of one sample)",
     lambda: ot.stem_finish_train(raw3, rawres, bias, bias, tt_, tres, lg, lb, 1e-5, film, B, CFG.L, HP, WP, h1, res),
     2 * Bp * C * 4 + 3 * Q * C * 4 + Q * (4 + C // 8))
rate(f"lead-time sum C={C}", lambda: ot.lead_sum(dY, B, CFG.L, HP, WP, torch.float32), (Q + Bp) * C * 4)
