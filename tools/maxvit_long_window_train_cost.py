"""Cost of one training step (forward + backward) of MaxViT(dim=128, depth=2) with the reference's defaults -- window 8 with
4 register tokens (S = 68 tokens per window), 32 heads x 32, dropout 0.1 -- on 12 fields of 48x40, in 'bf16' (mixed) and
'fp32' precision, next to the same network at window 7 (S = 53) on 12 fields of 49x42.  Prints the step time (CUDA events,
median of REPS steps) and the share of one traced step spent in the attention core backward (vg_attn_core_bwd; at window 7
in 'bf16' the fused attention's backward, vg_attn_bwd_fused).  The card's name and power limit are printed with the numbers.
Writes nothing.
usage: python tools/maxvit_long_window_train_cost.py [reps]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import synth
from vit_grid_model_b200 import MaxViT, _lib

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
N, DIM, DEPTH, HEADS, DH, CD, R = 12, 128, 2, 32, 32, 32, 4
GEOMS = {8: (48, 40), 7: (49, 42)}          # window -> map (6 x 5 and 7 x 6 windows)
CORE_BWD = ("vg_attn_core_bwd", "vg_attn_bwd_fused")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}   MaxViT(dim={DIM}, depth={DEPTH}, heads={HEADS}, dim_head={DH}, dropout 0.1), {N} fields, reps={REPS}")


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


for win, (H, W) in GEOMS.items():
    sd = synth.make_state_dict(synth.maxvit_multistage_spec(DIM, DEPTH, CD, HEADS, DH, win, 4, 0.25, R), seed=0)
    gen = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(N, DIM, H, W, device=dev, generator=gen)
    cond = torch.randn(N, CD, device=dev, generator=gen)
    dy = torch.randn(N, DIM, H, W, device=dev, generator=gen)
    for precision in ("bf16", "fp32"):
        m = MaxViT(dim=DIM, depth=DEPTH, cond_dim=CD, vit_window_size=win)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev).train().set_precision(precision)

        def step():
            for p in m.parameters():
                p.grad = None
            m(x, cond).backward(dy)
        for _ in range(3):
            step()
        t = [timed(step) for _ in range(REPS)]
        tag = f"[window {win}, S {R + win * win}, {H}x{W}, {precision}]"
        print(f"{tag} training step (forward + backward): {median(t):.2f} ms  [median of {REPS}; spread {min(t):.2f}..{max(t):.2f}]")
        _lib.TRACE = []
        step()
        torch.cuda.synchronize()
        total, core, calls = 0.0, 0.0, 0
        for name, _, e0, e1 in _lib.TRACE:
            ms = e0.elapsed_time(e1)
            total += ms
            if name in CORE_BWD:
                core += ms
                calls += 1
        _lib.TRACE = None
        print(f"{tag}   traced step {total:.2f} ms summed over every entry point; attention core backward {core:.2f} ms in "
              f"{calls} calls ({100 * core / total:.0f} %)")
        del m
