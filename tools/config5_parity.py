"""BASELINE configs[4] at full depth (512 ch, 32 x 64 heads, depth 4, 82x67): max rel err of every precision mode vs the CPU oracle."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from oracle import synth
from oracle.metnet3_oracle import metnet3_forward
from vit_grid_model_b200 import MetNet3

cfg = synth.GridConfig(dim=512, heads=32, dim_head=64, vit_depth=4)
sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=0)
x, ts, _ = synth.make_inputs(cfg, 1, seed=3)
t0 = time.perf_counter()
with torch.no_grad():
    ref = metnet3_forward(x, ts, sd, cfg)
print(f"oracle: {time.perf_counter() - t0:.1f} s", flush=True)
m = MetNet3(**cfg.metnet3_kwargs())
m.load_state_dict(sd, strict=True)
m = m.cuda().eval()
for mode in ("tf32", "tf32conv+fp32vit", "tf32_conv", "fp32"):
    if mode == "tf32conv+fp32vit":
        m.set_precision("tf32"); m.vit.set_precision("fp32")
    elif mode == "fp32conv+tf32vit":
        m.set_precision("fp32"); m.vit.set_precision("bf16")
    else:
        m.set_precision(mode)
    with torch.no_grad():
        y = m(x.cuda(), timestamps=ts.cuda())
        torch.cuda.synchronize(); t0 = time.perf_counter()
        y = m(x.cuda(), timestamps=ts.cuda())
        torch.cuda.synchronize(); dt = time.perf_counter() - t0
    e = ((y.cpu() - ref).abs().max() / ref.abs().max()).item()
    print(f"{mode:10s} rel err vs oracle {e:.3e}   {dt * 1e3:.1f} ms / 12 fields", flush=True)
