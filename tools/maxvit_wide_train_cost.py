"""Cost of one training step of the BASELINE configs[4] MaxViT backbone on its own: MaxViT(dim=512, heads=32, dim_head=64,
depth=4), 12 fields of 42x35, attention dropout 0.1, in 'bf16' (mixed) and 'fp32' precision.  Prints (1) the step time
(forward + backward, CUDA events, medians), (2) the time per entry point of one traced step for the kernels this backbone's
training added or generalised, (3) the memory-bound kernels alone, L2 flushed, with the bytes they must move and the rate.
The card's name and power limit are printed with the numbers.  Writes nothing.
usage: python tools/maxvit_wide_train_cost.py [reps]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import synth
from vit_grid_model_b200 import MaxViT, _lib
from vit_grid_model_b200 import ops_train as ot

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
N, H, W, DIM, DEPTH, HEADS, DH, CD = 12, 42, 35, 512, 4, 32, 64, 32
NEW = ("vg_attn_gather_bwd", "vg_attn_core_bwd", "vg_bn_bwd", "vg_dw3x3_fwd", "vg_dw3x3_wgrad", "vg_se_gate_train_fwd", "vg_se_bwd",
       "vg_field_dot", "vg_bn_stats", "vg_colsum", "vg_attn_out_bwd_gather", "vg_cond_mlp_bwd")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}   MaxViT(dim={DIM}, heads={HEADS}, dim_head={DH}, depth={DEPTH}), {N} fields of {H}x{W}, reps={REPS}")


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


sd = synth.make_state_dict(synth.maxvit_multistage_spec(DIM, DEPTH, CD, HEADS, DH, 7, 4, 0.25, 4), seed=0)
gen = torch.Generator(device=dev).manual_seed(1)
x = torch.randn(N, DIM, H, W, device=dev, generator=gen)
cond = torch.randn(N, CD, device=dev, generator=gen)
dy = torch.randn(N, DIM, H, W, device=dev, generator=gen)
for precision in ("bf16", "fp32"):
    m = MaxViT(dim=DIM, depth=DEPTH, cond_dim=CD, heads=HEADS, dim_head=DH, vit_window_size=7, num_register_tokens=4, dropout=0.1)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).train().set_precision(precision)

    def step():
        for p in m.parameters():
            p.grad = None
        m(x, cond).backward(dy)
    for _ in range(3):
        step()
    t = [timed(step) for _ in range(REPS)]
    print(f"[{precision}] training step (forward + backward): {median(t):.2f} ms  [median of {REPS}; spread {min(t):.2f}..{max(t):.2f}]")
    _lib.TRACE = []
    step()
    torch.cuda.synchronize()
    per, total = {}, 0.0
    for name, _, e0, e1 in _lib.TRACE:
        ms = e0.elapsed_time(e1)
        total += ms
        if name in NEW:
            c, s = per.get(name, (0, 0.0))
            per[name] = (c + 1, s + ms)
    _lib.TRACE = None
    print(f"[{precision}]   traced step: {total:.2f} ms summed over every entry point; of those:")
    for name, (c, s) in sorted(per.items(), key=lambda kv: -kv[1][1]):
        print(f"[{precision}]     {name:24s} {c:3d} calls {s:8.3f} ms")
    del m

# memory-bound kernels alone at the backbone's widths (rows M = N*H*W = 17,640; hidden 2048), L2 flushed before each call
M, HID = N * H * W, 4 * DIM
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB: evicts the 126 MB L2


def rate(label, fn, nbytes):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(max(REPS, 20)):
        flush.zero_()
        ts.append(timed(fn))
    t = median(ts)
    print(f"{label:44s} {t * 1e3:8.1f} us  {nbytes / 1e6:7.1f} MB  {nbytes / t / 1e6:6.0f} GB/s "
          f"({100 * nbytes / t / 1e6 / 7700:.0f} % of the 7.7 TB/s data-sheet HBM bandwidth)")


g = torch.Generator(device=dev).manual_seed(2)
raw, dout = torch.randn(M, HID, device=dev, generator=g), torch.randn(M, HID, device=dev, generator=g)
gamma, beta = torch.rand(HID, device=dev, generator=g) + 0.5, torch.randn(HID, device=dev, generator=g)
st = ot.bn_stats(raw, gamma, beta, 1e-5, 0.1, None, None)
dgam, dbet, draw = torch.zeros(HID, device=dev), torch.zeros(HID, device=dev), torch.empty_like(raw)
gate = torch.rand(N, HID, device=dev, generator=g)
fadd = torch.randn(N, HID, device=dev, generator=g)
# reduce pass reads dOut and raw, apply pass reads them again and writes draw
rate(f"bn_bwd C={HID} (GELU, squeeze-excite terms)",
     lambda: ot.bn_bwd(dout, raw, st, gamma, 1, dgam, dbet, fgate=gate, fadd=fadd, rows_per_field=H * W, out=draw), 5 * M * HID * 4)
rate(f"bn_bwd_frozen C={HID} (GELU)", lambda: ot.bn_bwd_frozen(dout, raw, st, 1, dgam, dbet, out=draw), 5 * M * HID * 4)
x4, d4 = raw.view(N, H, W, HID), dout.view(N, H, W, HID)
w9, ones, zeros = torch.randn(9, HID, device=dev, generator=g), torch.ones(HID, device=dev), torch.zeros(HID, device=dev)
out4 = torch.empty_like(x4)
rate(f"depthwise 3x3 C={HID} (forward / dgrad)", lambda: ot.dw3x3(x4, w9, ones, zeros, 0, out=out4), 2 * M * HID * 4)
dw9, db = torch.zeros(9, HID, device=dev), torch.zeros(HID, device=dev)
rate(f"depthwise 3x3 weight gradient C={HID}", lambda: ot.dw3x3_wgrad(x4, d4, dw9, db), 2 * M * HID * 4)
del raw, dout, draw, x4, d4, out4
C, S, nwin = DIM, 53, (H // 7) * (W // 7)
rows = N * nwin * S
xa = torch.randn(N, H, W, C, device=dev, generator=g)
reg = torch.randn(4, C, device=dev, generator=g)
film = torch.randn(N, 2 * C, device=dev, generator=g)
dtok, dxo = torch.randn(rows, C, device=dev, generator=g), torch.randn(N, H, W, C, device=dev, generator=g)
dreg, dfilm = torch.zeros(4, C, device=dev), torch.zeros(N, 2 * C, device=dev)
# reads x, dtok and dx_out, writes dx_in
rate(f"attn_gather_bwd C={C} (grid mode)", lambda: ot.attn_gather_bwd(xa, reg, film, dtok, dxo, None, 0.0, dreg, dfilm, 7, 4, True),
     (3 * M * C + rows * C) * 4)
