"""Run the attention core backward alone (for timing): the tcgen05 kernel on bf16 tensors (mode 3), the mma.sync kernel on
fp32 tensors (mode 2) and the exact-fp32 SIMT kernel (mode 0)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from vit_grid_model_b200 import ops_train as ot

N = int(sys.argv[1]) if len(sys.argv) > 1 else 96
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 3
H, W, w, R, heads, dh = 42, 35, 7, 4, 32, 32
rows = N * (H // w) * (W // w) * (R + w * w)
g = torch.Generator().manual_seed(0)
qkv = torch.randn(rows, 3 * heads * dh, generator=g).cuda()
datt = torch.randn(rows, heads * dh, generator=g).cuda()
qg, kg = torch.ones(heads * dh).cuda(), torch.ones(heads * dh).cuda()
tab = torch.randn(170, heads, generator=g).cuda()
dq, dk, dt = torch.zeros_like(qg), torch.zeros_like(kg), torch.zeros_like(tab)
for name, q, d, tf32 in (("tcgen05 bf16", qkv.bfloat16(), datt.bfloat16(), True), ("mma.sync fp32", qkv, datt, True),
                         ("SIMT fp32", qkv, datt, False)):
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ot.attn_core_bwd(q, d, qg, kg, tab, N, H, W, w, R, heads, dh, dq, dk, dt, tf32=tf32, want_att=tf32)
        e1.record()
        torch.cuda.synchronize()
    print(f"N={N} windows={N * 30} {name}: {e0.elapsed_time(e1):.3f} ms")
