"""The residual + fp32-copy variant of the conv kernel alone at bench shape (for timing)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from vit_grid_model_b200 import ops
N = int(sys.argv[1]) if len(sys.argv) > 1 else 768
HP, WP, C = 84, 70, 128
g = torch.Generator().manual_seed(0)
x = ops.pg_from_nchw(torch.randn(N, C, HP, WP, generator=g).cuda(), torch.bfloat16)
w = (torch.randn(C, 9 * C, generator=g) / 34).cuda().bfloat16()
b, ga, be = torch.zeros(C).cuda(), torch.ones(C).cuda(), torch.zeros(C).cuda()
res = torch.randn(x.shape[0], C, device="cuda")
out, out2 = torch.empty_like(x), torch.empty(x.shape[0], C, device="cuda")
for _ in range(5):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ops.conv3x3_ln(x, w, b, ga, be, 1e-5, None, res, out, N, HP, WP, out_copy=out2)
    e1.record(); torch.cuda.synchronize()
print(f"res+copy N={N}: {e0.elapsed_time(e1):.3f} ms")
