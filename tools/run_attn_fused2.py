"""Time the fused attention kernel alone on the 12hr-model map: python tools/run_attn_fused2.py N iters [grid]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from vit_grid_model_b200 import ops

N = int(sys.argv[1]) if len(sys.argv) > 1 else 96
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
grid = len(sys.argv) > 3 and sys.argv[3] == "grid"
H, W, C, heads, dh, w, R = 42, 35, 128, 32, 32, 7, 4
g = torch.Generator().manual_seed(0)
x = torch.randn(N, H, W, C, generator=g).cuda()
reg = (torch.randn(N, R, C, generator=g) if grid else torch.randn(R, C, generator=g)).cuda()
film = torch.randn(N, 2 * C, generator=g).cuda()
wqkv = (torch.randn(heads * 96, C, generator=g) / 11.3).half().cuda()
wout = (torch.randn(heads, C, dh, generator=g) / 32).cuda()
qg, kg = torch.ones(heads * dh).cuda(), torch.ones(heads * dh).cuda()
bias = torch.randn(170, heads, generator=g).cuda()
tab = ops.pack_head_tables(bias, qg, kg)
lb = ops.attn_logit_bound(bias, qg, kg, dh) if os.environ.get("NOMAX", "0") == "1" else 0.0      # NOMAX=1: softmax without the running maximum
best = 1e9
for _ in range(iters):
    xin = x.clone()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    y, r = ops.attn_fused(xin, reg, film, wqkv, wout, tab, w, R, grid, True, heads, dh, inplace=True, logit_bound=lb)
    e1.record()
    torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1))
gf = 2.0125 * N
print(f"logit_bound={lb:.1f} {'grid' if grid else 'block'} N={N} windows={N*30} best ms={best:.3f}  {gf / best:.1f} TFLOP/s algorithmic  finite={torch.isfinite(y).all().item()}")

dbg = torch.zeros(3 * 128 * 8 + 16 * 128 * 2, dtype=torch.int64, device="cuda")
os.environ["VG_ATTN2_DBG"] = hex(dbg.data_ptr())
ops.attn_fused(x.clone(), reg, film, wqkv, wout, tab, w, R, grid, True, heads, dh, inplace=True)
torch.cuda.synchronize()
del os.environ["VG_ATTN2_DBG"]
wsk = dbg.cpu()[3 * 128 * 8:].view(16, 128, 2)
d = dbg.cpu()[:3 * 128 * 8].view(3, 128, 8)
t0 = d[0, 0, 0].item()
names = ["start", "qkv_done", "staged(qk_ready)", "s_done", "bias+max", "exp+norm", "P buf free", "p_ready"]
for grp in (0, 1):
    print(f"group {grp}: head  " + "  ".join(f"{n:>10s}" for n in names))
    for j in list(range(grp, 12, 2)) + list(range(56 + grp, 72, 2)):
        row = d[grp, j]
        print(f"        {j:4d}  " + "  ".join(f"{(v.item() - t0):10d}" for v in row))
mn = ["iter start", "qkv deps ok", "QKV(j+1) issued", "S deps ok", "S(j) issued", "| p_ready(j) seen", "pv_done seen", "out issued"]
print("MMA warps: j  " + "  ".join(f"{n:>16s}" for n in mn))
for j in list(range(0, 12)) + list(range(58, 70)):
    row = d[2, j]
    print(f"      {j:4d}  " + "  ".join(f"{(row[i].item() - t0):16d}" for i in (0, 6, 1, 7, 2, 3, 4, 5)))
per = (d[0, 60, 7] - d[0, 40, 7]).item() / 20
print("steady-state cycles per head (group 0, heads 40..60):", per)

print("per-warp stamps (relative to group warp 0), heads 66..69: staged | p_ready   [warps: ch0 lg2,3,0,1 then ch1 lg2,3,0,1]")
for j in (66, 67, 68, 69):
    g = j & 1
    ws = wsk[g * 8:(g + 1) * 8, j]
    print(f"   head {j}: staged", [int(v - ws[0, 0]) for v in ws[:, 0]], " p_ready", [int(v - ws[0, 1]) for v in ws[:, 1]])
