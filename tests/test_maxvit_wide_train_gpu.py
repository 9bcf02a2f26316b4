"""Training of wide stand-alone MaxViT networks (GPU): the generalised kernels at 256 .. 512 channels, MBConv hidden widths up
to 2048 and dim_head 64 against float64 references, and the module -- y, x.grad, cond.grad, every parameter gradient and the
BatchNorm running buffers -- against float64 autograd through the oracle, in train() mode and in the frozen-BatchNorm eval()
graph, at 256, 384 and 512 channels and in a tuple-depth MaxViT whose stages widen the map 128 -> 256 -> 512.

Conventions (those of test_train_backward_kernels_gpu.py):
  * every reference is float64, on the GPU
  * every output a kernel must write completely starts as NaN; every accumulated output starts from a random tensor P and
    `out - P` is compared with the reference
  * errors are relative to the largest reference entry (rel_err) unless stated; each bound not taken from an existing rule
    states the error measured on a B200 next to it
"""
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle import maxvit_oracle as mo

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64, F32, BF16 = torch.float64, torch.float32, torch.bfloat16
WIN, R_REG = 7, 4
S_TOK = R_REG + WIN * WIN


def OT():
    from vit_grid_model_b200 import ops_train
    return ops_train


def call(name, *args):
    from vit_grid_model_b200 import _lib
    from vit_grid_model_b200.ops import _st
    _lib.call(name, *args, _st())


def note(**kv):
    """one line per measurement (pytest -s shows them; the measured values in the comments below come from these lines)"""
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0].split("::")[-1]
    print("MEASURE", test, " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in kv.items()))


def ptr(t):
    return None if t is None else t.data_ptr()


def rel_err(got, ref):
    """max |got - ref| / max |ref|, in float64 on the device"""
    got, ref = got.detach().to(DEV, F64), ref.detach().to(DEV, F64)
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, generator=g, device=DEV) * scale


def nan_like(shape, dtype=F32):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def prefill(shape, seed, scale=1.0):
    """the random P an accumulated output starts from, at 1/100 of the reference's largest entry"""
    return rnd(*shape, seed=seed, scale=0.01 * scale)


def _pixel_map(Hl, Wl, grid_mode):
    return (mo.grid_pixel_index if grid_mode else mo.block_pixel_index)(Hl, Wl, WIN).to(DEV)


# =========================================================================================== LayerNorm + FiLM backward
@pytest.mark.parametrize("reg_per_field", [False, True])
@pytest.mark.parametrize("grid_mode", [False, True])
@pytest.mark.parametrize("N,Hl,Wl", [(3, 42, 35), (1, 259, 259)])
@pytest.mark.parametrize("C", [256, 384, 512])
def test_attn_gather_bwd_wide(C, N, Hl, Wl, grid_mode, reg_per_field):
    """vg_attn_gather_bwd at C = 256, 384, 512 (a warp per row, C/32 channels per lane) in block and grid partition (stride 37
    at 259x259), registers shared (R,C) or per field (N,R,C): float64 autograd of the oracle's token sequence; dx_in = dx +
    dx_out at every pixel, dreg_in and dfilm accumulated.  With dtok = 0 the LayerNorm gradient is exactly zero, so dx_in must
    equal dx_out bit for bit at every window pixel: each pixel is written once, at its own address."""
    S, nwin = S_TOK, (Hl // WIN) * (Wl // WIN)
    x = rnd(N, Hl, Wl, C, seed=120) + rnd(C, seed=121)
    reg = rnd(*((N, R_REG, C) if reg_per_field else (R_REG, C)), seed=122)
    film = torch.cat([1 + 0.3 * rnd(N, C, seed=123), 0.3 * rnd(N, C, seed=124)], dim=1)
    dtok = rnd(N * nwin * S, C, seed=125)
    dx_out = rnd(N, Hl, Wl, C, seed=126)
    dreg_res = None if grid_mode else rnd(N, R_REG, C, seed=127)
    reg_scale = 0.0 if grid_mode else 1.0 / nwin
    xr, regr, filmr = (t.to(F64).requires_grad_(True) for t in (x, reg, film))
    pix = _pixel_map(Hl, Wl, grid_mode).reshape(-1)
    xs = xr.view(N, Hl * Wl, C)[:, pix].view(N, nwin, WIN * WIN, C)
    rege = (regr[:, None] if reg_per_field else regr[None, None]).expand(N, nwin, R_REG, C)
    tok = F.layer_norm(torch.cat([rege, xs], dim=2), (C,), eps=1e-5) * filmr[:, None, None, :C] + filmr[:, None, None, C:]
    loss = (tok * dtok.to(F64).view(N, nwin, S, C)).sum() + (xr * dx_out.to(F64)).sum()
    if dreg_res is not None:
        loss = loss + (rege * dreg_res.to(F64)[:, None]).sum() * reg_scale
    loss.backward()
    del tok, loss, xs, rege

    def run(dt):
        Pr, Pf = prefill(reg.shape, 128, regr.grad.abs().max().item()), prefill(film.shape, 129, filmr.grad.abs().max().item())
        dreg_in, dfilm, dx_in = Pr.clone(), Pf.clone(), nan_like(x.shape)
        call("vg_attn_gather_bwd", x.data_ptr(), reg.data_ptr(), int(reg_per_field), film.data_ptr(), dt.data_ptr(),
             dx_out.data_ptr(), ptr(dreg_res), reg_scale, dx_in.data_ptr(), dreg_in.data_ptr(), dfilm.data_ptr(),
             N, Hl, Wl, C, WIN, R_REG, int(grid_mode), 1e-5)
        torch.cuda.synchronize()
        return dx_in, dreg_in.double() - Pr.double(), dfilm.double() - Pf.double()
    dx_in, dreg, dfilm = run(dtok)
    e = dict(dx=rel_err(dx_in, xr.grad), dreg=rel_err(dreg, regr.grad), dfilm=rel_err(dfilm, filmr.grad))
    note(**e)
    # the existing rule of the 128-channel kernel (test_attn_gather_bwd): row-local fp32 LayerNorm backward, fp32 sums of 16
    # rows per warp and float atomics for dreg_in / dfilm
    assert e["dx"] < 1e-5 and e["dreg"] < 1e-5 and e["dfilm"] < 1e-5, e
    dx0, _, _ = run(torch.zeros_like(dtok))
    assert torch.equal(dx0, dx_out)


# =========================================================================================== attention core backward, dim_head 64
HEADS64, DH64 = 32, 64


def _rel_pos_index(win, R):
    W2 = 2 * win - 1
    t = torch.arange(win * win, device=DEV)
    a, b = t // win, t % win
    idx = torch.full((R + win * win, R + win * win), W2 * W2, dtype=torch.long, device=DEV)
    idx[R:, R:] = (a[:, None] - a[None, :] + win - 1) * W2 + (b[:, None] - b[None, :] + win - 1)
    return idx


def _core_bwd_ref(qkv, datt, qg, kg, bt, pmask, bf16_ops):
    """float64 backward of maxvit.py:189-213 on the [rows][3 inner] layout.  bf16_ops: round where the mode-2 kernel rounds --
    qh = q/|q| rs gq, kh, v, dO to bf16 (S = qh kh^T), P' = P mask and dS to bf16 in front of the products, the unit vectors of
    the RMSNorm backward taken from the rounded qh, kh; the bias gradient sums the unrounded dS.
    -> dqkv [rows][3 inner], dq_gamma, dk_gamma (heads*DH), dbias (table, heads)"""
    nw, H, D = qkv.shape[0] // S_TOK, HEADS64, DH64
    x = qkv.to(F64).view(nw, S_TOK, 3, H, D).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    dO = datt.to(F64).view(nw, S_TOK, H, D).permute(0, 2, 1, 3)
    rnd16 = (lambda t: t.to(BF16).to(F64)) if bf16_ops else (lambda t: t)
    inv_q = 1.0 / q.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    inv_k = 1.0 / k.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    rs = math.sqrt(D)
    gq = (torch.tensor(rs, dtype=F32, device=DEV) * qg).to(F64).view(H, 1, D) if bf16_ops else rs * qg.to(F64).view(H, 1, D)
    gk = (torch.tensor(rs, dtype=F32, device=DEV) * kg).to(F64).view(H, 1, D) if bf16_ops else rs * kg.to(F64).view(H, 1, D)
    qh, kh = rnd16(q * inv_q * gq), rnd16(k * inv_k * gk)
    vb, dOb = rnd16(v), rnd16(dO)
    idx = _rel_pos_index(WIN, R_REG)
    P = torch.softmax(qh @ kh.transpose(-1, -2) + bt.to(F64)[idx].permute(2, 0, 1), dim=-1)
    Mk = 1.0 if pmask is None else pmask
    dPm = (dOb @ vb.transpose(-1, -2)) * Mk
    dS = P * (dPm - (P * dPm).sum(-1, keepdim=True))
    dSb = rnd16(dS)
    dv = rnd16(P * Mk).transpose(-1, -2) @ dOb
    dqh, dkh = dSb @ kh, dSb.transpose(-1, -2) @ qh
    uq, uk = qh / gq, kh / gk
    dq = (dqh * gq - uq * (dqh * gq * uq).sum(-1, keepdim=True)) * inv_q
    dk = (dkh * gk - uk * (dkh * gk * uk).sum(-1, keepdim=True)) * inv_k
    dqg = (dqh * uq * rs).sum((0, 2)).reshape(-1)
    dkg = (dkh * uk * rs).sum((0, 2)).reshape(-1)
    dbias = torch.zeros(bt.shape, dtype=F64, device=DEV)
    dbias.index_add_(0, idx.reshape(-1), dS.sum(0).permute(1, 2, 0).reshape(S_TOK * S_TOK, H))
    dqkv = torch.stack([dq, dk, dv]).permute(1, 3, 0, 2, 4).reshape(nw * S_TOK, 3 * H * D)
    return dqkv, dqg, dkg, dbias


# mode 0 (exact fp32): the existing fp32 rule of test_train_kernels_gpu.py, 1e-4 of the largest reference entry (measured on a
# B200: 3.3e-6 at most).  Mode 2 against the bf16-rounding reference, worst of the six cases measured on a B200 (NVIDIA B200,
# 1000 W): dqkv 2.1e-3, dq_gamma 1.0e-3, dk_gamma 8.5e-4, dbias 7.4e-4 (fp32 accumulation order of the mma.sync tiles and the
# shared-memory atomics)
CORE_TOL = {0: dict(dqkv=1e-4, dq_gamma=1e-4, dk_gamma=1e-4, dbias=1e-4),
            2: dict(dqkv=8e-3, dq_gamma=4e-3, dk_gamma=3e-3, dbias=2.5e-3)}


@pytest.mark.parametrize("T", [0, 26])
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("N,Hl,Wl", [(3, 14, 21), (5, 7, 7), (2, 21, 35)])
def test_attn_core_bwd_dh64(N, Hl, Wl, mode, T):
    """vg_attn_core_bwd at dim_head 64, 32 heads: mode 0 (exact-fp32 SIMT, 172 KB of shared memory with dropout) and mode 2 (bf16
    mma.sync on fp32 tensors), without and with the probability dropout mask (read back through vg_dropout_mask_debug); 6
    windows per field, one window per field, and 15 (odd) windows per field.  dqkv written (NaN prefill), dq_gamma, dk_gamma and
    the bias table accumulated."""
    nwin = (Hl // WIN) * (Wl // WIN)
    inner = HEADS64 * DH64
    rows = N * nwin * S_TOK
    g = torch.Generator(device=DEV).manual_seed(3)
    qkv = torch.randn(rows, 3 * inner, device=DEV, generator=g)
    datt = torch.randn(rows, inner, device=DEV, generator=g)
    qg = 1 + 0.2 * torch.randn(inner, device=DEV, generator=g)
    kg = 1 + 0.2 * torch.randn(inner, device=DEV, generator=g)
    bt = 0.5 * torch.randn((2 * WIN - 1) ** 2 + 1, HEADS64, device=DEV, generator=g)
    drop = (4242, 1, T)
    pmask = None
    if T:
        pm, _ = OT().dropout_masks(drop, N * nwin, HEADS64, 128)
        pmask = pm[:, :, :S_TOK, :S_TOK].to(F64) * (256.0 / (256 - T))
    ref = _core_bwd_ref(qkv, datt, qg, kg, bt, pmask, bf16_ops=mode == 2)
    P = [prefill(t.shape, 130 + i, r.abs().max().item()) for i, (t, r) in enumerate(((qg, ref[1]), (kg, ref[2]), (bt, ref[3])))]
    dqg, dkg, dbt = (p.clone() for p in P)
    dqkv = nan_like(qkv.shape)
    call("vg_attn_core_bwd", qkv.data_ptr(), datt.data_ptr(), qg.data_ptr(), kg.data_ptr(), bt.data_ptr(), N, Hl, Wl, WIN, R_REG,
         HEADS64, DH64, dqkv.data_ptr(), dqg.data_ptr(), dkg.data_ptr(), dbt.data_ptr(), mode, None, drop[0], drop[1], drop[2])
    torch.cuda.synchronize()
    e = dict(dqkv=rel_err(dqkv, ref[0]), dq_gamma=rel_err(dqg.double() - P[0].double(), ref[1]),
             dk_gamma=rel_err(dkg.double() - P[1].double(), ref[2]), dbias=rel_err(dbt.double() - P[2].double(), ref[3]))
    note(**e)
    bad = {k: v for k, v in e.items() if not v < CORE_TOL[mode][k]}
    assert not bad, bad


def test_attn_core_bwd_tcgen05_stays_dim_head_32():
    """the tcgen05 kernel (mode 3) is built for dim_head 32 only and says so"""
    from vit_grid_model_b200 import _lib
    q = torch.zeros(S_TOK, 3 * 64, dtype=BF16, device=DEV)
    d = torch.zeros(S_TOK, 64, dtype=BF16, device=DEV)
    z = torch.zeros(4096, device=DEV)
    with pytest.raises(_lib.VitGridError, match="dim_head must be 32"):
        call("vg_attn_core_bwd", q.data_ptr(), d.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), 1, 7, 7, WIN, R_REG, 1, 64,
             q.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), 3, None, 0, 0, 0)


# =========================================================================================== BatchNorm backward
def _bn_input(M, C, seed):
    std = 0.5 + 1.5 * torch.rand(C, generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)
    off = torch.zeros(C, device=DEV)
    off[0::4], off[1::4] = 20.0, -20.0
    return rnd(M, C, seed=seed + 1) * std + off * std


@pytest.mark.parametrize("M,HW", [(882, 294), (282240, 1470)])
@pytest.mark.parametrize("C", [384, 1024, 1536, 2048])
def test_bn_bwd_wide(C, M, HW):
    """vg_bn_bwd (batch statistics) and vg_bn_bwd_frozen (running statistics) at C = 384, 1024, 1536 and 2048 (1536 and 2048: a
    thread per channel quad of a 1024-channel slice), as the MBConv calls them -- (act 0), (GELU with the squeeze-excite fgate /
    fadd, in place on dOut) -- against float64 autograd of F.batch_norm; 4 and 1,103 partials of 256 rows"""
    ot = OT()
    raw = _bn_input(M, C, 70)
    gamma, beta = 0.5 + rnd(C, seed=72).abs(), rnd(C, seed=73)
    r64 = raw.to(F64)
    m64, rs64 = r64.mean(0), (r64.var(0, unbiased=False) + 1e-5).rsqrt()
    del r64
    sc64 = gamma.to(F64) * rs64
    st = torch.stack([m64, rs64, sc64, beta.to(F64) - m64 * sc64]).float().contiguous()
    N = M // HW
    dOut = rnd(M, C, seed=75)
    fgate, fadd = torch.sigmoid(rnd(N, C, seed=76)), rnd(N, C, seed=77, scale=0.1)
    for frozen in (False, True):
        for act, with_se in ((0, False), (1, True)):
            r = raw.to(F64).requires_grad_(True)
            g64, b64 = gamma.to(F64).requires_grad_(True), beta.to(F64).requires_grad_(True)
            if frozen:
                y = F.batch_norm(r, st[0].to(F64), (1.0 / st[1].to(F64)) ** 2 - 1e-5, g64, b64, False, 0.0, 1e-5)
            else:
                y = F.batch_norm(r, None, None, g64, b64, True, 0.0, 1e-5)
            y = F.gelu(y) if act else y
            up = dOut.to(F64)
            if with_se:
                up = (up.view(N, HW, C) * fgate.to(F64)[:, None] + fadd.to(F64)[:, None]).view(M, C)
            y.backward(up)
            del y, up
            Pg, Pb = prefill((C,), 78, g64.grad.abs().max().item()), prefill((C,), 79, b64.grad.abs().max().item())
            dg, db = Pg.clone(), Pb.clone()
            kw = dict(fgate=fgate, fadd=fadd, rows_per_field=HW) if with_se else {}
            draw = dOut.clone() if with_se else nan_like((M, C))
            src = draw if with_se else dOut
            if frozen:
                ot.bn_bwd_frozen(src, raw, st, act, dg, db, out=draw, **kw)
            else:
                ot.bn_bwd(src, raw, st, gamma, act, dg, db, out=draw, **kw)
            torch.cuda.synchronize()
            e = dict(draw=rel_err(draw, r.grad), dgamma=rel_err(dg.double() - Pg.double(), g64.grad),
                     dbeta=rel_err(db.double() - Pb.double(), b64.grad))
            note(frozen=frozen, act=act, **e)
            # the existing rule of the 128 / 512-channel kernel (test_bn_act_bwd_colsum)
            assert e["draw"] < 2e-5 and e["dgamma"] < 1e-5 and e["dbeta"] < 1e-5, (frozen, act, e)
            del r, draw


# =========================================================================================== depthwise 3x3
@pytest.mark.parametrize("W", [16, 35, 259])
@pytest.mark.parametrize("C", [1024, 1536, 2048])
def test_dw3x3_wide(C, W):
    """the depthwise 3x3 of the training step at C = 1024, 1536, 2048 (512-channel slices over the grid): forward (scale 1,
    shift = bias) with its per-strip channel sums, data gradient (flipped taps), weight / bias gradient (accumulated), against
    float64 F.conv2d(groups=C).  Strips of 5 columns: W = 16, 35, 259 end on strips of 1, 5 and 4 columns."""
    ot = OT()
    N, H = 2, 7
    x, dY = rnd(N, C, H, W, seed=90), rnd(N, C, H, W, seed=91)
    w, b = rnd(C, 1, 3, 3, seed=92, scale=0.3), rnd(C, seed=93)
    xr, wr, br = (t.to(F64).requires_grad_(True) for t in (x, w, b))
    y64 = F.conv2d(xr, wr, br, padding=1, groups=C)
    y64.backward(dY.to(F64))
    x_cl, dY_cl = x.permute(0, 2, 3, 1).contiguous(), dY.permute(0, 2, 3, 1).contiguous()
    w9 = w.reshape(C, 9).t().contiguous()
    ones, zeros = torch.ones(C, device=DEV), torch.zeros(C, device=DEV)
    from vit_grid_model_b200 import _lib
    strips = _lib.load().vg_dw_strips(W)
    y, psum = nan_like((N, H, W, C)), nan_like((N, strips, C))
    call("vg_dw3x3_fwd", 1, x_cl.data_ptr(), w9.data_ptr(), ones.data_ptr(), b.data_ptr(), 0, y.data_ptr(), psum.data_ptr(), N, H, W, C)
    dx = nan_like((N, H, W, C))
    w9_flip = w9.flip(0).contiguous()
    call("vg_dw3x3_fwd", 1, dY_cl.data_ptr(), w9_flip.data_ptr(), ones.data_ptr(), zeros.data_ptr(), 0, dx.data_ptr(), None, N, H, W, C)
    ref_w9 = wr.grad.reshape(C, 9).t()
    Pw, Pb = prefill((9, C), 94, ref_w9.abs().max().item()), prefill((C,), 95, br.grad.abs().max().item())
    dw9, dbias = Pw.clone(), Pb.clone()
    ot.dw3x3_wgrad(x_cl, dY_cl, dw9, dbias)
    torch.cuda.synchronize()
    y_cl64 = y64.detach().permute(0, 2, 3, 1)
    ref_psum = torch.stack([y_cl64[:, :, 5 * s:5 * s + 5].sum((1, 2)) for s in range(strips)], dim=1)
    e = dict(y=rel_err(y, y_cl64), psum=rel_err(psum, ref_psum), dx=rel_err(dx.permute(0, 3, 1, 2), xr.grad),
             dw=rel_err(dw9.double() - Pw.double(), ref_w9), db=rel_err(dbias.double() - Pb.double(), br.grad))
    note(**e)
    # the existing rule of the 512-channel kernels (test_dw3x3_dgrad_and_wgrad): nine fp32 FMAs per output; fp32 sums over a
    # strip and then over the partials.  The strip sums add up to 35 outputs in fp32.
    assert e["y"] < 1e-6 and e["dx"] < 1e-6 and e["psum"] < 1e-5 and e["dw"] < 1e-5 and e["db"] < 1e-5, e


# =========================================================================================== squeeze-excite
@pytest.mark.parametrize("N,H,W,C", [(3, 14, 21, 2048), (1100, 7, 7, 2048), (48, 42, 35, 2048), (48, 42, 35, 1024),
                                     (1100, 7, 7, 1024)],
                         ids=["3-14-21", "1100-7-7", "48-42-35", "48-42-35-c1024", "1100-7-7-c1024"])
def test_squeeze_excite_wide(N, H, W, C):
    """maxvit.py:33-48 at C = 2048, se = 512 (512-channel networks) and C = 1024, se = 256 (256-channel networks): the gate
    with its saved intermediates on both branches of vg_se_gate_train_fwd (N <= 1024: field means + two dense-row passes, here
    also the 48-field fp32 inference chunk of BASELINE configs[4]; N = 1100: one block per field) and the backward (dW1, dW2
    accumulated, dmean written), from partial sums and intermediates derived in float64"""
    from vit_grid_model_b200 import _lib
    se = C // 4
    HW = H * W
    parts = _lib.load().vg_field_parts(HW)
    h3 = rnd(N, H, W, C, seed=100) + 0.5 * rnd(C, seed=101)
    dh4 = rnd(N, H, W, C, seed=102)
    W1, W2 = rnd(se, C, seed=103, scale=1 / math.sqrt(C)), rnd(C, se, seed=104, scale=4 / math.sqrt(se))
    rows = -(-HW // parts)
    h64, d64 = h3.view(N, HW, C).to(F64), dh4.view(N, HW, C).to(F64)
    psum = torch.stack([h64[:, k * rows:(k + 1) * rows].sum(1) for k in range(parts)], dim=1).float().contiguous()
    mean64 = h64.mean(1)
    hid64 = F.relu(mean64 @ W1.to(F64).t())
    gate64 = torch.sigmoid(hid64 @ W2.to(F64).t())
    gate, mean, hid = nan_like((N, C)), nan_like((N, C)), nan_like((N, se))
    call("vg_se_gate_train_fwd", psum.data_ptr(), N, parts, HW, W1.data_ptr(), W2.data_ptr(), C, se, gate.data_ptr(),
         mean.data_ptr(), hid.data_ptr())
    torch.cuda.synchronize()
    ef = dict(mean=rel_err(mean, mean64), hid=rel_err(hid, hid64), gate=rel_err(gate, gate64))
    mean32 = mean64.float()
    m = mean32.to(F64).requires_grad_(True)
    w1, w2 = W1.to(F64).requires_grad_(True), W2.to(F64).requires_grad_(True)
    hidr = F.relu(m @ w1.t())
    gr = torch.sigmoid(hidr @ w2.t())
    (h64 * gr[:, None, :] * d64).sum().backward()
    Pw1, Pw2 = prefill((se, C), 105, w1.grad.abs().max().item()), prefill((C, se), 106, w2.grad.abs().max().item())
    dW1, dW2 = Pw1.clone(), Pw2.clone()
    dmean = nan_like((N, C))
    work = torch.empty(N * ((parts + 1) * C + se), device=DEV)
    g32, hid32 = gr.detach().float().contiguous(), hidr.detach().float().contiguous()
    call("vg_se_bwd", dh4.data_ptr(), h3.data_ptr(), g32.data_ptr(), mean32.data_ptr(), hid32.data_ptr(), W1.data_ptr(),
         W2.data_ptr(), N, HW, C, se, dW1.data_ptr(), dW2.data_ptr(), dmean.data_ptr(), work.data_ptr(), work.numel())
    torch.cuda.synchronize()
    eb = dict(dmean=rel_err(dmean, m.grad / HW), dW1=rel_err(dW1.double() - Pw1.double(), w1.grad),
              dW2=rel_err(dW2.double() - Pw2.double(), w2.grad))
    note(**ef, **eb)
    # the existing rule of the 512-channel test (test_squeeze_excite_forward_and_backward): fp32 dot products of 2048 / 512 terms
    assert ef["mean"] < 1e-6 and ef["hid"] < 1e-5 and ef["gate"] < 1e-5, ef
    assert eb["dmean"] < 1e-5 and eb["dW1"] < 1e-5 and eb["dW2"] < 1e-5, eb


# =========================================================================================== the module
# (dim, depth, heads, dim_head): int depth = one stage at constant width; (1, 1, 1) = stages 128 -> 256 -> 512, both first
# layers widening the map (the last depth entry is dropped, as the reference's zip() does)
SHAPES = {"d256_h4_dh64": (256, 1, 4, 64), "d384_h6_dh64": (384, 1, 6, 64), "d512_h32_dh64_depth2": (512, 2, 32, 64),
          "tuple_128_256_512_dh32": (128, (1, 1, 1), 8, 32)}
N_FIELDS, H_MAP, W_MAP = 3, 14, 21


def _setup(shape, precision, seed=5, dropout=0.0):
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh = SHAPES[shape]
    sd = synth.make_state_dict(synth.maxvit_multistage_spec(dim, depth, 2, heads, dh, WIN, 4, 0.25, R_REG), seed=seed)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=WIN, num_register_tokens=R_REG,
               dropout=dropout)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().set_precision(precision)
    gen = torch.Generator().manual_seed(12)
    x = torch.randn(N_FIELDS, dim, H_MAP, W_MAP, generator=gen)
    cond = torch.randn(N_FIELDS, 2, generator=gen)
    dy = torch.randn(N_FIELDS, m.dim_out, H_MAP, W_MAP, generator=gen)
    return m, sd, x, cond, dy, heads, len(m.layers)


def _oracle(sd, x, cond, dy, heads, n_layers, training, monkeypatch=None, drop_masks=None):
    """float64 autograd through the oracle on the GPU -> (y, x.grad, cond.grad, {param: grad}, [(mean, unbiased var)] of every
    batch-statistic BatchNorm in call order)"""
    sd64 = {k: (v.to(DEV, F64).requires_grad_("running_" not in k) if v.is_floating_point() else v.to(DEV)) for k, v in sd.items()}
    x64, c64 = x.to(DEV, F64).requires_grad_(True), cond.to(DEV, F64).requires_grad_(True)
    stats = []
    if monkeypatch is not None:
        bn = F.batch_norm

        def recording(t, *a, **kw):                      # (input, running_mean, running_var, weight, bias, training, ...)
            if a[4]:
                d = t.detach()
                stats.append((d.mean((0, 2, 3)), d.var((0, 2, 3), unbiased=True)))
            return bn(t, *a, **kw)
        monkeypatch.setattr(mo.F, "batch_norm", recording)
    y = mo.maxvit_forward(x64, c64, sd64, depth=n_layers, heads=heads, window=WIN, num_reg=R_REG, training=training,
                          drop_masks=drop_masks)
    if monkeypatch is not None:
        monkeypatch.undo()
    y.backward(dy.to(DEV, F64))
    return y.detach(), x64.grad, c64.grad, {k: v.grad for k, v in sd64.items() if v.is_floating_point() and v.requires_grad}, stats


def _check_grads(pairs, fp32, G):
    """the bounds of test_maxvit_block_backward: relative L2 per tensor 2e-3 (fp32) / 6e-2 (bf16), and the rule of
    test_attention_dropout_forward_backward for dcond in bf16, 8e-2 -- two numbers per field, each the sum of the FiLM gradients of
    all tokens and channels, collect the rounding of the bf16 backward chain without averaging it away (measured on a B200: up to
    7.6e-2, the tuple-depth MaxViT in the eval() graph).  A conv bias in front of a batch-statistic BatchNorm has an analytically
    zero gradient: its rounding noise must stay far below the adjacent BatchNorm beta gradient (G: None in the frozen graph, where
    those biases have real gradients)"""
    bad, worst = [], 0.0
    for name, got, ref in pairs:
        g, rf = got.detach().to(DEV, F64), ref.to(DEV, F64)
        if G is not None and re.fullmatch(r"layers\.\d+\.0\.(fn\.)?[037]\.bias", name):
            beta = G[name[:-len("0.bias")] + str(int(name[-len("0.bias")]) + 1) + ".bias"].norm().item()
            if g.norm().item() > 1e-3 * beta:
                bad.append((name, g.norm().item(), beta))
            continue
        e = ((g - rf).norm() / max(rf.norm().item(), 1e-2)).item()
        if name == "dcond":
            e_dcond = e
        else:
            worst = max(worst, e)
        if e > (2e-3 if fp32 else (8e-2 if name == "dcond" else 6e-2)):
            bad.append((name, round(e, 5)))
    note(worst_l2=worst, dcond_l2=e_dcond)
    assert not bad, bad


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_maxvit_wide_train_step(shape, precision, monkeypatch):
    """MaxViT in train() mode through the public module: y, x.grad, cond.grad and every parameter gradient against float64
    autograd of the oracle (batch-statistic BatchNorm), the running buffers after the step (momentum 0.1, unbiased variance)
    and num_batches_tracked"""
    m, sd, x, cond, dy, heads, nl = _setup(shape, precision)
    m.train()
    oy, ogx, ogc, og, stats = _oracle(sd, x, cond, dy, heads, nl, True, monkeypatch)
    xg, cg = x.cuda().requires_grad_(True), cond.cuda().requires_grad_(True)
    y = m(xg, cg)
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    fp32 = precision == "fp32"
    ey = rel_err(y, oy)
    # the forward bound of test_maxvit_block_backward
    assert ey < (1e-4 if fp32 else 2e-2), ey
    named = dict(m.named_parameters())
    _check_grads([("dx", xg.grad, ogx), ("dcond", cg.grad, ogc)] + [(k, p.grad, og[k]) for k, p in named.items()], fp32,
                 {k: p.grad for k, p in named.items()})
    # running buffers: the BatchNorms in call order (layer by layer: 1, 4, 8); their inputs carry the forward error, so the
    # forward bound applies
    bns = [f"layers.{li}.0." + ("fn." if hasattr(m.layers[li][0], "fn") else "") + str(i) for li in range(nl) for i in (1, 4, 8)]
    assert len(stats) == len(bns)
    sdm = m.state_dict()
    er = 0.0
    for name, (mean, var) in zip(bns, stats):
        rm0, rv0 = sd[name + ".running_mean"].to(DEV, F64), sd[name + ".running_var"].to(DEV, F64)
        er = max(er, rel_err(sdm[name + ".running_mean"], 0.9 * rm0 + 0.1 * mean), rel_err(sdm[name + ".running_var"], 0.9 * rv0 + 0.1 * var))
        assert sdm[name + ".num_batches_tracked"].item() == sd[name + ".num_batches_tracked"].item() + 1
    note(y=ey, running=er)
    assert er < (1e-4 if fp32 else 2e-2), er


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_maxvit_wide_eval_input_grad(shape, precision):
    """the same graph in eval() mode when x requires grad: BatchNorm from the running buffers (frozen, nothing updated), no
    dropout even though the module's dropout is 0.1"""
    m, sd, x, cond, dy, heads, nl = _setup(shape, precision)
    m.eval()
    oy, ogx, ogc, og, _ = _oracle(sd, x, cond, dy, heads, nl, False)
    bufs = {k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k}
    xg, cg = x.cuda().requires_grad_(True), cond.cuda().requires_grad_(True)
    y = m(xg, cg)
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    assert all(torch.equal(v, m.state_dict()[k]) for k, v in bufs.items())
    fp32 = precision == "fp32"
    ey = rel_err(y, oy)
    note(y=ey)
    assert ey < (1e-4 if fp32 else 2e-2), ey
    _check_grads([("dx", xg.grad, ogx), ("dcond", cg.grad, ogc)] + [(k, p.grad, og[k]) for k, p in m.named_parameters()], fp32, None)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_maxvit_wide_attention_dropout(precision):
    """nn.Dropout at p = 0.25 on the attention probabilities and after to_out (maxvit.py:146,151) at 512 channels, 32 heads x 64:
    the un-fused path's masks exported through the test hook and fed to the oracle, so forward and every gradient must agree as
    without dropout (the bounds of test_attention_dropout_forward_backward)"""
    from vit_grid_model_b200 import train as tr
    p = 0.25
    m, sd, x, cond, dy, heads, nl = _setup("d512_h32_dh64_depth2", precision, dropout=p)
    m.train()
    dim = m.dim
    nwin = (H_MAP // WIN) * (W_MAP // WIN)
    seed, T = 123456789, tr.dropout_threshold(p)
    scale = 256.0 / (256 - T)
    masks = {}
    for li in range(nl):
        for ai in (1, 2):
            pm, om = OT().dropout_masks((seed, 2 * li + ai - 1, T), N_FIELDS * nwin, heads, dim)
            masks[(li, ai)] = (pm[:, :, :S_TOK, :S_TOK].to(F64) * scale, om[:, :S_TOK].to(F64) * scale)
    oy, ogx, ogc, og, _ = _oracle(sd, x, cond, dy, heads, nl, True, drop_masks=masks)
    xc, condc = x.permute(0, 2, 3, 1).contiguous().cuda(), cond.cuda()
    with torch.no_grad():
        yc, saved = tr.maxvit_train_forward(m, xc, condc, seed=seed)
        G = {k: torch.zeros_like(q) for k, q in m.named_parameters()}
        dcond = torch.zeros_like(condc)
        dxc = tr.maxvit_train_backward(m, saved, condc, dcond, dy.permute(0, 2, 3, 1).contiguous().cuda(), G, "")
    fp32 = precision == "fp32"
    ey = rel_err(yc.permute(0, 3, 1, 2), oy)
    note(y=ey)
    assert ey < (1e-4 if fp32 else 2e-2), ey
    _check_grads([("dx", dxc.permute(0, 3, 1, 2), ogx), ("dcond", dcond, ogc)] + [(k, G[k], og[k]) for k in G], fp32, G)
    with torch.no_grad():
        y2, _ = tr.maxvit_train_forward(m, xc, condc, seed=seed)
        y3, _ = tr.maxvit_train_forward(m, xc, condc, seed=seed + 1)
    assert torch.equal(yc, y2) and not torch.equal(yc, y3)
