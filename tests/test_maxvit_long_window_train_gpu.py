"""Training of MaxViT with windows of 65 .. 128 tokens (GPU), among them the reference's default window 8 with four register
tokens (S = 68): the 128-slot dropout counters, the forward kernels with dropout, both long-window core backward kernels (modes
0 and 2) against float64, and the module -- y, x.grad, cond.grad, every parameter gradient and the BatchNorm running buffers --
against float64 autograd through the oracle with the kernels' own dropout masks, in train() mode and in the frozen-BatchNorm
eval() graph.

Conventions (those of test_maxvit_wide_train_gpu.py):
  * every reference is float64, on the GPU
  * every output a kernel must write completely starts as NaN; every accumulated output starts from a random tensor P and
    `out - P` is compared with the reference
  * errors are relative to the largest reference entry (rel_err) unless stated; each bound not taken from an existing rule
    states the error measured on a B200 next to it
"""
import math
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle import maxvit_oracle as mo

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64, F32, BF16 = torch.float64, torch.float32, torch.bfloat16
FP32_TOL = 2e-5            # exact-fp32 outputs (test_maxvit_unfused_infer_gpu.FP32_TOL)
T_DROP = 26                # nn.Dropout(0.1): round(0.1 * 256)
# (win, R) -> S: 65, 68 (the reference default), 100, 128
LONG = {"S65_w8_R1": (8, 1), "S68_w8_R4": (8, 4), "S100_w10_R0": (10, 0), "S128_w11_R7": (11, 7)}


def O():
    from vit_grid_model_b200 import ops
    return ops


def OT():
    from vit_grid_model_b200 import ops_train
    return ops_train


def lib():
    from vit_grid_model_b200 import _lib
    return _lib


def call(name, *args):
    from vit_grid_model_b200.ops import _st
    lib().call(name, *args, _st())


def note(**kv):
    """one line per measurement (pytest -s shows them; the measured values in the comments below come from these lines)"""
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0].split("::")[-1]
    print("MEASURE", test, " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in kv.items()))


def rel_err(got, ref):
    """max |got - ref| / max |ref|, in float64 on the device"""
    got, ref = got.detach().to(DEV, F64), ref.detach().to(DEV, F64)
    assert not torch.isnan(got).any(), "NaN in the output: an entry was not written"
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, generator=g, device=DEV) * scale


def nan_like(shape, dtype=F32):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def prefill(shape, seed, scale=1.0):
    """the random P an accumulated output starts from, at 1/100 of the reference's largest entry"""
    return rnd(*shape, seed=seed, scale=0.01 * scale)


def geom(win, nwin_per_field):
    """(Hl, Wl) with 1, 6 or 15 windows per field"""
    X, Y = {1: (1, 1), 6: (2, 3), 15: (3, 5)}[nwin_per_field]
    return X * win, Y * win


# =========================================================================================== dropout counters
def np_drop_hash(seed, a, b):
    """vg_rng.cuh drop_hash in uint32 arithmetic"""
    M = np.uint64(0xFFFFFFFF)
    a, b = np.asarray(a, np.uint64), np.asarray(b, np.uint64)
    x = (a * np.uint64(0x9E3779B1) + b * np.uint64(0x85EBCA77) + np.uint64(seed)) & M
    x ^= x >> np.uint64(16); x = (x * np.uint64(0x85EBCA6B)) & M
    x ^= x >> np.uint64(13); x = (x * np.uint64(0xC2B2AE35)) & M
    x ^= x >> np.uint64(16)
    return x


def np_masks(seed, salt, T, n_windows, heads, C, row_stride, head_stride):
    """the masks restated: row id wdx * row_stride + i, probability group salt * 8192 + h * head_stride + g, to_out group
    salt * 8192 + 4096 + g; byte k of a hash is key / channel 4g + k, kept when >= T"""
    slots = row_stride
    w = np.arange(n_windows, dtype=np.uint64)[:, None, None, None]
    h = np.arange(heads, dtype=np.uint64)[None, :, None, None]
    i = np.arange(slots, dtype=np.uint64)[None, None, :, None]
    j = np.arange(slots, dtype=np.uint64)[None, None, None, :]
    rid = w * np.uint64(row_stride) + i
    grp = np.uint64(salt * 8192) + h * np.uint64(head_stride) + j // np.uint64(4)
    pm = ((np_drop_hash(seed, rid, grp) >> (np.uint64(8) * (j % np.uint64(4)))) & np.uint64(255)) >= T
    c = np.arange(C, dtype=np.uint64)[None, None, :]
    rid_o = np.arange(n_windows, dtype=np.uint64)[:, None, None] * np.uint64(row_stride) + np.arange(slots, dtype=np.uint64)[None, :, None]
    om = ((np_drop_hash(seed, rid_o, np.uint64(salt * 8192 + 4096) + c // np.uint64(4)) >> (np.uint64(8) * (c % np.uint64(4))))
          & np.uint64(255)) >= T
    return pm.astype(np.uint8), om.astype(np.uint8)


def test_dropout_mask_counters():
    """vg_dropout_mask_debug against the formula: slots = 64 keeps the ids (64, 16) and is the default call; slots = 128 uses
    (128, 32).  The keep rate is 1 - T/256, and token 64 of window w no longer shares the counter of token 0 of window w + 1"""
    seed, salt, T, nw, heads, C = 987654321, 3, T_DROP, 6, 5, 128
    pm64, om64 = OT().dropout_masks((seed, salt, T), nw, heads, C)
    pm64b, om64b = OT().dropout_masks((seed, salt, T), nw, heads, C, slots=64)
    pm128, om128 = OT().dropout_masks((seed, salt, T), nw, heads, C, slots=128)
    torch.cuda.synchronize()
    assert torch.equal(pm64, pm64b) and torch.equal(om64, om64b)
    rp, ro = np_masks(seed, salt, T, nw, heads, C, 64, 16)
    assert np.array_equal(pm64.cpu().numpy(), rp) and np.array_equal(om64.cpu().numpy(), ro)
    rp, ro = np_masks(seed, salt, T, nw, heads, C, 128, 32)
    assert np.array_equal(pm128.cpu().numpy(), rp) and np.array_equal(om128.cpu().numpy(), ro)
    keep = dict(prob=pm128.double().mean().item(), out=om128.double().mean().item())
    note(**keep)
    assert all(abs(v - (1 - T / 256)) < 5e-3 for v in keep.values()), keep
    for w in range(nw - 1):
        assert not torch.equal(pm128[w, :, 64], pm128[w + 1, :, 0]) and not torch.equal(om128[w, 64], om128[w + 1, 0])
    with pytest.raises(lib().VitGridError, match="slots"):
        OT().dropout_masks((seed, salt, T), 1, 1, C, slots=96)
    with pytest.raises(lib().VitGridError, match="heads"):
        OT().dropout_masks((seed, salt, T), 1, 129, C, slots=128)


def prob_masks(drop, n_windows, heads, S):
    """(Nw, heads, S, S) float64 probability masks * scale of a window of S > 64 tokens"""
    pm, _ = OT().dropout_masks(drop, n_windows, heads, 128, slots=128)
    return pm[:, :, :S, :S].to(F64) * (256.0 / (256 - drop[2]))


# =========================================================================================== forward kernels
def _core_operands(N, Hl, Wl, win, R, heads, dh, seed):
    S, nwin = R + win * win, (Hl // win) * (Wl // win)
    inner = heads * dh
    qkv = rnd(N * nwin * S, 3 * inner, seed=seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    qg = 0.5 + torch.rand(inner, device=DEV, generator=g)
    kg = 0.5 + torch.rand(inner, device=DEV, generator=g)
    bt = rnd((2 * win - 1) ** 2 + 1, heads, seed=seed + 2)
    return qkv, qg, kg, bt


def _core_fwd_ref(qkv, qg, kg, bt, S, win, R, heads, dh, pmask):
    """float64 maxvit.py:189-213 with the probability dropout -> [rows][heads*dh]"""
    nw = qkv.shape[0] // S
    x = qkv.to(F64).view(nw, S, 3, heads, dh).permute(2, 0, 3, 1, 4)
    rs = math.sqrt(dh)
    qh = F.normalize(x[0], dim=-1) * rs * qg.to(F64).view(heads, 1, dh)
    kh = F.normalize(x[1], dim=-1) * rs * kg.to(F64).view(heads, 1, dh)
    P = torch.softmax(qh @ kh.transpose(-1, -2) + bt.to(F64)[mo.rel_pos_indices(win, R).to(DEV)].permute(2, 0, 1), dim=-1)
    return ((P * pmask) @ x[2]).permute(0, 2, 1, 3).reshape(nw * S, heads * dh)


@pytest.mark.parametrize("dh", [32, 64])
@pytest.mark.parametrize("case", list(LONG))
def test_attn_core_fwd_long_dropout(case, dh):
    """vg_attn_core_fwd with dropout at S = 65 .. 128 (the SIMT kernel, 128-slot masks) against float64 with the exported masks;
    codes 2 and 4 with dropout run the same kernel: bit-equal to code 1"""
    win, R = LONG[case]
    S, heads, N = R + win * win, 8, 2
    Hl, Wl = geom(win, 6)
    nwin = 6
    drop = (20261022, 5, T_DROP)
    qkv, qg, kg, bt = _core_operands(N, Hl, Wl, win, R, heads, dh, seed=11)
    out = nan_like((qkv.shape[0], heads * dh))
    O().attn_core(qkv, qg, kg, bt, N, Hl, Wl, win, R, heads, dh, out=out, drop=drop)
    ref = _core_fwd_ref(qkv, qg, kg, bt, S, win, R, heads, dh, prob_masks(drop, N * nwin, heads, S))
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    note(rel=e)
    assert e <= FP32_TOL, e                 # the fp32 rule of test_attn_core_simt_dropout (measured on a B200: 1.8e-6 at most)
    for kw in (dict(x3=True), dict(tf32=True)):
        assert torch.equal(out, O().attn_core(qkv, qg, kg, bt, N, Hl, Wl, win, R, heads, dh, drop=drop, **kw))


def test_attn_core_fwd_long_rejects():
    """S = 129 is too long with or without dropout; dropout at S > 64 takes at most 128 heads"""
    qkv, qg, kg, bt = _core_operands(1, 11, 11, 11, 8, 4, 32, seed=13)
    with pytest.raises(lib().VitGridError, match="too long"):
        O().attn_core(qkv, qg, kg, bt, 1, 11, 11, 11, 8, 4, 32, drop=(1, 0, T_DROP))
    z = torch.zeros(4, device=DEV)
    with pytest.raises(lib().VitGridError, match="heads"):
        call("vg_attn_core_fwd", 1, z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), 1, 8, 8, 8, 4, 129, 32, z.data_ptr(),
             1, 0, T_DROP)


@pytest.mark.parametrize("case", ["S68_w8_R4", "S128_w11_R7"])
def test_attn_out_long_dropout(case):
    """vg_attn_out_fwd with to_out dropout at S = 68 and 128 (block partition, register rows to reg_out): the 128-slot out-mask
    fed to the float64 reference; x_out and reg_out start as NaN"""
    win, R = LONG[case]
    S, N, C, inner = R + win * win, 2, 256, 512
    Hl, Wl = geom(win, 6)
    nwin = 6
    drop = (777, 5, T_DROP)
    attn, W = rnd(N * nwin * S, inner, seed=21), rnd(C, inner, seed=22, scale=1 / math.sqrt(inner))
    x_in, reg = rnd(N, Hl, Wl, C, seed=23), rnd(R, C, seed=24)
    x_out = nan_like(x_in.shape)
    x_out, reg_out = O().attn_out(attn, W, x_in, reg, win, R, False, True, x_out=x_out, drop=drop)
    om = OT().dropout_masks(drop, N * nwin, 1, C, slots=128)[1][:, :S].to(F64) * (256.0 / (256 - T_DROP))
    torch.cuda.synchronize()
    proj = (attn.to(F64) @ W.to(F64).t()).view(N, nwin, S, C) * om.view(N, nwin, S, C)
    x_ref = x_in.to(F64).reshape(N, Hl * Wl, C).clone()
    pix = mo.block_pixel_index(Hl, Wl, win).reshape(-1).to(DEV)
    x_ref[:, pix] += proj[:, :, R:].reshape(N, nwin * win * win, C)
    reg_ref = proj[:, :, :R] + reg.to(F64)[None, None]
    # the fp32 rule of test_attn_out_dropout: FP32_TOL of the largest projection entry plus one rounding of the residual add
    # (measured on a B200: 0.052 of that allowance at most)
    fm = proj.abs().max().item()
    e = dict(x=((x_out.to(F64).view(N, Hl * Wl, C) - x_ref).abs() / (FP32_TOL * fm + 2.0 ** -24 * x_ref.abs())).max().item(),
             reg=((reg_out.to(F64).view(N, nwin, R, C) - reg_ref).abs() / (FP32_TOL * fm + 2.0 ** -24 * reg_ref.abs())).max().item())
    note(**e)
    assert not torch.isnan(x_out).any() and not torch.isnan(reg_out).any()
    assert e["x"] <= 1.0 and e["reg"] <= 1.0, e


def test_attn_out_bwd_gather_long_dropout():
    """vg_attn_out_bwd_gather at S = 68 with the to_out mask: window rows gather dx_out, register rows dreg * reg_scale, times
    the 128-slot mask * scale -- one fp32 product per element (of fp32 operands), so bit-equal to the float64 product rounded
    to fp32"""
    win, R = LONG["S68_w8_R4"]
    S, N, C = R + win * win, 3, 256
    Hl, Wl = geom(win, 6)
    nwin = 6
    drop = (4242, 7, T_DROP)
    dx_out, dreg = rnd(N, Hl, Wl, C, seed=31), rnd(N, R, C, seed=32)
    reg_scale = 1.0 / nwin
    dproj = OT().attn_out_bwd_gather(dx_out, dreg, reg_scale, win, R, False, drop=drop)
    scale32 = torch.tensor(256.0 / (256 - T_DROP), dtype=F32).item()       # the kernel's scale is an fp32 number
    om = OT().dropout_masks(drop, N * nwin, 1, C, slots=128)[1][:, :S].to(F64) * scale32
    torch.cuda.synchronize()
    pix = mo.block_pixel_index(Hl, Wl, win).reshape(-1).to(DEV)
    g = torch.empty(N, nwin, S, C, dtype=F64, device=DEV)
    g[:, :, R:] = dx_out.to(F64).view(N, Hl * Wl, C)[:, pix].view(N, nwin, win * win, C)
    g[:, :, :R] = (dreg.float() * reg_scale).to(F64)[:, None]
    ref = (g.view(N * nwin, S, C) * om).float()
    assert torch.equal(dproj.view(N * nwin, S, C), ref)


# =========================================================================================== core backward
def _core_bwd_ref(qkv, datt, qg, kg, bt, S, win, R, heads, D, pmask, bf16_ops):
    """float64 backward of maxvit.py:189-213 on the [rows][3 inner] layout (test_maxvit_wide_train_gpu._core_bwd_ref at any
    window).  bf16_ops: round where the mode-2 kernels round -- qh, kh, v, dO to bf16, P' = P mask and dS to bf16 in front of
    the products, the unit vectors of the RMSNorm backward taken from the rounded qh, kh; the bias gradient sums the unrounded dS.
    -> dqkv [rows][3 inner], dq_gamma, dk_gamma (heads*D), dbias (table, heads)"""
    nw, H = qkv.shape[0] // S, heads
    x = qkv.to(F64).view(nw, S, 3, H, D).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    dO = datt.to(F64).view(nw, S, H, D).permute(0, 2, 1, 3)
    rnd16 = (lambda t: t.to(BF16).to(F64)) if bf16_ops else (lambda t: t)
    inv_q = 1.0 / q.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    inv_k = 1.0 / k.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    rs = math.sqrt(D)
    gq = (torch.tensor(rs, dtype=F32, device=DEV) * qg).to(F64).view(H, 1, D) if bf16_ops else rs * qg.to(F64).view(H, 1, D)
    gk = (torch.tensor(rs, dtype=F32, device=DEV) * kg).to(F64).view(H, 1, D) if bf16_ops else rs * kg.to(F64).view(H, 1, D)
    qh, kh = rnd16(q * inv_q * gq), rnd16(k * inv_k * gk)
    vb, dOb = rnd16(v), rnd16(dO)
    idx = mo.rel_pos_indices(win, R).to(DEV)
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
    dbias.index_add_(0, idx.reshape(-1), dS.sum(0).permute(1, 2, 0).reshape(S * S, H))
    dqkv = torch.stack([dq, dk, dv]).permute(1, 3, 0, 2, 4).reshape(nw * S, 3 * H * D)
    return dqkv, dqg, dkg, dbias


# mode 0 (exact fp32): the existing fp32 rule of test_attn_core_bwd_dh64, 1e-4 of the largest reference entry (measured on an
# NVIDIA B200 at 1000 W: 3.6e-6 at most).  Mode 2 against the bf16-rounding reference: the bounds of test_attn_core_bwd_dh64
# (64-key kernel); the worst of the 48 long-window cases measured on the same card: dqkv 2.7e-3, dq_gamma 7.9e-4, dk_gamma
# 8.3e-4, dbias 1.5e-3
CORE_TOL = {0: dict(dqkv=1e-4, dq_gamma=1e-4, dk_gamma=1e-4, dbias=1e-4),
            2: dict(dqkv=8e-3, dq_gamma=4e-3, dk_gamma=3e-3, dbias=2.5e-3)}


def _run_core_bwd(case, dh, mode, T, nwin, heads=8, N=2, seed=3):
    win, R = LONG[case]
    S = R + win * win
    Hl, Wl = geom(win, nwin)
    inner = heads * dh
    rows = N * nwin * S
    g = torch.Generator(device=DEV).manual_seed(seed)
    qkv = torch.randn(rows, 3 * inner, device=DEV, generator=g)
    datt = torch.randn(rows, inner, device=DEV, generator=g)
    qg = 1 + 0.2 * torch.randn(inner, device=DEV, generator=g)
    kg = 1 + 0.2 * torch.randn(inner, device=DEV, generator=g)
    bt = 0.5 * torch.randn((2 * win - 1) ** 2 + 1, heads, device=DEV, generator=g)
    drop = (4242, 1, T)
    pmask = prob_masks(drop, N * nwin, heads, S) if T else None
    ref = _core_bwd_ref(qkv, datt, qg, kg, bt, S, win, R, heads, dh, pmask, bf16_ops=mode == 2)
    P = [prefill(t.shape, 130 + i, r.abs().max().item()) for i, (t, r) in enumerate(((qg, ref[1]), (kg, ref[2]), (bt, ref[3])))]
    dqg, dkg, dbt = (p.clone() for p in P)
    dqkv = nan_like(qkv.shape)
    call("vg_attn_core_bwd", qkv.data_ptr(), datt.data_ptr(), qg.data_ptr(), kg.data_ptr(), bt.data_ptr(), N, Hl, Wl, win, R,
         heads, dh, dqkv.data_ptr(), dqg.data_ptr(), dkg.data_ptr(), dbt.data_ptr(), mode, None, drop[0], drop[1], drop[2])
    torch.cuda.synchronize()
    return dict(dqkv=rel_err(dqkv, ref[0]), dq_gamma=rel_err(dqg.double() - P[0].double(), ref[1]),
                dk_gamma=rel_err(dkg.double() - P[1].double(), ref[2]), dbias=rel_err(dbt.double() - P[2].double(), ref[3]))


@pytest.mark.parametrize("nwin", [1, 6, 15])
@pytest.mark.parametrize("T", [0, T_DROP])
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("dh", [32, 64])
@pytest.mark.parametrize("case", list(LONG))
def test_attn_core_bwd_long(case, dh, mode, T, nwin):
    """vg_attn_core_bwd at S = 65, 68, 100 and 128: mode 0 (exact-fp32 SIMT, resident keys and streamed query blocks) and mode 2
    (bf16 mma.sync on fp32 tensors, 8 warps, keys in two halves), dim_head 32 and 64, without and with the probability dropout
    mask (128 slots, read back through vg_dropout_mask_debug), 1, 6 and 15 windows per field.  dqkv written (NaN prefill),
    dq_gamma, dk_gamma and the bias table accumulated onto non-zero values"""
    e = _run_core_bwd(case, dh, mode, T, nwin)
    note(**e)
    bad = {k: v for k, v in e.items() if not v < CORE_TOL[mode][k]}
    assert not bad, bad


def test_attn_core_bwd_long_rejects():
    """S = 129 in modes 0 and 2; dropout at S > 64 with 129 heads; mode 3 (the tcgen05 kernel) keeps S <= 64; att_out needs
    S <= 64"""
    z = torch.zeros(64, device=DEV)
    zp = z.data_ptr()

    def run(win, R, heads, dh, mode, T, att=None):
        call("vg_attn_core_bwd", zp, zp, zp, zp, zp, 1, win, win, win, R, heads, dh, zp, zp, zp, zp, mode, att, 1, 0, T)
    for mode in (0, 2):
        with pytest.raises(lib().VitGridError, match="sequence 129 > 128"):
            run(11, 8, 4, 32, mode, 0)
        with pytest.raises(lib().VitGridError, match="heads"):
            run(8, 4, 129, 32, mode, T_DROP)
    with pytest.raises(lib().VitGridError, match="sequence 68 > 64"):
        run(8, 4, 4, 32, 3, 0)
    with pytest.raises(lib().VitGridError, match="att_out"):
        run(8, 4, 4, 32, 2, 0, att=zp)


# =========================================================================================== the module
# (dim, depth, heads, dim_head, window, registers): the reference defaults (dim 128, depth 2, 32 x 32, window 8, 4 registers);
# 256 channels at 4 x 64; a tuple-depth stage 128 -> 256 (its first layer widens the map); window 11 with 7 registers (S = 128)
SHAPES = {"default_d128_depth2": (128, 2, 32, 32, 8, 4), "d256_h4_dh64_w8": (256, 1, 4, 64, 8, 4),
          "tuple_128_256_w8": (128, (2, 1), 8, 32, 8, 4), "d128_h4_dh64_w11_R7": (128, 1, 4, 64, 11, 7)}
N_FIELDS = 3


def _setup(shape, precision, seed=5):
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh, win, R = SHAPES[shape]
    sd = synth.make_state_dict(synth.maxvit_multistage_spec(dim, depth, 2, heads, dh, win, 4, 0.25, R), seed=seed)
    kw = {} if shape.startswith("default") else dict(heads=heads, dim_head=dh, vit_window_size=win, num_register_tokens=R)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, **kw)          # every other argument at its reference default (dropout 0.1)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().set_precision(precision)
    Hl, Wl = (16, 24) if win == 8 else (22, 33)
    gen = torch.Generator().manual_seed(12)
    x = torch.randn(N_FIELDS, dim, Hl, Wl, generator=gen)
    cond = torch.randn(N_FIELDS, 2, generator=gen)
    dy = torch.randn(N_FIELDS, m.dim_out, Hl, Wl, generator=gen)
    return m, sd, x, cond, dy


def _oracle(m, sd, x, cond, dy, training, monkeypatch=None, drop_masks=None):
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
    y = mo.maxvit_forward(x64, c64, sd64, depth=len(m.layers), heads=m.heads, window=m.vit_window_size,
                          num_reg=m.num_register_tokens, training=training, drop_masks=drop_masks)
    if monkeypatch is not None:
        monkeypatch.undo()
    y.backward(dy.to(DEV, F64))
    return y.detach(), x64.grad, c64.grad, {k: v.grad for k, v in sd64.items() if v.is_floating_point() and v.requires_grad}, stats


def _check_grads(pairs, fp32, G):
    """the bounds of test_maxvit_wide_train_gpu._check_grads: relative L2 per tensor 2e-3 (fp32) / 6e-2 (bf16), dcond in bf16
    8e-2; a conv bias in front of a batch-statistic BatchNorm (analytically zero gradient) must stay far below the adjacent
    BatchNorm beta gradient (G: None in the frozen graph)"""
    bad, worst, e_dcond = [], 0.0, 0.0
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


def _train_masks(m, seed, n_windows):
    """the kernels' masks of one training step (salt 2 li + 0 / 1 for block / grid attention), 128 slots, as the oracle's
    drop_masks"""
    S = m.num_register_tokens + m.vit_window_size ** 2
    T = 26
    scale = 256.0 / (256 - T)
    masks = {}
    for li in range(len(m.layers)):
        C = m.layers[li][1].to_out[0].weight.shape[0]
        for ai in (1, 2):
            pm, om = OT().dropout_masks((seed, 2 * li + ai - 1, T), n_windows, m.heads, C, slots=128)
            masks[(li, ai)] = (pm[:, :, :S, :S].to(F64) * scale, om[:, :S].to(F64) * scale)
    return masks


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_maxvit_long_window_train_step(shape, precision, monkeypatch):
    """MaxViT in train() mode through the public module with nn.Dropout(0.1) on: the kernels' masks fed to the float64 oracle;
    y, x.grad, cond.grad and every parameter gradient, the running buffers after the step and num_batches_tracked.  The same
    dropout seed gives the same bits, the next seed another output"""
    from vit_grid_model_b200 import train as tr
    m, sd, x, cond, dy = _setup(shape, precision)
    assert m.num_register_tokens + m.vit_window_size ** 2 > 64
    m.train()
    s0 = 1234567
    seed = (s0 * 1103515245 + 12345) & 0x7FFFFFFF                # MaxViT.next_dropout_seed after _dropout_state = s0
    assert tr.dropout_threshold(0.1) == 26
    nwin = (x.shape[2] // m.vit_window_size) * (x.shape[3] // m.vit_window_size)
    masks = _train_masks(m, seed, N_FIELDS * nwin)
    oy, ogx, ogc, og, stats = _oracle(m, sd, x, cond, dy, True, monkeypatch, drop_masks=masks)
    m._dropout_state = s0
    xg, cg = x.cuda().requires_grad_(True), cond.cuda().requires_grad_(True)
    y = m(xg, cg)
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    fp32 = precision == "fp32"
    ey = rel_err(y, oy)
    # the forward bound of test_maxvit_block_backward (measured on a B200: 5.1e-3 at most, bf16; gradients: worst relative L2
    # 2.3e-2, dcond 4.0e-2; running buffers 2.1e-3)
    assert ey < (1e-4 if fp32 else 2e-2), ey
    named = dict(m.named_parameters())
    _check_grads([("dx", xg.grad, ogx), ("dcond", cg.grad, ogc)] + [(k, p.grad, og[k]) for k, p in named.items()], fp32,
                 {k: p.grad for k, p in named.items()})
    nl = len(m.layers)
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
    with torch.no_grad():
        m._dropout_state = s0
        y2 = m(x.cuda(), cond.cuda())
        y3 = m(x.cuda(), cond.cuda())
    assert torch.equal(y.detach(), y2) and not torch.equal(y2, y3)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_maxvit_long_window_eval_input_grad(shape, precision):
    """the same networks in eval() mode when x requires grad: BatchNorm from the running buffers (frozen, nothing updated), no
    dropout even though the module's dropout is 0.1"""
    m, sd, x, cond, dy = _setup(shape, precision)
    m.eval()
    oy, ogx, ogc, og, _ = _oracle(m, sd, x, cond, dy, False)
    bufs = {k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k}
    xg, cg = x.cuda().requires_grad_(True), cond.cuda().requires_grad_(True)
    y = m(xg, cg)
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    assert all(torch.equal(v, m.state_dict()[k]) for k, v in bufs.items())
    fp32 = precision == "fp32"
    ey = rel_err(y, oy)
    note(y=ey)
    # the bounds of test_maxvit_wide_eval_input_grad (measured on a B200: y 6.8e-3, worst relative L2 3.4e-2, dcond 4.6e-2, bf16)
    assert ey < (1e-4 if fp32 else 2e-2), ey
    _check_grads([("dx", xg.grad, ogx), ("dcond", cg.grad, ogc)] + [(k, p.grad, og[k]) for k, p in m.named_parameters()], fp32, None)
