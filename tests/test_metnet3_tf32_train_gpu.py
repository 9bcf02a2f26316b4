"""Training MetNet3 in the 'tf32_conv' precision (fp32 storage, tf32 convolutions, exact-fp32 MaxViT training kernels) at 128,
256, 384 and 512 channels (GPU).

Kernels at the wide widths against float64: the wide conv block's training forward (vg_conv3x3_ln_wide_train_fwd: out, xhat,
rstd, ReLU mask), the wide stem finish (vg_stem_finish_wide_train_fwd), the wide Block backward (vg_conv_ln_bwd_wide,
vg_conv_ln_param_grads_wide), head backward / lead-time sum / per-field sum / ConvTranspose gather at C > 128, and the tf32
3x3 data / weight gradients with nine taps.  Written outputs are prefilled with NaN, accumulated ones with nonzero values.
Module: one training step of MetNet3 against float64 autograd through the oracle (prediction, every parameter gradient per
tensor, the MaxViT BatchNorm running buffers against the oracle's batch statistics), x.grad and every parameter gradient in
train() and eval() mode, smoke runs and the precisions that stay unbuilt.
Every bound is at most 4x the value measured on a B200 (power limit 1000 W), which is given beside it."""
import os
import re
import sys

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import synth
from oracle import maxvit_oracle as mo
from oracle.metnet3_oracle import metnet3_forward

pytestmark = pytest.mark.gpu

F64 = torch.float64
DEV = "cuda"
WIDTHS = (256, 384, 512)
# a 384-channel network (6 x 64 heads) and the configs[4] head layout at 512 channels with three input time steps
CFG_WIDE384 = synth.GridConfig(T=3, C=24, H=26, W=25, dim=384, L=2, heads=6, dim_head=64)
CFG_WIDE512_T3 = synth.GridConfig(T=3, C=24, H=26, W=25, dim=512, L=2, heads=32, dim_head=64)
MODULE_CFGS = {128: synth.CFG_SMALL128, 256: synth.CFG_WIDE256, 384: CFG_WIDE384, 512: CFG_WIDE512_T3}


def note(**kv):
    """measured values (printed with -s) for the bounds' comments"""
    print("MEASURED", kv)


def o():
    from vit_grid_model_b200 import ops
    return ops


def call(name, *args):
    from vit_grid_model_b200 import _lib
    _lib.call(name, *args, torch.cuda.current_stream().cuda_stream)


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def rnd(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=gen(seed), device=DEV) * scale


def rel(got, ref):
    g, r = got.double(), ref.double()
    return ((g - r).abs().max() / r.abs().max().clamp_min(1e-30)).item()


def tf32(t):
    """truncate fp32 to the tf32 operand the tensor cores read (the low 13 mantissa bits dropped)"""
    return (t.float().contiguous().view(torch.int32) & -8192).view(torch.float32)


def pg_nan(N, HP, WP, C):
    return torch.full((o().pg_pixels(N, HP, WP), C), float("nan"), device=DEV)


def pg(x):
    return o().pg_from_nchw(x, torch.float32)


def unpg(buf, N, HP, WP):
    return o().pg_to_nchw(buf, N, HP, WP)


def pad_mask(N, HP, WP):
    """True at the PG positions that are pads"""
    m = torch.ones(o().pg_pixels(N, HP, WP), dtype=torch.bool, device=DEV)
    inner = m[:N * (HP + 1) * (WP + 1)].view(N, HP + 1, WP + 1)[:, 1:, 1:]
    inner.fill_(False)
    return m


def mask_bits(z):
    """(N,C,H,W) bool -> (N,H,W,C/32) int32 words, bit c%32 of word c/32"""
    N, C, H, W = z.shape
    b = z.permute(0, 2, 3, 1).reshape(N, H, W, C // 32, 32).long()
    w = (b << torch.arange(32, device=DEV)).sum(-1)
    return (w & 0xFFFFFFFF).to(torch.int64)


def pg_words(words, N, HP, WP):
    """kernel mask [q][C/32] int32 -> (N,HP,WP,C/32) int64 words of the frame pixels"""
    K = words.shape[1]
    v = words.view(N * (HP + 1) + 1, WP + 1, K)[:N * (HP + 1)].view(N, HP + 1, WP + 1, K)[:, 1:, 1:]
    return v.long() & 0xFFFFFFFF


# ------------------------------------------------------------------------------------------ wide conv block, training forward
FWD_GEOMS = {"1x14x14": (1, 14, 14), "2x84x70": (2, 84, 70), "wp78": (2, 14, 78), "wp79": (2, 13, 79)}


def _conv_ln_ref(x, w, bias, g, b, eps, film, res, dtype):
    """float64 reference of the Block (metnet3.py:110-126): -> out, xhat, rstd, pre-activation z"""
    if dtype == 2:
        x, w = tf32(x), tf32(w)
    v = F.conv2d(x.double(), w.double(), padding=1) + bias.double().view(1, -1, 1, 1)
    mean = v.mean(1, keepdim=True)
    var = (v - mean).pow(2).mean(1, keepdim=True)
    rstd = var.clamp_min(eps).rsqrt()
    xhat = (v - mean) * rstd
    z = xhat * g.double().view(1, -1, 1, 1) + b.double().view(1, -1, 1, 1)
    if film is not None:
        C = x.shape[1]
        z = z * (film[:, :C].double().view(-1, C, 1, 1) + 1) + film[:, C:].double().view(-1, C, 1, 1)
    y = z.clamp_min(0)
    if res is not None:
        y = y + res.double()
    return y, xhat, rstd[:, 0], z


@pytest.mark.parametrize("dtype", [1, 2])
@pytest.mark.parametrize("variant", ["film", "res"])
@pytest.mark.parametrize("geom", list(FWD_GEOMS))
@pytest.mark.parametrize("C", (128,) + WIDTHS)
def test_wide_train_fwd(C, geom, variant, dtype):
    N, HP, WP = FWD_GEOMS[geom]
    _wide_train_fwd_case(C, N, HP, WP, variant, dtype)


def test_wide_train_fwd_518():
    _wide_train_fwd_case(256, 1, 518, 518, "film", 2)


def _wide_train_fwd_case(C, N, HP, WP, variant, dtype):
    from vit_grid_model_b200.metnet3 import _pack_conv3x3
    eps = 1e-5
    x = rnd(N, C, HP, WP, seed=C + HP)
    x[-1, :, :HP // 2] = 0.0                         # the conv output of these rows is the constant bias: variance clamp
    w = rnd(C, C, 3, 3, seed=2, scale=(C * 9) ** -0.5)
    bias = torch.full((C,), 0.1, device=DEV)
    g, b = 1 + 0.2 * rnd(C, seed=3), 0.1 * rnd(C, seed=4)
    film = 0.5 * rnd(N, 2 * C, seed=5) if variant == "film" else None
    res = rnd(N, C, HP, WP, seed=6) if variant == "res" else None
    xp = pg(x)
    Q = xp.shape[0]
    out, xhat = pg_nan(N, HP, WP, C), pg_nan(N, HP, WP, C)
    copy = pg_nan(N, HP, WP, C) if variant == "res" else None
    rstd = torch.full((Q,), float("nan"), device=DEV)
    mask = torch.full((Q, C // 32), -1, dtype=torch.int32, device=DEV)
    scratch = torch.empty(Q * C * (2 if dtype == 1 else 1), device=DEV)
    Wt = _pack_conv3x3(w, torch.float32)
    resp = pg(res) if res is not None else None
    call("vg_conv3x3_ln_wide_train_fwd", dtype, xp.data_ptr(), C, Wt.data_ptr(), bias.data_ptr(), g.data_ptr(), b.data_ptr(), eps,
         o()._p(film), o()._p(resp), 0, out.data_ptr(), o()._p(copy), xhat.data_ptr(), rstd.data_ptr(), mask.data_ptr(), N, HP, WP,
         scratch.data_ptr(), scratch.numel())
    torch.cuda.synchronize()
    y, xh, rs, z = _conv_ln_ref(x, w, bias, g, b, eps, film, res, dtype)
    pads = pad_mask(N, HP, WP)
    for t in (out, xhat):
        assert (t[pads] == 0).all()
    assert (rstd[pads] == 0).all() and (mask[pads] == 0).all()
    e_out, e_xh = rel(unpg(out, N, HP, WP), y), rel(unpg(xhat, N, HP, WP), xh)
    rs_k = rstd[:N * (HP + 1) * (WP + 1)].view(N, HP + 1, WP + 1)[:, 1:, 1:]
    e_rs = rel(rs_k, rs)
    if copy is not None:
        assert torch.equal(copy, out)
    assert torch.isclose(rs_k[-1, :HP // 2 - 1], torch.tensor(eps ** -0.5, device=DEV), rtol=1e-6).all()   # clamped rows
    # mask: bit-exact wherever the pre-activation is not within rounding of 0
    safe = (z.abs() > 1e-4 * z.abs().max()).permute(0, 2, 3, 1)
    got = pg_words(mask, N, HP, WP)
    gb = ((got.unsqueeze(-1) >> torch.arange(32, device=DEV)) & 1).reshape(N, HP, WP, C).bool()
    ref = (z > 0).permute(0, 2, 3, 1)
    assert (gb[safe] == ref[safe]).all()
    note(test="wide_train_fwd", C=C, N=N, HP=HP, WP=WP, variant=variant, dtype=dtype, out=e_out, xhat=e_xh, rstd=e_rs)
    # operands truncated to tf32 (dtype 2) make every product exact: both modes are fp32 accumulations of exact products
    assert e_out < 1e-5 and e_xh < 1e-5 and e_rs < 1e-5       # measured on a B200: out 5.7e-6, xhat 6.1e-6, rstd 4.2e-8


# ------------------------------------------------------------------------------------------ wide stem finish, training
@pytest.mark.parametrize("C", WIDTHS)
def test_wide_stem_finish_train(C):
    B, L, HP, WP, eps = 2, 12, 14, 28, 1e-5
    N = B * L
    raw3, rawres = pg(rnd(B, C, HP, WP, seed=1)), pg(rnd(B, C, HP, WP, seed=2))
    b3, b1 = 0.1 * rnd(C, seed=3), 0.1 * rnd(C, seed=4)
    tt, tres = 0.3 * rnd(N, 9, C, seed=5), 0.3 * rnd(N, C, seed=6)
    g, be = 1 + 0.2 * rnd(C, seed=7), 0.1 * rnd(C, seed=8)
    film = 0.5 * rnd(N, 2 * C, seed=9)
    h1, res, xhat = pg_nan(N, HP, WP, C), pg_nan(N, HP, WP, C), pg_nan(N, HP, WP, C)
    Q = h1.shape[0]
    rstd = torch.full((Q,), float("nan"), device=DEV)
    mask = torch.full((Q, C // 32), -1, dtype=torch.int32, device=DEV)
    call("vg_stem_finish_wide_train_fwd", 1, raw3.data_ptr(), rawres.data_ptr(), b3.data_ptr(), b1.data_ptr(), tt.data_ptr(),
         tres.data_ptr(), g.data_ptr(), be.data_ptr(), eps, film.data_ptr(), B, L, HP, WP, C, h1.data_ptr(), res.data_ptr(),
         xhat.data_ptr(), rstd.data_ptr(), mask.data_ptr())
    torch.cuda.synchronize()
    # per field n = b*L + l: v = raw3[b] + b3 + tt[n][case(h, w)] over the nine border cases
    ry = torch.ones(HP, dtype=torch.long, device=DEV); ry[0], ry[-1] = 0, 2
    rx = torch.ones(WP, dtype=torch.long, device=DEV); rx[0], rx[-1] = 0, 2
    case = (ry.view(-1, 1) * 3 + rx.view(1, -1))                                             # (HP, WP)
    bi = torch.arange(N, device=DEV) // L
    r3 = unpg(raw3, B, HP, WP).double()[bi] + b3.double().view(1, -1, 1, 1)
    t = tt.double()[:, case].permute(0, 3, 1, 2)                                             # (N, C, HP, WP)
    v = r3 + t
    mean = v.mean(1, keepdim=True)
    rs = (v - mean).pow(2).mean(1, keepdim=True).clamp_min(eps).rsqrt()
    xh = (v - mean) * rs
    z = (xh * g.double().view(1, -1, 1, 1) + be.double().view(1, -1, 1, 1)) * (film[:, :C].double().view(N, C, 1, 1) + 1) \
        + film[:, C:].double().view(N, C, 1, 1)
    rres = unpg(rawres, B, HP, WP).double()[bi] + b1.double().view(1, -1, 1, 1) + tres.double().view(N, C, 1, 1)
    pads = pad_mask(N, HP, WP)
    assert (h1[pads] == 0).all() and (xhat[pads] == 0).all() and (rstd[pads] == 0).all() and (mask[pads] == 0).all()
    e = dict(h1=rel(unpg(h1, N, HP, WP), z.clamp_min(0)), res=rel(unpg(res, N, HP, WP), rres), xhat=rel(unpg(xhat, N, HP, WP), xh),
             rstd=rel(rstd[:N * (HP + 1) * (WP + 1)].view(N, HP + 1, WP + 1)[:, 1:, 1:], rs[:, 0]))
    note(test="wide_stem_finish_train", C=C, **e)
    assert max(e.values()) < 7e-7                                # measured on a B200: <= 1.8e-7 (xhat)
    safe = (z.abs() > 1e-5 * z.abs().max()).permute(0, 2, 3, 1)
    got = pg_words(mask, N, HP, WP)
    gb = ((got.unsqueeze(-1) >> torch.arange(32, device=DEV)) & 1).reshape(N, HP, WP, C).bool()
    assert (gb[safe] == (z > 0).permute(0, 2, 3, 1)[safe]).all()


# ------------------------------------------------------------------------------------------ wide Block backward
BWD_GEOMS = {"3x14x14": (3, 14, 14), "2x84x70": (2, 84, 70)}


@pytest.mark.parametrize("with_film", [True, False])
@pytest.mark.parametrize("geom", list(BWD_GEOMS))
@pytest.mark.parametrize("C", (128,) + WIDTHS)
def test_wide_block_bwd(C, geom, with_film):
    """dconv, the per-field sums A/B/D, the border sums and the parameter gradients.  3 x 14x14: 225 pixels per field, so field
    boundaries fall inside the 256-pixel blocks and the last block is partial; one field has clamped rows (rstd = eps^-1/2)"""
    N, HP, WP = BWD_GEOMS[geom]
    eps = 1e-5
    dy = rnd(N, C, HP, WP, seed=11)
    v = rnd(N, C, HP, WP, seed=12)
    xh = (v - v.mean(1, keepdim=True)) / v.std(1, unbiased=False, keepdim=True)
    rs = 0.5 + torch.rand(N, HP, WP, generator=gen(13), device=DEV)
    rs[1, : HP // 2] = eps ** -0.5                                 # clamped rows: no variance gradient
    zmask = torch.rand(N, C, HP, WP, generator=gen(14), device=DEV) > 0.4
    g, b = 1 + 0.2 * rnd(C, seed=15), 0.1 * rnd(C, seed=16)
    film = 0.5 * rnd(N, 2 * C, seed=17) if with_film else None
    dyp, xhp = pg(dy), pg(xh)
    Q = dyp.shape[0]
    rstd = torch.zeros(Q, device=DEV)
    rstd[:N * (HP + 1) * (WP + 1)].view(N, HP + 1, WP + 1)[:, 1:, 1:] = rs
    words = torch.zeros(Q, C // 32, dtype=torch.int64, device=DEV)
    words[:N * (HP + 1) * (WP + 1)].view(N, HP + 1, WP + 1, C // 32)[:, 1:, 1:] = mask_bits(zmask)
    mask = ((words + 2 ** 31) % 2 ** 32 - 2 ** 31).to(torch.int32)           # the same 32 bits as signed words
    dconv = pg_nan(N, HP, WP, C)
    sums = 0.25 * torch.ones(3, N, C, device=DEV)                  # accumulated outputs: nonzero start
    border = 0.5 * torch.ones(N, 8, C, device=DEV)
    call("vg_conv_ln_bwd_wide", C, dyp.data_ptr(), xhp.data_ptr(), rstd.data_ptr(), mask.data_ptr(), g.data_ptr(), o()._p(film), eps,
         dconv.data_ptr(), sums[0].data_ptr(), sums[1].data_ptr(), sums[2].data_ptr(), border.data_ptr(), N, HP, WP)
    dg, db, dbias = torch.full((C,), 0.5, device=DEV), torch.full((C,), -0.5, device=DEV), torch.full((C,), 0.25, device=DEV)
    dfilm = torch.full((N, 2 * C), float("nan"), device=DEV)
    call("vg_conv_ln_param_grads_wide", sums[0].data_ptr(), sums[1].data_ptr(), sums[2].data_ptr(), N, C, g.data_ptr(), b.data_ptr(),
         o()._p(film), dg.data_ptr(), db.data_ptr(), dbias.data_ptr(), dfilm.data_ptr())
    torch.cuda.synchronize()
    # float64 reference
    s = (film[:, :C].double().view(N, C, 1, 1) + 1) if with_film else torch.ones(1, C, 1, 1, dtype=F64, device=DEV)
    dz = dy.double() * zmask
    x64, r64 = xh.double(), rs.double().unsqueeze(1)
    dx = dz * g.double().view(1, -1, 1, 1) * s
    s1 = dx.mean(1, keepdim=True)
    s2 = (dx * x64).mean(1, keepdim=True) * (rs.unsqueeze(1) < eps ** -0.5 * (1 - 1e-6))
    ref = r64 * (dx - s1 - x64 * s2)
    A, Bs, D = (dz * x64).sum((2, 3)), dz.sum((2, 3)), ref.sum((2, 3))
    bref = torch.stack([ref[:, :, 0].sum(-1), ref[:, :, -1].sum(-1), ref[:, :, :, 0].sum(-1), ref[:, :, :, -1].sum(-1),
                        ref[:, :, 0, 0], ref[:, :, 0, -1], ref[:, :, -1, 0], ref[:, :, -1, -1]], 1)
    sv = s[:, :, 0, 0].expand(N, C)
    # the parameter gradients read the kernel's own (accumulated) sums
    sA, sB, sD = sums[0].double(), sums[1].double(), sums[2].double()
    e = dict(dconv=rel(unpg(dconv, N, HP, WP), ref), A=rel(sums[0] - 0.25, A), B=rel(sums[1] - 0.25, Bs), D=rel(sums[2] - 0.25, D),
             border=rel(border - 0.5, bref), dg=rel(dg - 0.5, (sA * sv).sum(0)), db=rel(db + 0.5, (sB * sv).sum(0)),
             dbias=rel(dbias - 0.25, sD.sum(0)))
    e["dfilm"] = rel(dfilm, torch.cat([sA * g.double() + sB * b.double(), sB], 1))
    assert (dconv[pad_mask(N, HP, WP)] == 0).all()
    note(test="wide_block_bwd", C=C, geom=geom, film=with_film, **e)
    assert max(e.values()) < 1e-6, e                               # measured on a B200: <= 3.8e-7 (border sums)


# ------------------------------------------------------------------------------------------ small backward kernels at C > 128
@pytest.mark.parametrize("C", WIDTHS)
def test_head_bwd_wide(C):
    N, HP, WP, H, Wd, pt, pl, std = 3, 28, 28, 26, 25, 1, 1, 7.5
    h = rnd(N, C, HP, WP, seed=21)
    w = rnd(C, seed=22)
    dpred = rnd(N, H, Wd, seed=23)
    dH = pg_nan(N, HP, WP, C)
    dw, db = torch.full((C,), 0.5, device=DEV), torch.full((1,), 0.5, device=DEV)
    call("vg_head_bwd_wide", 1, dpred.data_ptr(), pg(h).data_ptr(), w.data_ptr(), std, N, HP, WP, C, H, Wd, pt, pl, dH.data_ptr(),
         dw.data_ptr(), db.data_ptr())
    torch.cuda.synchronize()
    d = torch.zeros(N, HP, WP, dtype=F64, device=DEV)
    d[:, pt:pt + H, pl:pl + Wd] = dpred.double() * std
    e = dict(dH=rel(unpg(dH, N, HP, WP), d.unsqueeze(1) * w.double().view(1, -1, 1, 1)),
             dw=rel(dw - 0.5, (h.double() * d.unsqueeze(1)).sum((0, 2, 3))), db=rel(db - 0.5, d.sum().view(1)))
    assert (dH[pad_mask(N, HP, WP)] == 0).all()
    note(test="head_bwd_wide", C=C, **e)
    assert max(e.values()) < 6e-7                                # measured on a B200: <= 1.5e-7 (dw)


@pytest.mark.parametrize("C", WIDTHS)
def test_lead_sum_and_field_sum_wide(C):
    B, L, HP, WP = 2, 3, 28, 28
    N = B * L
    x = rnd(N, C, HP, WP, seed=31)
    xp = pg(x)
    out = pg_nan(B, HP, WP, C)
    call("vg_lead_sum_wide", 1, 1, xp.data_ptr(), out.data_ptr(), B, L, HP, WP, C)
    fs = 0.5 * torch.ones(N, C, device=DEV)
    call("vg_pg_field_sum_wide", xp.data_ptr(), fs.data_ptr(), N, HP, WP, C)
    torch.cuda.synchronize()
    e = dict(lead=rel(unpg(out, B, HP, WP), x.double().view(B, L, C, HP, WP).sum(1)), field=rel(fs - 0.5, x.double().sum((2, 3))))
    assert (out[pad_mask(B, HP, WP)] == 0).all()
    note(test="lead_field_sum_wide", C=C, **e)
    assert max(e.values()) < 6e-7                                # measured on a B200: <= 1.5e-7 (field sums)


@pytest.mark.parametrize("C", WIDTHS)
def test_convT2_bwd_gather_wide(C):
    N, Hl, Wl = 2, 14, 14
    dup = rnd(N, C, 2 * Hl, 2 * Wl, seed=41)
    G = torch.full((N * Hl * Wl, 4 * C), float("nan"), device=DEV)
    dbias = torch.full((C,), 0.5, device=DEV)
    call("vg_convT2_bwd_gather", 1, pg(dup).data_ptr(), G.data_ptr(), dbias.data_ptr(), N, Hl, Wl, C)
    torch.cuda.synchronize()
    ref = dup.view(N, C, Hl, 2, Wl, 2).permute(0, 2, 4, 3, 5, 1).reshape(N * Hl * Wl, 4 * C)
    assert torch.equal(G, ref)
    e = rel(dbias - 0.5, dup.double().sum((0, 2, 3)))
    note(test="convT2_bwd_gather_wide", C=C, dbias=e)
    assert e < 1.1e-6                                            # measured on a B200: 2.8e-7


# ------------------------------------------------------------------------------------------ tf32 3x3 data / weight gradients
def _shift_rows(A, s):
    out = torch.zeros_like(A)
    M = A.shape[0]
    if s >= 0:
        out[:M - s] = A[s:]
    else:
        out[-s:] = A[:M + s]
    return out


@pytest.mark.parametrize("integer", [True, False])
@pytest.mark.parametrize("C,Ca", [(256, 256), (512, 512), (512, 640)])
def test_tf32_dgrad_wgrad_nine_taps(C, Ca, integer):
    """C -> C block shapes and the stem shape (Ca = c_pad 640 input channels of the 12-hour model): the data gradient
    (ops.gemm, negated shifts) and the weight gradient (vg_wgrad) in tf32.  Integer operands are exact in tf32 and every
    partial sum is an integer below 2^24: bit-exact."""
    from vit_grid_model_b200 import ops_train as ot
    N, HP, WP = 2, 28, 28
    shifts = o().conv_tap_shifts(WP)
    nshifts = tuple(-s for s in shifts)
    M = o().pg_pixels(N, HP, WP)
    pads = pad_mask(N, HP, WP)

    def make(cols, seed):
        t = (torch.randint(-3, 4, (M, cols), generator=gen(seed), device=DEV).float() if integer else rnd(M, cols, seed=seed))
        t[pads] = 0
        return t
    dY, A = make(C, 51), make(Ca, 52)
    dW = torch.full((C, 9 * Ca), float("nan"), device=DEV)
    ot.wgrad(dY, A, dW, ntaps=9, tap_shift=shifts, beta=0.0, tf32=True)
    Wt = (torch.randint(-3, 4, (Ca, 9 * C), generator=gen(53), device=DEV).float() if integer else rnd(Ca, 9 * C, seed=53))
    dX = o().gemm(dY, Wt, ntaps=9, tap_shift=nshifts, out_f32=True, tf32=True)
    torch.cuda.synchronize()
    d64, a64, w64 = tf32(dY).double(), tf32(A).double(), tf32(Wt).double()
    refW = torch.cat([d64.t() @ _shift_rows(a64, s) for s in shifts], 1)
    refX = sum(_shift_rows(d64, s) @ w64[:, t * C:(t + 1) * C].t() for t, s in enumerate(nshifts))
    if integer:
        assert torch.equal(dW, refW.float()) and torch.equal(dX, refX.float())
        return
    e = dict(wgrad=rel(dW, refW), dgrad=rel(dX, refX))
    note(test="tf32_dgrad_wgrad", C=C, Ca=Ca, **e)
    assert e["wgrad"] < 5e-6 and e["dgrad"] < 5e-5                 # measured on a B200: wgrad <= 1.7e-6, dgrad <= 1.4e-5


# ------------------------------------------------------------------------------------------ module
def _model(cfg, precision="tf32_conv", train=True, seed=0, dropout=0.0, stn=False):
    from vit_grid_model_b200 import MetNet3, MetNet3_with_stn_imgs
    m = (MetNet3_with_stn_imgs if stn else MetNet3)(**cfg.metnet3_kwargs(), dropout=dropout)
    m.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=seed), strict=True)
    m = m.cuda().set_precision(precision)
    return m.train() if train else m.eval()


def _oracle(cfg, x, ts, dpred, training, seed=0, stn=False, monkeypatch=None):
    """float64 autograd through the oracle on the GPU -> (pred, x.grad, {param: grad}, the oracle's state dict (buffers as given),
    [(mean, unbiased var)] of every batch-statistic BatchNorm in call order, recorded when monkeypatch is given)"""
    sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=seed)
    for k, v in sd.items():
        if v.is_floating_point():
            sd[k] = v.to(DEV, F64)
            if "running_" not in k and k != "pm25_boundaries":
                sd[k].requires_grad_(True)
        else:
            sd[k] = v.to(DEV)
    stats = []
    if monkeypatch is not None:
        bn = mo.F.batch_norm

        def recording(t, *a, **kw):                      # (input, running_mean, running_var, weight, bias, training, ...)
            if a[4]:
                d = t.detach()
                stats.append((d.mean((0, 2, 3)), d.var((0, 2, 3), unbiased=True)))
            return bn(t, *a, **kw)
        monkeypatch.setattr(mo.F, "batch_norm", recording)
    x64 = x.detach().to(DEV, F64).requires_grad_(True)
    pred = metnet3_forward(x64, ts.cpu(), sd, cfg, training=training, stn_imgs=stn)
    if monkeypatch is not None:
        monkeypatch.undo()
    pred.backward(dpred.to(DEV, F64))
    return pred.detach(), x64.grad, {k: v.grad for k, v in sd.items() if v.is_floating_point() and v.requires_grad}, sd, stats


def _inputs(cfg, B=2, seed=31):
    x, ts, _ = synth.make_inputs(cfg, B, seed=seed)
    dpred = torch.randn(B, cfg.L, cfg.H, cfg.W, generator=torch.Generator().manual_seed(seed + 1))
    return x, ts, dpred


PRE_BN_BIAS = re.compile(r"(vit\.layers\.\d+\.0\.(?:fn\.)?)([037])\.bias")


def _check_grads(pairs, grads, frozen, bound_l2, bound_cos, label):
    """Per tensor: relative L2 error (floor 1e-2 on the reference norm, as in test_train_gpu.py), max error (same floor) and
    cosine (tensors with a reference norm above 1e-2) against float64; every tensor must be inside bound_l2 and bound_cos.  A conv
    bias in front of a batch-statistic BatchNorm has an analytically zero gradient in train() mode: its norm must stay below 7e-6
    of the adjacent BatchNorm beta gradient instead (measured on a B200: <= 1.7e-6) (in the frozen eval() graph those biases have real gradients).  Also returns
    the global relative L2 over every tensor."""
    bad, worst_l2, worst_max, worst_cos, worst_bias, num, den = [], ("", 0.0), 0.0, ("", 1.0), 0.0, 0.0, 0.0
    for name, got, ref in pairs:
        g, r = got.detach().to(DEV, F64), ref.to(DEV, F64)
        num += (g - r).pow(2).sum().item()
        den += r.pow(2).sum().item()
        m = PRE_BN_BIAS.fullmatch(name)
        if m and not frozen:
            beta = grads[m.group(1) + str(int(m.group(2)) + 1) + ".bias"].norm().item()
            worst_bias = max(worst_bias, g.norm().item() / beta)
            if g.norm().item() > 7e-6 * beta:
                bad.append((name, "pre-BN bias", g.norm().item(), beta))
            continue
        el2 = (g - r).norm().item() / max(r.norm().item(), 1e-2)
        emax = (g - r).abs().max().item() / max(r.abs().max().item(), 1e-2)
        cos = (torch.dot(g.reshape(-1), r.reshape(-1)) / (g.norm() * r.norm()).clamp_min(1e-30)).item() if r.norm() > 1e-2 else 1.0
        worst_max = max(worst_max, emax)
        if el2 > worst_l2[1]:
            worst_l2 = (name, el2)
        if cos < worst_cos[1]:
            worst_cos = (name, cos)
        if el2 > bound_l2 or cos < bound_cos:
            bad.append((name, round(el2, 5), round(cos, 6)))
    gl2 = (num / den) ** 0.5
    note(test=label, worst_l2=worst_l2, worst_max=worst_max, worst_cos=worst_cos, pre_bn_bias_ratio=worst_bias, global_l2=gl2)
    assert not bad, bad[:20]
    return gl2


# (prediction, per-tensor relative L2, per-tensor cosine) of one tf32_conv step.  Measured on a B200 at 1000 W -- prediction; worst
# per-tensor L2 (tensor); lowest cosine (tensor); global L2; running buffers:
#   128: 2.1e-3; 6.3e-2 (resnet2.blocks.0.block1.norm.b); 0.99801 (same); 4.2e-2; 2.6e-4
#   256: 7.0e-3; 0.236 (condition_model_time.2.weight); 0.99296 (resnet2.blocks.1.block1.proj.bias); 7.3e-2; 3.1e-4
#   384: 4.4e-3; 0.187 (condition_model_time.2.weight); 0.99572 (same); 4.7e-2; 2.1e-4
#   512: 3.3e-3; 0.110 (condition_lead_time.weight); 0.99499 (same); 4.8e-2; 2.5e-4
# For scale, the same 128-channel step in 'fp32' measures global L2 2.7e-3, worst tensor 8.0e-3; in 'bf16' 0.139 and 0.243.
# The worst tensors are the small time-embedding tables, each entry a sum over every pixel of the stem's time channels.
STEP_BOUNDS = {128: (8e-3, 0.25, 0.992), 256: (2.8e-2, 0.5, 0.98), 384: (1.7e-2, 0.5, 0.985), 512: (1.3e-2, 0.3, 0.985)}
# x.grad tests, (C, train): measured worst per-tensor L2 / lowest cosine -- 256 train 0.236 / 0.99296, eval 6.1e-2 / 0.99886;
# 512 train 0.110 / 0.99499, eval 8.7e-2 / 0.99923
XGRAD_BOUNDS = {(256, True): (0.5, 0.98), (256, False): (0.2, 0.996), (512, True): (0.3, 0.985), (512, False): (0.25, 0.997)}


@pytest.mark.parametrize("C", [128, 256, 384, 512])
def test_tf32_conv_train_step(C, monkeypatch):
    """prediction, every parameter gradient (per tensor) and the MaxViT BatchNorm running buffers (momentum 0.1, unbiased
    variance of the batch statistics the oracle computes) against float64 autograd of the oracle, num_batches_tracked + 1"""
    cfg = MODULE_CFGS[C]
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg)
    pred = m(x.cuda(), timestamps=ts.cuda())
    pred.backward(dpred.cuda())
    torch.cuda.synchronize()
    opred, _, og, osd, stats = _oracle(cfg, x, ts, dpred, True, monkeypatch=monkeypatch)
    e_pred = rel(pred, opred)
    bpred, bl2, bcos = STEP_BOUNDS[C]
    grads = {k: p.grad for k, p in m.named_parameters()}
    _check_grads([(k, grads[k], og[k]) for k in og], grads, False, bl2, bcos, f"tf32_conv_train_step C={C}")
    # running buffers: the MaxViT BatchNorms in call order (layer by layer: 1, 4, 8)
    bns = [f"vit.layers.{li}.0." + ("fn." if hasattr(m.vit.layers[li][0], "fn") else "") + str(i)
           for li in range(len(m.vit.layers)) for i in (1, 4, 8)]
    assert len(stats) == len(bns)
    sdm = m.state_dict()
    e_run = 0.0
    for name, (mean, var) in zip(bns, stats):
        rm0, rv0 = osd[name + ".running_mean"], osd[name + ".running_var"]
        e_run = max(e_run, rel(sdm[name + ".running_mean"], 0.9 * rm0 + 0.1 * mean), rel(sdm[name + ".running_var"], 0.9 * rv0 + 0.1 * var))
        assert sdm[name + ".num_batches_tracked"].item() == osd[name + ".num_batches_tracked"].item() + 1, name
    note(test="tf32_conv_train_step", C=C, pred=e_pred, running=e_run)
    assert e_pred < bpred and e_run < 1.2e-3, (e_pred, e_run)


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("C", [256, 512])
def test_tf32_conv_x_grad(C, train):
    """x.grad and every parameter gradient, per tensor, in train() mode and in the frozen-BatchNorm eval() graph"""
    cfg = MODULE_CFGS[C]
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, train=train)
    xg = x.cuda().requires_grad_(True)
    pred = m(xg, timestamps=ts.cuda())
    assert pred.grad_fn is not None
    pred.backward(dpred.cuda())
    torch.cuda.synchronize()
    _, ogx, og, _, _ = _oracle(cfg, x, ts, dpred, train)
    grads = {k: p.grad for k, p in m.named_parameters()}
    bl2, bcos = XGRAD_BOUNDS[(C, train)]
    _check_grads([("x", xg.grad, ogx)] + [(k, grads[k], og[k]) for k in og], grads, not train, bl2, bcos,
                 f"tf32_conv_x_grad C={C} train={train}")


def test_tf32_conv_stn_variant():
    cfg = synth.GridConfig(T=3, C=25, H=26, W=25, dim=256, L=2, vit_depth=2, heads=4, dim_head=64)
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, stn=True)
    pred = m(x.cuda().clone(), timestamps=ts.cuda())
    pred.backward(dpred.cuda())
    torch.cuda.synchronize()
    opred, _, og, _, _ = _oracle(cfg, x, ts, dpred, True, stn=True)
    grads = {k: p.grad for k, p in m.named_parameters()}
    e_pred = rel(pred, opred)
    note(test="tf32_conv_stn", pred=e_pred)
    assert e_pred < 3.6e-2                                           # measured on a B200: 9.2e-3
    # measured on a B200: worst per-tensor L2 0.131 (condition_lead_time.weight), lowest cosine 0.99288
    _check_grads([(k, grads[k], og[k]) for k in og], grads, False, 0.35, 0.975, "tf32_conv_stn")


def test_tf32_conv_default_dropout_finite():
    cfg = synth.CFG_WIDE256
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, dropout=0.1)
    pred = m(x.cuda(), timestamps=ts.cuda())
    pred.backward(dpred.cuda())
    assert torch.isfinite(pred).all() and all(torch.isfinite(p.grad).all() for p in m.parameters())


def test_tf32_conv_flat_adamw_512_loss_decreases():
    """a few optimiser steps at 512 channels on the configs[4] head layout (32 x 64, two input time steps: the stem's c_pad of
    64 runs its weight gradient as exact-fp32 products)"""
    from vit_grid_model_b200 import FlatAdamW, focal_r_loss
    cfg = synth.CFG_WIDE512
    x, ts, _ = synth.make_inputs(cfg, 2, seed=61)
    target = torch.rand(2, cfg.L, cfg.H, cfg.W, generator=torch.Generator().manual_seed(62)) * 40
    m = _model(cfg)
    opt = FlatAdamW(m, lr=1e-5)
    losses = []
    for _ in range(4):
        opt.zero_grad()
        loss = focal_r_loss(m(x.cuda(), timestamps=ts.cuda()), target.cuda())
        loss.backward()
        opt.step()
        losses.append(loss.item())
    note(test="flat_adamw_512", losses=losses)
    assert all(torch.isfinite(torch.tensor(losses))) and losses[-1] < losses[0]


def test_unbuilt_precisions_still_raise():
    cfg = synth.CFG_WIDE256
    x, ts, _ = _inputs(cfg)
    for precision in ("tf32", "bf16_all", "fp32", "bf16"):
        m = _model(cfg, precision)
        with pytest.raises(NotImplementedError):
            m(x.cuda(), timestamps=ts.cuda())
    m = _model(synth.CFG_SMALL128, "bf16_all")
    x, ts, _ = _inputs(synth.CFG_SMALL128)
    with pytest.raises(NotImplementedError):
        m(x.cuda(), timestamps=ts.cuda())
    with pytest.raises(NotImplementedError):
        m.set_precision("tf32")(x.cuda(), timestamps=ts.cuda())

