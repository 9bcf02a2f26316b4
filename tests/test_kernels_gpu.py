"""Per-kernel parity (GPU): every libvitgrid entry point, called through the C ABI, against the CPU oracle /
a plain fp32 PyTorch statement of the same op on identical seeded inputs.

Tolerances: fp32 mode 1e-4 relative (max-abs error / max-abs reference); bf16 mode 1e-2 (2e-2 where the
reference output itself is rounded to bf16).  Index work is bit-exact.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle import maxvit_oracle as mo
from oracle import metnet3_oracle as m3o

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.bfloat16]
TOL = {torch.float32: 1e-4, torch.bfloat16: 1.5e-2}
# GEMM modes: (storage dtype, tf32 tensor cores?) -> tolerance of a single GEMM against fp32
GEMM_MODES = [(torch.float32, False), (torch.bfloat16, False), (torch.float32, True)]
GEMM_TOL = {(torch.float32, False): 2e-5, (torch.bfloat16, False): 6e-3, (torch.float32, True): 1.5e-3}


def ops():
    from vit_grid_model_b200 import ops as _ops
    return _ops


def rel_err(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def q(t, dtype):
    """round a CPU fp32 tensor to what the device path will see"""
    return t.to(dtype).float()


# ------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("mode", GEMM_MODES)
@pytest.mark.parametrize("M,K,N", [(1000, 128, 128), (4099, 512, 384), (130, 1024, 128), (20000, 128, 3072), (300, 96, 256)])
def test_gemm_plain(mode, M, K, N):
    dtype, tf32 = mode
    if not tf32 and K % 64:
        pytest.skip("bf16 / SIMT K blocks are 64 wide; only the tf32 path takes K % 32 == 0")
    o = ops()
    A, W = q(rnd(M, K, seed=1), dtype), q(rnd(N, K, seed=2) / math.sqrt(K), dtype)
    out = o.gemm(A.cuda().to(dtype), W.cuda().to(dtype), tf32=tf32)
    assert rel_err(out, A @ W.t()) < GEMM_TOL[mode]


@pytest.mark.parametrize("mode", GEMM_MODES)
def test_gemm_bn_gelu_residual(mode):
    dtype, tf32 = mode
    o = ops()
    M, K, N = 3000, 128, 512
    A, W = q(rnd(M, K, seed=1), dtype), q(rnd(N, K, seed=2) / math.sqrt(K), dtype)
    scale, shift, res = 0.5 + torch.rand(N), rnd(N, seed=4), q(rnd(M, N, seed=5), dtype)
    out = o.gemm(A.cuda().to(dtype), W.cuda().to(dtype), scale=scale.cuda(), shift=shift.cuda(), act=1,
                 res=res.cuda().to(dtype), tf32=tf32)
    ref = F.gelu((A @ W.t()) * scale + shift) + res
    assert rel_err(out, ref) < (2e-3 if tf32 else TOL[dtype])


@pytest.mark.parametrize("dtype", DTYPES)
def test_gemm_per_batch_weights(dtype):
    o = ops()
    nb, rows, K, N = 5, 300, 128, 128
    A = q(rnd(nb * rows, K, seed=1), dtype)
    W = q(rnd(nb, N, K, seed=2) / math.sqrt(K), dtype)
    out = o.gemm(A.cuda().to(dtype), W.reshape(nb * N, K).cuda().to(dtype), rows_per_batch=rows, b_rows_per_batch=N)
    ref = torch.einsum("brk,bnk->brn", A.view(nb, rows, K), W).reshape(nb * rows, N)
    assert rel_err(out, ref) < (2e-5 if dtype == torch.float32 else 6e-3)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("N,H,W,Ca", [(2, 12, 10, 128), (3, 28, 28, 64), (1, 84, 70, 192)])
def test_conv3x3_as_shifted_gemm(dtype, N, H, W, Ca):
    """raw 3x3/pad-1 convolution over the padded-grid layout == F.conv2d"""
    o = ops()
    x = q(rnd(N, Ca, H, W, seed=3), dtype)
    w = q(rnd(128, Ca, 3, 3, seed=4) / math.sqrt(9 * Ca), dtype)
    xp = o.pg_from_nchw(x.cuda(), dtype)
    wt = w.permute(0, 2, 3, 1).reshape(128, 9 * Ca).contiguous().cuda().to(dtype)
    out = o.gemm(xp, wt, ntaps=9, tap_shift=o.conv_tap_shifts(W), out_f32=True)
    got = o.pg_to_nchw(out, N, H, W)
    assert rel_err(got, F.conv2d(x, w, padding=1)) < (2e-5 if dtype == torch.float32 else 6e-3)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("with_film,with_res", [(True, False), (False, True)])
def test_conv3x3_ln_block(dtype, with_film, with_res):
    """metnet3.py:110-126 Block (+ residual) fused epilogue; pads of the output must be exactly zero"""
    o = ops()
    N, H, W, C = 3, 14, 28, 128
    x = q(rnd(N, C, H, W, seed=3), dtype)
    w = q(rnd(C, C, 3, 3, seed=4) / math.sqrt(9 * C), dtype)
    b, g, be = rnd(C, seed=5, scale=0.1), 0.5 + torch.rand(C), rnd(C, seed=7, scale=0.1)
    film = rnd(N, 2 * C, seed=8, scale=0.3) if with_film else None
    res = q(rnd(N, C, H, W, seed=9), dtype) if with_res else None
    out = torch.full((o.pg_pixels(N, H, W), C), 7.0, dtype=dtype, device="cuda")
    o.conv3x3_ln(o.pg_from_nchw(x.cuda(), dtype), w.permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous().cuda().to(dtype),
                 b.cuda(), g.cuda(), be.cuda(), 1e-5, None if film is None else film.cuda(),
                 None if res is None else o.pg_from_nchw(res.cuda(), dtype), out, N, H, W)
    h = m3o.chan_layer_norm(F.conv2d(x, w, b, padding=1), g.view(1, C, 1, 1), be.view(1, C, 1, 1))
    if with_film:
        h = h * (film[:, :C, None, None] + 1) + film[:, C:, None, None]
    h = F.relu(h)
    if with_res:
        h = h + res
    assert rel_err(o.pg_to_nchw(out, N, H, W), h) < TOL[dtype]
    # pad positions are zero
    full = out.float().view(N * (H + 1) + 1, W + 1, C)
    assert full[:, 0].abs().max().item() == 0.0
    assert full[::H + 1].abs().max().item() == 0.0


# ------------------------------------------------------------------------------------------ input side
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("layout", ["contiguous", "channels_last_view"])
def test_prepare(dtype, layout):
    o = ops()
    cfg = synth.CFG_SMALL128
    x, ts, _ = synth.make_inputs(cfg, 2)
    xd = x.cuda()
    if layout == "channels_last_view":      # the eval driver's permuted view (evaluation_vit.py:248-249)
        xd = x.permute(0, 3, 4, 1, 2).contiguous().cuda().permute(0, 3, 4, 1, 2)
    cpad = (cfg.T * cfg.C + 63) // 64 * 64
    out = o.prepare(xd, cfg.pads, cfg.HP, cfg.WP, cpad, cfg.pm25_mean, cfg.pm25_std, dtype)
    ref = x.clone()
    pm = torch.tensor([4, 10, 16, 22])
    ref[:, :, pm] = (ref[:, :, pm] - cfg.pm25_mean) / cfg.pm25_std
    ref = F.pad(ref, cfg.pads).reshape(2, cfg.T * cfg.C, cfg.HP, cfg.WP)
    got = o.pg_to_nchw(out, 2, cfg.HP, cfg.WP)
    assert got[:, cfg.T * cfg.C:].abs().max().item() == 0.0
    if dtype == torch.float32:
        assert torch.equal(got[:, :cfg.T * cfg.C].cpu(), ref)
    else:
        assert torch.equal(got[:, :cfg.T * cfg.C].cpu(), ref.to(dtype))


def test_time_terms_match_explicit_conv():
    """analytic time-channel term == the 3x3 / 1x1 convolution of the constant time channels (Q1, Q2 included)"""
    o = ops()
    cfg = synth.CFG_SMALL128
    B = 3
    sd = synth.make_state_dict(synth.metnet3_spec(cfg))
    x, ts, _ = synth.make_inputs(cfg, B)
    net_in, cond = m3o.prepare_input(x, ts, sd, cfg)
    w3, w1 = sd["resnet1.blocks.0.block1.proj.weight"], sd["resnet1.blocks.0.res_conv.weight"]
    cd = cfg.T * cfg.C
    t_only = net_in[:, cd:]
    ref3 = F.conv2d(t_only, w3[:, cd:], padding=1)             # (N,128,HP,WP)
    ref1 = F.conv2d(t_only, w1[:, cd:])
    temb, cond_d, tt, tres = o.time_terms(ts.cuda(), B, cfg.L, sd["condition_lead_time.weight"].cuda(),
                                          *[sd[f"condition_model_time.{i}.weight"].cuda() for i in range(3)],
                                          w3.cuda().contiguous(), w1.cuda().contiguous(), cd, cfg.dim)
    assert torch.equal(cond_d.cpu(), cond)
    assert torch.equal(temb.cpu(), net_in[:, cd:, 0, 0])
    HP, WP = cfg.HP, cfg.WP
    rows = {0: 0, 1: HP // 2, 2: HP - 1}
    cols = {0: 0, 1: WP // 2, 2: WP - 1}
    for ry in range(3):
        for rx in range(3):
            assert rel_err(tt[:, ry * 3 + rx], ref3[:, :, rows[ry], cols[rx]]) < 1e-5
    assert rel_err(tres, ref1[:, :, 3, 3]) < 1e-5


def test_cond_mlps():
    o = ops()
    g = torch.Generator().manual_seed(3)
    cond = torch.randn(7, 2, generator=g)
    W0, b0 = torch.randn(256, 2, generator=g), torch.randn(256, generator=g)
    W1, b1 = torch.randn(256, 256, generator=g) / 16, torch.randn(256, generator=g)
    got = o.cond_mlp(cond.cuda(), W0.cuda(), b0.cuda(), pre_relu=True)
    assert rel_err(got, F.linear(F.relu(cond), W0, b0)) < 1e-5
    got = o.cond_mlp(cond.cuda(), W0.cuda(), b0.cuda(), W1.cuda(), b1.cuda())
    assert rel_err(got, F.linear(F.silu(F.linear(cond, W0, b0)), W1, b1)) < 1e-5


# ------------------------------------------------------------------------------------------ MBConv pieces
@pytest.mark.parametrize("dtype,out_dtype", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16),
                                             (torch.bfloat16, torch.float32)])
def test_pool2(dtype, out_dtype):
    o = ops()
    x = q(rnd(3, 128, 14, 28, seed=1), dtype)
    got = o.pool2(o.pg_from_nchw(x.cuda(), dtype), 3, 14, 28, out_dtype=out_dtype)
    assert got.dtype == out_dtype
    assert torch.equal(got.float().cpu().permute(0, 3, 1, 2), F.max_pool2d(x, 2, 2))


@pytest.mark.parametrize("dtype", DTYPES)
def test_dwconv_bn_gelu_and_se(dtype):
    o = ops()
    N, H, W, C, se = 3, 14, 21, 512, 128
    x = q(rnd(N, C, H, W, seed=1), dtype)
    w, scale, shift = rnd(C, 1, 3, 3, seed=2) / 3, 0.5 + torch.rand(C), rnd(C, seed=4, scale=0.1)
    out, psum = o.dw3x3_bnact(x.permute(0, 2, 3, 1).contiguous().cuda().to(dtype),
                              w.reshape(C, 9).t().contiguous().cuda(), scale.cuda(), shift.cuda())
    ref = F.gelu(F.conv2d(x, w, padding=1, groups=C) * scale.view(1, C, 1, 1) + shift.view(1, C, 1, 1))
    assert rel_err(out.permute(0, 3, 1, 2), ref) < TOL[dtype]
    assert rel_err(psum.sum(1) / (H * W), ref.mean(dim=(2, 3))) < 1e-4
    W1, W2 = rnd(se, C, seed=5) / math.sqrt(C), rnd(C, se, seed=6) / math.sqrt(se)
    gate = o.se_gate(psum, H * W, W1.cuda(), W2.cuda())
    gref = torch.sigmoid(F.linear(F.relu(F.linear(ref.mean(dim=(2, 3)), W1)), W2))
    assert rel_err(gate, gref) < 1e-4
    o.se_scale_(out, gate)
    assert rel_err(out.permute(0, 3, 1, 2), ref * gref[:, :, None, None]) < TOL[dtype]


# ------------------------------------------------------------------------------------------ attention
def _attn_sd(dim, heads, dh, w, r, seed):
    spec = {k[len("layers.0.1."):]: v for k, v in synth.maxvit_spec(dim, 1, 2, heads, dh, w, 4, 0.25, r).items()
            if k.startswith("layers.0.1.")}
    return synth.make_state_dict(spec, seed=seed)


@pytest.mark.parametrize("mode", GEMM_MODES)
@pytest.mark.parametrize("grid_mode", [False, True])
def test_attention_layer(mode, grid_mode):
    """gather+LN+FiLM -> QKV GEMM -> core -> out-proj(+residual, scatter) == oracle attention + residual"""
    dtype, tf32 = mode
    o = ops()
    N, H, W, C, heads, dh, w, R = 2, 14, 21, 128, 32, 32, 7, 4
    sd = _attn_sd(C, heads, dh, w, R, seed=7)
    x = q(rnd(N, H, W, C, seed=1), dtype)
    cond = rnd(N, 2, seed=2)
    reg = rnd(N, R, C, seed=3) if grid_mode else rnd(R, C, seed=3)
    nwin = (H // w) * (W // w)
    idx = (mo.grid_pixel_index if grid_mode else mo.block_pixel_index)(H, W, w).reshape(-1)
    flat = x.reshape(N, H * W, C)
    tok = flat[:, idx].reshape(N * nwin, w * w, C)
    regs = reg.repeat_interleave(nwin, 0) if grid_mode else reg[None].expand(N * nwin, R, C)
    seq = torch.cat([regs, tok], dim=1)
    # the oracle sees the same rounded weights the device uses
    sdq = dict(sd)
    for k in ("to_qkv.weight", "to_out.0.weight"):
        sdq[k] = q(sd[k], dtype)
    ref = mo.attention(seq, cond, sdq, "", heads=heads, window=w, num_reg=R) + seq
    ref_x = torch.empty_like(flat)
    ref_x[:, idx] = ref[:, R:].reshape(N, nwin * w * w, C)

    gamma, beta = mo.film(cond, sd, "")
    film = torch.cat([gamma, beta], dim=1).cuda().contiguous()
    xd = x.cuda().to(dtype)
    tokens = o.attn_gather(xd, reg.cuda(), film, w, R, grid_mode)
    qkv = o.gemm(tokens, sd["to_qkv.weight"].cuda().to(dtype), tf32=tf32)
    att = o.attn_core(qkv, sd["q_norm.gamma"].reshape(-1).cuda(), sd["k_norm.gamma"].reshape(-1).cuda(),
                      sd["rel_pos_bias.weight"].cuda(), N, H, W, w, R, heads, dh)
    x_out, reg_out = o.attn_out(att, sd["to_out.0.weight"].cuda().to(dtype), xd, reg.cuda(), w, R, grid_mode, True, tf32=tf32)
    tol = {(torch.float32, False): 1e-4, (torch.bfloat16, False): 2e-2, (torch.float32, True): 3e-3}[mode]
    assert rel_err(x_out.reshape(N, H * W, C), ref_x) < tol
    assert rel_err(reg_out, ref[:, :R]) < tol
    mean = o.reg_mean(reg_out, N, nwin)
    assert rel_err(mean, reg_out.view(N, nwin, R, C).mean(1)) < 1e-5


@pytest.mark.parametrize("grid_mode", [False, True])
@pytest.mark.parametrize("N,H,W", [(2, 14, 21), (5, 7, 7), (3, 42, 35)])
def test_attention_fused(grid_mode, N, H, W):
    """the one-kernel attention layer (tf32 projections, bf16 PV) == oracle attention + residual.
    (5,7,7): odd number of windows -> a half-empty last tile; (3,42,35): the 12hr model's map."""
    o = ops()
    C, heads, dh, w, R = 128, 32, 32, 7, 4
    sd = _attn_sd(C, heads, dh, w, R, seed=9)
    x = rnd(N, H, W, C, seed=1)
    cond = rnd(N, 2, seed=2)
    reg = rnd(N, R, C, seed=3) if grid_mode else rnd(R, C, seed=3)
    nwin = (H // w) * (W // w)
    idx = (mo.grid_pixel_index if grid_mode else mo.block_pixel_index)(H, W, w).reshape(-1)
    flat = x.reshape(N, H * W, C)
    tok = flat[:, idx].reshape(N * nwin, w * w, C)
    regs = reg.repeat_interleave(nwin, 0) if grid_mode else reg[None].expand(N * nwin, R, C)
    seq = torch.cat([regs, tok], dim=1)
    ref = mo.attention(seq, cond, sd, "", heads=heads, window=w, num_reg=R) + seq
    ref_x = torch.empty_like(flat)
    ref_x[:, idx] = ref[:, R:].reshape(N, nwin * w * w, C)
    gamma, beta = mo.film(cond, sd, "")
    film = torch.cat([gamma, beta], dim=1).cuda().contiguous()
    inner = heads * dh
    wq = sd["to_qkv.weight"]
    wqkv_h = torch.stack([wq[i * inner:(i + 1) * inner].reshape(heads, dh, C) for i in range(3)], dim=1).reshape(heads * 96, C)
    wout_h = sd["to_out.0.weight"].reshape(C, heads, dh).permute(1, 0, 2).contiguous()
    head_tab = o.pack_head_tables(sd["rel_pos_bias.weight"], sd["q_norm.gamma"], sd["k_norm.gamma"]).cuda()
    x_out, reg_out = o.attn_fused(x.cuda(), reg.cuda(), film, wqkv_h.contiguous().cuda(), wout_h.cuda(), head_tab,
                                  w, R, grid_mode, True, heads, dh)
    assert rel_err(x_out.reshape(N, H * W, C), ref_x) < 4e-3
    assert rel_err(reg_out, ref[:, :R]) < 4e-3
    # the same softmax without the running maximum (the caller's logit bound proves exp2 stays inside fp32)
    bound = o.attn_logit_bound(sd["rel_pos_bias.weight"].cuda(), sd["q_norm.gamma"].cuda(), sd["k_norm.gamma"].cuda(), dh)
    assert 0 < bound <= 115
    x_nm, reg_nm = o.attn_fused(x.cuda(), reg.cuda(), film, wqkv_h.contiguous().cuda(), wout_h.cuda(), head_tab,
                                w, R, grid_mode, True, heads, dh, logit_bound=bound)
    assert rel_err(x_nm.reshape(N, H * W, C), ref_x) < 4e-3 and rel_err(reg_nm, ref[:, :R]) < 4e-3
    assert rel_err(x_nm, x_out) < 1e-3


@pytest.mark.parametrize("grid_mode", [False, True])
@pytest.mark.parametrize("drop", [(0, 0, 0), (1234, 3, 26)])
def test_attention_fused_is_deterministic(grid_mode, drop):
    """race detector: the fused kernel hands operands between four warp roles through TMEM / shared memory (P, X and O_h are
    TMEM operands, S runs a head ahead); every repeat on the same input must be bit-identical -- a missing wait (e.g. the
    out-projection reading O_h before PV retired) shows up as differing repeats.  24 fields: several tiles per CTA."""
    o = ops()
    N, H, W, C, heads, dh, w, R = 24, 42, 35, 128, 32, 32, 7, 4
    x = rnd(N, H, W, C, seed=11).cuda()
    reg = (rnd(N, R, C, seed=12) if grid_mode else rnd(R, C, seed=12)).cuda()
    film = rnd(N, 2 * C, seed=13).cuda()
    wqkv = (rnd(heads * 96, C, seed=14) / 11.3).cuda()
    wout = (rnd(heads, C, dh, seed=15) / 32).cuda()
    qg, kg = (0.5 + torch.rand(heads * dh)).cuda(), (0.5 + torch.rand(heads * dh)).cuda()
    tab = o.pack_head_tables(rnd(170, heads, seed=16).cuda(), qg, kg)
    ref = None
    for _ in range(6):
        y, r = o.attn_fused(x, reg, film, wqkv, wout, tab, w, R, grid_mode, True, heads, dh, drop=drop, logit_bound=0.0 if drop[2] else 110.0)
        torch.cuda.synchronize()
        if ref is None:
            ref = (y.clone(), r.clone())
        else:
            assert torch.equal(y, ref[0]) and torch.equal(r, ref[1])
    assert torch.isfinite(ref[0]).all()


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 6e-3), ("bf16_all", 3e-2)])
def test_maxvit_module(precision, tol):
    """MaxViT nn.Module (reference API) vs oracle, depth 2 (second MBConv is residual)"""
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh, w, R, N, H, W = 128, 2, 32, 32, 7, 4, 3, 14, 21
    sd = synth.make_state_dict(synth.maxvit_spec(dim, depth, 2, heads, dh, w, 4, 0.25, R), seed=5)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=w, num_register_tokens=R)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval().set_precision(precision)
    x, cond = rnd(N, dim, H, W, seed=1), rnd(N, 2, seed=2)
    with torch.no_grad():
        y = m(x.cuda(), cond.cuda())
    ref = mo.maxvit_forward(x, cond, sd, depth=depth, heads=heads, window=w, num_reg=R)
    assert y.shape == ref.shape and y.dtype == torch.float32
    assert rel_err(y, ref) < tol


@pytest.mark.parametrize("dim,heads,dh,w,R,H,W", [(256, 4, 64, 7, 4, 14, 21), (512, 32, 64, 7, 4, 14, 14), (128, 3, 32, 8, 1, 16, 24),
                                                   (384, 6, 64, 7, 2, 7, 14), (128, 5, 32, 7, 4, 14, 21)])
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1.5e-2)])   # tf32 logits: the q.k scale grows with dim_head
def test_maxvit_module_other_widths(dim, heads, dh, w, R, H, W, precision, tol):
    """MaxViT at the widths / head sizes of BASELINE configs[4] (dim 512, dim_head 64) and other constructor arguments the
    reference accepts (window 8, one register token, heads * dim_head != dim, an odd head count at the fused kernel's
    width): the general (un-fused) attention path"""
    from vit_grid_model_b200 import MaxViT
    depth, N = 2, 2
    sd = synth.make_state_dict(synth.maxvit_spec(dim, depth, 2, heads, dh, w, 4, 0.25, R), seed=7)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=w, num_register_tokens=R)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval().set_precision(precision)
    x, cond = rnd(N, dim, H, W, seed=1), rnd(N, 2, seed=2)
    with torch.no_grad():
        y = m(x.cuda(), cond.cuda())
    ref = mo.maxvit_forward(x, cond, sd, depth=depth, heads=heads, window=w, num_reg=R)
    assert rel_err(y, ref) < tol


# ------------------------------------------------------------------------------------------ decoder side
@pytest.mark.parametrize("dtype,tf32,out_dtype", [(torch.float32, False, torch.float32), (torch.bfloat16, False, torch.bfloat16),
                                                  (torch.float32, True, torch.bfloat16)])
def test_convT2(dtype, tf32, out_dtype):
    o = ops()
    N, Hl, Wl, C = 2, 7, 14, 128
    x = q(rnd(N, C, Hl, Wl, seed=1), dtype)
    w, b = q(rnd(C, C, 2, 2, seed=2) / math.sqrt(C), dtype), rnd(C, seed=3, scale=0.1)
    out = torch.zeros(o.pg_pixels(N, 2 * Hl, 2 * Wl), C, dtype=out_dtype, device="cuda")
    o.convT2(x.permute(0, 2, 3, 1).contiguous().cuda().to(dtype),
             w.permute(2, 3, 1, 0).reshape(4 * C, C).contiguous().cuda().to(dtype), b.cuda(), out, tf32=tf32)
    ref = F.conv_transpose2d(x, w, b, stride=2)
    assert rel_err(o.pg_to_nchw(out, N, 2 * Hl, 2 * Wl), ref) < TOL[out_dtype]


def test_conv3x3_ln_fp32_skip_copy_and_fused_head():
    """bf16 block with an fp32 residual, an fp32 output copy and the 1x1 head fused into the epilogue"""
    o = ops()
    cfg = synth.CFG_SMALL128
    N, H, W, C, dtype = 3, cfg.HP, cfg.WP, 128, torch.bfloat16
    x = q(rnd(N, C, H, W, seed=3), dtype)
    w = q(rnd(C, C, 3, 3, seed=4) / math.sqrt(9 * C), dtype)
    b, g, be = rnd(C, seed=5, scale=0.1), 0.5 + torch.rand(C), rnd(C, seed=7, scale=0.1)
    res = rnd(N, C, H, W, seed=9)
    hw, hb = rnd(C, seed=11) / math.sqrt(C), 0.2
    h = F.relu(m3o.chan_layer_norm(F.conv2d(x, w, b, padding=1), g.view(1, C, 1, 1), be.view(1, C, 1, 1))) + res
    pl, pr, pt, pb = cfg.pads
    ref_head = (F.conv2d(h[..., pt:H - pb, pl:W - pr], hw.view(1, C, 1, 1)) + hb).squeeze(1) * cfg.pm25_std + cfg.pm25_mean
    wt = w.permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous().cuda().to(dtype)
    xp, rp = o.pg_from_nchw(x.cuda(), dtype), o.pg_from_nchw(res.cuda(), torch.float32)
    out = torch.empty(o.pg_pixels(N, H, W), C, dtype=dtype, device="cuda")
    copy = torch.empty(o.pg_pixels(N, H, W), C, dtype=torch.float32, device="cuda")
    o.conv3x3_ln(xp, wt, b.cuda(), g.cuda(), be.cuda(), 1e-5, None, rp, out, N, H, W, out_copy=copy)
    assert rel_err(o.pg_to_nchw(copy, N, H, W), h) < 2e-3                  # only the conv operands are bf16
    assert torch.equal(out.float(), copy.to(dtype).float())                # bf16 output == rounded fp32 copy
    pred = torch.empty(N, cfg.H, cfg.W, dtype=torch.float32, device="cuda")
    o.conv3x3_ln(xp, wt, b.cuda(), g.cuda(), be.cuda(), 1e-5, None, rp, None, N, H, W,
                 head=(hw.cuda(), hb, cfg.pm25_std, cfg.pm25_mean, cfg.H, cfg.W, cfg.pads, pred))
    assert rel_err(pred, ref_head) < 2e-3


def test_conv3x3_ln_copy_tma_store_is_repeatable_and_matches_output():
    """The fp32 copy of the conv output leaves through TMA tensor stores from the residual chunk buffers (csrc/vg_epilogue.cuh).
    It must give the same bits launch after launch, on a buffer large enough for many tiles per CTA (a buffer-reuse race
    between the store, the refill and the next chunk would show), write every element, and agree with the bf16 output, which
    leaves the same epilogue registers; the bf16 output must not change when the copy is requested."""
    o = ops()
    N, H, W, C, dtype = 40, 84, 70, 128, torch.bfloat16
    g_ = torch.Generator(device="cuda").manual_seed(5)
    xp = o.pg_from_nchw(torch.randn(N, C, H, W, device="cuda", generator=g_), dtype)
    wt = (torch.randn(C, 9 * C, device="cuda", generator=g_) / math.sqrt(9 * C)).to(dtype)
    b, g, be = (torch.randn(C, device="cuda", generator=g_) * 0.1 for _ in range(3))
    g = g + 1.0
    rp = torch.randn(xp.shape[0], C, device="cuda", generator=g_)
    ref_out = ref_copy = None
    for rep in range(6):
        out = torch.empty_like(xp)
        copy = torch.full((xp.shape[0], C), float("nan"), dtype=torch.float32, device="cuda")
        o.conv3x3_ln(xp, wt, b, g, be, 1e-5, None, rp, out, N, H, W, out_copy=copy)
        torch.cuda.synchronize()
        if ref_out is None:
            ref_out, ref_copy = out, copy
        else:
            assert torch.equal(out, ref_out) and torch.equal(copy, ref_copy), rep
    assert torch.isfinite(ref_copy).all()
    assert torch.equal(ref_out, ref_copy.to(dtype))
    out = torch.empty_like(xp)
    o.conv3x3_ln(xp, wt, b, g, be, 1e-5, None, rp, out, N, H, W)
    torch.cuda.synchronize()
    assert torch.equal(out, ref_out)


@pytest.mark.parametrize("dtype", DTYPES)
def test_head(dtype):
    o = ops()
    cfg = synth.CFG_SMALL128
    N, C = 3, 128
    h = q(rnd(N, C, cfg.HP, cfg.WP, seed=1), dtype)
    w, b = rnd(C, seed=2) / math.sqrt(C), 0.3
    got = o.head(o.pg_from_nchw(h.cuda(), dtype), w.cuda(), b, cfg.pm25_std, cfg.pm25_mean, N, cfg.HP, cfg.WP, cfg.H,
                 cfg.W, cfg.pads)
    pl, pr, pt, pb = cfg.pads
    ref = (F.conv2d(h[..., pt:cfg.HP - pb, pl:cfg.WP - pr], w.view(1, C, 1, 1)) + b).squeeze(1) * cfg.pm25_std + cfg.pm25_mean
    assert rel_err(got, ref) < 1e-5


def test_focal_r_forward_backward():
    from oracle.focal_r_oracle import focal_r, focal_r_grad
    from vit_grid_model_b200 import focal_r_loss
    g = torch.Generator().manual_seed(0)
    p = (torch.rand(4, 12, 82, 67, generator=g) * 60)
    t = (torch.rand(4, 12, 82, 67, generator=g) * 60)
    for mse in (False, True):
        pd = p.cuda().requires_grad_(True)
        loss = focal_r_loss(pd, t.cuda(), mse=mse)
        loss.backward()
        assert abs(loss.item() - focal_r(p.double(), t.double(), mse=mse).item()) / focal_r(p, t, mse=mse).item() < 1e-4
        assert rel_err(pd.grad, focal_r_grad(p, t, mse=mse)) < 1e-4


# ------------------------------------------------------------------------------------------ API corners (round 2)
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_multistage_maxvit_golden_from_reference(golden, precision, tol):
    """MaxViT(depth=(2, 1)) from width 64: ONE stage 64 -> 128 of two layers (the reference's zip() drops the last depth entry,
    maxvit.py:240-262); the first MBConv widens the map and has no residual"""
    from vit_grid_model_b200 import MaxViT
    f = golden("maxvit_multistage.pt")
    m = MaxViT(dim=f["dim"], depth=f["depth"], cond_dim=2, heads=f["heads"], dim_head=f["dim_head"], vit_window_size=f["window"],
               num_register_tokens=f["num_reg"])
    assert list(m.state_dict().keys()) == f["keys"]
    sd = synth.make_state_dict(synth.maxvit_multistage_spec(f["dim"], f["depth"], 2, f["heads"], f["dim_head"], f["window"], 4, 0.25,
                                                            f["num_reg"]), seed=f["seed"])
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval().set_precision(precision)
    with torch.no_grad():
        y = m(f["x"].cuda(), f["cond"].cuda())
    assert y.shape == f["y"].shape and rel_err(y, f["y"]) < tol


@pytest.mark.parametrize("variant,cond_dim", [("film", 2), ("nocond", None)])
def test_standalone_attention_golden_from_reference(golden, variant, cond_dim):
    """Attention.forward(x, cond) called on its own (maxvit.py:170-219), with FiLM and with cond_dim=None"""
    from vit_grid_model_b200 import Attention
    f = golden("attention_standalone.pt")
    a = Attention(dim=f["dim"], cond_dim=cond_dim, heads=f["heads"], dim_head=f["dim_head"], dropout=0.1, window_size=f["window"],
                  num_registers=f["num_reg"])
    a.load_state_dict(synth.make_state_dict(synth.attention_spec(f["dim"], cond_dim, f["heads"], f["dim_head"], f["window"]), seed=f["seed"]),
                      strict=True)
    a = a.cuda().eval()
    y = a(f["x"].cuda(), f["cond"].cuda())
    assert y.shape == f[variant].shape and rel_err(y, f[variant]) < 1e-4


def test_maxvit_module_trains_standalone():
    """MaxViT.forward in train() mode is differentiable (x, cond, parameters) like the reference module under autograd"""
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh, w, R, N, H, W = 128, 1, 32, 32, 7, 4, 2, 14, 21
    sd = synth.make_state_dict(synth.maxvit_spec(dim, depth, 2, heads, dh, w, 4, 0.25, R), seed=5)
    for v in sd.values():
        if v.is_floating_point() and v.dim() > 0:
            v.requires_grad_(True)
    x, cond, dy = rnd(N, dim, H, W, seed=1).requires_grad_(True), rnd(N, 2, seed=2).requires_grad_(True), rnd(N, dim, H, W, seed=3)
    ref = mo.maxvit_forward(x, cond, {k: v for k, v in sd.items()}, depth=depth, heads=heads, window=w, num_reg=R, training=True)
    ref.backward(dy)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=w, num_register_tokens=R, dropout=0.0)
    m.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=True)
    m = m.cuda().train().set_precision("fp32")
    xc, cc = x.detach().cuda().requires_grad_(True), cond.detach().cuda().requires_grad_(True)
    y = m(xc, cc)
    y.backward(dy.cuda())
    assert rel_err(y, ref) < 1e-4
    assert rel_err(xc.grad, x.grad) < 1e-3 and rel_err(cc.grad, cond.grad) < 1e-3
    for k, p in m.named_parameters():
        if "running_" in k or sd[k].grad is None:
            continue
        if k.endswith((".0.0.bias", ".0.3.bias", ".0.7.bias")):
            continue                                            # conv bias in front of a batch-statistic BatchNorm: zero gradient
        assert rel_err(p.grad, sd[k].grad) < 2e-3, k


# ---- fp32-accurate projections on the tf32 tensor cores (the MaxViT side of precision 'tf32_conv') --------------------------
def test_split3_tf32_layout_is_bit_exact():
    """vg_split3_tf32: hi = the operand with the 13 low mantissa bits cleared, lo = x - hi (exact in fp32), laid out [hi|hi|lo] for
    the left operand and [hi|lo|hi] for the weights"""
    x = rnd(37, 64, seed=3).cuda()
    hi = (x.view(torch.int32) & -8192).view(torch.float32)
    lo = x - hi
    assert torch.equal(ops().split3_tf32(x, 0), torch.cat([hi, hi, lo], 1))
    assert torch.equal(ops().split3_tf32(x, 1), torch.cat([hi, lo, hi], 1))


@pytest.mark.parametrize("M,K,N", [(777, 128, 384), (2120, 512, 1536), (300, 2048, 512)])
def test_gemm_3xtf32_is_fp32_accurate(M, K, N):
    """one tf32 GEMM over the split operands against a float64 product.  Tolerance: 1.5 * (3K/8) * 2^-24 + 1e-6 of the largest
    output -- the truncating fp32 accumulation of the tensor core over 3K/8 instructions is what is left once the operand rounding
    is gone (measured 3e-6 at K=128, 8e-6 at 512, 3e-5 at 2048; plain tf32 8e-4; the SIMT kernel 1e-6) -- and at least 20x closer
    than plain tf32, with the fused epilogue (BN scale/shift + GELU + residual) intact"""
    A, W = rnd(M, K, seed=1).cuda(), (rnd(N, K, seed=2) / math.sqrt(K)).cuda()
    ref = A.double() @ W.double().t()
    scale = ref.abs().max().item()
    err_x3 = (ops().gemm(A, W, x3=True).double() - ref).abs().max().item() / scale
    err_simt = (ops().gemm(A, W).double() - ref).abs().max().item() / scale
    err_tf32 = (ops().gemm(A, W, tf32=True).double() - ref).abs().max().item() / scale
    tol = 1.5 * (3 * K / 8) * 2.0 ** -24 + 1e-6
    assert err_simt < 3e-6 and err_x3 < tol, (err_x3, err_simt, tol)
    assert err_tf32 > 20 * err_x3, (err_tf32, err_x3)
    s, t, r = (1 + 0.1 * rnd(N, seed=4)).cuda(), rnd(N, seed=5).cuda(), rnd(M, N, seed=6).cuda()
    got = ops().gemm(A, W, scale=s, shift=t, act=1, res=r, x3=True)
    want = F.gelu(ref * s.double() + t.double()) + r.double()
    assert (got.double() - want).abs().max().item() / want.abs().max().item() < 2 * tol


@pytest.mark.parametrize("N,cd,hid,od", [(12, 2, 1024, 1024), (12, 512, 2048, 1024), (5, 67, 1024, 256), (1, 512, 1024, 1024)])
def test_cond_mlp_wide_rows_path(N, cd, hid, od):
    """few fields x wide FiLM layers (configs[4]) go through two vg_dense_rows_fwd passes: same numbers as Linear -> SiLU -> Linear"""
    c = rnd(N, cd, seed=1).cuda()
    W0, b0 = (rnd(hid, cd, seed=2) / math.sqrt(cd)).cuda(), rnd(hid, seed=3).cuda()
    W1, b1 = (rnd(od, hid, seed=4) / math.sqrt(hid)).cuda(), rnd(od, seed=5).cuda()
    want = F.linear(F.silu(F.linear(c.double(), W0.double(), b0.double())), W1.double(), b1.double())
    assert rel_err(ops().cond_mlp(c, W0, b0, W1, b1), want) < 1e-5


def test_se_gate_wide_rows_path():
    """squeeze-excite gate at configs[4]'s widths (12 fields, 2048 channels, 512 hidden): mean -> Linear -> ReLU -> Linear -> sigmoid"""
    N, parts, C, se, HW = 12, 13, 2048, 512, 1590
    psum = rnd(N, parts, C, seed=1, scale=30.0).cuda()
    W1, W2 = (rnd(se, C, seed=2) / math.sqrt(C)).cuda(), (rnd(C, se, seed=3) / math.sqrt(se)).cuda()
    mean = psum.double().sum(1) / HW
    want = torch.sigmoid(F.linear(F.relu(F.linear(mean, W1.double())), W2.double()))
    assert rel_err(ops().se_gate(psum, HW, W1, W2), want) < 1e-5


@pytest.mark.parametrize("dh,heads", [(64, 8), (32, 4)])
@pytest.mark.parametrize("N,H,W,w,R", [(2, 14, 21, 7, 4), (1, 16, 24, 8, 0), (3, 7, 7, 7, 4)])
def test_attn_core_tensor_core_variants_match_exact_fp32(dh, heads, N, H, W, w, R):
    """the mma.sync core (3xTF32 split products for fp32 tensors = precision 'tf32_conv'; single tf32 products for bf16 tensors) against
    the exact-fp32 SIMT core on the same qkv: 2e-5 (split) and 1e-2 (bf16 storage) of the largest output"""
    o = ops()
    S, nwin = w * w + R, (H // w) * (W // w)
    qkv = rnd(N * nwin * S, 3 * heads * dh, seed=1).cuda()
    qg, kg = (1 + 0.2 * rnd(heads * dh, seed=2)).cuda(), (1 + 0.2 * rnd(heads * dh, seed=3)).cuda()
    bt = rnd((2 * w - 1) ** 2 + 1, heads, seed=4).cuda()
    exact = o.attn_core(qkv, qg, kg, bt, N, H, W, w, R, heads, dh)
    split = o.attn_core(qkv, qg, kg, bt, N, H, W, w, R, heads, dh, x3=True)
    assert rel_err(split, exact) < 2e-5
    q16 = qkv.bfloat16()
    exact16 = o.attn_core(q16.float(), qg, kg, bt, N, H, W, w, R, heads, dh)
    assert rel_err(o.attn_core(q16, qg, kg, bt, N, H, W, w, R, heads, dh), exact16) < 1e-2
    assert rel_err(o.attn_core(qkv, qg, kg, bt, N, H, W, w, R, heads, dh, tf32=True), exact) < 1e-2      # fp32 storage, single tf32 products


def test_attn_core_split_output_is_the_split_of_the_plain_output():
    """dtype code 6: the core writes its rows as [hi | hi | lo] -- bit for bit what vg_split3_tf32 makes of the plain (code 2) output"""
    o = ops()
    N, H, W, w, R, heads, dh = 2, 14, 21, 7, 4, 8, 64
    qkv = rnd(N * 6 * (w * w + R), 3 * heads * dh, seed=1).cuda()
    qg, kg = (1 + 0.2 * rnd(heads * dh, seed=2)).cuda(), (1 + 0.2 * rnd(heads * dh, seed=3)).cuda()
    bt = rnd((2 * w - 1) ** 2 + 1, heads, seed=4).cuda()
    plain = o.attn_core(qkv, qg, kg, bt, N, H, W, w, R, heads, dh, x3=True)
    split = o.attn_core(qkv, qg, kg, bt, N, H, W, w, R, heads, dh, x3=True, split_out=True)
    assert torch.equal(split, o.split3_tf32(plain, 0))


def test_new_entry_points_reject_bad_arguments():
    """error behaviour of the C ABI: bad codes come back as VitGridError with vg_last_error()'s text, nothing is launched"""
    from vit_grid_model_b200 import _lib
    o = ops()
    x = rnd(8, 64, seed=1).cuda()
    with pytest.raises(_lib.VitGridError, match="pattern"):
        o.split3_tf32(x, 2)
    out = torch.empty(8, 4, device="cuda")
    with pytest.raises(_lib.VitGridError, match="activation"):
        _lib.call("vg_dense_rows_fwd", x.data_ptr(), 8, 64, 0, x.data_ptr(), None, 4, 7, out.data_ptr(), None)
    qkv = rnd(53, 3 * 64, seed=2).cuda()
    with pytest.raises(_lib.VitGridError, match="dtype code"):
        _lib.call("vg_attn_core_fwd", 3, qkv.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), 1, 7, 7, 7, 4, 1, 64, out.data_ptr(), 0, 0, 0, None)
