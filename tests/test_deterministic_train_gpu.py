"""Deterministic training backward under torch.use_deterministic_algorithms(True) (GPU).

Kernels: every vg_*_det entry point, reached through the ops_train wrappers with the flag on, (1) gives identical bits when it
runs twice on the same inputs, and (2) agrees with its atomic twin (the flag off) to fp32 reduction-order error; the atomic twins
are checked against float64 in test_train_backward_kernels_gpu.py / test_metnet3_tf32_train_gpu.py, and the plain sums here are
also checked against float64 directly.  Accumulated outputs start from nonzero values.

Modules: a MetNet3 training step in 'fp32' (dropout 0.1, one FlatAdamW step) and the eval() x.grad graph run twice from one
state dict and one torch.manual_seed give identical loss, prediction, gradients, x.grad, BatchNorm buffers and parameters, and
agree with float64 autograd through the oracle; so do MetNet3 steps in 'bf16' and 'tf32_conv' at 128, 256 and 512 channels, and
stand-alone MaxViT steps (512 channels / 32 x 64 heads, and the reference default window 8 with 4 register tokens) in 'bf16'
and 'fp32'."""
import contextlib
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import synth

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64 = torch.float64


def ot():
    from vit_grid_model_b200 import ops_train
    return ops_train


def ops():
    from vit_grid_model_b200 import ops
    return ops


def note(**kv):
    print("MEASURED", kv)


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def rnd(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=gen(seed), device=DEV) * scale


def rel(got, ref):
    g, r = got.double(), ref.double()
    return ((g - r).abs().max() / r.abs().max().clamp_min(1e-30)).item()


@contextlib.contextmanager
def deterministic(on=True, warn_only=False):
    prev, prev_w = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_w)


def three_ways(fn, bound, label, **info):
    """fn() -> list of output tensors.  The flag on twice: identical bits; against the flag off: within `bound` (max error relative
    to the largest reference magnitude, per tensor).  -> the deterministic outputs"""
    with deterministic(False):
        ref = [t.clone() for t in fn()]
    with deterministic(True):
        a = [t.clone() for t in fn()]
    with deterministic(True, warn_only=True):
        b = [t.clone() for t in fn()]
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    errs = [rel(x, r) for x, r in zip(a, ref)]
    note(test=label, **info, vs_atomic=max(errs))
    assert max(errs) < bound, errs
    return a


# ------------------------------------------------------------------------------------------ MetNet3 Block backward
BLOCK_GEOMS = {"3x14x14": (3, 14, 14),           # 225 pixels per field: field boundaries inside blocks, a partial last block
               "192x6x7": (192, 6, 7),           # 56 pixels per field: a warp spans several fields
               "1x518x518": (1, 518, 518)}


def _block_inputs(N, HP, WP, C, xdtype, seed=11):
    Q = ops().pg_pixels(N, HP, WP)
    dY = rnd(Q, C, seed=seed)
    xhat = rnd(Q, C, seed=seed + 1).to(xdtype)
    rstd = 0.5 + torch.rand(Q, generator=gen(seed + 2), device=DEV)
    rstd[: Q // 7] = 1e-5 ** -0.5                            # clamped rows: no variance gradient
    mask = torch.randint(-2 ** 31, 2 ** 31 - 1, (Q, C // 32), generator=gen(seed + 3), device=DEV, dtype=torch.int64).to(torch.int32)
    g = 1 + 0.2 * rnd(C, seed=seed + 4)
    film = 0.5 * rnd(N, 2 * C, seed=seed + 5)
    return dY, (xhat, rstd, mask), g, film


@pytest.mark.parametrize("geom", list(BLOCK_GEOMS))
@pytest.mark.parametrize("dt", ["bf16_bf16", "bf16_f32", "f32_f32"])
def test_conv_ln_bwd_det(geom, dt):
    N, HP, WP = BLOCK_GEOMS[geom]
    xdt = torch.bfloat16 if dt.startswith("bf16") else torch.float32
    odt = torch.bfloat16 if dt.endswith("bf16") else torch.float32
    dY, saved, g, film = _block_inputs(N, HP, WP, 128, xdt)
    want_border = odt == torch.float32

    def run():
        dconv, sums, border = ot().conv_ln_bwd(dY, saved, g, film, 1e-5, N, HP, WP, odt, want_border=want_border)
        return [dconv.float(), sums] + ([border] if want_border else [])
    out = three_ways(run, 2e-5, "conv_ln_bwd", geom=geom, dt=dt)
    assert torch.isfinite(out[1]).all()


@pytest.mark.parametrize("geom", ["3x14x14", "192x6x7"])
@pytest.mark.parametrize("C", [256, 384, 512])
def test_conv_ln_bwd_wide_det(geom, C):
    N, HP, WP = BLOCK_GEOMS[geom]
    dY, saved, g, film = _block_inputs(N, HP, WP, C, torch.float32, seed=21)

    def run():
        dconv, sums, border = ot().conv_ln_bwd(dY, saved, g, film, 1e-5, N, HP, WP, torch.float32, want_border=True)
        return [dconv, sums, border]
    three_ways(run, 2e-5, "conv_ln_bwd_wide", geom=geom, C=C)


# ------------------------------------------------------------------------------------------ small reductions
@pytest.mark.parametrize("C", [128, 512])
@pytest.mark.parametrize("hdt", [torch.bfloat16, torch.float32])
def test_head_bwd_det(C, hdt):
    N, HP, WP, H, W, pads, std = 3, 28, 28, 26, 25, (1, 2, 1, 1), 7.5
    h = rnd(ops().pg_pixels(N, HP, WP), C, seed=31).to(hdt)
    w = rnd(C, seed=32)
    dpred = rnd(N, H, W, seed=33)

    def run():
        dw, db = torch.full((C,), 0.5, device=DEV), torch.full((1,), 0.5, device=DEV)
        dH = ot().head_bwd(dpred, h, w, std, N, HP, WP, H, W, pads, dw, db)
        return [dH, dw, db]
    dH, dw, db = three_ways(run, 1e-5, "head_bwd", C=C, dtype=str(hdt))
    d = torch.zeros(N, HP, WP, dtype=F64, device=DEV)
    d[:, 1:1 + H, 1:1 + W] = dpred.double() * std
    hf = ops().pg_to_nchw(h.float(), N, HP, WP).double()
    e = dict(dw=rel(dw - 0.5, (hf * d.unsqueeze(1)).sum((0, 2, 3))), db=rel(db - 0.5, d.sum().view(1)))
    note(test="head_bwd_f64", C=C, **e)
    assert max(e.values()) < 6e-7


@pytest.mark.parametrize("C", [128, 512])
def test_convT2_bwd_gather_det(C):
    N, Hl, Wl = 2, 14, 14
    dup = rnd(N, C, 2 * Hl, 2 * Wl, seed=41)
    dupp = ops().pg_from_nchw(dup, torch.float32)

    def run():
        dbias = torch.full((C,), 0.5, device=DEV)
        G = ot().convT2_bwd_gather(dupp, N, Hl, Wl, C, torch.float32, dbias)
        return [G, dbias]
    G, dbias = three_ways(run, 1e-5, "convT2_bwd_gather", C=C)
    e = rel(dbias - 0.5, dup.double().sum((0, 2, 3)))
    note(test="convT2_bwd_gather_f64", C=C, dbias=e)
    assert e < 1.1e-6


@pytest.mark.parametrize("N", [1, 192])
@pytest.mark.parametrize("C", [128, 512])
def test_pg_field_sum_det(N, C):
    HP, WP = (518, 518) if N == 1 else (8, 9)
    x = rnd(N, C, HP, WP, seed=51)
    xp = ops().pg_from_nchw(x, torch.float32)
    (fs,) = three_ways(lambda: [ot().pg_field_sum(xp, N, HP, WP)], 1e-5, "pg_field_sum", N=N, C=C)
    e = rel(fs, x.double().sum((2, 3)))
    note(test="pg_field_sum_f64", N=N, C=C, err=e)
    assert e < 1e-6


@pytest.mark.parametrize("M,C", [(100003, 96), (4099, 512)])
def test_colsum_det(M, C):
    x = rnd(M, C, seed=61)

    def run():
        out = torch.full((C,), 0.25, device=DEV)
        ot().colsum(x, out)
        return [out]
    (out,) = three_ways(run, 1e-5, "colsum", M=M, C=C)
    e = rel(out - 0.25, x.double().sum(0))
    note(test="colsum_f64", M=M, C=C, err=e)
    assert e < 1e-6


def test_time_terms_and_embed_bwd_det():
    B, L, le, te, Cout, c_data = 4, 6, 8, 4, 128, 75
    N, ntc = B * L, le + 3 * te
    c_in = c_data + ntc
    border, sumD, tres = rnd(N, 8, Cout, seed=71), rnd(N, Cout, seed=72), rnd(N, Cout, seed=73)
    temb, w3, w1 = rnd(N, ntc, seed=74), rnd(Cout, c_in, 3, 3, seed=75), rnd(Cout, c_in, 1, 1, seed=76)
    ts = torch.zeros(B, 7, 4, device=DEV)
    ts[:, 6, 1] = torch.tensor([0, 12, 12, 3], dtype=torch.float32)
    ts[:, 6, 2] = torch.tensor([5, 5, 31, 0], dtype=torch.float32)
    ts[:, 6, 3] = torch.tensor([24, 1, 1, 1], dtype=torch.float32)
    dcond = rnd(N, le, seed=77)

    def run():
        dw3, dw1, db1 = torch.full_like(w3, 0.5), torch.full_like(w1, 0.5), torch.full((Cout,), 0.5, device=DEV)
        dtemb = ot().time_terms_bwd(border, sumD, tres, temb, w3, w1, c_data, dw3, dw1, db1)
        tabs = [torch.full((L + 1, le), 0.5, device=DEV), torch.full((13, te), 0.5, device=DEV),
                torch.full((32, te), 0.5, device=DEV), torch.full((25, te), 0.5, device=DEV)]
        ot().time_embed_bwd(dtemb, dcond, ts, B, L, le, te, *tabs)
        return [dw3, dw1, db1, dtemb] + tabs
    out = three_ways(run, 1e-5, "time_terms_embed_bwd")
    e = rel(out[2] - 0.5, tres.double().sum(0))
    note(test="time_terms_db1_f64", err=e)
    assert e < 1e-6


# ------------------------------------------------------------------------------------------ attention
# (win, R, Hl, Wl): S = 16, 53, 64 (the 64-slot kernels), 68 (the reference default 8x8 + 4 registers) and 128 (the long-window
# kernels); two or more windows per field
ATTN_CASES = {"S16_w4_R0": (4, 0, 16, 16), "S53_w7_R4": (7, 4, 14, 21), "S64_w8_R0": (8, 0, 16, 24), "S68_w8_R4": (8, 4, 16, 24),
              "S128_w11_R7": (11, 7, 22, 33)}


def _core_operands(case, heads, dh, N=2):
    win, R, Hl, Wl = ATTN_CASES[case]
    S, nwin = win * win + R, (Hl // win) * (Wl // win)
    rows, inner = N * nwin * S, heads * dh
    qkv, datt = rnd(rows, 3 * inner, seed=81), rnd(rows, inner, seed=82)
    qg, kg = 1 + 0.1 * rnd(inner, seed=83), 1 + 0.1 * rnd(inner, seed=84)
    bt = 0.1 * rnd((2 * win - 1) ** 2 + 1, heads, seed=85)
    return win, R, Hl, Wl, S, nwin, qkv, datt, qg, kg, bt


@pytest.mark.parametrize("drop", [(0, 0, 0), (1234, 3, 26)])
@pytest.mark.parametrize("dh", [32, 64])
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("case", list(ATTN_CASES))
def test_attn_core_bwd_det(case, mode, dh, drop):
    """modes 0 (exact-fp32 SIMT; S > 64: the long-window kernel) and 2 (bf16 mma.sync; S > 64: its long-window kernel): bits twice,
    the atomic twin, and float64 -- the bias-table gradient of dbias_gather's offset arithmetic included -- within the bounds of
    the atomic kernels (test_maxvit_long_window_train_gpu.CORE_TOL)"""
    from test_maxvit_long_window_train_gpu import CORE_TOL, _core_bwd_ref
    N, heads = 2, 4
    win, R, Hl, Wl, S, nwin, qkv, datt, qg, kg, bt = _core_operands(case, heads, dh, N)

    def run():
        dqg, dkg, dbt = torch.full_like(qg, 0.5), torch.full_like(kg, 0.5), torch.full_like(bt, 0.5)
        dqkv = ot().attn_core_bwd(qkv, datt, qg, kg, bt, N, Hl, Wl, win, R, heads, dh, dqg, dkg, dbt, tf32=mode == 2, drop=drop)
        return [dqkv, dqg, dkg, dbt]
    dqkv, dqg, dkg, dbt = three_ways(run, 2e-5 if mode == 0 else 1e-4, "attn_core_bwd", case=case, mode=mode, dh=dh, drop=drop[2])
    pmask = None
    if drop[2]:
        pm, _ = ot().dropout_masks(drop, N * nwin, heads, 128, slots=64 if S <= 64 else 128)
        pmask = pm[:, :, :S, :S].to(F64) * (256.0 / (256 - drop[2]))
    ref = _core_bwd_ref(qkv, datt, qg, kg, bt, S, win, R, heads, dh, pmask, bf16_ops=mode == 2)
    e = dict(dqkv=rel(dqkv, ref[0]), dq_gamma=rel(dqg - 0.5, ref[1]), dk_gamma=rel(dkg - 0.5, ref[2]), dbias=rel(dbt - 0.5, ref[3]))
    note(test="attn_core_bwd_f64", case=case, mode=mode, dh=dh, drop=drop[2], **e)
    bad = {k: v for k, v in e.items() if not v < CORE_TOL[mode][k]}
    assert not bad, bad


@pytest.mark.parametrize("drop", [(0, 0, 0), (1234, 3, 26)])
@pytest.mark.parametrize("case", ["S16_w4_R0", "S53_w7_R4", "S64_w8_R0"])
def test_attn_core_bwd_tc_det(case, drop):
    """mode 3 (the tcgen05 kernel on bf16 tensors, S <= 64, dim_head 32, att re-materialised): bits twice and the atomic twin"""
    N, heads, dh = 2, 4, 32
    win, R, Hl, Wl, S, nwin, qkv, datt, qg, kg, bt = _core_operands(case, heads, dh, N)
    qkv16, datt16 = qkv.to(torch.bfloat16), datt.to(torch.bfloat16)

    def run():
        dqg, dkg, dbt = torch.full_like(qg, 0.5), torch.full_like(kg, 0.5), torch.full_like(bt, 0.5)
        dqkv, att = ot().attn_core_bwd(qkv16, datt16, qg, kg, bt, N, Hl, Wl, win, R, heads, dh, dqg, dkg, dbt, want_att=True, drop=drop)
        return [dqkv.float(), att.float(), dqg, dkg, dbt]
    three_ways(run, 1e-4, "attn_core_bwd_tc", case=case, drop=drop[2])


@pytest.mark.parametrize("reg_per_field", [False, True])
@pytest.mark.parametrize("C", [128, 512])
@pytest.mark.parametrize("grid_mode", [0, 1])
def test_attn_gather_bwd_det(grid_mode, C, reg_per_field):
    N, Hl, Wl, win, R = 3, 14, 21, 7, 4
    S, nwin = win * win + R, (Hl // win) * (Wl // win)
    x, film = rnd(N, Hl, Wl, C, seed=91), 0.5 * rnd(N, 2 * C, seed=92)
    reg = rnd(N, R, C, seed=93) if reg_per_field else rnd(R, C, seed=93)
    dtok, dx_out, dreg_res = rnd(N * nwin * S, C, seed=94), rnd(N, Hl, Wl, C, seed=95), rnd(N, R, C, seed=96)

    def run():
        dreg_in, dfilm = torch.full_like(reg, 0.5), torch.full((N, 2 * C), 0.5, device=DEV)
        dx_in = ot().attn_gather_bwd(x, reg, film, dtok, dx_out, dreg_res, 0.5, dreg_in, dfilm, win, R, grid_mode)
        return [dx_in, dreg_in, dfilm]
    three_ways(run, 1e-5, "attn_gather_bwd", grid_mode=grid_mode, C=C, reg_per_field=reg_per_field)


# ------------------------------------------------------------------------------------------ module steps
def _metnet3(cfg, precision, dropout, train=True):
    from vit_grid_model_b200 import MetNet3
    m = MetNet3(**cfg.metnet3_kwargs(), dropout=dropout)
    m.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
    m = m.cuda().set_precision(precision)
    return m.train() if train else m.eval()


def _metnet3_step(cfg, precision, train=True):
    """one FlatAdamW step (train) or x.grad of the frozen graph (eval) -> every tensor the step produces"""
    from vit_grid_model_b200 import FlatAdamW, focal_r_loss
    x, ts, _ = synth.make_inputs(cfg, 2, seed=31)
    target = torch.rand(2, cfg.L, cfg.H, cfg.W, generator=torch.Generator().manual_seed(32)) * 40
    torch.manual_seed(1234)
    m = _metnet3(cfg, precision, 0.1, train)
    opt = FlatAdamW(m, lr=1e-4)
    xg = x.cuda().requires_grad_(True)
    pred = m(xg, timestamps=ts.cuda())
    loss = focal_r_loss(pred, target.cuda())
    loss.backward()
    out = {"loss": loss.detach().clone(), "pred": pred.detach().clone(), "x.grad": xg.grad.clone()}
    out.update({"grad." + k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None})
    if train:
        opt.step()
        out.update({"param." + k: p.detach().clone() for k, p in m.named_parameters()})
    out.update({"buffer." + k: b.clone() for k, b in m.named_buffers()})
    torch.cuda.synchronize()
    return out


def _assert_identical(a, b):
    assert a.keys() == b.keys()
    bad = [k for k in a if not torch.equal(a[k], b[k])]
    assert not bad, bad[:10]


MODULE_STEPS = {                          # (config, precision): the widths and precisions training is built for
    "128_bf16": (synth.CFG_SMALL128, "bf16"), "128_fp32": (synth.CFG_SMALL128, "fp32"), "128_tf32_conv": (synth.CFG_SMALL128, "tf32_conv"),
    "256_tf32_conv": (synth.CFG_WIDE256, "tf32_conv"), "512_tf32_conv": (synth.CFG_WIDE512, "tf32_conv")}


@pytest.mark.parametrize("step", list(MODULE_STEPS))
def test_metnet3_step_is_bit_reproducible(step):
    cfg, precision = MODULE_STEPS[step]
    with deterministic(True):
        a = _metnet3_step(cfg, precision, True)
        b = _metnet3_step(cfg, precision, True)
    _assert_identical(a, b)
    assert all(torch.isfinite(v).all() for v in a.values())


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_metnet3_eval_x_grad_is_bit_reproducible(precision):
    cfg = synth.CFG_SMALL128
    with deterministic(True):
        a = _metnet3_step(cfg, precision, False)
        b = _metnet3_step(cfg, precision, False)
    _assert_identical(a, b)


def test_metnet3_fp32_det_step_matches_float64():
    """the deterministic step's gradients against float64 autograd through the oracle (dropout off), with the per-tensor rule of
    test_metnet3_tf32_train_gpu._check_grads and the figures that file records for this 128-channel fp32 step with atomics: global
    relative L2 2.7e-3, worst tensor 8.0e-3 (resnet2.blocks.0.block1.norm.b / proj.bias).  Measured for the deterministic step on
    a B200 at 1000 W: global 2.703e-3, worst tensor 8.04e-3 (resnet2.blocks.0.block1.proj.bias), i.e. the same figures; the
    bounds keep those two figures at their recorded two digits"""
    from oracle.metnet3_oracle import metnet3_forward
    from test_metnet3_tf32_train_gpu import _check_grads
    cfg = synth.CFG_SMALL128
    x, ts, _ = synth.make_inputs(cfg, 2, seed=31)
    dpred = torch.randn(2, cfg.L, cfg.H, cfg.W, generator=torch.Generator().manual_seed(32))
    m = _metnet3(cfg, "fp32", 0.0)
    with deterministic(True):
        pred = m(x.cuda(), timestamps=ts.cuda())
        pred.backward(dpred.cuda())
    sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=0)
    for k, v in sd.items():
        if v.is_floating_point():
            sd[k] = v.to(DEV, F64)
            if "running_" not in k and k != "pm25_boundaries":
                sd[k].requires_grad_(True)
        else:
            sd[k] = v.to(DEV)
    ref = metnet3_forward(x.to(DEV, F64), ts.cpu(), sd, cfg, training=True)
    ref.backward(dpred.to(DEV, F64))
    grads = {k: p.grad for k, p in m.named_parameters()}
    pairs = [(k, grads[k], sd[k].grad) for k in grads if sd[k].grad is not None]
    e_pred = rel(pred.detach(), ref.detach())
    note(test="metnet3_fp32_det_vs_f64", pred=e_pred)
    gl2 = _check_grads(pairs, grads, False, 8.05e-3, 0.9999, "metnet3_fp32_det")
    assert e_pred < 1e-4 and gl2 < 2.75e-3, (e_pred, gl2)


MAXVIT_STEPS = {                          # (dim, depth, heads, dim_head, window, registers, precision)
    "512_32x64_w7_bf16": (512, 2, 32, 64, 7, 4, "bf16"), "512_32x64_w7_fp32": (512, 2, 32, 64, 7, 4, "fp32"),
    "128_w8_R4_bf16": (128, 2, 32, 32, 8, 4, "bf16"), "128_w8_R4_fp32": (128, 2, 32, 32, 8, 4, "fp32")}


def _maxvit_step(shape, train=True):
    """one training step of a stand-alone MaxViT (dropout 0.1 as the reference default, an AdamW step) -> every tensor it produces"""
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh, win, R, precision = MAXVIT_STEPS[shape]
    sd = synth.make_state_dict(synth.maxvit_multistage_spec(dim, depth, 2, heads, dh, win, 4, 0.25, R), seed=5)
    torch.manual_seed(4321)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=win, num_register_tokens=R, dropout=0.1)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().set_precision(precision)
    m = m.train() if train else m.eval()
    g = torch.Generator().manual_seed(12)
    Hl, Wl = (2 * win, 3 * win)
    x = torch.randn(3, dim, Hl, Wl, generator=g).cuda().requires_grad_(True)
    cond = torch.randn(3, 2, generator=g).cuda()
    dy = torch.randn(3, m.dim_out, Hl, Wl, generator=g).cuda()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-4, foreach=False)
    y = m(x, cond)
    loss = (y * dy).sum()
    loss.backward()
    out = {"loss": loss.detach().clone(), "y": y.detach().clone(), "x.grad": x.grad.clone()}
    out.update({"grad." + k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None})
    if train:
        opt.step()
        out.update({"param." + k: p.detach().clone() for k, p in m.named_parameters()})
    out.update({"buffer." + k: b.clone() for k, b in m.named_buffers()})
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("shape", list(MAXVIT_STEPS))
def test_maxvit_step_is_bit_reproducible(shape):
    with deterministic(True):
        a = _maxvit_step(shape)
        b = _maxvit_step(shape)
    _assert_identical(a, b)
    assert all(torch.isfinite(v).all() for v in a.values())


def test_maxvit_eval_x_grad_is_bit_reproducible():
    with deterministic(True):
        a = _maxvit_step("128_w8_R4_fp32", train=False)
        b = _maxvit_step("128_w8_R4_fp32", train=False)
    _assert_identical(a, b)
