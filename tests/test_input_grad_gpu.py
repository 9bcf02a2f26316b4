"""Gradients with respect to the input grids (GPU): the adjoint of the input preparation (vg_prepare_bwd), BatchNorm backward
with running statistics (vg_bn_bwd_frozen), and x.grad of MetNet3 / MetNet3_with_stn_imgs / MaxViT in train() mode and in
eval() mode (the frozen-BatchNorm graph, built only when the input requires grad), against float64 autograd through the
CPU oracle.  The oracle is functional and clones x first, so x.grad there is the reference module's input gradient."""
import math
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


def lib():
    from vit_grid_model_b200 import _lib
    return _lib


def ops():
    from vit_grid_model_b200 import ops as o
    return o


# ------------------------------------------------------------------------------------------ vg_prepare_bwd
def _frame(B, T, C, H, W):
    ph, pw = (14 - H) % 14, (14 - W) % 14
    return H + ph, W + pw, (pw // 2, pw - pw // 2, ph // 2, ph - ph // 2), (T * C + 63) // 64 * 64


def _prepare_bwd_raw(g, B, T, C, H, W, pads, HP, WP, std, extra, fill):
    """the ABI on an output prefilled with `fill` (every element must be overwritten)"""
    dx = torch.full((B, T, C, H, W), fill, dtype=torch.float32, device=g.device)
    pl, _, pt, _ = pads
    lib().call("vg_prepare_bwd", g.data_ptr(), B, T, C, H, W, pt, pl, HP, WP, g.shape[1], float(std), int(extra), dx.data_ptr(),
               torch.cuda.current_stream().cuda_stream)
    return dx


PREP_GEOMS = {                            # (B, T, H, W): the 12-hour model's 82x67 grid, an odd small grid, the 512x512 domain
    "12hr": (2, 25, 82, 67),
    "odd": (3, 3, 13, 11),
    "512": (1, 25, 512, 512),
}


@pytest.mark.parametrize("stn", [False, True])
@pytest.mark.parametrize("geom", list(PREP_GEOMS))
def test_prepare_bwd_is_the_adjoint_of_prepare(geom, stn):
    o = ops()
    B, T, H, W = PREP_GEOMS[geom]
    C = 25 if stn else 24                                     # MetNet3_with_stn_imgs: variable 24, standardised too
    extra = 24 if stn else -1
    HP, WP, pads, cpad = _frame(B, T, C, H, W)
    std = 15.0
    gen = torch.Generator(device="cuda").manual_seed(7)
    rows = o.pg_pixels(B, HP, WP)
    g = torch.randn(rows, cpad, device="cuda", generator=gen)  # pad rows / columns and channels >= T*C hold values too
    dx = _prepare_bwd_raw(g, B, T, C, H, W, pads, HP, WP, std, extra, float("nan"))
    assert not torch.isnan(dx).any()
    # direct: the frame pixels of the first T*C channels, PM2.5 channels (and the station image) divided by std -- within
    # half an ulp of the float64 quotient (the kernel divides once, correctly rounded)
    pl, _, pt, _ = pads
    ref = g.view(B * (HP + 1) + 1, WP + 1, cpad)[:B * (HP + 1)].view(B, HP + 1, WP + 1, cpad)[:, 1 + pt:1 + pt + H, 1 + pl:1 + pl + W, :T * C]
    ref = ref.permute(0, 3, 1, 2).reshape(B, T, C, H, W).double()
    pm = [4, 10, 16, 22] + ([24] if stn else [])
    ref[:, :, pm] /= float(torch.tensor(std, dtype=torch.float32))
    err = (dx.double() - ref).abs()
    half_ulp = 0.5 * (torch.nextafter(dx.abs(), torch.tensor(math.inf, device="cuda")) - dx.abs()).double()
    assert bool((err <= half_ulp).all()), err.max().item()
    del ref, err, half_ulp
    # adjoint identity <prepare(x), g> = <x, prepare_bwd(g)> (the linear part of prepare: mean 0)
    x = torch.randn(B, T, C, H, W, device="cuda", generator=gen)
    xs = x.clone()
    if stn:
        o.standardise_channel_(xs, 24, 0.0, std)
    px = o.prepare(xs, pads, HP, WP, cpad, 0.0, std, torch.float32)
    lhs = (px.double() * g.double()).sum().item()
    rhs = (x.double() * dx.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-6 * (px.double().abs() * g.double().abs()).sum().item(), (lhs, rhs)


# ------------------------------------------------------------------------------------------ vg_bn_bwd_frozen
@pytest.mark.parametrize("gated", [False, True])
@pytest.mark.parametrize("M,C", [(282240, 128), (282240, 512), (147, 128), (147, 512)])
def test_bn_bwd_frozen_matches_autograd(M, C, gated):
    """M = 282,240 = 192 fields x 42 x 35 pixels: the MBConv rows of a 16-sample training step at the 12-hour geometry"""
    from vit_grid_model_b200 import ops_train as ot
    gen = torch.Generator(device="cuda").manual_seed(M + C)
    nf = 192 if M > 1000 else 3
    raw = torch.randn(M, C, device="cuda", generator=gen) * 1.5 + 0.3
    dout = torch.randn(M, C, device="cuda", generator=gen)
    bn = torch.nn.BatchNorm2d(C).cuda().eval()
    with torch.no_grad():
        bn.weight.copy_(0.5 + torch.rand(C, device="cuda", generator=gen))
        bn.bias.copy_(0.1 * torch.randn(C, device="cuda", generator=gen))
        bn.running_mean.copy_(0.3 * torch.randn(C, device="cuda", generator=gen))
        bn.running_var.copy_(0.5 + 2 * torch.rand(C, device="cuda", generator=gen))
    fgate = torch.rand(nf, C, device="cuda", generator=gen) if gated else None
    fadd = 0.1 * torch.randn(nf, C, device="cuda", generator=gen) if gated else None
    st = ot.bn_frozen_stats(bn)
    dgamma = torch.zeros(C, device="cuda")
    dbeta = torch.zeros(C, device="cuda")
    draw = ot.bn_bwd_frozen(dout, raw, st, 1, dgamma, dbeta, fgate=fgate, fadd=fadd, rows_per_field=M // nf if gated else 0)
    # float64 autograd of F.batch_norm(training=False) -> GELU
    r64 = raw.double().requires_grad_(True)
    w64 = bn.weight.detach().double().requires_grad_(True)
    b64 = bn.bias.detach().double().requires_grad_(True)
    y = F.gelu(F.batch_norm(r64, bn.running_mean.double(), bn.running_var.double(), w64, b64, False, 0.0, bn.eps))
    g = dout.double()
    if gated:
        g = g * fgate.double().repeat_interleave(M // nf, 0) + fadd.double().repeat_interleave(M // nf, 0)
    y.backward(g)
    for name, got, ref in (("draw", draw, r64.grad), ("dgamma", dgamma, w64.grad), ("dbeta", dbeta, b64.grad)):
        e = ((got.double() - ref).abs().max() / ref.abs().max()).item()
        assert e < 1e-5, (name, e)


# ------------------------------------------------------------------------------------------ MetNet3
def _model(cfg, precision, train, seed=0, stn=False, dropout=0.0):
    from vit_grid_model_b200 import MetNet3, MetNet3_with_stn_imgs
    cls = MetNet3_with_stn_imgs if stn else MetNet3
    m = cls(**cfg.metnet3_kwargs(), dropout=dropout)
    m.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=seed), strict=True)
    m = m.cuda().set_precision(precision)
    return m.train() if train else m.eval()


def _oracle(cfg, x, ts, dpred, training, seed=0, stn=False):
    """float64 autograd through the oracle -> (pred, x.grad, {param: grad})"""
    sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=seed)
    for k, v in sd.items():
        if v.is_floating_point():
            sd[k] = v.double()
            if "running_" not in k and k != "pm25_boundaries":
                sd[k].requires_grad_(True)
    x64 = x.detach().cpu().double().requires_grad_(True)
    pred = metnet3_forward(x64, ts.cpu(), sd, cfg, training=training, stn_imgs=stn)
    pred.backward(dpred.cpu().double())
    return pred.detach(), x64.grad, {k: v.grad for k, v in sd.items() if v.requires_grad}


def _errs(got, ref):
    g, r = got.detach().double().cpu(), ref.double()
    emax = ((g - r).abs().max() / max(r.abs().max().item(), 1e-2)).item()
    el2 = ((g - r).norm() / max(r.norm().item(), 1e-2)).item()
    cos = (torch.dot(g.reshape(-1), r.reshape(-1)) / (g.norm() * r.norm()).clamp_min(1e-30)).item()
    return emax, el2, cos


def _check_fp32(pairs):
    """the fp32 gradient bounds of test_train_gpu.py: max error < 2e-2 and L2 < 5e-3 of the tensor's largest entry / norm"""
    bad = []
    for name, got, ref in pairs:
        emax, el2, _ = _errs(got, ref)
        if emax > 2e-2 or el2 > 5e-3:
            bad.append((name, round(emax, 6), round(el2, 6)))
    assert not bad, bad[:20]


def _check_mixed(pairs):
    """the mixed-precision gradient bounds of test_train_gpu.py: per-tensor cosine >= 0.95, global relative L2 < 0.2"""
    bad, num, den = [], 0.0, 0.0
    for name, got, ref in pairs:
        g, r = got.detach().double().cpu(), ref.double()
        num += (g - r).pow(2).sum().item()
        den += r.pow(2).sum().item()
        _, _, cos = _errs(got, ref)
        if r.norm().item() > 1e-2 and cos < 0.95:
            bad.append((name, round(cos, 4)))
    assert not bad, bad[:20]
    assert (num / den) ** 0.5 < 0.2, (num / den) ** 0.5


def _same(a, b):
    """equal up to the run-to-run rounding of the backward: several of its sums (LayerNorm / head / embedding / attention
    parameter gradients, dfilm) are float atomics whose order varies between launches, so two identical steps agree to
    ~1e-7 of the largest entry (measured on a B200: <= 5.8e-7 of max(|b|, 1)), not bit for bit"""
    return ((a - b).abs().max() <= 1e-5 * max(b.abs().max().item(), 1.0)).item()


def _inputs(cfg, B=2, seed=31):
    x, ts, _ = synth.make_inputs(cfg, B, seed=seed)
    dpred = torch.randn(B, cfg.L, cfg.H, cfg.W, generator=torch.Generator().manual_seed(seed + 1))
    return x, ts, dpred


def test_train_mode_x_grad_fp32():
    cfg = synth.CFG_SMALL128
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, "fp32", True)
    xg = x.cuda().requires_grad_(True)
    m(xg, timestamps=ts.cuda()).backward(dpred.cuda())
    m0 = _model(cfg, "fp32", True)                     # the same step without x.requires_grad
    m0(x.cuda(), timestamps=ts.cuda()).backward(dpred.cuda())
    torch.cuda.synchronize()
    g0 = {k: p.grad for k, p in m0.named_parameters()}
    for k, p in m.named_parameters():
        zb = re.fullmatch(r"(vit\.layers\.\d+\.0\.(?:fn\.)?)([037])\.bias", k)
        if zb:
            # conv bias in front of a batch-statistic BatchNorm: the gradient is analytically zero and both runs hold the rounding
            # noise of an atomic column sum (~1e-4 here), which differs from run to run; as in test_train_kernels_gpu.py it must
            # stay far below the BatchNorm beta gradient next to it (measured on a B200: noise norm 1.9e-3 .. 3.7e-3 against beta
            # gradient norms of 2.4e3 .. 3.0e3, ratio <= 1.3e-6)
            beta = g0[zb.group(1) + str(int(zb.group(2)) + 1) + ".bias"].norm().item()
            assert max(p.grad.norm().item(), g0[k].norm().item()) < 1e-3 * beta, (k, p.grad.norm().item(), beta)
        else:
            assert _same(p.grad, g0[k]), k                         # measured: <= 1.7e-6 of max(|g|, 1)
    _, gx, _ = _oracle(cfg, x, ts, dpred, True)
    _check_fp32([("x", xg.grad, gx)])                          # measured on a B200: max 8.2e-3, L2 2.8e-3


def _eval_state(m):
    return ({k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k},
            m._dropout_state, getattr(m.vit, "_dropout_state", None))


def test_eval_mode_x_grad_fp32():
    cfg = synth.CFG_SMALL128
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, "fp32", False, dropout=0.1)
    m.next_dropout_seed()                              # a seed state that a wrong advance would change
    with torch.no_grad():
        y_inf = m(x.cuda(), timestamps=ts.cuda())
    bufs, s0, s1 = _eval_state(m)

    def run():
        for p in m.parameters():
            p.grad = None
        xg = x.cuda().requires_grad_(True)
        pred = m(xg, timestamps=ts.cuda())
        assert pred.grad_fn is not None
        pred.backward(dpred.cuda())
        torch.cuda.synchronize()
        return pred.detach(), xg.grad, {k: p.grad.clone() for k, p in m.named_parameters()}

    pred, gx, grads = run()
    assert ((pred - y_inf).abs().max() / y_inf.abs().max()).item() < 1e-4
    bufs1, t0, t1 = _eval_state(m)
    assert (t0, t1) == (s0, s1)
    for k, v in bufs.items():
        assert torch.equal(v, bufs1[k]), k
    pred2, gx2, grads2 = run()                         # the forward is deterministic: identical bits
    assert torch.equal(pred, pred2) and _same(gx, gx2)
    assert [k for k in grads if not _same(grads[k], grads2[k])] == []
    _, ogx, ograds = _oracle(cfg, x, ts, dpred, False)
    # measured on a B200: x max 1.2e-3, L2 3.7e-4; worst parameter max 3.4e-3, L2 1.0e-3
    _check_fp32([("x", gx, ogx)] + [(k, grads[k], ograds[k]) for k in grads])


@pytest.mark.parametrize("train", [True, False])
def test_mixed_precision_x_grad(train):
    cfg = synth.CFG_SMALL128
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, "bf16", train)
    xg = x.cuda().requires_grad_(True)
    m(xg, timestamps=ts.cuda()).backward(dpred.cuda())
    torch.cuda.synchronize()
    _, ogx, ograds = _oracle(cfg, x, ts, dpred, train)
    # measured on a B200: train() min cosine 0.975 (x 0.990), global L2 0.139; eval() min cosine 0.993 (x 0.995), global L2 0.059
    _check_mixed([("x", xg.grad, ogx)] + [(k, p.grad, ograds[k]) for k, p in m.named_parameters()])


@pytest.mark.parametrize("train", [True, False])
def test_permuted_view_receives_its_gradient(train):
    """the channels-last view of evaluation_vit.py:248-249 gets the same x.grad as the contiguous tensor"""
    cfg = synth.CFG_SMALL128
    x, ts, dpred = _inputs(cfg)
    grads = []
    for view in (False, True):
        m = _model(cfg, "fp32", train)
        if view:
            base = x.permute(0, 3, 4, 1, 2).contiguous().cuda().requires_grad_(True)
            xin = base.permute(0, 3, 4, 1, 2)
            assert not xin.is_contiguous()
        else:
            base = xin = x.cuda().requires_grad_(True)
        m(xin, timestamps=ts.cuda()).backward(dpred.cuda())
        grads.append(base.grad.permute(0, 3, 4, 1, 2) if view else base.grad)
    assert _same(grads[0], grads[1])


def test_stn_variant_leaf_raises_and_non_leaf_matches_oracle():
    cfg = synth.CFG_STN_SMALL128
    x, ts, dpred = _inputs(cfg)
    m = _model(cfg, "fp32", False, stn=True)
    leaf = x.cuda().requires_grad_(True)
    with pytest.raises(RuntimeError, match="leaf Variable that requires grad"):
        m(leaf, timestamps=ts.cuda())
    assert torch.equal(leaf.detach().cpu(), x)                    # refused before the tensor was touched
    raw = x.cuda().requires_grad_(True)
    m(raw * 1.0, timestamps=ts.cuda()).backward(dpred.cuda())
    torch.cuda.synchronize()
    _, ogx, ograds = _oracle(cfg, x, ts, dpred, False, stn=True)
    # measured on a B200: x max 6.7e-6 (variable 24: 3.9e-6), worst parameter max 9.3e-6
    _check_fp32([("x", raw.grad, ogx), ("x[:, :, 24]", raw.grad[:, :, 24], ogx[:, :, 24])]
                + [(k, p.grad, ograds[k]) for k, p in m.named_parameters()])


def test_eval_without_input_grad_is_the_inference_path():
    cfg = synth.CFG_SMALL128
    x, ts, _ = _inputs(cfg)
    for precision in ("bf16", "fp32"):
        m = _model(cfg, precision, False)
        with torch.no_grad():
            y0 = m(x.cuda(), timestamps=ts.cuda())
        y1 = m(x.cuda(), timestamps=ts.cuda())                   # grad mode on, parameters require grad, x does not
        assert y1.grad_fn is None and not y1.requires_grad
        assert torch.equal(y0, y1)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_standalone_maxvit_eval_input_grad(precision):
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh, w, r, N, H, W = 128, 2, 32, 32, 7, 4, 3, 14, 21
    sd = synth.make_state_dict(synth.maxvit_spec(dim, depth, 2, heads, dh, w, 4, 0.25, r), seed=5)
    gen = torch.Generator().manual_seed(12)
    x = torch.randn(N, dim, H, W, generator=gen)
    cond = torch.randn(N, 2, generator=gen)
    dy = torch.randn(N, dim, H, W, generator=gen)
    sd64 = {k: (v.double().requires_grad_("running_" not in k) if v.is_floating_point() else v) for k, v in sd.items()}
    x64, c64 = x.double().requires_grad_(True), cond.double().requires_grad_(True)
    mo.maxvit_forward(x64, c64, sd64, depth=depth, heads=heads, window=w, num_reg=r, training=False).backward(dy.double())
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=w, num_register_tokens=r)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval().set_precision(precision)
    bufs = {k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k}
    xg, cg = x.cuda().requires_grad_(True), cond.cuda().requires_grad_(True)
    m(xg, cg).backward(dy.cuda())
    torch.cuda.synchronize()
    assert all(torch.equal(v, m.state_dict()[k]) for k, v in bufs.items())
    pairs = [("dx", xg.grad, x64.grad), ("dcond", cg.grad, c64.grad)] + [(k, p.grad, sd64[k].grad) for k, p in m.named_parameters()]
    if precision == "fp32":
        _check_fp32(pairs)                                     # measured on a B200: worst max 1.6e-5, L2 1.3e-5
    else:
        _check_mixed(pairs)                                    # measured on a B200: min cosine 0.9992, global L2 2.6e-2
