"""Per-kernel parity of the training kernels (GPU), through the C ABI, against PyTorch autograd of the same op.

Gradient tolerances: fp32 mode 1e-4 (relative to the largest reference entry), tf32 2e-3, bf16 1.5e-2.
"""
import math
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import metnet3_oracle as m3o

pytestmark = pytest.mark.gpu

MODES = [(torch.float32, False), (torch.bfloat16, False), (torch.float32, True)]
WTOL = {(torch.float32, False): 2e-5, (torch.bfloat16, False): 1e-2, (torch.float32, True): 2e-3}


def O():
    from vit_grid_model_b200 import ops
    return ops


def OT():
    from vit_grid_model_b200 import ops_train
    return ops_train


def rel_err(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("M,N,Ca", [(5000, 128, 128), (3001, 512, 128), (4099, 128, 512), (2500, 3072, 128), (70000, 128, 1024)])
def test_wgrad_plain(mode, M, N, Ca):
    dtype, tf32 = mode
    dY, A = rnd(M, N, seed=1).to(dtype), rnd(M, Ca, seed=2).to(dtype)
    ref = dY.float().t() @ A.float()
    dW = torch.zeros(N, Ca, device="cuda")
    OT().wgrad(dY.cuda(), A.cuda(), dW, tf32=tf32, beta=0.0)
    assert rel_err(dW, ref) < WTOL[mode]
    OT().wgrad(dY.cuda(), A.cuda(), dW, tf32=tf32, beta=1.0)          # accumulate
    assert rel_err(dW, 2 * ref) < WTOL[mode]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("Nf,H,W", [(2, 12, 10), (3, 28, 28)])
def test_wgrad_conv3x3(mode, Nf, H, W):
    """3x3 weight gradient over the padded-grid layout vs autograd of F.conv2d"""
    dtype, tf32 = mode
    o = O()
    x = rnd(Nf, 128, H, W, seed=3).to(dtype).float()
    dy = rnd(Nf, 128, H, W, seed=4).to(dtype).float()
    w = torch.zeros(128, 128, 3, 3, requires_grad=True)
    F.conv2d(x, w, padding=1).backward(dy)
    xp, dyp = o.pg_from_nchw(x.cuda(), dtype), o.pg_from_nchw(dy.cuda(), dtype)
    dW = torch.zeros(128, 9 * 128, device="cuda")
    OT().wgrad(dyp, xp, dW, ntaps=9, tap_shift=o.conv_tap_shifts(W), tf32=tf32, beta=0.0)
    got = dW.view(128, 9, 128).permute(0, 2, 1).reshape(128, 128, 3, 3)
    assert rel_err(got, w.grad) < WTOL[mode]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("with_film,with_res", [(True, False), (False, True)])
def test_conv_block_backward(dtype, with_film, with_res):
    """Block (conv3x3 -> ChanLayerNorm -> FiLM -> ReLU (+res)) forward with saves + full backward vs autograd"""
    o, ot = O(), OT()
    N, H, W, C = 3, 12, 10, 128
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    x = rnd(N, C, H, W, seed=1).to(dtype).float().requires_grad_(True)
    w = (rnd(C, C, 3, 3, seed=2) / math.sqrt(9 * C)).to(dtype).float().requires_grad_(True)
    b = rnd(C, seed=3, scale=0.1).requires_grad_(True)
    g = (0.5 + torch.rand(C, generator=torch.Generator().manual_seed(4))).requires_grad_(True)
    be = rnd(C, seed=5, scale=0.1).requires_grad_(True)
    film = rnd(N, 2 * C, seed=6, scale=0.3).requires_grad_(True) if with_film else None
    res = rnd(N, C, H, W, seed=7).requires_grad_(True) if with_res else None
    dy = rnd(N, C, H, W, seed=8)
    h = m3o.chan_layer_norm(F.conv2d(x, w, b, padding=1), g.view(1, C, 1, 1), be.view(1, C, 1, 1))
    if with_film:
        h = h * (film[:, :C, None, None] + 1) + film[:, C:, None, None]
    y = F.relu(h)
    if with_res:
        y = y + res
    y.backward(dy)
    # device path
    xp = o.pg_from_nchw(x.detach().cuda(), dtype)
    Wt = w.detach().permute(0, 2, 3, 1).reshape(C, 9 * C).to(dtype).cuda().contiguous()
    out = o.pg_empty(N, H, W, C, dtype, "cuda")
    resp = o.pg_from_nchw(res.detach().cuda(), torch.float32) if with_res else None
    filmd = film.detach().cuda() if with_film else None
    gd, bed, bd = g.detach().cuda(), be.detach().cuda(), b.detach().cuda()
    _, saved = ot.conv3x3_ln_train(xp, Wt, bd, gd, bed, 1e-5, filmd, resp, out, N, H, W)
    assert rel_err(o.pg_to_nchw(out, N, H, W), y) < (1e-4 if dtype == torch.float32 else 1.5e-2)
    dyp = o.pg_from_nchw(dy.cuda(), torch.float32)
    dconv, sums, _ = ot.conv_ln_bwd(dyp, saved, gd, filmd, 1e-5, N, H, W, dtype)
    dg, db, dbias = (torch.zeros(C, device="cuda") for _ in range(3))
    dfilm = ot.conv_ln_param_grads(sums, N, gd, bed, filmd, dg, db, dbias, with_film)
    assert rel_err(dg, g.grad) < tol and rel_err(db, be.grad) < tol and rel_err(dbias, b.grad) < tol
    if with_film:
        assert rel_err(dfilm, film.grad) < tol
    dW = torch.zeros(C, 9 * C, device="cuda")
    ot.wgrad(dconv, xp, dW, ntaps=9, tap_shift=o.conv_tap_shifts(W), beta=0.0)
    assert rel_err(dW.view(C, 9, C).permute(0, 2, 1).reshape(C, C, 3, 3), w.grad) < tol
    Wd = w.detach().permute(1, 2, 3, 0).reshape(C, 9 * C).to(dtype).cuda().contiguous()          # [ci][tap][co]
    dx = o.gemm(dconv, Wd, ntaps=9, tap_shift=tuple(-s for s in o.conv_tap_shifts(W)), out_f32=True)
    assert rel_err(o.pg_to_nchw(dx, N, H, W), x.grad) < tol


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_maxvit_block_backward(precision):
    """MaxViT (depth 2: MBConv without and with residual, block + grid attention, register tokens) in train() mode:
    forward and every gradient vs autograd through the CPU oracle (batch-statistic BatchNorm)."""
    from oracle import synth
    from oracle import maxvit_oracle as mo
    from vit_grid_model_b200 import MaxViT
    from vit_grid_model_b200 import train as tr
    dim, depth, heads, dh, w, r, N, H, W = 128, 2, 32, 32, 7, 4, 3, 14, 21
    sd = synth.make_state_dict(synth.maxvit_spec(dim, depth, 2, heads, dh, w, 4, 0.25, r), seed=5)
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k:
            v.requires_grad_(True)
    x = rnd(N, dim, H, W, seed=12).requires_grad_(True)
    cond = rnd(N, 2, seed=13).requires_grad_(True)
    dy = rnd(N, dim, H, W, seed=14)
    y = mo.maxvit_forward(x, cond, sd, depth=depth, heads=heads, window=w, num_reg=r, training=True)
    y.backward(dy)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=w, num_register_tokens=r, dropout=0.0)
    m.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=True)
    m = m.cuda().train().set_precision(precision)
    xc = x.detach().permute(0, 2, 3, 1).contiguous().cuda()
    condc = cond.detach().cuda()
    with torch.no_grad():
        yc, saved = tr.maxvit_train_forward(m, xc, condc)
        G = {k: torch.zeros_like(p) for k, p in m.named_parameters()}
        dcond = torch.zeros_like(condc)
        dxc = tr.maxvit_train_backward(m, saved, condc, dcond, dy.permute(0, 2, 3, 1).contiguous().cuda(), G, "")
    fp32 = precision == "fp32"
    assert rel_err(yc.permute(0, 3, 1, 2), y) < (1e-4 if fp32 else 2e-2)
    tol = 2e-3 if fp32 else 6e-2
    bad = []
    for name, got, ref in [("dx", dxc.permute(0, 3, 1, 2), x.grad), ("dcond", dcond, cond.grad)] + [(k, G[k], sd[k].grad) for k in G]:
        g, rf = got.detach().float().cpu(), ref
        if re.fullmatch(r"layers\.\d+\.0\.(fn\.)?[037]\.bias", name):
            # conv bias in front of a batch-statistic BatchNorm: the gradient is analytically zero; both sides hold
            # rounding noise only, which must stay far below the BatchNorm beta gradient next to it
            beta = G[name[:-len("0.bias")] + str(int(name[-len("0.bias")]) + 1) + ".bias"].norm().item()
            if g.norm().item() > 1e-3 * beta:
                bad.append((name, g.norm().item(), beta))
            continue
        e = ((g - rf).norm() / max(rf.norm().item(), 1e-2)).item()
        if e > tol:
            bad.append((name, round(e, 5)))
    assert not bad, bad


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_attention_dropout_forward_backward(precision):
    """nn.Dropout on the attention probabilities and after to_out (maxvit.py:146,151), train() mode: the kernels' counter-based
    masks are exported through the test hook and fed to the oracle, so forward and every gradient must agree as without dropout;
    the keep rate must match the quantised probability.  'bf16': the fused kernel + bf16 backward chain; 'fp32': the un-fused
    exact-fp32 kernels, which apply the same masks."""
    from oracle import synth
    from oracle import maxvit_oracle as mo
    from vit_grid_model_b200 import MaxViT
    from vit_grid_model_b200 import train as tr
    dim, depth, heads, dh, w, r, N, H, W, p = 128, 1, 32, 32, 7, 4, 2, 14, 21, 0.25
    S, nwin = r + w * w, (H // w) * (W // w)
    sd = synth.make_state_dict(synth.maxvit_spec(dim, depth, 2, heads, dh, w, 4, 0.25, r), seed=7)
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k:
            v.requires_grad_(True)
    x = rnd(N, dim, H, W, seed=21).requires_grad_(True)
    cond = rnd(N, 2, seed=22).requires_grad_(True)
    dy = rnd(N, dim, H, W, seed=23)
    seed, T = 123456789, tr.dropout_threshold(p)
    scale = 256.0 / (256 - T)
    masks = {}
    for ai, salt in ((1, 0), (2, 1)):
        pm, om = OT().dropout_masks((seed, salt, T), N * nwin, heads, dim)
        keep = pm[:, :, :S, :S].float().mean().item()
        assert abs(keep - (1 - T / 256)) < 5e-3, keep
        masks[(0, ai)] = (pm[:, :, :S, :S].float().cpu() * scale, om[:, :S].float().cpu() * scale)
    y = mo.maxvit_forward(x, cond, sd, depth=depth, heads=heads, window=w, num_reg=r, training=True, drop_masks=masks)
    y.backward(dy)
    m = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=w, num_register_tokens=r, dropout=p)
    m.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=True)
    m = m.cuda().train().set_precision(precision)
    fp32 = precision == "fp32"
    xc, condc = x.detach().permute(0, 2, 3, 1).contiguous().cuda(), cond.detach().cuda()
    with torch.no_grad():
        yc, saved = tr.maxvit_train_forward(m, xc, condc, seed=seed)
        G = {k: torch.zeros_like(q) for k, q in m.named_parameters()}
        dcond = torch.zeros_like(condc)
        dxc = tr.maxvit_train_backward(m, saved, condc, dcond, dy.permute(0, 2, 3, 1).contiguous().cuda(), G, "")
    assert rel_err(yc.permute(0, 3, 1, 2), y) < (1e-4 if fp32 else 2e-2)
    bad = []
    for name, got, ref in [("dx", dxc.permute(0, 3, 1, 2), x.grad), ("dcond", dcond, cond.grad)] + [(k, G[k], sd[k].grad) for k in G]:
        if re.fullmatch(r"layers\.\d+\.0\.(fn\.)?[037]\.bias", name):
            continue
        g, rf = got.detach().float().cpu(), ref
        e = ((g - rf).norm() / max(rf.norm().item(), 1e-2)).item()
        # the attention backward chain (tokens, qkv, datt, dqkv, att) is held in bf16; dcond -- two numbers per field, each the
        # sum of the FiLM gradients of all tokens and channels -- collects that rounding without averaging it away
        if e > (2e-3 if fp32 else (8e-2 if name == "dcond" else 6e-2)):
            bad.append((name, round(e, 5)))
    assert not bad, bad
    # a different seed gives a different mask, the same seed the same output
    with torch.no_grad():
        y2, _ = tr.maxvit_train_forward(m, xc, condc, seed=seed)
        y3, _ = tr.maxvit_train_forward(m, xc, condc, seed=seed + 1)
    assert torch.equal(yc, y2) and not torch.equal(yc, y3)


def _attn_core_autograd(qkv, datt, qg, kg, bt, nw, S, win, R, heads, dh, pmask=None):
    """fp32 autograd of maxvit.py:189-213 (+ dropout mask on the probabilities) on the [rows][3*inner] layout of the kernels"""
    inner = heads * dh
    x = qkv.float().view(nw, S, 3, heads, dh).permute(2, 0, 3, 1, 4).detach().requires_grad_(True)   # (3, windows, h, S, d)
    qg_ = qg.view(heads, 1, dh).detach().requires_grad_(True)
    kg_ = kg.view(heads, 1, dh).detach().requires_grad_(True)
    bt_ = bt.detach().requires_grad_(True)
    qh = F.normalize(x[0], dim=-1) * (dh ** 0.5) * qg_
    kh = F.normalize(x[1], dim=-1) * (dh ** 0.5) * kg_
    W2 = 2 * win - 1
    idx = torch.full((S, S), W2 * W2, dtype=torch.long)
    for i in range(R, S):
        for j in range(R, S):
            a, b = divmod(i - R, win)
            c, d = divmod(j - R, win)
            idx[i, j] = (a - c + win - 1) * W2 + (b - d + win - 1)
    prob = (qh @ kh.transpose(-1, -2) + bt_[idx.to(bt.device)].permute(2, 0, 1)).softmax(-1)
    if pmask is not None:
        prob = prob * pmask
    out = (prob @ x[2]).permute(0, 2, 1, 3).reshape(nw * S, inner)
    out.backward(datt.float())
    return x.grad.permute(1, 3, 0, 2, 4).reshape(nw * S, 3 * inner), out.detach(), qg_.grad.reshape(-1), kg_.grad.reshape(-1), bt_.grad


@pytest.mark.parametrize("Hl,Wl,N,T", [(14, 21, 3, 0), (21, 35, 2, 0), (21, 35, 2, 64), (7, 7, 5, 26), (14, 14, 12, 26)])
def test_attn_core_bwd_tcgen05(Hl, Wl, N, T):
    """The tcgen05 attention-core backward (csrc/vg_attn_bwd_tc.cu: bf16 tensors, two windows per M=128 tile) against fp32 autograd
    of the same bf16 inputs and against the mma.sync kernel (mode 2) on those inputs widened to fp32, its outputs rounded to bf16;
    even and odd window counts (an odd count leaves the second half of a field's last tile empty), one window per field, with and
    without the dropout masks (read back from the kernels' own test hook)."""
    win, R, heads, dh = 7, 4, 32, 32
    S, nwin, inner = R + win * win, (Hl // win) * (Wl // win), heads * dh
    rows = N * nwin * S
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn(rows, 3 * inner, device="cuda", generator=g).to(torch.bfloat16)
    datt = torch.randn(rows, inner, device="cuda", generator=g).to(torch.bfloat16)
    qg = 1 + 0.2 * torch.randn(inner, device="cuda", generator=g)
    kg = 1 + 0.2 * torch.randn(inner, device="cuda", generator=g)
    bt = 0.5 * torch.randn((2 * win - 1) ** 2 + 1, heads, device="cuda", generator=g)
    drop = (4242, 1, T)
    pmask = None
    if T:
        pm, _ = OT().dropout_masks(drop, N * nwin, heads, 128)
        pmask = pm[:, :, :S, :S].float() * (256.0 / (256 - T))
    ref = _attn_core_autograd(qkv, datt, qg, kg, bt, N * nwin, S, win, R, heads, dh, pmask)

    def launch(q, d):
        dqg, dkg, dbt = torch.zeros_like(qg), torch.zeros_like(kg), torch.zeros_like(bt)
        dqkv, att = OT().attn_core_bwd(q, d, qg, kg, bt, N, Hl, Wl, win, R, heads, dh, dqg, dkg, dbt, tf32=True, want_att=True, drop=drop)
        torch.cuda.synchronize()
        return [dqkv, att, dqg, dkg, dbt]
    tc = launch(qkv, datt)
    mma = launch(qkv.float(), datt.float())
    mma[0], mma[1] = mma[0].cpu().to(torch.bfloat16), mma[1].cpu().to(torch.bfloat16)     # round to nearest, as bf16 outputs are
    names = ["dqkv", "att", "dq_gamma", "dk_gamma", "dbias"]
    l2 = lambda a, b: ((a.float().cpu() - b.float().cpu()).norm() / b.float().cpu().norm().clamp_min(1e-12)).item()
    for nm, got, prev, rf in zip(names, tc, mma, ref):
        assert torch.isfinite(got.float()).all(), nm
        # L2: 1.2e-2 (bf16 operands and bf16 output tensors; measured 6e-3 .. 1e-2 for both kernels), never worse than 1.15x the
        # mma.sync kernel; largest single deviation: 3e-2 of the largest reference entry
        e_tc, e_mma = l2(got, rf), l2(prev, rf)
        assert e_tc < 1.2e-2 and e_tc < 1.15 * e_mma + 1e-4, (nm, e_tc, e_mma)
        assert rel_err(got, rf) < 3e-2, (nm, rel_err(got, rf), rel_err(prev, rf))
    # the kernel is deterministic in everything but the order of its global atomics: repeated launches must give the same bits (a
    # hand-over race -- e.g. the item flush reusing the P' / dS blocks before the last product has retired -- shows up here)
    for _ in range(12):
        dqkv2, att2, dqg, dkg, dbt = launch(qkv, datt)
        assert torch.equal(dqkv2, tc[0]) and torch.equal(att2, tc[1])
        assert rel_err(dbt, tc[4]) < 1e-4 and rel_err(dqg, tc[2]) < 1e-4


def test_repeatable_launches_of_the_pipelined_kernels():
    """Kernels with producer / consumer hand-overs through shared memory must give the same bits launch after launch:
    the LayerNorm backward (per-warp bulk-copy ring), the store-epilogue GEMM with sixteen epilogue warps (16-bit plain store and
    BN + GELU fp16 output) and the conv data gradient through the halo kernel."""
    o, ot = O(), OT()
    g_ = torch.Generator(device="cuda").manual_seed(11)
    # LN backward on a PG buffer whose pixel count is not a multiple of four (the last group is read without the ring)
    N, HP, WP, C = 7, 29, 23, 128
    npix = o.pg_pixels(N, HP, WP)
    dY = torch.randn(npix, C, device="cuda", generator=g_)
    xhat = torch.randn(npix, C, device="cuda", generator=g_).to(torch.bfloat16)
    rstd = torch.rand(npix, device="cuda", generator=g_) + 0.5
    mask = torch.randint(0, 2 ** 31 - 1, (npix, 4), device="cuda", generator=g_, dtype=torch.int32)
    ln_g = torch.randn(C, device="cuda", generator=g_)
    film = torch.randn(N, 2 * C, device="cuda", generator=g_) * 0.1
    ref = None
    for _ in range(6):
        dconv, sums, _b = ot.conv_ln_bwd(dY, (xhat, rstd, mask), ln_g, film, 1e-5, N, HP, WP, torch.bfloat16)
        torch.cuda.synchronize()
        if ref is None:
            ref = (dconv, sums)
        else:
            assert torch.equal(dconv, ref[0])
            assert rel_err(sums, ref[1]) < 1e-5                      # float atomics: order-dependent in the last bits only
    # GEMMs
    M, K = 20000, 128
    A = torch.randn(M, K, device="cuda", generator=g_)
    for (Nn, kw, dt) in ((3072, dict(), torch.bfloat16), (512, dict(scale=torch.rand(512, device="cuda") + 0.5, shift=torch.randn(512, device="cuda"), act=1, tf32=True, out_dtype=torch.float16), torch.float32)):
        Wm = (torch.randn(Nn, K, device="cuda", generator=g_) / math.sqrt(K)).to(dt)
        first = None
        for _ in range(6):
            out = o.gemm(A.to(dt), Wm, **kw)
            torch.cuda.synchronize()
            first = out if first is None else first
            assert torch.equal(out, first)
        refm = A.to(dt).float() @ Wm.float().t()
        if "act" in kw:
            refm = F.gelu(refm * kw["scale"] + kw["shift"])
        assert rel_err(first, refm) < 1.5e-2
    # conv data gradient (halo kernel, flipped taps)
    Nf, H, W = 5, 28, 21
    dconv = o.pg_from_nchw(torch.randn(Nf, C, H, W, device="cuda", generator=g_), torch.bfloat16)
    Wd = (torch.randn(C, 9 * C, device="cuda", generator=g_) / 34).to(torch.bfloat16)
    res = torch.randn(dconv.shape[0], C, device="cuda", generator=g_)
    first = None
    for _ in range(6):
        dx = o.gemm(dconv, Wd, ntaps=9, tap_shift=tuple(-s for s in o.conv_tap_shifts(W)), res=res, out_f32=True)
        torch.cuda.synchronize()
        first = dx if first is None else first
        assert torch.equal(dx, first)
