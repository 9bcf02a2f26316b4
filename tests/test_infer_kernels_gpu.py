"""Per-kernel parity of the inference kernels (GPU) against float64 PyTorch, at the geometry bench.py measures (the 12-hour
model: 84x70 frames, L = 12, B = 64, i.e. 768 fields in one call; MaxViT at 42x35) and at the edges where the kernels change
path: fewer rows than one 256-row tile, many tiles per CTA, the last frame width of the halo conv kernel (WP = 78) and the
first of the generic tcgen05 path (WP = 79), the 518x518 domain, fp32 buffers larger than 2^31 bytes, per-field weights over
1,470 rows (not a multiple of the 256-row tile), the nine border cases of the stem's time term, and the LayerNorm's
var.clamp(eps) branch.

Conventions of this file:
  * every reference is float64 (on the GPU, with torch's own ops), built from the operands rounded exactly as the device sees
    them (bf16 / fp16 via .to(dtype)), so what is left is the kernel's arithmetic, not the storage format's
  * tf32 contractions run twice: once on operands that are tf32-representable (the low 13 mantissa bits clear: whether the
    tensor core truncates or rounds, they are exact, and the bound is the fp32 one), and once on plain fp32 operands with
    the rounding-agnostic bound 2 * 2^-10 * sum|a||b| per element on top (propagated through the LayerNorm where one follows)
  * every output the kernel must write completely starts as NaN; pads of padded-grid (PG) outputs must be exactly 0.0
  * comparisons are per field (a bad field must not be averaged away): fp32 outputs within 2e-5 of the field's largest
    entry; 16-bit outputs within half an ulp of the float64 result plus the fp32 arithmetic's own error (rounded to nearest:
    rounding toward zero fails); selections and copies bit-exact
"""
import ctypes
import math
import os
from functools import lru_cache

import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle import maxvit_oracle as mo
from oracle import metnet3_oracle as m3o

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64 = torch.float64
BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
FP32_TOL = 2e-5           # fp32 outputs: max |err| / max |ref| per field
TF32_U = 2.0 ** -10        # tf32 keeps 10 explicit mantissa bits; 2 * TF32_U * sum|a||b| bounds rounding or truncation


def O():
    from vit_grid_model_b200 import ops
    return ops


def call(name, *args):
    from vit_grid_model_b200 import _lib
    from vit_grid_model_b200.ops import _st
    _lib.call(name, *args, _st())


def note(**kv):
    """one line per measurement (pytest -s shows them; the numbers in DESIGN.md come from these lines)"""
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0].split("::")[-1]
    print("MEASURE", test, " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in kv.items()))


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, generator=g, device=DEV) * scale


def tf32_exact(t):
    """t with the 13 low mantissa bits cleared: a tf32 operand the tensor core takes exactly"""
    return (t.contiguous().view(torch.int32) & -8192).view(F32)


def nan_like(shape, dtype=F32):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def pg_frame(buf, N, HP, WP):
    """(N,HP,WP,C) view of the frame pixels of a PG buffer (no copy)"""
    C = buf.shape[-1]
    return buf.view(N * (HP + 1) + 1, WP + 1, C)[:N * (HP + 1)].view(N, HP + 1, WP + 1, C)[:, 1:, 1:]


def pg_field(buf, n, HP, WP):
    """(HP,WP,C) frame of field n of a PG buffer"""
    C = buf.shape[-1]
    return buf.view(-1, WP + 1, C)[n * (HP + 1) + 1:(n + 1) * (HP + 1)][:, 1:]


def pg_pads(buf, N, HP, WP):
    """every pad entry of a PG buffer (column 0 of every row, and the separator rows)"""
    C = buf.shape[-1]
    v = buf.view(N * (HP + 1) + 1, WP + 1, C)
    return torch.cat([v[:, 0].reshape(-1), v[::HP + 1, 1:].reshape(-1)])


def pg_nan(N, HP, WP, C, dtype=F32):
    return nan_like((O().pg_pixels(N, HP, WP), C), dtype)


def assert_pads_zero(buf, N, HP, WP):
    p = pg_pads(buf, N, HP, WP).float()
    assert torch.equal(p, torch.zeros_like(p)), "a pad is not 0.0"


def f32_ratio(got, ref, extra=None, tol=FP32_TOL):
    """got, ref: (N, ...) -> (worst over fields of max |err| / (tol * max|ref of field| + extra), worst per-field rel error).
    extra: an element-wise absolute allowance (the tf32 operand bound) or None."""
    got, ref = got.to(DEV, F64), ref.to(DEV, F64)
    N = ref.shape[0]
    err = (got - ref).abs().reshape(N, -1)
    fmax = ref.abs().reshape(N, -1).amax(1, keepdim=True).clamp_min(1e-300)
    allow = tol * fmax + (0 if extra is None else extra.to(DEV, F64).reshape(N, -1))
    ratio = (err / allow).amax().item()
    assert not torch.isnan(got).any(), "NaN in the output"
    return ratio, (err.amax(1, keepdim=True) / fmax).amax().item()


def rn16(got, ref64, err_abs=0.0):
    """largest |got - ref| / (ulp / 2 + err_abs) of 16-bit results got against the float64 reference: <= 1 means got is the
    reference rounded to nearest, up to the fp32 arithmetic's own absolute error err_abs (scalar or element-wise) in front of
    the rounding.  (A bound of one ulp would let rounding toward zero pass.)  The ulp is the larger of got's and the rounded
    reference's."""
    dt = got.dtype
    r = ref64.to(DEV).to(dt).to(F64)
    g = got.to(DEV, F64)
    assert not torch.isnan(g).any(), "NaN in the output"
    _, e = torch.frexp(torch.maximum(r.abs(), g.abs()))
    bits, tiny = (8, 2.0 ** -133) if dt == BF16 else (11, 2.0 ** -24)
    ulp = torch.ldexp(torch.ones_like(r), e - bits).clamp_min(tiny)
    return ((g - ref64.to(DEV, F64)).abs() / (0.5 * ulp + torch.as_tensor(err_abs, dtype=F64, device=DEV))).max().item()


def per_field_abs_allow(ref, tol=FP32_TOL):
    """(N, ...) -> tol * max|ref| of each field, broadcastable to ref"""
    N = ref.shape[0]
    return tol * ref.abs().reshape(N, -1).amax(1).view(N, *([1] * (ref.dim() - 1)))


def ln_error_bound(h, delta, G, eps):
    """element-wise bound of the ChanLayerNorm output error when its input h (N,C,H,W) carries an error |d| <= delta:
    |d xhat_c| <= rstd (|d_c| + max_c|d| (1 + |xhat_c|)), times |G_c| (the LayerNorm gain with FiLM folded in)"""
    mean = h.mean(1, keepdim=True)
    rstd = h.var(1, unbiased=False, keepdim=True).clamp(min=eps).rsqrt()
    xhat = (h - mean) * rstd
    D = delta.amax(1, keepdim=True)
    return G.abs() * rstd * (delta + D * (1 + xhat.abs()))


# =========================================================================================== conv block, 128 channels
# (N, HP, WP, head pads (left, right, top, bottom)).  The 12-hour pads and the small128 pads are both (1, 2, 1, 1); the other
# geometries use asymmetric pads so that a swap of pad_left / pad_top or of a pad with its opposite side shows.
CONV_GEOMS = {
    "n1_14x14": (1, 14, 14, (2, 1, 0, 3)),          # 15*15 + 15 = 240 PG rows: less than one 256-row tile
    "n40_84x70": (40, 84, 70, synth.CFG_12HR.pads),  # 241,471 rows = 944 tiles on 148 SMs: 6 or 7 per CTA
    "small128": (3, 28, 28, synth.CFG_SMALL128.pads),
    "wp78": (3, 28, 78, (0, 3, 2, 1)),               # 256 + 2 (WP + 2) = 416: the widest frame of the halo kernel
    "wp79": (3, 28, 79, (3, 0, 1, 2)),               # 418 rows: the generic tcgen05 conv + LN epilogue
    "n1_518": (1, 518, 518, (3, 3, 3, 3)),           # BASELINE configs[3]'s domain
}
CONV_DTYPES = {0: "bf16", 1: "fp32", 2: "tf32"}
EPS = 1e-5


def _conv_operands(code, N, HP, WP, C, seed):
    """seeded operands of one conv block, rounded to what the device sees.  Rows 0-3 of every frame are zero, and the conv
    bias is O(1e-3): at the frame pixels of rows 0-2 the conv output is the bias alone, whose variance over the channels
    (about 1e-6) is below eps, so the LayerNorm takes its var.clamp(eps) branch there."""
    x = rnd(N, C, HP, WP, seed=seed)
    x[:, :, :4] = 0
    w = rnd(C, C, 3, 3, seed=seed + 1, scale=1 / math.sqrt(9 * C))
    if code == 0:
        x, w = x.to(BF16).float(), w.to(BF16).float()
    elif code == 2:
        x, w = tf32_exact(x), tf32_exact(w)
    b = rnd(C, seed=seed + 2, scale=1e-3)
    g = 1.0 + 0.5 * torch.rand(C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 3))
    be = rnd(C, seed=seed + 4, scale=0.1)
    film = rnd(N, 2 * C, seed=seed + 5, scale=0.3)
    res = rnd(N, C, HP, WP, seed=seed + 6)
    return x, w, b, g, be, film, res


@lru_cache(maxsize=1)
def _conv_case(code, geom, C=128, seed=10):
    N, HP, WP, pads = CONV_GEOMS[geom] if isinstance(geom, str) else geom
    x, w, b, g, be, film, res = _conv_operands(code, N, HP, WP, C, seed)
    h64 = F.conv2d(x.to(F64), w.to(F64), b.to(F64), padding=1)
    return (N, HP, WP, pads), (x, w, b, g, be, film, res), h64


def _block_ref(h64, g, be, film, res):
    """ChanLayerNorm (oracle) -> FiLM -> ReLU -> + residual, float64 NCHW"""
    C = h64.shape[1]
    y = m3o.chan_layer_norm(h64, g.to(F64).view(1, C, 1, 1), be.to(F64).view(1, C, 1, 1), EPS)
    G = g.to(F64).view(1, C, 1, 1).expand(h64.shape[0], C, 1, 1)
    if film is not None:
        f = film.to(F64)
        y = y * (f[:, :C, None, None] + 1) + f[:, C:, None, None]
        G = G * (f[:, :C, None, None] + 1)
    y = F.relu(y)
    if res is not None:
        y = y + res.to(F64)
    return y, G


def _head_ref(y64, hw, hb, HP, WP, pads, std, mean):
    pl, pr, pt, pb = pads
    z = torch.einsum("nchw,c->nhw", y64[:, :, pt:HP - pb, pl:WP - pr], hw.to(F64))
    return (z + hb) * std + mean


def _run_conv_block(code, geom, epi, C=128):
    """one conv block call for epilogue `epi`; returns the measured ratios (each must be <= 1)"""
    o = O()
    (N, HP, WP, pads), (x, w, b, g, be, film, res), h64 = _conv_case(code, geom, C)
    adt = BF16 if code == 0 else F32
    use_film = epi == "film"
    res_f32 = code == 0 and epi in ("res32_copy_tma1", "head_only", "head_out")
    use_res = epi not in ("film", "copy_thread_stores")
    want_copy = "copy" in epi
    resq = None
    if use_res:
        resq = res if (res_f32 or code != 0) else res.to(BF16).float()
    y64, G = _block_ref(h64, g, be, film if use_film else None, resq)
    # element-wise allowance: fp32 accumulation over 9 * C terms, and for tf32 on plain fp32 operands the operand bound
    acc = per_field_abs_allow(y64)
    xp = o.pg_from_nchw(x, adt)
    wt = w.permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous().to(adt)
    rp = None if resq is None else o.pg_from_nchw(resq, F32 if res_f32 else adt)
    out = None if epi == "head_only" else pg_nan(N, HP, WP, C, adt)
    copy = pg_nan(N, HP, WP, C) if want_copy else None
    head = pred = None
    pl, pr, pt, pb = pads
    H, W = HP - pt - pb, WP - pl - pr
    if epi.startswith("head"):
        hw, hb, std, mean = rnd(C, seed=31, scale=1 / math.sqrt(C)), 0.2, 15.0, 20.0
        pred = nan_like((N, H, W))
        head = (hw, hb, std, mean, H, W, pads, pred)
    o.conv3x3_ln(xp, wt, b, g, be, EPS, film if use_film else None, rp, out, N, HP, WP, out_copy=copy, head=head, tf32=code == 2)
    torch.cuda.synchronize()
    yref = y64.permute(0, 2, 3, 1)
    r = {}
    if out is not None:
        got = pg_frame(out, N, HP, WP)
        if adt == BF16:
            r["out_rn"] = rn16(got, yref, acc.permute(0, 2, 3, 1))
        else:
            r["out"], r["out_rel"] = f32_ratio(got, yref)
        assert_pads_zero(out, N, HP, WP)
    if copy is not None:
        r["copy"], r["copy_rel"] = f32_ratio(pg_frame(copy, N, HP, WP), yref)
        assert_pads_zero(copy, N, HP, WP)
        if out is not None:
            assert torch.equal(out.float(), copy.to(adt).float()), "output != (rounded) fp32 copy"
    if pred is not None:
        pref = _head_ref(y64, hw, hb, HP, WP, pads, std, mean)
        # the head sums 128 block outputs: allow 2e-5 of sum |w||y| per pixel (times std) on the block's own allowance
        zabs = torch.einsum("nchw,c->nhw", y64[:, :, pt:HP - pb, pl:WP - pr].abs(), hw.abs().to(F64)) * std
        r["head"], r["head_rel"] = f32_ratio(pred, pref, extra=FP32_TOL * zabs, tol=0.0)
        r["head_rel"] = ((pred.to(F64) - pref).abs().amax() / (pref - mean).abs().amax()).item()
    return r


@pytest.mark.parametrize("geom", list(CONV_GEOMS))
@pytest.mark.parametrize("code", list(CONV_DTYPES), ids=list(CONV_DTYPES.values()))
@pytest.mark.parametrize("epi", ["film", "res", "res32_copy_tma1", "copy_thread_stores", "head_only", "head_out"])
def test_conv3x3_ln(code, geom, epi):
    """metnet3.py:110-126 Block (+ the ResnetBlock residual, + the fused 1x1 head) in the three conv dtypes: 0 = bf16 operands
    (halo kernel up to WP = 78, generic tcgen05 above), 1 = exact fp32 (SIMT), 2 = fp32 storage with tf32 tcgen05 (here on
    tf32-representable operands: the bound is the fp32 one; test_conv3x3_ln_tf32_plain_operands covers rounding).  The fp32
    copy of the output leaves through TMA tensor stores with an fp32 residual (res32_copy_tma1, halo kernel), and through
    per-thread stores without a residual (copy_thread_stores)."""
    if epi.startswith("res32_copy") and code != 0:
        pytest.skip("the fp32 residual is the bf16 block's skip connection")
    r = _run_conv_block(code, geom, epi)
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)


def test_conv3x3_ln_tf32_plain_operands():
    """dtype 2 on plain fp32 operands at 84x70 (6 fields): within the rounding-agnostic tf32 bound, propagated through the
    LayerNorm.  tcgen05 kind::tf32 truncates its operands: against the operands truncated to tf32 (x & -8192) the output is
    within the fp32 bound (measured 2.3e-6 on a B200), against the exact operands it is not (3.7e-4).  Both are asserted, so a
    quiet fall-back to the exact-fp32 SIMT kernel (about 2e-6 against the exact operands) fails here."""
    o = O()
    N, HP, WP, C = 6, 84, 70, 128
    x = rnd(N, C, HP, WP, seed=41)
    x[:, :, :4] = 0
    w = rnd(C, C, 3, 3, seed=42, scale=1 / math.sqrt(9 * C))
    b, be = rnd(C, seed=43, scale=1e-3), rnd(C, seed=44, scale=0.1)
    g = 1.0 + 0.5 * torch.rand(C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(45))
    film = rnd(N, 2 * C, seed=46, scale=0.3)
    out = pg_nan(N, HP, WP, C)
    o.conv3x3_ln(o.pg_from_nchw(x, F32), w.permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous(), b, g, be, EPS, film, None, out,
                 N, HP, WP, tf32=True)
    torch.cuda.synchronize()
    h64 = F.conv2d(x.to(F64), w.to(F64), b.to(F64), padding=1)
    y64, G = _block_ref(h64, g, be, film, None)
    delta = 2 * TF32_U * F.conv2d(x.abs().to(F64), w.abs().to(F64), padding=1)
    extra = ln_error_bound(h64, delta, G, EPS).permute(0, 2, 3, 1)
    got = pg_frame(out, N, HP, WP)
    ratio, rel = f32_ratio(got, y64.permute(0, 2, 3, 1), extra=extra)
    ht = F.conv2d(tf32_exact(x).to(F64), tf32_exact(w).to(F64), b.to(F64), padding=1)
    ratio_trunc, rel_trunc = f32_ratio(got, _block_ref(ht, g, be, film, None)[0].permute(0, 2, 3, 1))
    note(ratio=ratio, rel=rel, ratio_truncation_model=ratio_trunc, rel_truncation_model=rel_trunc)
    assert_pads_zero(out, N, HP, WP)
    assert ratio <= 1.0
    assert ratio_trunc <= 1.0 and rel > 5 * FP32_TOL, (ratio_trunc, rel)


@pytest.mark.parametrize("with_res", [True, False], ids=["copy_tma", "copy_thread_stores"])
def test_conv3x3_ln_headline_batch(with_res):
    """bench.py's size: 768 fields at 84x70, bf16 with the fp32 copy, then the fused head: with the fp32 residual (the copy
    is stored by TMA) and without a residual (the copy is stored by the threads).  The fp32 buffers are 4,634,951 x 128 x 4 B =
    2.37 GB; a field spans 85 x 71 rows of 512 B, so field 694 straddles 2^31 bytes and fields 695 and up lie past it.
    Fields 0, 1, 383, 694, 695, 766 and 767 against float64; over the whole buffers every pad is 0.0 and nothing is NaN."""
    o = O()
    N, HP, WP, C = 768, 84, 70, 128
    pads = synth.CFG_12HR.pads
    pl, pr, pt, pb = pads
    H, W = HP - pt - pb, WP - pl - pr
    xp = torch.zeros(o.pg_pixels(N, HP, WP), C, dtype=BF16, device=DEV)
    g_ = torch.Generator(device=DEV).manual_seed(51)
    pg_frame(xp, N, HP, WP).copy_(torch.randn(N, HP, WP, C, device=DEV, generator=g_).to(BF16))
    rp = None
    if with_res:
        rp = torch.zeros(o.pg_pixels(N, HP, WP), C, device=DEV)
        pg_frame(rp, N, HP, WP).copy_(torch.randn(N, HP, WP, C, device=DEV, generator=g_))
    w = rnd(C, C, 3, 3, seed=52, scale=1 / math.sqrt(9 * C)).to(BF16).float()
    b, be = rnd(C, seed=53, scale=0.1), rnd(C, seed=54, scale=0.1)
    g = 1.0 + 0.5 * torch.rand(C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(55))
    wt = w.permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous().to(BF16)
    out = pg_nan(N, HP, WP, C, BF16)
    copy = pg_nan(N, HP, WP, C)
    assert copy.numel() * 4 > 2 ** 31
    o.conv3x3_ln(xp, wt, b, g, be, EPS, None, rp, out, N, HP, WP, out_copy=copy)
    hw, hb, std, mean = rnd(C, seed=56, scale=1 / math.sqrt(C)), 0.2, synth.CFG_12HR.pm25_std, synth.CFG_12HR.pm25_mean
    pred = nan_like((N, H, W))
    o.conv3x3_ln(xp, wt, b, g, be, EPS, None, rp, None, N, HP, WP, head=(hw, hb, std, mean, H, W, pads, pred))
    torch.cuda.synchronize()
    assert not torch.isnan(out).any() and not torch.isnan(copy).any() and not torch.isnan(pred).any()
    assert_pads_zero(out, N, HP, WP)
    assert_pads_zero(copy, N, HP, WP)
    worst = {}
    for n in (0, 1, 383, 694, 695, 766, 767):
        xn = pg_field(xp, n, HP, WP).permute(2, 0, 1)[None].to(F64)
        rn = pg_field(rp, n, HP, WP).permute(2, 0, 1)[None].to(F64) if with_res else None
        y64, _ = _block_ref(F.conv2d(xn, w.to(F64), b.to(F64), padding=1), g, be, None, rn)
        yref = y64.permute(0, 2, 3, 1)
        rc, relc = f32_ratio(pg_field(copy, n, HP, WP)[None], yref)
        ro = rn16(pg_field(out, n, HP, WP)[None], yref, per_field_abs_allow(yref))
        pref = _head_ref(y64, hw, hb, HP, WP, pads, std, mean)
        zabs = torch.einsum("nchw,c->nhw", y64[:, :, pt:HP - pb, pl:WP - pr].abs(), hw.abs().to(F64)) * std
        rh, _ = f32_ratio(pred[n:n + 1], pref, extra=FP32_TOL * zabs, tol=0.0)
        worst[n] = (rc, relc, ro, rh)
    note(**{f"f{n}_copy_rel": v[1] for n, v in worst.items()}, copy=max(v[0] for v in worst.values()),
         out_rn=max(v[2] for v in worst.values()), head=max(v[3] for v in worst.values()))
    for n, (rc, relc, ro, rh) in worst.items():
        assert rc <= 1.0 and ro <= 1.0 and rh <= 1.0, (n, rc, relc, ro, rh)


# =========================================================================================== wide conv block and stem
@pytest.mark.parametrize("C", [256, 384, 512])
@pytest.mark.parametrize("code", list(CONV_DTYPES), ids=list(CONV_DTYPES.values()))
@pytest.mark.parametrize("epi", ["film", "res", "res32_copy_tma1", "head_only", "head_out"])
def test_conv3x3_ln_wide(C, code, epi):
    """vg_conv3x3_ln_wide_fwd (n_start_channels 256 / 384 / 512, BASELINE configs[4]): shifted-row GEMM + row-wise LayerNorm /
    FiLM / ReLU / residual / copy / head, at 2 fields of 28x35"""
    if epi.startswith("res32_copy") and code != 0:
        pytest.skip("the fp32 residual and the fp32 copy are the bf16 block's skip connection")
    r = _run_conv_block(code, (2, 28, 35, (1, 2, 3, 0)), epi, C=C)
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)


def _stem_operands(B, L, HP, WP, C, seed):
    N = B * L
    npix = O().pg_pixels(B, HP, WP)
    raw3 = rnd(npix, C, seed=seed)                 # pads hold values too (the stem GEMM computes them): they must be ignored
    rawres = rnd(npix, C, seed=seed + 1)
    bias3, bias1 = rnd(C, seed=seed + 2, scale=0.1), rnd(C, seed=seed + 3, scale=0.1)
    tt = rnd(N, 9, C, seed=seed + 4)               # nine distinct border cases per field
    tres = rnd(N, C, seed=seed + 5)
    g = 1.0 + 0.5 * torch.rand(C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 6))
    be = rnd(C, seed=seed + 7, scale=0.1)
    film = rnd(N, 2 * C, seed=seed + 8, scale=0.3)
    return raw3, rawres, bias3, bias1, tt, tres, g, be, film


def _stem_ref(B, L, HP, WP, C, raw3, rawres, bias3, bias1, tt, tres, g, be, film):
    """per field n = b L + l: h1 = ReLU(FiLM(ChanLayerNorm(raw3[b] + bias3 + tt[n][case(y, x)]))), res = rawres[b] + bias1 + tres[n];
    case = 3 ry + rx with ry / rx = 0 at the first row / column, 2 at the last, 1 inside"""
    N = B * L
    bidx = torch.arange(N, device=DEV) // L
    r3 = pg_frame(raw3, B, HP, WP).to(F64)[bidx]                       # (N,HP,WP,C)
    rr = pg_frame(rawres, B, HP, WP).to(F64)[bidx]
    ry = torch.ones(HP, dtype=torch.long, device=DEV)
    ry[0], ry[-1] = 0, 2
    rx = torch.ones(WP, dtype=torch.long, device=DEV)
    rx[0], rx[-1] = 0, 2
    case = ry[:, None] * 3 + rx[None, :]                               # (HP,WP)
    tterm = tt.to(F64)[:, case]                                        # (N,HP,WP,C)
    v = (r3 + bias3.to(F64) + tterm).permute(0, 3, 1, 2)
    h1, _ = _block_ref(v, g, be, film, None)
    res = rr + bias1.to(F64) + tres.to(F64)[:, None, None, :]
    return h1.permute(0, 2, 3, 1), res


@pytest.mark.parametrize("h1_dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("C,B,L,HP,WP", [(128, 4, 12, 84, 70), (256, 2, 3, 28, 35), (384, 2, 3, 28, 35), (512, 2, 3, 28, 35)])
def test_stem_finish(h1_dtype, C, B, L, HP, WP):
    """vg_stem_finish_fwd (C = 128, the lead-time dedup: field n = b L + l reads sample b) and vg_stem_finish_wide_fwd, with
    distinct per-field tt / tres / FiLM.  Each of the nine border cases of the time term (the four corners, the four edges and
    the interior) has its own tt row, so the whole-field comparison checks every one of them."""
    o = O()
    N = B * L
    ops_in = _stem_operands(B, L, HP, WP, C, seed=60 + C)
    raw3, rawres, bias3, bias1, tt, tres, g, be, film = ops_in
    h1 = pg_nan(N, HP, WP, C, h1_dtype)
    res = pg_nan(N, HP, WP, C)
    o.stem_finish(raw3, rawres, bias3, bias1, tt, tres, g, be, EPS, film, B, L, HP, WP, h1, res)
    torch.cuda.synchronize()
    h1ref, resref = _stem_ref(B, L, HP, WP, C, *ops_in)
    got = pg_frame(h1, N, HP, WP)
    r = {}
    if h1_dtype == BF16:
        r["h1_rn"] = rn16(got, h1ref, per_field_abs_allow(h1ref))
    else:
        r["h1"], r["h1_rel"] = f32_ratio(got, h1ref)
    # res: a sum of three fp32 terms (two roundings)
    rgot = pg_frame(res, N, HP, WP)
    rabs = pg_frame(rawres, B, HP, WP).abs().to(F64)[torch.arange(N, device=DEV) // L] + bias1.abs().to(F64) + \
        tres.abs().to(F64)[:, None, None, :]
    r["res"] = ((rgot.to(F64) - resref).abs() / (2 * 2.0 ** -24 * rabs + 1e-30)).max().item()
    note(**r)
    assert_pads_zero(h1, N, HP, WP)
    assert_pads_zero(res, N, HP, WP)
    for k, v_ in r.items():
        if not k.endswith("_rel"):
            assert v_ <= 1.0, (k, r)


@pytest.mark.parametrize("mode", ["bf16", "tf32_exact", "tf32_plain"])
@pytest.mark.parametrize("kind", ["conv3x3", "res_conv"])
def test_stem_gemm(mode, kind):
    """the per-sample stem GEMMs of the 12-hour model at 84x70, B = 4, Ca = 640 (600 data channels padded to 64): the raw
    3x3 conv (9 taps) and the 1x1 res_conv, fp32 outputs.  On plain fp32 operands the tf32 path must also be within the fp32
    bound of the operands truncated to tf32, and outside it against the exact operands (measured 1.6e-5 / 2.1e-6 against 7.8e-4 /
    8.0e-4 on a B200), as in test_conv3x3_ln_tf32_plain_operands"""
    o = O()
    B, HP, WP, Ca, Co = 4, 84, 70, 640, 128
    x = rnd(B, Ca, HP, WP, seed=71)
    k = 3 if kind == "conv3x3" else 1
    w = rnd(Co, Ca, k, k, seed=72, scale=1 / math.sqrt(k * k * Ca))
    dt = BF16 if mode == "bf16" else F32
    if mode == "bf16":
        x, w = x.to(BF16).float(), w.to(BF16).float()
    elif mode == "tf32_exact":
        x, w = tf32_exact(x), tf32_exact(w)
    xp = o.pg_from_nchw(x, dt)
    wt = w.permute(0, 2, 3, 1).reshape(Co, k * k * Ca).contiguous().to(dt)
    if kind == "conv3x3":
        out = o.gemm(xp, wt, ntaps=9, tap_shift=o.conv_tap_shifts(WP), out_f32=True, tf32=mode != "bf16")
    else:
        out = o.gemm(xp, wt, out_f32=True, tf32=mode != "bf16")
    torch.cuda.synchronize()
    assert out.dtype == F32 and torch.isfinite(out).all()
    ref = F.conv2d(x.to(F64), w.to(F64), padding=k // 2).permute(0, 2, 3, 1)
    extra = None
    if mode == "tf32_plain":
        extra = 2 * TF32_U * F.conv2d(x.abs().to(F64), w.abs().to(F64), padding=k // 2).permute(0, 2, 3, 1)
    got = pg_frame(out, B, HP, WP)
    # the 3x3 GEMM sums K = 5,760 products: measured 7.7e-6 (bf16) and 1.6e-5 (tf32) of the largest entry on a B200, the
    # tensor core's truncating fp32 accumulation over K / 8 (tf32) or K / 16 (bf16) instructions; the 2e-5 bound holds
    ratio, rel = f32_ratio(got, ref, extra=extra)
    r = dict(ratio=ratio, rel=rel)
    if mode == "tf32_plain":
        reft = F.conv2d(tf32_exact(x).to(F64), tf32_exact(w).to(F64), padding=k // 2).permute(0, 2, 3, 1)
        r["ratio_truncation_model"], r["rel_truncation_model"] = f32_ratio(got, reft)
    note(**r)
    assert ratio <= 1.0
    if mode == "tf32_plain":
        assert r["ratio_truncation_model"] <= 1.0 and rel > 5 * FP32_TOL, r


# =========================================================================================== MBConv chain, default precision
MB_N, MB_H, MB_W, MB_C, MB_HID = 24, 42, 35, 128, 512


def _gelu64(z):
    return F.gelu(z)                       # erf form (nn.GELU() default, maxvit.py:90,93)


@pytest.mark.parametrize("operands", ["tf32_exact", "plain"])
def test_mbconv_expand_tf32_fp16_out(operands):
    """1x1 expand of precision 'bf16' (maxvit.py:88-90): fp32 A, tf32 tcgen05, folded BN scale / shift, GELU, fp16 output
    (out_f32 = 3), at 24 fields of 42x35"""
    o = O()
    M = MB_N * MB_H * MB_W
    A = rnd(M, MB_C, seed=81)
    W = rnd(MB_HID, MB_C, seed=82, scale=1 / math.sqrt(MB_C))
    if operands == "tf32_exact":
        A, W = tf32_exact(A), tf32_exact(W)
    s = 0.5 + torch.rand(MB_HID, device=DEV, generator=torch.Generator(device=DEV).manual_seed(83))
    t = rnd(MB_HID, seed=84, scale=0.5)
    out = o.gemm(A, W, scale=s, shift=t, act=1, tf32=True, out_dtype=F16)
    torch.cuda.synchronize()
    assert out.dtype == F16
    z = A.to(F64) @ W.to(F64).t()
    ref = _gelu64(z * s.to(F64) + t.to(F64))
    sabs = A.abs().to(F64) @ W.abs().to(F64).t()
    # fp32 arithmetic: accumulation over 128 terms + the epilogue, times |s| and GELU's slope (<= 1.13)
    err = 1.13 * s.abs().to(F64) * (FP32_TOL * sabs)
    if operands == "plain":
        err = err + 1.13 * s.abs().to(F64) * 2 * TF32_U * sabs
    r = dict(rn=rn16(out, ref, err))
    if operands == "plain":
        reft = _gelu64((tf32_exact(A).to(F64) @ tf32_exact(W).to(F64).t()) * s.to(F64) + t.to(F64))
        r["rn_truncation_model"] = rn16(out, reft, 1.13 * s.abs().to(F64) * FP32_TOL * sabs)
    note(**r)
    assert r["rn"] <= 1.0
    if operands == "plain":                  # kind::tf32 truncates (measured 0.93 of the bound against the truncated operands)
        assert r["rn_truncation_model"] <= 1.0, r


def _dw_operands(N, H, W, C, dtype, seed):
    x = rnd(N, H, W, C, seed=seed).to(dtype)
    w = rnd(C, 1, 3, 3, seed=seed + 1, scale=1 / 3)
    s = 0.5 + torch.rand(C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 2))
    t = rnd(C, seed=seed + 3, scale=0.1)
    return x, w, s, t


def _dw_ref(x, w, s, t):
    C = x.shape[-1]
    z = F.conv2d(x.to(F64).permute(0, 3, 1, 2), w.to(F64), padding=1, groups=C)
    zabs = F.conv2d(x.abs().to(F64).permute(0, 3, 1, 2), w.abs().to(F64), padding=1, groups=C)
    y = _gelu64(z * s.to(F64).view(1, C, 1, 1) + t.to(F64).view(1, C, 1, 1))
    return y.permute(0, 2, 3, 1), (1.13 * s.abs().to(F64).view(1, C, 1, 1) * zabs).permute(0, 2, 3, 1)


@pytest.mark.parametrize("N", [MB_N, 768])
def test_mbconv_dw_fp16_se_chain(N):
    """the default-precision MBConv chain after the expand, kernel by kernel at 42x35 (128 -> 512 -> 128):
    vg_dw3x3_fwd in fp16 with GELU and the squeeze-excite partial sums, se_gate, vg_se_fold_weights to fp16 (bit-exact), and
    the fp16-operand GEMM (dtype 3) with per-field weights over 1,470 rows per field, folded BN and the fp32 residual.
    N = 768: the headline batch (fields 0, 1, 383, 766, 767 compared)"""
    o = O()
    H, W, C, Co, HW = MB_H, MB_W, MB_HID, MB_C, MB_H * MB_W
    x, w, s, t = _dw_operands(N, H, W, C, F16, seed=91)
    w9 = w.reshape(C, 9).t().contiguous()
    out = nan_like((N, H, W, C), F16)
    out, psum = o.dw3x3_bnact(x, w9, s, t, out=out)
    torch.cuda.synchronize()
    fields = list(range(N)) if N <= 24 else [0, 1, 383, 766, 767]
    fi = torch.tensor(fields, device=DEV)
    yref, yabs = _dw_ref(x[fi], w, s, t)
    r = dict(dw_rn=rn16(out[fi], yref, FP32_TOL * yabs))
    # psum: per field and channel, the strips' partial sums add up to the sum of the GELU outputs over the 1,470 pixels
    assert psum.shape == (N, o._lib.load().vg_dw_strips(W), C) and torch.isfinite(psum).all()
    tot = psum[fi].to(F64).sum(1)
    tref = yref.sum((1, 2))
    r["psum"] = ((tot - tref).abs() / (FP32_TOL * yref.abs().sum((1, 2)))).max().item()
    # squeeze-excite gate on the kernel's own partial sums
    se = C // 4
    W1, W2 = rnd(se, C, seed=95, scale=1 / math.sqrt(C)), rnd(C, se, seed=96, scale=1 / math.sqrt(se))
    gate = o.se_gate(psum, HW, W1, W2)
    gref = torch.sigmoid(F.linear(F.relu(F.linear(psum.to(F64).sum(1) / HW, W1.to(F64))), W2.to(F64)))
    r["gate"], r["gate_rel"] = f32_ratio(gate, gref)
    # per-field projection weights W * gate, rounded once to fp16: bit-exact
    Wp = rnd(Co, C, seed=97, scale=1 / math.sqrt(C))
    wn = o.se_fold_weights(Wp, gate, dtype=F16)
    assert torch.equal(wn, (Wp[None] * gate[:, None, :]).to(F16).reshape(N * Co, C))
    wn32 = o.se_fold_weights(Wp, gate, dtype=F32)
    assert torch.equal(wn32, (Wp[None] * gate[:, None, :]).reshape(N * Co, C))
    # dtype-3 GEMM: fp16 operands, per-field weights (rows_per_batch = 1,470), BN scale / shift, fp32 residual, fp32 out
    sp = 0.5 + torch.rand(Co, device=DEV, generator=torch.Generator(device=DEV).manual_seed(98))
    tp = rnd(Co, seed=99, scale=0.1)
    xres = rnd(N * HW, Co, seed=100)
    y = nan_like((N * HW, Co))
    o.gemm(out.view(N * HW, C), wn, rows_per_batch=HW, b_rows_per_batch=Co, scale=sp, shift=tp, res=xres, out=y, out_f32=True)
    torch.cuda.synchronize()
    A = out.view(N, HW, C)[fi].to(F64)
    Wf = wn.view(N, Co, C)[fi].to(F64)
    yr = torch.einsum("nrk,nok->nro", A, Wf) * sp.to(F64) + tp.to(F64) + xres.view(N, HW, Co)[fi].to(F64)
    r["proj"], r["proj_rel"] = f32_ratio(y.view(N, HW, Co)[fi], yr)
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("C,N,H,W", [(1536, 2, 14, 21), (2048, 2, 14, 21), (1024, 2, 14, 21), (1024, 48, 42, 35), (2048, 48, 42, 35)],
                         ids=["1536", "2048", "1024", "1024_n48_42x35", "2048_n48_42x35"])
def test_dw3x3_bnact_wide_hidden(dtype, C, N, H, W):
    """vg_dw3x3_bnact_fwd at hidden widths where 128 % (C / 4) != 0 (dims 256, 384 and 512 x expansion 4), with its per-row
    channel sums, and vg_se_scale_fwd in place.  C = 1024 is the one width where a block of 256 threads holds two pixel lanes
    per row (C / 8 = 128 channel groups) whose partial sums the block adds up; at W = 35 the two lanes get 18 and 17 pixels.
    48 fields of 42x35: the configs[4] chunk"""
    o = O()
    x, w, s, t = _dw_operands(N, H, W, C, dtype, seed=110)
    out = nan_like((N, H, W, C), dtype)
    out, psum = o.dw3x3_bnact(x, w.reshape(C, 9).t().contiguous(), s, t, out=out)
    torch.cuda.synchronize()
    yref, yabs = _dw_ref(x, w, s, t)
    r = {}
    if dtype == BF16:
        r["dw_rn"] = rn16(out, yref, FP32_TOL * yabs)
    else:
        r["dw"], r["dw_rel"] = f32_ratio(out, yref, extra=FP32_TOL * yabs)
    assert psum.shape == (N, H, C)
    r["psum"] = ((psum.to(F64) - yref.sum(2)).abs() / (FP32_TOL * yref.abs().sum(2))).max().item()
    gate = torch.rand(N, C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(115))
    before = out.clone()
    o.se_scale_(out, gate)
    assert torch.equal(out, (before.float() * gate[:, None, None, :]).to(dtype))
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)


# =========================================================================================== decoder and the smaller pieces
@pytest.mark.parametrize("N,HP,WP", [(4, 84, 70), (1, 518, 518)])
@pytest.mark.parametrize("dtype,out_dtype", [(F32, F32), (BF16, BF16), (BF16, F32)], ids=["fp32", "bf16", "bf16_to_fp32"])
def test_pool2(N, HP, WP, dtype, out_dtype):
    """MaxPool2d(2,2) PG -> channels-last, bit-exact (bf16 -> fp32 widens exactly)"""
    o, C = O(), 128
    x = rnd(N, C, HP, WP, seed=120).to(dtype)
    out = nan_like((N, HP // 2, WP // 2, C), out_dtype)
    call("vg_pool2_fwd", o.DT_CODE[dtype], int(out_dtype != dtype), o.pg_from_nchw(x, dtype).data_ptr(), out.data_ptr(), N, HP, WP, C)
    torch.cuda.synchronize()
    assert torch.equal(out, F.max_pool2d(x.float(), 2, 2).permute(0, 2, 3, 1).to(out_dtype))


CONVT_MODES = {   # the decoder's ConvTranspose2d as each precision runs it (metnet3.py:315)
    "bf16_mixed": (F32, True, BF16, True),     # precision 'bf16': tf32 MaxViT output -> bf16 decoder input + fp32 skip copy
    "bf16_all": (BF16, False, BF16, False),
    "fp32": (F32, False, F32, False),
}


@pytest.mark.parametrize("N,Hl,Wl", [(4, 42, 35), (1, 259, 259)])
@pytest.mark.parametrize("mode", list(CONVT_MODES))
def test_convT2(N, Hl, Wl, mode):
    """ConvTranspose2d(k=2, s=2) + depth-to-space into a PG buffer: the kernel writes the frame only, so the pads the caller
    zeroed must stay 0.0 and every frame entry (NaN before) must be written.  tf32 on tf32-representable operands."""
    o, C = O(), 128
    xdt, tf32, odt, with_copy = CONVT_MODES[mode]
    x = rnd(N, Hl, Wl, C, seed=130)
    w = rnd(C, C, 2, 2, seed=131, scale=1 / math.sqrt(C))
    x, w = (tf32_exact(x), tf32_exact(w)) if tf32 else (x.to(xdt).float(), w.to(xdt).float())
    b = rnd(C, seed=132, scale=0.1)
    HP, WP = 2 * Hl, 2 * Wl
    frame_nan = o.pg_from_nchw(torch.full((N, 1, HP, WP), float("nan"), device=DEV), F32)   # NaN in the frame, 0 at pads
    out = frame_nan.expand(-1, C).to(odt).contiguous()
    copy = frame_nan.expand(-1, C).contiguous() if with_copy else None
    o.convT2(x.to(xdt), w.permute(2, 3, 1, 0).reshape(4 * C, C).contiguous().to(xdt), b, out, tf32=tf32, out_copy=copy)
    torch.cuda.synchronize()
    ref = F.conv_transpose2d(x.permute(0, 3, 1, 2).to(F64), w.to(F64), b.to(F64), stride=2).permute(0, 2, 3, 1)
    rabs = F.conv_transpose2d(x.permute(0, 3, 1, 2).abs().to(F64), w.abs().to(F64), b.abs().to(F64), stride=2).permute(0, 2, 3, 1)
    r = {}
    got = pg_frame(out, N, HP, WP)
    if odt == BF16:
        r["out_rn"] = rn16(got, ref, FP32_TOL * rabs)
    else:
        r["out"], r["out_rel"] = f32_ratio(got, ref, extra=FP32_TOL * rabs)
    assert_pads_zero(out, N, HP, WP)
    if copy is not None:
        r["copy"], r["copy_rel"] = f32_ratio(pg_frame(copy, N, HP, WP), ref, extra=FP32_TOL * rabs)
        assert_pads_zero(copy, N, HP, WP)
        assert torch.equal(out.float(), copy.to(BF16).float())
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)


@pytest.mark.parametrize("N,nwin", [(24, 30), (2, 1369)])
def test_reg_mean(N, nwin):
    """mean of the register tokens over the windows (42x35: 30 windows; 259x259: 1,369)"""
    RC = 4 * 128
    x = 1.0 + rnd(N, nwin, RC, seed=140)
    out = nan_like((N, RC))
    call("vg_reg_mean_fwd", x.data_ptr(), out.data_ptr(), N, nwin, RC)
    torch.cuda.synchronize()
    ratio, rel = f32_ratio(out, x.to(F64).mean(1))
    note(ratio=ratio, rel=rel)
    assert ratio <= 1.0


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
def test_prepare_12hr(dtype):
    """metnet3.py:356-387 at the 12-hour geometry (25 x 24 channels of 82x67 -> 84x70 PG with 640 channels), bit-exact,
    every pad and every channel above T*C exactly 0.0"""
    o = O()
    cfg = synth.CFG_12HR
    B, Cpad = 2, 640
    x = rnd(B, cfg.T, cfg.C, cfg.H, cfg.W, seed=150, scale=10.0) + 20.0
    out = pg_nan(B, cfg.HP, cfg.WP, Cpad, dtype)
    strides = (ctypes.c_longlong * 5)(*x.stride())
    pl, pr, pt, pb = cfg.pads
    call("vg_prepare_fwd", o.DT_CODE[dtype], x.data_ptr(), strides, B, cfg.T, cfg.C, cfg.H, cfg.W, pt, pl, cfg.HP, cfg.WP, Cpad,
         float(cfg.pm25_mean), float(cfg.pm25_std), out.data_ptr())
    torch.cuda.synchronize()
    ref = x.cpu()                       # on the host: torch's CUDA division by a Python scalar multiplies by the reciprocal
    pm = torch.tensor([4, 10, 16, 22])
    ref[:, :, pm] = (ref[:, :, pm] - cfg.pm25_mean) / cfg.pm25_std
    ref = F.pad(ref, cfg.pads).reshape(B, cfg.T * cfg.C, cfg.HP, cfg.WP).permute(0, 2, 3, 1)
    got = pg_frame(out, B, cfg.HP, cfg.WP).cpu()
    assert torch.equal(got[..., :cfg.T * cfg.C], ref.to(dtype))
    assert torch.equal(got[..., cfg.T * cfg.C:].float(), torch.zeros_like(got[..., cfg.T * cfg.C:].float()))
    assert_pads_zero(out, B, cfg.HP, cfg.WP)


# =========================================================================================== fused attention, many tiles per CTA
def _attn_sd(dim, heads, dh, w, r, seed):
    spec = {k[len("layers.0.1."):]: v for k, v in synth.maxvit_spec(dim, 1, 2, heads, dh, w, 4, 0.25, r).items()
            if k.startswith("layers.0.1.")}
    return synth.make_state_dict(spec, seed=seed)


@pytest.mark.parametrize("bound", [False, True], ids=["running_max", "logit_bound"])
@pytest.mark.parametrize("grid_mode", [False, True], ids=["block", "grid"])
def test_attention_fused_many_tiles(grid_mode, bound):
    """the one-kernel attention layer at 24 fields of 42x35 (720 windows: several tiles per CTA) against the float64 oracle,
    per field: the output x + attn(x) within 4e-3 of the field's largest entry (fp16 QKV and X, bf16 P and V), and the
    attention term alone (x_out - x) within 4e-3 of its own largest entry: the residual does not hide it (measured 2.6e-3,
    2.3e-3 and 2.7e-3 on a B200)"""
    o = O()
    N, H, W, C, heads, dh, w, R = 24, 42, 35, 128, 32, 32, 7, 4
    sd = _attn_sd(C, heads, dh, w, R, seed=9)
    x = torch.randn(N, H, W, C, generator=torch.Generator().manual_seed(161))
    cond = torch.randn(N, 2, generator=torch.Generator().manual_seed(162))
    reg = torch.randn(*((N, R, C) if grid_mode else (R, C)), generator=torch.Generator().manual_seed(163))
    nwin = (H // w) * (W // w)
    idx = (mo.grid_pixel_index if grid_mode else mo.block_pixel_index)(H, W, w).reshape(-1)
    flat = x.reshape(N, H * W, C).double()
    tok = flat[:, idx].reshape(N * nwin, w * w, C)
    regd = reg.double()
    regs = regd.repeat_interleave(nwin, 0) if grid_mode else regd[None].expand(N * nwin, R, C)
    seq = torch.cat([regs, tok], dim=1)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    att = mo.attention(seq, cond.double(), sd64, "", heads=heads, window=w, num_reg=R)
    att_x = torch.empty_like(flat)
    att_x[:, idx] = att[:, R:].reshape(N, nwin * w * w, C)
    gamma, beta = mo.film(cond, sd, "")
    film = torch.cat([gamma, beta], dim=1).to(DEV).contiguous()
    inner = heads * dh
    wq = sd["to_qkv.weight"]
    wqkv_h = torch.stack([wq[i * inner:(i + 1) * inner].reshape(heads, dh, C) for i in range(3)], dim=1).reshape(heads * 96, C)
    wout_h = sd["to_out.0.weight"].reshape(C, heads, dh).permute(1, 0, 2).contiguous()
    head_tab = o.pack_head_tables(sd["rel_pos_bias.weight"], sd["q_norm.gamma"], sd["k_norm.gamma"]).to(DEV)
    lb = 0.0
    if bound:
        lb = o.attn_logit_bound(sd["rel_pos_bias.weight"].to(DEV), sd["q_norm.gamma"].to(DEV), sd["k_norm.gamma"].to(DEV), dh)
    xd = x.to(DEV)
    x_out, reg_out = o.attn_fused(xd, reg.to(DEV), film, wqkv_h.contiguous().to(DEV), wout_h.to(DEV), head_tab, w, R, grid_mode,
                                  True, heads, dh, logit_bound=lb)
    torch.cuda.synchronize()
    ref_x = (flat + att_x).to(DEV)
    r = {}
    r["x"], r["x_rel"] = f32_ratio(x_out.reshape(N, H * W, C), ref_x, tol=4e-3)
    r["reg"], r["reg_rel"] = f32_ratio(reg_out.view(N, nwin, R, C), (seq[:, :R] + att[:, :R]).view(N, nwin, R, C).to(DEV), tol=4e-3)
    r["attn"], r["attn_rel"] = f32_ratio((x_out.reshape(N, H * W, C) - xd.reshape(N, H * W, C)), att_x.to(DEV), tol=4e-3)
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)
