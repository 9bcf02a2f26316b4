"""Per-kernel parity of the un-fused MaxViT inference chain (GPU) against float64, at the chunk BASELINE configs[4] runs in
fp32 (max_fields = 48 fields of 42x35: 76,320 token rows, 46,080 (window, head) blocks of 32 heads x 64) and at the edges where
the kernels change path.  Every MaxViT layer takes this chain when MaxViT.fused_attn_applies is false: every wide network
(256 / 384 / 512 channels, dim_head 64; 3xTF32 projections and the split tensor-core core by default), set_precision("fp32")
at any width, the tf32 / bf16 modes at wide widths, and the forward of the fp32 training step.

  attention : vg_attn_gather_fwd -> QKV vg_gemm_fwd -> vg_attn_core_fwd -> vg_attn_out_fwd (out-projection + residual + scatter)
  MBConv    : 3xTF32 expand + BN + GELU -> (depthwise, squeeze-excite: test_infer_kernels_gpu.py, test_maxvit_wide_train_gpu.py)
              -> vg_se_fold_weights -> per-field 3xTF32 projection + BN + residual

Conventions (those of test_infer_kernels_gpu.py):
  * every reference is float64 on the GPU, built from the operands as the device sees them (bf16 via .to(dtype))
  * every output the kernel must write completely starts as NaN
  * comparisons are per field, and per (window, head) for the attention core: a bad field or window is not averaged away
  * each GEMM runs twice: on small-integer operands, where every sum is exact (in 3xTF32 the lo halves are 0), so the output
    must be bit-equal across the whole tensor -- every tile, slice, field boundary and scatter target -- and on Gaussian
    operands, within an existing rule: FP32_TOL of the field's largest entry (exact fp32), 1.5 (3K/8) 2^-24 + 1e-6 (3xTF32,
    test_gemm_3xtf32_is_fp32_accurate), + 2 * 2^-10 * sum|a||b| (plain tf32), half an ulp plus the fp32 error (16-bit outputs).
    Bounds without such a rule are at most 4x the value measured on a B200, stated next to them.
"""
import math
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle import maxvit_oracle as mo

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64, F32, BF16 = torch.float64, torch.float32, torch.bfloat16
FP32_TOL = 2e-5            # exact-fp32 outputs: max |err| / max |ref| per field
TF32_U = 2.0 ** -10         # 2 * TF32_U * sum|a||b| bounds the tf32 operand rounding or truncation
WIN, R_REG, EPS = 7, 4, 1e-5
S_TOK = R_REG + WIN * WIN
# the configs[4] fp32 chunk: 48 fields of 42x35, 512 channels, 32 heads x 64
CH_N, CH_H, CH_W, CH_C, CH_HEADS, CH_DH = 48, 42, 35, 512, 32, 64
CH_NWIN = (CH_H // WIN) * (CH_W // WIN)
CH_ROWS = CH_N * CH_NWIN * S_TOK          # 76,320


def O():
    from vit_grid_model_b200 import ops
    return ops


def OT():
    from vit_grid_model_b200 import ops_train
    return ops_train


def note(**kv):
    """one line per measurement (pytest -s shows them; the measured values in the comments below come from these lines)"""
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0].split("::")[-1]
    print("MEASURE", test, " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in kv.items()))


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, generator=g, device=DEV) * scale


def ints(*shape, seed=0, lo=-2, hi=2):
    """small integers as fp32: exact in tf32 and bf16, and every sum of the tests below stays far below 2^24"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(lo, hi + 1, shape, generator=g, device=DEV).float()


def nan_like(shape, dtype=F32):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def tf32_trunc(t):
    """t rounded to fp32, then the 13 low mantissa bits cleared (what the tensor core reads of an fp32 operand)"""
    return (t.float().contiguous().view(torch.int32) & -8192).view(F32).to(t.dtype)


def x3_tol(K):
    """the 3xTF32 rule: the truncating fp32 accumulation of the tensor core over 3K/8 instructions"""
    return 1.5 * (3 * K / 8) * 2.0 ** -24 + 1e-6


def field_max(ref, N):
    """(N, ...) -> max |ref| of each field, broadcastable to ref"""
    return ref.abs().reshape(N, -1).amax(1).view(N, *([1] * (ref.dim() - 1)))


def ratio(got, ref, allow):
    """largest |got - ref| / allow (element-wise allowance); NaN anywhere in got fails"""
    g = got.to(F64)
    assert not torch.isnan(g).any(), "NaN in the output: an entry was not written"
    return ((g - ref).abs() / allow).max().item()


def field_rel(got, ref, N):
    """worst over the fields of max |err| / max |ref| of the field"""
    err = (got.to(F64) - ref).abs().reshape(N, -1).amax(1)
    return (err / ref.abs().reshape(N, -1).amax(1).clamp_min(1e-300)).max().item()


def rn16(got, ref64, err_abs=0.0):
    """largest |got - ref| / (ulp / 2 + err_abs) of 16-bit results (test_infer_kernels_gpu.rn16): <= 1 means got is the
    reference rounded to nearest, up to the fp32 arithmetic's own error err_abs in front of the rounding"""
    dt = got.dtype
    r = ref64.to(dt).to(F64)
    g = got.to(F64)
    assert not torch.isnan(g).any(), "NaN in the output"
    _, e = torch.frexp(torch.maximum(r.abs(), g.abs()))
    bits, tiny = (8, 2.0 ** -133) if dt == BF16 else (11, 2.0 ** -24)
    ulp = torch.ldexp(torch.ones_like(r), e - bits).clamp_min(tiny)
    return ((g - ref64).abs() / (0.5 * ulp + torch.as_tensor(err_abs, dtype=F64, device=DEV))).max().item()


def pixel_map(Hl, Wl, grid_mode, win=WIN):
    """(nwin * win^2,) flat pixel of every window token, windows x-major (the oracle's index maps)"""
    return (mo.grid_pixel_index if grid_mode else mo.block_pixel_index)(Hl, Wl, win).reshape(-1).to(DEV)


# =========================================================================================== gather + QKV projection
GATHER_GEOMS = {"n48_42x35_block": (48, 42, 35, False), "n48_42x35_grid": (48, 42, 35, True), "n1_259x259_grid": (1, 259, 259, True)}
GATHER_DTYPES = {"fp32": (F32, F32), "bf16": (BF16, BF16), "fp32_to_bf16": (F32, BF16)}


def _gather_operands(N, Hl, Wl, C, grid_mode, seed):
    """x with a per-channel offset (the LayerNorm's mean matters), registers shared (block) or per field (grid), FiLM rows"""
    x = rnd(N, Hl, Wl, C, seed=seed) + rnd(C, seed=seed + 1)
    reg = rnd(*((N, R_REG, C) if grid_mode else (R_REG, C)), seed=seed + 2)
    film = torch.cat([1 + 0.3 * rnd(N, C, seed=seed + 3), 0.3 * rnd(N, C, seed=seed + 4)], dim=1).contiguous()
    return x, reg, film


def _gather_ref(x, reg, film, grid_mode):
    """(N, nwin, S, C): (registers ++ window tokens) -> LayerNorm without affine -> raw FiLM (maxvit.py:137, 187)"""
    N, Hl, Wl, C = x.shape
    nwin = (Hl // WIN) * (Wl // WIN)
    xs = x.to(F64).reshape(N, Hl * Wl, C)[:, pixel_map(Hl, Wl, grid_mode)].view(N, nwin, WIN * WIN, C)
    r = reg.to(F64)
    rege = (r[:, None] if reg.dim() == 3 else r[None, None]).expand(N, nwin, R_REG, C)
    f = film.to(F64)
    return F.layer_norm(torch.cat([rege, xs], dim=2), (C,), eps=EPS) * f[:, None, None, :C] + f[:, None, None, C:]


@pytest.mark.parametrize("dt", list(GATHER_DTYPES))
@pytest.mark.parametrize("geom", list(GATHER_GEOMS))
@pytest.mark.parametrize("C", [128, 256, 384, 512])
def test_attn_gather(C, geom, dt):
    """vg_attn_gather_fwd at C = 128 .. 512: block partition with shared register tokens, grid partition with per-field ones
    (stride 37 at 259x259); fp32 -> fp32, bf16 -> bf16 and fp32 -> bf16 tokens.  Every token row is NaN-prefilled and
    compared per field"""
    o = O()
    N, Hl, Wl, grid_mode = GATHER_GEOMS[geom]
    xdt, odt = GATHER_DTYPES[dt]
    x, reg, film = _gather_operands(N, Hl, Wl, C, grid_mode, seed=10 + C)
    x = x.to(xdt)
    nwin = (Hl // WIN) * (Wl // WIN)
    out = nan_like((N * nwin * S_TOK, C), odt)
    o.attn_gather(x, reg, film, WIN, R_REG, grid_mode, eps=EPS, out=out)
    torch.cuda.synchronize()
    ref = _gather_ref(x, reg, film, grid_mode)
    got = out.view(N, nwin, S_TOK, C)
    if odt == BF16:
        r = dict(rn=rn16(got, ref, FP32_TOL * field_max(ref, N)))
    else:
        r = dict(ratio=ratio(got, ref, FP32_TOL * field_max(ref, N)), rel=field_rel(got, ref, N))
    note(**r)
    assert max(v for k, v in r.items() if k != "rel") <= 1.0, r


QKV_MODES = {"simt_fp32": dict(), "tf32": dict(tf32=True), "x3": dict(x3=True), "x3_cached": dict(x3=True)}
FIELDS = (0, CH_N // 2, CH_N - 1)          # first, middle and last field of the chunk


@pytest.mark.parametrize("operands", ["int", "gauss"])
@pytest.mark.parametrize("mode", list(QKV_MODES))
def test_qkv_projection_chunk(mode, operands):
    """the QKV projection of the configs[4] chunk, ops.gemm(tokens, W_qkv): 76,320 x 6,144 over K = 512 in SIMT fp32, plain
    tf32 and 3xTF32 (x3=True, splitting the weights per call or from a cached Wt_x3).  Integer operands: the whole output
    bit-equal to the exact product.  Gaussian: the gathered tokens of 48 fields; the rows of the first, a middle and the last
    field against float64"""
    o = O()
    M, K, Nout = CH_ROWS, CH_C, 3 * CH_HEADS * CH_DH
    if operands == "int":
        A, W = ints(M, K, seed=31), ints(Nout, K, seed=32)
    else:
        x, reg, film = _gather_operands(CH_N, CH_H, CH_W, K, False, seed=33)
        A = o.attn_gather(x, reg, film, WIN, R_REG, False, eps=EPS)
        W = rnd(Nout, K, seed=34, scale=1 / math.sqrt(K))
    kw = dict(QKV_MODES[mode])
    if mode == "x3_cached":
        kw["Wt_x3"] = o.split3_tf32(W, 1)
    out = nan_like((M, Nout))
    o.gemm(A, W, out=out, **kw)
    torch.cuda.synchronize()
    if operands == "int":
        assert torch.equal(out.to(F64), A.to(F64) @ W.to(F64).t()), "integer QKV projection not exact"
        return
    rows = torch.cat([torch.arange(f * CH_NWIN * S_TOK, (f + 1) * CH_NWIN * S_TOK, device=DEV) for f in FIELDS])
    n = len(FIELDS)
    a64 = A[rows].to(F64)
    ref = (a64 @ W.to(F64).t()).view(n, -1, Nout)
    got = out[rows].view(n, -1, Nout)
    tol = x3_tol(K) if mode.startswith("x3") else FP32_TOL
    allow = tol * field_max(ref, n)
    if mode == "tf32":
        allow = allow + 2 * TF32_U * (a64.abs() @ W.to(F64).abs().t()).view(n, -1, Nout)
    r = dict(ratio=ratio(got, ref, allow), rel=field_rel(got, ref, n))
    note(**r)
    assert r["ratio"] <= 1.0, r


# =========================================================================================== attention core
def _core_operands(N, Hl, Wl, win, R, heads, dh, seed, zero_token=None):
    """qkv rows [q | k | v] of every (window, token), the two RMSNorm gains U(0.5, 1.5) (synth 'pos') and the bias table;
    zero_token: a token whose q and k are zero in every window and head (F.normalize's eps branch)"""
    S, nwin = R + win * win, (Hl // win) * (Wl // win)
    inner = heads * dh
    qkv = rnd(N * nwin * S, 3 * inner, seed=seed)
    if zero_token is not None:
        qkv.view(N * nwin, S, 3 * inner)[:, zero_token, :2 * inner] = 0
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    qg = 0.5 + torch.rand(inner, device=DEV, generator=g)
    kg = 0.5 + torch.rand(inner, device=DEV, generator=g)
    bt = rnd((2 * win - 1) ** 2 + 1, heads, seed=seed + 2)
    return qkv, qg, kg, bt


def _core_ref(qkv, qg, kg, bt, S, win, R, heads, dh, pmask=None, tf32_ops=False):
    """float64 maxvit.py:189-213 per (window, head) -> (nw * heads, S * dh).  pmask: dropout of the probabilities (scaled,
    applied after the softmax; the normaliser is not dropped).  tf32_ops: round where the single-product tensor-core kernel
    rounds -- q-hat, K-hat, P and V truncated to tf32"""
    nw = qkv.shape[0] // S
    x = qkv.to(F64).view(nw, S, 3, heads, dh).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    rs = math.sqrt(dh)
    qh = F.normalize(q, dim=-1) * rs * qg.to(F64).view(heads, 1, dh)
    kh = F.normalize(k, dim=-1) * rs * kg.to(F64).view(heads, 1, dh)
    if tf32_ops:
        qh, kh, v = tf32_trunc(qh), tf32_trunc(kh), tf32_trunc(v)
    idx = mo.rel_pos_indices(win, R).to(DEV)
    P = torch.softmax(qh @ kh.transpose(-1, -2) + bt.to(F64)[idx].permute(2, 0, 1), dim=-1)
    del qh, kh
    if tf32_ops:
        P = tf32_trunc(P)
    if pmask is not None:
        P = P * pmask
    return (P @ v).reshape(nw * heads, S * dh)


def _per_block(out, S, heads, dh):
    """(nw * S, heads * dh) kernel output -> (nw * heads, S * dh)"""
    nw = out.shape[0] // S
    return out.view(nw, S, heads, dh).permute(0, 2, 1, 3).reshape(nw * heads, S * dh)


def block_rel(got, ref):
    """worst over the (window, head) blocks of max |err| / max |ref| of the block"""
    g = got.to(F64)
    assert not torch.isnan(g).any(), "NaN in the output: an entry was not written"
    return ((g - ref).abs().amax(1) / ref.abs().amax(1).clamp_min(1e-300)).max().item()


# per (window, head), of the block's largest entry.  Codes 1 (exact-fp32 SIMT) and 2 (3xTF32 mma.sync) keep the fp32 rule
# (measured 3.5e-6 and 1.05e-5 at the chunk).  Codes 4 (single tf32 products, fp32 storage) and 0 (bf16 storage) against the
# reference that truncates q-hat, K-hat, P and V to tf32: at most 4x the worst value measured on an NVIDIA B200 at 1000 W --
# code 4 2.9e-3 (the chunk; 5.9e-3 against the exact operands), code 0 3.9e-3 (the chunk; 3.7e-3 for the SIMT kernel on bf16
# storage at S = 128, where the bf16 output rounding dominates)
CORE_BOUND = {1: FP32_TOL, 2: FP32_TOL, 4: 1e-2, 0: 1.5e-2}


@pytest.mark.parametrize("code", [1, 2, 4, 0, 6])
def test_attn_core_chunk(code):
    """vg_attn_core_fwd on the configs[4] chunk: 48 fields of 42x35, w 7, R 4 (S = 53: the last four-key group holds three pad
    keys), 32 heads x 64 = 46,080 (window, head) blocks, every one compared.  Code 6 (the output rows as the 3xTF32 left
    operand [hi | hi | lo]) is bit for bit split3_tf32 of code 2's output"""
    o = O()
    qkv, qg, kg, bt = _core_operands(CH_N, CH_H, CH_W, WIN, R_REG, CH_HEADS, CH_DH, seed=41)
    geo = (CH_N, CH_H, CH_W, WIN, R_REG, CH_HEADS, CH_DH)
    inner = CH_HEADS * CH_DH
    if code == 6:
        plain = o.attn_core(qkv, qg, kg, bt, *geo, out=nan_like((CH_ROWS, inner)), x3=True)
        split = o.attn_core(qkv, qg, kg, bt, *geo, x3=True, split_out=True)
        torch.cuda.synchronize()
        assert torch.equal(split, o.split3_tf32(plain, 0))
        return
    src = qkv.to(BF16) if code == 0 else qkv
    out = nan_like((CH_ROWS, inner), src.dtype)
    o.attn_core(src, qg, kg, bt, *geo, out=out, x3=code == 2, tf32=code == 4)
    torch.cuda.synchronize()
    ref = _core_ref(src, qg, kg, bt, S_TOK, WIN, R_REG, CH_HEADS, CH_DH, tf32_ops=code in (4, 0))
    r = dict(rel=block_rel(_per_block(out, S_TOK, CH_HEADS, CH_DH), ref))
    if code in (4, 0):        # against the exact operands: what the tf32 rounding model accounts for
        r["rel_exact_operands"] = block_rel(_per_block(out, S_TOK, CH_HEADS, CH_DH),
                                            _core_ref(src, qg, kg, bt, S_TOK, WIN, R_REG, CH_HEADS, CH_DH))
    note(**r)
    assert r["rel"] <= CORE_BOUND[code], r


@pytest.mark.parametrize("N,Hl,Wl", [(48, 42, 35), (1, 259, 259)])
def test_attn_core_12hr_heads_fp32(N, Hl, Wl):
    """the 12-hour model's heads (32 x 32, inner 1,024) in exact fp32 (code 1, the SIMT kernel) at 48 fields of 42x35 and at
    1 x 259x259 (1,369 windows)"""
    o = O()
    heads, dh = 32, 32
    qkv, qg, kg, bt = _core_operands(N, Hl, Wl, WIN, R_REG, heads, dh, seed=51)
    out = nan_like((qkv.shape[0], heads * dh))
    o.attn_core(qkv, qg, kg, bt, N, Hl, Wl, WIN, R_REG, heads, dh, out=out)
    torch.cuda.synchronize()
    r = dict(rel=block_rel(_per_block(out, S_TOK, heads, dh), _core_ref(qkv, qg, kg, bt, S_TOK, WIN, R_REG, heads, dh)))
    note(**r)
    assert r["rel"] <= CORE_BOUND[1], r


# (N, Hl, Wl, win, R): S = 64 is the largest sequence of the mma.sync kernel (w 8, no registers: every query row tile full);
# S = 65 falls to the SIMT kernel even for codes 2 and 4; S = 128 is the SIMT kernel's largest; S = 27 (w 5, R 2) leaves one
# real key in its last four-key group
CORE_EDGES = {"S64_w8_R0": (2, 16, 24, 8, 0), "S65_w8_R1": (2, 16, 24, 8, 1), "S128_w11_R7": (2, 22, 11, 11, 7),
              "S27_w5_R2": (3, 10, 15, 5, 2)}


@pytest.mark.parametrize("code", [1, 2, 4, 0])
@pytest.mark.parametrize("dh", [32, 64])
@pytest.mark.parametrize("edge", list(CORE_EDGES))
def test_attn_core_edges(edge, dh, code):
    """vg_attn_core_fwd where it changes path, with one token whose q and k are zero in every window and head (F.normalize's
    eps branch: its scores are the bias alone, and it is a zero key for every query).  Above S = 64 codes 2 and 4 run the
    SIMT kernel: bit-equal to code 1"""
    o = O()
    N, Hl, Wl, win, R = CORE_EDGES[edge]
    heads = 4
    S = R + win * win
    qkv, qg, kg, bt = _core_operands(N, Hl, Wl, win, R, heads, dh, seed=61, zero_token=R + 3)
    src = qkv.to(BF16) if code == 0 else qkv
    out = nan_like((qkv.shape[0], heads * dh), src.dtype)
    o.attn_core(src, qg, kg, bt, N, Hl, Wl, win, R, heads, dh, out=out, x3=code == 2, tf32=code == 4)
    torch.cuda.synchronize()
    ref = _core_ref(src, qg, kg, bt, S, win, R, heads, dh, tf32_ops=S <= 64 and code in (4, 0))
    r = dict(rel=block_rel(_per_block(out, S, heads, dh), ref))
    note(**r)
    if S > 64 and code in (2, 4):
        assert torch.equal(out, o.attn_core(qkv, qg, kg, bt, N, Hl, Wl, win, R, heads, dh)), "S > 64 must run the SIMT kernel"
    assert r["rel"] <= (CORE_BOUND[1] if S > 64 and code in (2, 4) else CORE_BOUND[code]), r


def test_attn_core_rejects_long_sequence():
    """S = 129 (w 11, R 8) is one more than the SIMT kernel's largest sequence: VitGridError, nothing launched"""
    from vit_grid_model_b200 import _lib
    o = O()
    qkv, qg, kg, bt = _core_operands(1, 11, 11, 11, 8, 4, 32, seed=71)
    with pytest.raises(_lib.VitGridError, match="too long"):
        o.attn_core(qkv, qg, kg, bt, 1, 11, 11, 11, 8, 4, 32)


@pytest.mark.parametrize("dh", [32, 64])
def test_attn_core_simt_dropout(dh):
    """nn.Dropout on the probabilities (maxvit.py:146) at T = 26 (p = 26/256) in the SIMT kernel, the forward of the fp32
    training step: the kernel's masks, exported through vg_dropout_mask_debug, fed to the float64 reference.  Probabilities are
    dropped (and scaled) after the normalisation; the normaliser is not dropped.  Codes 2 and 4 with dropout run the same SIMT
    kernel: bit-equal"""
    o = O()
    N, Hl, Wl, heads, T = 4, 14, 21, 32, 26
    nwin = (Hl // WIN) * (Wl // WIN)
    drop = (20261021, 3, T)
    qkv, qg, kg, bt = _core_operands(N, Hl, Wl, WIN, R_REG, heads, dh, seed=81)
    out = nan_like((qkv.shape[0], heads * dh))
    o.attn_core(qkv, qg, kg, bt, N, Hl, Wl, WIN, R_REG, heads, dh, out=out, drop=drop)
    pm = OT().dropout_masks(drop, N * nwin, heads, 128)[0][:, :, :S_TOK, :S_TOK].to(F64) * (256.0 / (256 - T))
    torch.cuda.synchronize()
    ref = _core_ref(qkv, qg, kg, bt, S_TOK, WIN, R_REG, heads, dh, pmask=pm)
    r = dict(rel=block_rel(_per_block(out, S_TOK, heads, dh), ref), kept=pm.ne(0).double().mean().item())
    note(**r)
    assert r["rel"] <= CORE_BOUND[1], r
    for kw in (dict(x3=True), dict(tf32=True)):
        assert torch.equal(out, o.attn_core(qkv, qg, kg, bt, N, Hl, Wl, WIN, R_REG, heads, dh, drop=drop, **kw))


# =========================================================================================== out-projection + scatter
# (N, Hl, Wl, C, inner, win, R)
OUT_SHAPES = {"c512_chunk": (CH_N, CH_H, CH_W, CH_C, CH_HEADS * CH_DH, WIN, R_REG),
              "c128_n48": (48, 42, 35, 128, 1024, WIN, R_REG),
              "c128_n1_259x259": (1, 259, 259, 128, 1024, WIN, R_REG),
              "c256_w8_R0": (2, 16, 24, 256, 512, 8, 0)}
OUT_CODES = ["fp32", "tf32", "x3", "x3_split", "bf16"]


def _out_ref(attn, W, x_in, reg, N, Hl, Wl, C, win, R, grid_mode, out_mask=None):
    """float64 x_in + to_out(attn) scattered through the inverse partition map, and the register rows + reg_in; proj alone"""
    S, nwin = R + win * win, (Hl // win) * (Wl // win)
    proj = (attn.to(F64) @ W.to(F64).t()).view(N, nwin, S, C)
    if out_mask is not None:
        proj = proj * out_mask.view(N, nwin, S, C)
    x_ref = x_in.to(F64).reshape(N, Hl * Wl, C).clone()
    pix = pixel_map(Hl, Wl, grid_mode, win)
    x_ref[:, pix] += proj[:, :, R:].reshape(N, nwin * win * win, C)
    r = reg.to(F64)
    reg_ref = proj[:, :, :R] + (r[:, None] if reg.dim() == 3 else r[None, None])
    return x_ref.view(N, Hl, Wl, C), reg_ref, proj


def _run_attn_out(code, attn, W, x_in, reg, N, Hl, Wl, win, R, grid_mode, drop=(0, 0, 0)):
    """ops.attn_out in dtype code `code` into a NaN-prefilled x_out.  Block mode: ops.attn_out allocates reg_out itself, so the
    same launch runs again through vg_attn_out_fwd with NaN-prefilled x_out and reg_out, and must give the same bits"""
    from vit_grid_model_b200 import _lib
    o = O()
    x_out = nan_like(x_in.shape, x_in.dtype)
    kw = dict(x_out=x_out, drop=drop)
    a_dev, w_dev, tf32 = attn, W, code != "fp32" and code != "bf16"
    if code == "tf32":
        kw["tf32"] = True
    elif code == "x3":
        kw["x3"] = True
        a_dev, w_dev = o.split3_tf32(attn, 0), o.split3_tf32(W, 1)
    elif code == "x3_split":                              # the rows attn_core(split_out=True) writes, and the cached weight split
        a_dev, w_dev = o.split3_tf32(attn, 0), o.split3_tf32(W, 1)
        attn = a_dev
        kw.update(attn_is_split=True, Wt_x3=w_dev)
    want_reg = not grid_mode
    x_out, reg_out = o.attn_out(attn, W, x_in, reg, win, R, grid_mode, want_reg, **kw)
    if want_reg:
        x2, reg2 = nan_like(x_in.shape, x_in.dtype), nan_like(reg_out.shape)
        C = x_in.shape[-1]
        scratch = torch.empty(a_dev.shape[0] * C, device=DEV) if code == "fp32" else None
        _lib.call("vg_attn_out_fwd", o._gemm_code(a_dev.dtype, tf32), a_dev.data_ptr(), a_dev.shape[1], w_dev.data_ptr(),
                  x_in.data_ptr(), reg.data_ptr(), int(reg.dim() == 3), reg2.data_ptr(), x2.data_ptr(), N, Hl, Wl, C, win, R,
                  int(grid_mode), int(drop[0]), int(drop[1]), int(drop[2]), None if scratch is None else scratch.data_ptr(),
                  0 if scratch is None else scratch.numel(), o._st())
        torch.cuda.synchronize()
        assert torch.equal(x2, x_out) and torch.equal(reg2, reg_out), "vg_attn_out_fwd is not deterministic"
        x_out, reg_out = x2, reg2
    torch.cuda.synchronize()
    return x_out, reg_out


@pytest.mark.parametrize("operands", ["int", "gauss"])
@pytest.mark.parametrize("partition", ["block_reg_out", "grid"])
@pytest.mark.parametrize("code", OUT_CODES)
@pytest.mark.parametrize("shape", list(OUT_SHAPES))
def test_attn_out(shape, code, partition, operands):
    """vg_attn_out_fwd: to_out GEMM whose epilogue adds the residual and scatters every window token to its pixel (block: the
    register rows to reg_out with the shared reg_in; grid: per-field reg_in, no reg_out), in SIMT fp32, plain tf32, 3xTF32
    (x3=True, and attn_is_split=True with the cached weight split) and bf16.  x_out and reg_out start as NaN: every pixel and
    register row is written.  Integer operands: bit-equal everywhere; Gaussian: per field"""
    N, Hl, Wl, C, inner, win, R = OUT_SHAPES[shape]
    grid_mode = partition == "grid"
    if N == 1 and not grid_mode:
        pytest.skip("259x259 is a grid-attention geometry here (stride 37)")
    S, nwin = R + win * win, (Hl // win) * (Wl // win)
    rows = N * nwin * S
    make = (lambda *s, seed: ints(*s, seed=seed)) if operands == "int" else rnd
    attn = make(rows, inner, seed=91)
    W = make(C, inner, seed=92) if operands == "int" else rnd(C, inner, seed=92, scale=1 / math.sqrt(inner))
    x_in = make(N, Hl, Wl, C, seed=93)
    reg = make(*((N, R, C) if grid_mode else (R, C)), seed=94)
    if code == "bf16":
        attn, W, x_in = attn.to(BF16), W.to(BF16), x_in.to(BF16)
    x_out, reg_out = _run_attn_out(code, attn, W, x_in, reg, N, Hl, Wl, win, R, grid_mode)
    x_ref, reg_ref, proj = _out_ref(attn, W, x_in, reg, N, Hl, Wl, C, win, R, grid_mode)
    if operands == "int":
        assert torch.equal(x_out, x_ref.to(x_out.dtype)), "integer x_out not exact"
        if reg_out is not None:
            assert torch.equal(reg_out.view(N, nwin, R, C), reg_ref.float()), "integer reg_out not exact"
        return
    # element-wise allowance: the projection's rule of the field's largest projection entry (+ the tf32 operand bound), plus
    # the one fp32 rounding of the residual add
    pix = pixel_map(Hl, Wl, grid_mode, win)
    tol = x3_tol(inner) if code.startswith("x3") else FP32_TOL
    fm = field_max(proj, N).view(N, 1, 1, 1)
    allow_x = tol * fm + 2.0 ** -24 * x_ref.abs()
    if code == "tf32":
        pa = (attn.abs().to(F64) @ W.abs().to(F64).t()).view(N, nwin, S, C)
        ex = torch.zeros_like(x_ref).view(N, Hl * Wl, C)
        ex[:, pix] = pa[:, :, R:].reshape(N, nwin * win * win, C)
        allow_x = allow_x + 2 * TF32_U * ex.view_as(x_ref)
    r = {}
    if code == "bf16":
        r["x_rn"] = rn16(x_out, x_ref, FP32_TOL * fm)
    else:
        r["x"] = ratio(x_out, x_ref, allow_x)
    # the attention term alone, x_out - x_in, of its own largest entry: the residual does not hide it
    proj_x = torch.zeros_like(x_ref).view(N, Hl * Wl, C)
    proj_x[:, pix] = proj[:, :, R:].reshape(N, nwin * win * win, C)
    r["attn_term_rel"] = field_rel(x_out.to(F64) - x_in.to(F64), proj_x.view_as(x_ref), N)
    if reg_out is not None and R:
        allow_r = tol * fm + 2.0 ** -24 * reg_ref.abs()
        if code == "tf32":
            allow_r = allow_r + 2 * TF32_U * pa[:, :, :R]
        r["reg"] = ratio(reg_out.view(N, nwin, R, C), reg_ref, allow_r)
    note(**r)
    bad = {k: v for k, v in r.items() if not k.endswith("_rel") and not v <= 1.0}
    assert not bad, r


@pytest.mark.parametrize("code", ["fp32", "x3"])
def test_attn_out_dropout(code):
    """nn.Dropout after to_out, before the residual (maxvit.py:151, 310) at T = 26: the kernel's out-mask [window][token][C],
    exported through vg_dropout_mask_debug, fed to the float64 reference; register rows are dropped too"""
    N, Hl, Wl, C, inner, T = 4, 14, 21, 512, 2048, 26
    nwin = (Hl // WIN) * (Wl // WIN)
    drop = (777, 5, T)
    attn, W = rnd(N * nwin * S_TOK, inner, seed=101), rnd(C, inner, seed=102, scale=1 / math.sqrt(inner))
    x_in, reg = rnd(N, Hl, Wl, C, seed=103), rnd(R_REG, C, seed=104)
    x_out, reg_out = _run_attn_out(code, attn, W, x_in, reg, N, Hl, Wl, WIN, R_REG, False, drop=drop)
    om = OT().dropout_masks(drop, N * nwin, 1, C)[1][:, :S_TOK].to(F64) * (256.0 / (256 - T))
    x_ref, reg_ref, proj = _out_ref(attn, W, x_in, reg, N, Hl, Wl, C, WIN, R_REG, False, out_mask=om)
    tol = x3_tol(inner) if code == "x3" else FP32_TOL
    fm = field_max(proj, N).view(N, 1, 1, 1)
    r = dict(x=ratio(x_out, x_ref, tol * fm + 2.0 ** -24 * x_ref.abs()),
             reg=ratio(reg_out.view(N, nwin, R_REG, C), reg_ref, tol * fm + 2.0 ** -24 * reg_ref.abs()),
             kept=om.ne(0).double().mean().item())
    note(**r)
    assert r["x"] <= 1.0 and r["reg"] <= 1.0, r


# =========================================================================================== MBConv at wide widths
MB_FIELDS, MB_HW = 48, 42 * 35


@pytest.mark.parametrize("operands", ["int", "gauss"])
@pytest.mark.parametrize("C,hid", [(256, 1024), (384, 1536), (512, 2048)])
def test_mbconv_expand_x3(C, hid, operands):
    """the MBConv 1x1 expand of precision 'fp32_x3' (the MaxViT side of 'tf32_conv') at 48 x 1,470 rows: 3xTF32, folded BN
    scale / shift, GELU.  Integer operands (integer scale / shift, no GELU: every value exact): bit-equal.  Gaussian, with
    GELU: within 2 x the 3xTF32 rule of the field's largest output (the epilogue rule of test_gemm_3xtf32_is_fp32_accurate)"""
    o = O()
    M = MB_FIELDS * MB_HW
    if operands == "int":
        A, W = ints(M, C, seed=111), ints(hid, C, seed=112)
        s, t = ints(hid, seed=113, lo=1, hi=2), ints(hid, seed=114, lo=-8, hi=8)
        out = nan_like((M, hid))
        o.gemm(A, W, scale=s, shift=t, act=0, x3=True, out=out)
        torch.cuda.synchronize()
        assert torch.equal(out.to(F64), (A.to(F64) @ W.to(F64).t()) * s.to(F64) + t.to(F64))
        return
    A, W = rnd(M, C, seed=115), rnd(hid, C, seed=116, scale=1 / math.sqrt(C))
    s = 0.5 + torch.rand(hid, device=DEV, generator=torch.Generator(device=DEV).manual_seed(117))
    t = rnd(hid, seed=118, scale=0.5)
    out = nan_like((M, hid))
    o.gemm(A, W, scale=s, shift=t, act=1, x3=True, out=out)
    torch.cuda.synchronize()
    ref = F.gelu((A.to(F64) @ W.to(F64).t()) * s.to(F64) + t.to(F64)).view(MB_FIELDS, MB_HW, hid)
    got = out.view(MB_FIELDS, MB_HW, hid)
    r = dict(ratio=ratio(got, ref, 2 * x3_tol(C) * field_max(ref, MB_FIELDS)), rel=field_rel(got, ref, MB_FIELDS))
    note(**r)
    assert r["ratio"] <= 1.0, r


# (N, H, W, hidden, Cout, residual): the projection of 256 / 384 / 512-channel layers at the chunk; the widening first layer of a
# 256 -> 512 stage (hidden 4 x 512, no residual); 2 x 259x259 at 128 channels (67,081 rows per field)
PROJ_CASES = {"c256": (48, 42, 35, 1024, 256, True), "c384": (48, 42, 35, 1536, 384, True), "c512": (48, 42, 35, 2048, 512, True),
              "widen_256_to_512": (48, 42, 35, 2048, 512, False), "c128_n2_259x259": (2, 259, 259, 512, 128, True)}


@pytest.mark.parametrize("operands", ["int", "gauss"])
@pytest.mark.parametrize("case", list(PROJ_CASES))
def test_se_fold_and_field_projection_x3(case, operands):
    """maxvit.py:302-304 in fp32_x3: vg_se_fold_weights in fp32 (per-field weights W * gate, bit-exact), then the per-field
    3xTF32 projection -- rows_per_batch = H*W (1,470: not a multiple of the 256-row tile), b_rows_per_batch = Cout, K = 3 x
    hidden -- with BN scale / shift and the fp32 residual.  Distinct gates per field, so a field given another field's weights
    shows.  Integer operands (integer gates, scale and shift): bit-equal; Gaussian: per field, 2 x the 3xTF32 rule"""
    o = O()
    N, H, W_, hid, Cout, residual = PROJ_CASES[case]
    HW = H * W_
    if operands == "int":
        h2, Wp = ints(N * HW, hid, seed=121), ints(Cout, hid, seed=122)
        gate = ints(N, hid, seed=123, lo=1, hi=3)
        s, t = ints(Cout, seed=124, lo=1, hi=2), ints(Cout, seed=125, lo=-8, hi=8)
        res = ints(N * HW, Cout, seed=126) if residual else None
    else:
        h2, Wp = rnd(N * HW, hid, seed=127), rnd(Cout, hid, seed=128, scale=1 / math.sqrt(hid))
        gate = torch.rand(N, hid, device=DEV, generator=torch.Generator(device=DEV).manual_seed(129))
        s = 0.5 + torch.rand(Cout, device=DEV, generator=torch.Generator(device=DEV).manual_seed(130))
        t = rnd(Cout, seed=131, scale=0.1)
        res = rnd(N * HW, Cout, seed=132) if residual else None
    wn = o.se_fold_weights(Wp, gate, dtype=F32)
    assert torch.equal(wn, (Wp[None] * gate[:, None, :]).reshape(N * Cout, hid))
    y = nan_like((N * HW, Cout))
    o.gemm(h2, wn, rows_per_batch=HW, b_rows_per_batch=Cout, scale=s, shift=t, res=res, out=y, out_f32=True, x3=True)
    torch.cuda.synchronize()
    ref = torch.einsum("nrk,nok->nro", h2.view(N, HW, hid).to(F64), wn.view(N, Cout, hid).to(F64)) * s.to(F64) + t.to(F64)
    if res is not None:
        ref = ref + res.view(N, HW, Cout).to(F64)
    got = y.view(N, HW, Cout)
    if operands == "int":
        assert torch.equal(got.to(F64), ref), "integer per-field projection not exact"
        return
    r = dict(ratio=ratio(got, ref, 2 * x3_tol(hid) * field_max(ref, N)), rel=field_rel(got, ref, N))
    note(**r)
    assert r["ratio"] <= 1.0, r


# =========================================================================================== one layer at the chunk
# per field, of the field's largest output: fp32 the module bound of the MaxViT tests (measured 6.2e-6); fp32_x3 4x the value
# measured on an NVIDIA B200 at 1000 W, 1.13e-4
LAYER_BOUND = {"fp32": 1e-4, "fp32_x3": 4.5e-4}


@pytest.mark.parametrize("precision", ["fp32", "fp32_x3"])
def test_maxvit_layer_chunk(precision):
    """MaxViT(dim=512, heads=32, dim_head=64, depth=1).forward_cl on the 48-field chunk against mo.maxvit_forward in float64
    on the device, per field: the host glue the per-kernel tests bypass -- split-weight caching, the conditioning MLP and
    squeeze-excite routing at these widths, the register mean between block and grid attention"""
    from vit_grid_model_b200 import MaxViT
    dim, heads, dh = CH_C, CH_HEADS, CH_DH
    sd = synth.make_state_dict(synth.maxvit_multistage_spec(dim, 1, 2, heads, dh, WIN, 4, 0.25, R_REG), seed=141)
    m = MaxViT(dim=dim, depth=1, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=WIN, num_register_tokens=R_REG)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval().set_precision(precision)
    assert not m.fused_attn_applies(dim)
    gen = torch.Generator().manual_seed(142)
    x = torch.randn(CH_N, dim, CH_H, CH_W, generator=gen).to(DEV)
    cond = torch.randn(CH_N, 2, generator=gen).to(DEV)
    with torch.no_grad():
        y = m.forward_cl(x.permute(0, 2, 3, 1).contiguous(), cond)
        y = m.forward_cl(x.permute(0, 2, 3, 1).contiguous(), cond)      # the second call runs on the cached packed weights
    torch.cuda.synchronize()
    sd64 = {k: (v.to(DEV, F64) if v.is_floating_point() else v.to(DEV)) for k, v in sd.items()}
    with torch.no_grad():
        ref = mo.maxvit_forward(x.to(F64), cond.to(F64), sd64, depth=1, heads=heads, window=WIN, num_reg=R_REG)
    got = y.permute(0, 3, 1, 2)
    assert not torch.isnan(got).any()
    r = dict(rel=field_rel(got, ref, CH_N))
    note(**r)
    assert r["rel"] <= LAYER_BOUND[precision], r
