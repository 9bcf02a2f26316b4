"""Per-kernel parity of the tensor-core kernels of the mixed-precision training step (GPU) against float64 PyTorch, at the
size the step runs them: 192 fields of 84x70 (16 samples x 12 lead times; MaxViT at 42x35: 305,280 attention token rows,
282,240 MBConv rows), the 518x518 domain of BASELINE configs[3], and the edges where the kernels change path (fewer rows
than one tile, the last frame width of the halo conv kernel WP = 78 and the first of the generic tcgen05 path WP = 79,
reduction slices that end one row into a K step, column groups that straddle the taps of the 640-channel stem, dW tiles
that are half full).

Conventions of this file:
  * every contraction runs twice.  The exact run uses small-integer operands: every product and every partial sum is an
    integer below 2^24 (asserted per case), so fp32 accumulation is exact in any order and any split, and the fp32 result
    must be bit-equal to the float64 reference (a 16-bit result where it fits: |sum| <= 256 for bf16).  That checks every
    index: slices, taps, column groups, partial tiles, TMA out-of-bounds fill, the beta accumulate, the residual add.  The
    numeric run uses seeded Gaussian operands rounded as the device sees them, and checks the rounding:
      - fp32 outputs within FP32_TOL of the largest entry of their field (or row block; for weight gradients, of their
        128-row n-tile: at 10^6 rows the worst-case sum|a||b| bound is far above the result);
      - 16-bit outputs within half an ulp of the float64 result plus the fp32 arithmetic's own error (rounded to nearest);
      - tf32 on plain fp32 operands: within 2 * 2^-10 * sum|a||b| more, and within the fp32 bound against the operands
        truncated to tf32 (tcgen05 kind::tf32 truncates)
  * every output the kernel must write completely starts as NaN (integer outputs: all bits set); accumulated outputs start
    from an integer prefill
  * references are built once per case (lru_cache of one entry: the next case frees the previous one) on the GPU
"""
import math
import os
from functools import lru_cache

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64 = torch.float64
BF16, F32 = torch.bfloat16, torch.float32
FP32_TOL = 2e-5            # fp32 outputs: max |err| / max |ref| per field
TF32_U = 2.0 ** -10
EXACT_LIMIT = 2 ** 24      # integers up to here are exact in fp32
EPS = 1e-5
# rstd, element-wise relative (exact / numeric run): measured 4.3e-7 / 7.0e-6 on a B200
RSTD_TOL = {True: 1.5e-6, False: 2.5e-5}


def O():
    from vit_grid_model_b200 import ops
    return ops


def OT():
    from vit_grid_model_b200 import ops_train
    return ops_train


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


def rint(*shape, seed=0, lo=-2, hi=2):
    """integers in [lo, hi] as fp32"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(lo, hi + 1, shape, generator=g, device=DEV).float()


def tf32_exact(t):
    """t with the 13 low mantissa bits cleared: a tf32 operand the tensor core takes exactly"""
    return (t.contiguous().view(torch.int32) & -8192).view(F32)


def nan_like(shape, dtype=F32):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def prefill(shape, seed):
    """the integer dW an accumulating (beta = 1) weight gradient starts from"""
    return rint(*shape, seed=seed, lo=-4, hi=4)


def pg_frame(buf, N, HP, WP):
    """(N,HP,WP,C) view of the frame pixels of a PG buffer (no copy)"""
    C = buf.shape[-1]
    return buf.view(N * (HP + 1) + 1, WP + 1, C)[:N * (HP + 1)].view(N, HP + 1, WP + 1, C)[:, 1:, 1:]


def pg_pads(buf, N, HP, WP):
    """every pad entry of a PG buffer (column 0 of every row, and the separator rows)"""
    C = buf.shape[-1]
    v = buf.view(N * (HP + 1) + 1, WP + 1, C)
    return torch.cat([v[:, 0].reshape(-1), v[::HP + 1, 1:].reshape(-1)])


def pg_nan(N, HP, WP, C, dtype=F32):
    return nan_like((O().pg_pixels(N, HP, WP), C), dtype)


def pg_from_nchw(x, dtype):
    return O().pg_from_nchw(x, dtype)


def assert_pads_zero(buf, N, HP, WP, what):
    p = pg_pads(buf, N, HP, WP).float()
    assert torch.equal(p, torch.zeros_like(p)), f"a pad of {what} is not 0"


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
    the rounding.  The ulp is the larger of got's and the rounded reference's."""
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


def assert_exact(got, ref, what):
    got = got.to(DEV, F64)
    bad = (got != ref.to(DEV, F64)) | torch.isnan(got)
    if bad.any():
        i = bad.reshape(-1).nonzero()[0].item()
        raise AssertionError(f"{what}: {bad.sum().item()} entries differ from the exact result; first at flat index {i}: "
                             f"{got.reshape(-1)[i].item()} != {ref.reshape(-1)[i].item()}")


def check_ratios(r):
    note(**r)
    for k, v in r.items():
        if not k.endswith("_rel"):
            assert v <= 1.0, (k, r)


# (N, HP, WP) of the training step's conv blocks and their path edges
GEOMS = {
    "n1_14x14": (1, 14, 14),          # 15*15 + 15 = 240 PG rows: less than one tile
    "n192_84x70": (192, 84, 70),      # the bench.py train line: 1,158,791 rows, about 30 tiles per CTA
    "wp78": (3, 28, 78),              # the widest frame of the halo kernel (256 + 2 (WP + 2) = 416 rows)
    "wp79": (3, 28, 79),              # the first of the generic tcgen05 GEMM (EPI_CONV_LN_TRAIN / EPI_STORE)
    "n2_518x518": (2, 518, 518),      # BASELINE configs[3]'s domain
}


# =========================================================================================== A. conv block forward with saves
@lru_cache(maxsize=1)
def _fwd_case(geom, exact, C=128):
    """operands and float64 reference of one conv block: -> (x, w, b, g, be, film, res, pre64 (N,HP,WP,C), xhat64, rstd64).
    Rows 0-3 of every frame of x are zero; in the numeric run the conv bias is O(1e-3), so at the frame pixels of rows 0-2
    the conv output is the bias alone, whose variance over the channels (about 1e-6) is below eps: the LayerNorm takes its
    var.clamp(eps) branch there."""
    N, HP, WP = GEOMS[geom]
    if exact:
        x, w, b = rint(N, C, HP, WP, seed=1), rint(C, C, 3, 3, seed=2), rint(C, seed=3, lo=-3, hi=3)
        assert 9 * C * 2 * 2 + 3 < EXACT_LIMIT
    else:
        x = rnd(N, C, HP, WP, seed=1).to(BF16).float()
        w = rnd(C, C, 3, 3, seed=2, scale=1 / math.sqrt(9 * C)).to(BF16).float()
        b = rnd(C, seed=3, scale=1e-3)
    x[:, :, :4] = 0
    g = 1.0 + 0.5 * torch.rand(C, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    be = rnd(C, seed=5, scale=0.1)
    film = rnd(N, 2 * C, seed=6, scale=0.3)
    res = rnd(N, C, HP, WP, seed=7)
    h = F.conv2d(x.to(F64), w.to(F64), b.to(F64), padding=1).permute(0, 2, 3, 1)         # (N,HP,WP,C)
    mean = h.mean(-1, keepdim=True)
    rstd = h.var(-1, unbiased=False, keepdim=True).clamp(min=EPS).rsqrt()
    xhat = (h - mean) * rstd
    del h, mean
    return x, w, b, g, be, film, res, xhat, rstd[..., 0]


def _mask_bits(mask):
    """(Q,4) int32 ReLU mask -> (Q,128) bool (bit c % 32 of word c // 32)"""
    c = torch.arange(128, device=DEV)
    return ((mask[:, c // 32] >> (c % 32)) & 1).bool()


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "numeric"])
@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("launch", ["film", "res32_copy"])
def test_conv3x3_ln_train_fwd(launch, geom, exact):
    """vg_conv3x3_ln_train_fwd in bf16 (conv_halo_kernel<1> up to WP = 78, gemm_tc_kernel<EPI_CONV_LN_TRAIN> above) in the
    two calls of train._resblock_train_fwd: block1 with FiLM and no residual, block2 with the fp32 residual and the fp32
    copy (TMA residual loads and TMA copy stores in the halo kernel).  out / copy as the inference kernels are checked;
    the saves: xhat = the float64 xhat rounded to bf16, rstd within the fp32 bound, the ReLU mask = (pre-ReLU > 0) of the
    float64 reference wherever the pre-ReLU value is farther from 0 than its error bound, and exactly consistent with the
    kernel's own output; xhat, rstd and the mask words are 0 at pads.  The exact run (integer x, W, bias) makes the
    conv sum exact: xhat and rstd are then held to the fp32 LayerNorm arithmetic alone."""
    N, HP, WP = GEOMS[geom]
    C = 128
    o = O()
    x, w, b, g, be, film, res, xhat64, rstd64 = _fwd_case(geom, exact)
    use_film = launch == "film"
    G = g.to(F64)
    pre = xhat64 * G + be.to(F64)
    if use_film:
        f = film.to(F64)[:, None, None, :]
        pre = pre * (f[..., :C] + 1) + f[..., C:]
        G = G * (f[..., :C] + 1)
    y = pre.clamp_min(0)
    resq = None
    if not use_film:
        resq = res.permute(0, 2, 3, 1)
        y = y + resq.to(F64)
    # element-wise allowances: the conv sum's fp32 accumulation (numeric run only) and the LayerNorm's fp32 arithmetic
    acc_tol = 0.0 if exact else FP32_TOL
    ln_tol = 2e-6
    xp = pg_from_nchw(x, BF16)
    wt = w.permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous().to(BF16)
    rp = None if resq is None else pg_from_nchw(res, F32)
    Q = xp.shape[0]
    out = pg_nan(N, HP, WP, C, BF16)
    copy = None if use_film else pg_nan(N, HP, WP, C)
    xhat = nan_like((Q, C), BF16)
    rstd = nan_like((Q,))
    mask = torch.full((Q, 4), -1, dtype=torch.int32, device=DEV)
    call("vg_conv3x3_ln_train_fwd", o.DT_CODE[BF16], xp.data_ptr(), C, wt.data_ptr(), b.data_ptr(), g.data_ptr(),
         be.data_ptr(), EPS, film.data_ptr() if use_film else None, None if rp is None else rp.data_ptr(), int(rp is not None),
         out.data_ptr(), None if copy is None else copy.data_ptr(), xhat.data_ptr(), rstd.data_ptr(), mask.data_ptr(),
         N, HP, WP, None, 0)
    torch.cuda.synchronize()
    r = {}
    allow_y = per_field_abs_allow(y, acc_tol + ln_tol)
    r["out_rn"] = rn16(pg_frame(out, N, HP, WP), y, allow_y)
    assert_pads_zero(out, N, HP, WP, "out")
    if copy is not None:
        r["copy"], r["copy_rel"] = f32_ratio(pg_frame(copy, N, HP, WP), y, tol=acc_tol + ln_tol)
        assert_pads_zero(copy, N, HP, WP, "the fp32 copy")
        assert torch.equal(out.float(), copy.to(BF16).float()), "output != (rounded) fp32 copy"
    r["xhat_rn"] = rn16(pg_frame(xhat, N, HP, WP), xhat64, per_field_abs_allow(xhat64, acc_tol + ln_tol))
    assert_pads_zero(xhat, N, HP, WP, "xhat")
    rg = pg_frame(rstd.view(-1, 1), N, HP, WP)[..., 0].to(F64)
    assert not torch.isnan(rg).any()
    # rstd, element-wise relative: in the exact run the variance carries the fp32 LayerNorm arithmetic alone
    r["rstd"] = ((rg - rstd64).abs() / (rstd64 * RSTD_TOL[exact])).max().item()
    assert_pads_zero(rstd.view(-1, 1), N, HP, WP, "rstd")
    assert_pads_zero(mask, N, HP, WP, "the ReLU mask")
    bits = _mask_bits(mask)
    fb = pg_frame(bits, N, HP, WP)
    # the mask against the float64 pre-ReLU value, where its sign is certain: the LayerNorm output's error is bounded by
    # allow_y (the same allowance out is held to)
    sure = pre.abs() > 2 * allow_y
    assert sure.float().mean().item() > 0.95
    wrong = (fb != (pre > 0)) & sure
    assert not wrong.any(), f"{wrong.sum().item()} ReLU mask bits disagree with the float64 sign of the pre-ReLU value"
    # self-consistency, exact: the bit is what the kernel's own ReLU saw
    if use_film:
        assert torch.equal(bits, out.float() > 0), "mask bit != (out > 0)"
    else:
        d = copy - rp
        ulp = torch.ldexp(torch.ones_like(rp), torch.frexp(rp)[1] - 24)
        clear = d.abs() > ulp
        assert torch.equal(bits[clear], (d > 0)[clear]), "mask bit != (copy - res > 0)"
    check_ratios(r)


# =========================================================================================== B. conv data gradient
@lru_cache(maxsize=1)
def _dgrad_case(geom, exact, C=128):
    """dconv (NCHW, what conv_ln_bwd writes: zeros at pads once packed), w (non-symmetric), the residual dOut and the float64
    input gradient of F.conv2d (NHWC) without the residual"""
    N, HP, WP = GEOMS[geom]
    if exact:
        dc, w, res = rint(N, C, HP, WP, seed=11), rint(C, C, 3, 3, seed=12), rint(N, C, HP, WP, seed=13, lo=-8, hi=8)
        assert 9 * C * 2 * 2 + 8 < EXACT_LIMIT
    else:
        dc = rnd(N, C, HP, WP, seed=11).to(BF16).float()
        w = rnd(C, C, 3, 3, seed=12, scale=1 / math.sqrt(9 * C)).to(BF16).float()
        res = rnd(N, C, HP, WP, seed=13)
    assert not torch.equal(w, w.flip(2, 3))
    dx = F.conv_transpose2d(dc.to(F64), w.to(F64), padding=1).permute(0, 2, 3, 1)
    return dc, w, res, dx


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "numeric"])
@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("with_res", [False, True], ids=["dt1", "dx_plus_dOut"])
def test_conv3x3_dgrad(with_res, geom, exact):
    """the conv data gradient of train._resblock_train_bwd: ops.gemm(dconv, _pack_dgrad3x3(w), 9 negated tap shifts, fp32
    out) without the residual (dt1) and with the fp32 residual dOut (dx); conv_halo_kernel<2> (flipped taps) up to WP = 78,
    the generic gemm_tc_kernel<EPI_STORE> at WP = 79 and 518.  Frame pixels against the float64 input gradient of F.conv2d
    (+ dOut): bit-exact in the exact run, within the fp32 bound otherwise.  Every row must be written (the output starts
    as NaN); what the pads hold is not part of the contract, since every reader of a gradient ignores pads (DESIGN.md §3)."""
    from vit_grid_model_b200.train import _pack_dgrad3x3
    N, HP, WP = GEOMS[geom]
    C = 128
    o = O()
    dc, w, res, dx64 = _dgrad_case(geom, exact)
    ref = dx64
    rp = None
    if with_res:
        rp = pg_from_nchw(res, F32)
        ref = dx64 + res.permute(0, 2, 3, 1).to(F64)
    dcp = pg_from_nchw(dc, BF16)
    out = pg_nan(N, HP, WP, C)
    nshifts = tuple(-s for s in o.conv_tap_shifts(WP))
    o.gemm(dcp, _pack_dgrad3x3(w, BF16), ntaps=9, tap_shift=nshifts, res=rp, out=out, out_f32=True)
    torch.cuda.synchronize()
    assert not torch.isnan(out).any(), "a row of the data gradient was not written"
    got = pg_frame(out, N, HP, WP)
    if exact:
        assert_exact(got, ref, "dgrad")
        note(exact=1)
    else:
        ratio, rel = f32_ratio(got, ref)
        check_ratios(dict(ratio=ratio, ratio_rel=rel))


# =========================================================================================== C. weight gradient
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def wgrad_plan(M, Ntot, Ca, ntaps, kt=64):
    """host copy of wgrad_plan (csrc/vg_wgrad.cu) for the tensor-core paths: -> (ksplit, rows_per_split)"""
    n_tiles = (Ntot + 127) // 128
    col_tiles = ntaps * (Ca // 128)
    acc = 3 if (ntaps == 9 and Ca == 128) else min(col_tiles, 4)
    units = n_tiles * ((col_tiles + acc - 1) // acc)
    want = max(1, min(_sms() // units, (M + 8 * kt - 1) // (8 * kt), 64))
    rps = (M + want - 1) // want
    rps = (rps + kt - 1) // kt * kt
    return (M + rps - 1) // rps, rps


def _edge_rows(last):
    """M for Ntot = Ca = 128, one tap, bf16: 64 reduction slices of 640 rows, the last one `last` rows long"""
    M = 63 * 640 + last
    assert wgrad_plan(M, 128, 128, 1) == (64, 640), wgrad_plan(M, 128, 128, 1)
    return M


# name -> (dY rows layout, Ntot, Ca, ntaps, tf32).  "pg": PG buffers of N fields (the conv / stem weight gradients, dY zero
# at pads); an int: that many plain rows.
WGRAD_CASES = {
    "conv3x3_n192_84x70": (("pg", 192, 84, 70), 128, 128, 9, False),
    "conv3x3_n12_518x518": (("pg", 12, 518, 518), 128, 128, 9, False),     # M = 3,232,851: the largest reduction
    "stem3x3_ca640_b16": (("pg", 16, 84, 70), 128, 640, 9, False),         # 45 column tiles in groups of 4 (straddling taps)
    "stem3x3_ca640_b1": (("pg", 1, 84, 70), 128, 640, 9, False),
    "res_conv_ca640_b16": (("pg", 16, 84, 70), 128, 640, 1, False),        # 5 column tiles: 4 + 1
    "to_out_305280": (305280, 128, 1024, 1, False),              # attention rows of 192 fields of 42x35
    "to_qkv_305280": (305280, 3072, 128, 1, False),
    "mbconv_proj_282240_tf32": (282240, 128, 512, 1, True),
    "mbconv_expand_282240_tf32": (282240, 512, 128, 1, True),
    "convT_282240_tf32": (282240, 512, 128, 1, True),
    "ntot64": (5000, 64, 128, 1, False),                                   # the only n-tile is half full
    "ntot192": (5000, 192, 256, 1, False),                                 # the last n-tile is half full
    "m37": (37, 128, 128, 1, False),                                       # one partial K step
    "last_slice_1_row": ("edge1", 128, 128, 1, False),
    "last_slice_kt_minus_1_rows": ("edge63", 128, 128, 1, False),
}


@lru_cache(maxsize=1)
def _wgrad_case(name, exact):
    """-> (dY, A (device dtype), tap shifts, float64 reference [Ntot][ntaps*Ca], and for tf32 on plain operands the
    reference of the truncated operands and sum |a||b|)"""
    layout, Ntot, Ca, ntaps, tf32 = WGRAD_CASES[name]
    if isinstance(layout, tuple):
        _, N, HP, WP = layout
        M = O().pg_pixels(N, HP, WP)
        shifts = O().conv_tap_shifts(WP) if ntaps == 9 else (0,)
    else:
        M = _edge_rows(int(layout[4:])) if isinstance(layout, str) else layout
        shifts = (0,)
    dt = F32 if tf32 else BF16
    if exact:
        dY, A = rint(M, Ntot, seed=21), rint(M, Ca, seed=22)
        assert 2 * 2 * M < EXACT_LIMIT, M
    else:
        dY, A = rnd(M, Ntot, seed=21), rnd(M, Ca, seed=22)
        if not tf32:
            dY, A = dY.to(BF16).float(), A.to(BF16).float()
    if isinstance(layout, tuple):                       # PG: dY is zero at pads, as conv_ln_bwd / lead_sum write it
        _, N, HP, WP = layout
        keep = pg_from_nchw(torch.ones(N, 1, HP, WP, device=DEV), F32)
        dY *= keep
        A *= keep                                       # the activations are zero at pads too
        del keep

    def ref_of(dY, A):
        d64 = dY.to(F64)
        cols = []
        for s in shifts:                                # A[m + s], zero outside [0, M) (TMA out-of-bounds fill)
            a = torch.zeros_like(A, dtype=F64)
            lo, hi = max(0, -s), min(M, M - s)
            a[lo:hi] = A[lo + s:hi + s].to(F64)
            cols.append(d64.t() @ a)
            del a
        return torch.cat(cols, 1)
    ref = ref_of(dY, A)
    extra = None
    if tf32 and not exact:
        extra = (ref_of(tf32_exact(dY), tf32_exact(A)), ref_of(dY.abs(), A.abs()))
    return dY.to(dt), A.to(dt), shifts, ref, extra


def _ntile_ratio(got, ref, tol):
    """max over 128-row n-tiles of dW of max |err| / (tol * max |ref| of the tile)"""
    Ntot = ref.shape[0]
    nt = (Ntot + 127) // 128
    err = (got.to(F64) - ref).abs()
    worst, rel = 0.0, 0.0
    for t in range(nt):
        e, m = err[t * 128:(t + 1) * 128].max().item(), ref[t * 128:(t + 1) * 128].abs().max().item()
        worst, rel = max(worst, e / (tol * m)), max(rel, e / m)
    return worst, rel


# numeric run: max |err| / max |ref| per 128-row n-tile, bound (measured on a B200).  The error grows with the rows one CTA
# accumulates in TMEM (the tensor core's fp32 accumulation truncates): 3,232,851 rows in 21 slices (518x518) and 305,280 rows
# in 6 slices (to_qkv: 24 n-tiles leave 6 slices for 148 SMs) measure the most.  tf32: against the operands truncated to tf32.
WGRAD_TOL = {
    "conv3x3_n192_84x70": 1e-4,           # 2.5e-5
    "conv3x3_n12_518x518": 2e-4,          # 7.3e-5
    "stem3x3_ca640_b16": 3e-5,            # 9.1e-6
    "stem3x3_ca640_b1": 2e-6,             # 5.6e-7
    "res_conv_ca640_b16": 5e-6,           # 1.6e-6
    "to_out_305280": 2e-5,                # 5.3e-6
    "to_qkv_305280": 2e-4,                # 7.7e-5
    "mbconv_proj_282240_tf32": 4e-5,      # 1.0e-5
    "mbconv_expand_282240_tf32": 5e-5,    # 1.9e-5
    "convT_282240_tf32": 5e-5,            # 1.9e-5
    "ntot64": 2e-6,                       # 6.4e-7
    "ntot192": 2e-6,                      # 5.4e-7
    "m37": 4e-7,                          # 1.1e-7
    "last_slice_1_row": 2e-6,             # 7.5e-7
    "last_slice_kt_minus_1_rows": 2e-6,   # 7.6e-7
}


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "numeric"])
@pytest.mark.parametrize("name", list(WGRAD_CASES))
def test_wgrad(name, exact):
    """ops_train.wgrad (wgrad_tc_kernel<0> bf16, <1> tf32, + wgrad_reduce_kernel) at every shape the training step launches,
    at its real row count, and at the edges of the entry point: with beta = 0 into a NaN-filled dW, and with beta = 1 onto
    an integer prefill"""
    layout, Ntot, Ca, ntaps, tf32 = WGRAD_CASES[name]
    dY, A, shifts, ref, extra = _wgrad_case(name, exact)
    M = dY.shape[0]
    if isinstance(layout, str):
        ks, rps = wgrad_plan(M, Ntot, Ca, ntaps)
        assert M - (ks - 1) * rps == int(layout[4:])
    dW = nan_like((Ntot, ntaps * Ca))
    OT().wgrad(dY, A, dW, ntaps=ntaps, tap_shift=shifts, beta=0.0, tf32=tf32)
    P = prefill((Ntot, ntaps * Ca), seed=23)
    dW1 = P.clone()
    OT().wgrad(dY, A, dW1, ntaps=ntaps, tap_shift=shifts, beta=1.0, tf32=tf32)
    torch.cuda.synchronize()
    assert not torch.isnan(dW).any(), "dW not written everywhere"
    if exact:
        assert_exact(dW, ref, "dW (beta = 0)")
        assert_exact(dW1, ref + P.to(F64), "dW (beta = 1)")
        note(exact=1)
        return
    tol = WGRAD_TOL[name]
    r = {}
    if tf32:
        reft, sabs = extra
        r["trunc"], r["trunc_rel"] = _ntile_ratio(dW, reft, tol)
        r["plain"] = ((dW.to(F64) - ref).abs() / (tol * ref.abs().amax() + 2 * TF32_U * sabs)).max().item()
        r["trunc_beta1"], _ = _ntile_ratio(dW1.to(F64) - P.to(F64), reft, tol)
    else:
        r["ntile"], r["ntile_rel"] = _ntile_ratio(dW, ref, tol)
        r["ntile_beta1"], _ = _ntile_ratio(dW1.to(F64) - P.to(F64), ref, tol)
    check_ratios(r)


@pytest.mark.parametrize("beta", [0.0, 1.0, 0.5])
def test_wgrad_empty_reduction(beta):
    """M = 0: the sum over no rows is zero, so dW = beta * dW as for any M (a NaN-filled dW with beta = 0 becomes 0)"""
    Ntot, Ca = 128, 256
    dY, A = torch.empty(0, Ntot, dtype=BF16, device=DEV), torch.empty(0, Ca, dtype=BF16, device=DEV)
    P = prefill((Ntot, Ca), seed=24)
    dW = nan_like((Ntot, Ca)) if beta == 0.0 else P.clone()
    OT().wgrad(dY, A, dW, beta=beta)
    torch.cuda.synchronize()
    assert torch.equal(dW, torch.zeros_like(P) if beta == 0.0 else beta * P)


# =========================================================================================== F. GEMMs of the backward chains
# name -> (M, K, N, operand dtype (None: tf32 on fp32), output dtype, residual).  MaxViT at 42x35: 192 fields x 30 windows x
# 53 tokens = 305,280 attention rows (bf16 chain, train._attention_train_bwd); 192 x 1,470 = 282,240 MBConv / ConvTranspose
# rows (tf32, train.maxvit_train_backward / metnet3_train_backward).
GEMM_CASES = {
    "qkv_remat_bf16_n3072": (305280, 128, 3072, BF16, BF16, False),
    "datt_bf16_n1024": (305280, 128, 1024, BF16, BF16, False),
    "dtok_k3072_fp32": (305280, 3072, 128, BF16, F32, False),
    "mbconv_dh4_tf32_n512": (282240, 128, 512, None, F32, False),
    "mbconv_dx_tf32_k512_res": (282240, 512, 128, None, F32, True),
    "convT_dlow_tf32_k512": (282240, 512, 128, None, F32, False),
}
ROWS_PER_BLOCK = {305280: 1590, 282240: 1470}      # one field's rows


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "numeric"])
@pytest.mark.parametrize("name", list(GEMM_CASES))
def test_backward_gemm(name, exact):
    """ops.gemm as the backward chains call it, at the step's row count: the attention chain's bf16 GEMMs (QKV
    re-materialisation and datt with bf16 out, dtok over K = 3,072 with fp32 out), the MBConv 1x1 data gradients in tf32
    (the expand's with the fp32 residual) and the ConvTranspose data gradient (K = 512, tf32).  Row blocks of one field."""
    M, K, N, dt, odt, with_res = GEMM_CASES[name]
    tf32 = dt is None
    if exact:
        # bf16 out: operands in {-1, 0, 1} keep |sum| <= 128, where bf16 is exact
        lim = 1 if odt == BF16 else 2
        A, W = rint(M, K, seed=31, lo=-lim, hi=lim), rint(N, K, seed=32, lo=-lim, hi=lim)
        res = rint(M, N, seed=33, lo=-8, hi=8) if with_res else None
        assert K * lim * lim + 8 < EXACT_LIMIT and (odt != BF16 or K * lim * lim <= 256)
    else:
        A, W = rnd(M, K, seed=31), rnd(N, K, seed=32, scale=1 / math.sqrt(K))
        if not tf32:
            A, W = A.to(dt).float(), W.to(dt).float()
        res = rnd(M, N, seed=33) if with_res else None
    ddt = F32 if tf32 else dt
    out = nan_like((M, N), odt)
    O().gemm(A.to(ddt), W.to(ddt), res=res, out=out, out_f32=odt == F32, tf32=tf32)
    torch.cuda.synchronize()
    nb = M // ROWS_PER_BLOCK[M]
    ref = A.to(F64) @ W.to(F64).t()
    if res is not None:
        ref += res.to(F64)
    if exact:
        assert_exact(out, ref, name)
        note(exact=1)
        return
    r = {}
    if odt == BF16:
        r["rn"] = rn16(out.view(nb, -1, N), ref.view(nb, -1, N), per_field_abs_allow(ref.view(nb, -1, N)))
    elif tf32:
        sabs = A.abs().to(F64) @ W.abs().to(F64).t()
        r["plain"], r["plain_rel"] = f32_ratio(out.view(nb, -1, N), ref.view(nb, -1, N), extra=2 * TF32_U * sabs.view(nb, -1, N))
        del sabs
        reft = tf32_exact(A).to(F64) @ tf32_exact(W).to(F64).t()
        if res is not None:
            reft += res.to(F64)
        r["trunc"], r["trunc_rel"] = f32_ratio(out.view(nb, -1, N), reft.view(nb, -1, N))
    else:
        r["ratio"], r["ratio_rel"] = f32_ratio(out.view(nb, -1, N), ref.view(nb, -1, N))
    check_ratios(r)


# =========================================================================================== D. attention core backward, tcgen05
WIN, R_REG, HEADS, DH = 7, 4, 32, 32
S_TOK = R_REG + WIN * WIN
LOG2E = 1.0 / math.log(2.0)
ATTN_BWD_CASES = {           # name -> (fields, Hl, Wl, dropout threshold T)
    "n192_42x35_T0": (192, 42, 35, 0),          # 6,144 (field, head) items on the persistent CTAs, 15 tiles per item
    "n192_42x35_T26": (192, 42, 35, 26),        # the training step's attention dropout 0.1
    "n2_259x259_T26": (2, 259, 259, 26),        # 1,369 windows: the last tile of every item is half empty (configs[3])
    "n1_7x7_T26": (1, 7, 7, 26),                # one window
}
# largest error beyond the half-ulp rounding of the bf16 outputs, relative to the largest entry of its (window, head) block
# (dqkv, att) or of its head (gamma and bias gradients).  Measured on a B200 over the cases below: dq 1.1e-2, dk 1.5e-2,
# dv 7.3e-3, att 1.5e-2; dq_gamma 2.7e-4, dk_gamma 2.3e-4, dbias 3.0e-4.  The block errors are the reference's, not the
# kernel's: it rounds q^ and K" from float64 where the kernel rounds its fp32 rsqrtf products, and at a near-tie one K"
# entry (about 12, bf16 ulp 1/16) moves a logit of these peaked softmaxes by 1e-2.  With one window per field (7x7, 32
# blocks, no tie met) the same comparison measures 6e-5 (dq) and 2e-6 or less (dk, dv, att).
ATTN_BWD_TOL = {"dq": 3e-2, "dk": 3e-2, "dv": 3e-2, "att": 3e-2, "dq_gamma": 1e-3, "dk_gamma": 1e-3, "dbias": 1e-3}


def _rel_pos_index(win, R):
    """(S, S) index into the relative-position bias table (maxvit.py:158-168): the last entry for pairs with a register token"""
    W2 = 2 * win - 1
    t = torch.arange(win * win, device=DEV)
    a, b = t // win, t % win
    idx = torch.full((R + win * win, R + win * win), W2 * W2, dtype=torch.long, device=DEV)
    idx[R:, R:] = (a[:, None] - a[None, :] + win - 1) * W2 + (b[:, None] - b[None, :] + win - 1)
    return idx


def _attn_bwd_ref(qkv, datt, qg, kg, bt, pmask):
    """float64 backward of maxvit.py:189-213 for a run of windows, rounded where vg_attn_bwd_tc.cu rounds: q^ = q / |q| and
    K" = log2e rs^2 gq gk k / |k| to bf16 (S = q^ K" in the exp2 domain), P' = P mask and dS to bf16 in front of the four
    output products; the bias gradient sums the unrounded dS.  qkv [rows][3 inner], datt [rows][inner] (bf16), pmask
    (windows, heads, S, S) with the 1 / (1 - p) scale, or None.  -> dq, dk, dv, att (windows, heads, S, DH), dG (heads, DH)
    = sum over the rows of dK" u_k, dbias (table entries, heads)"""
    nw = qkv.shape[0] // S_TOK
    x = qkv.to(F64).view(nw, S_TOK, 3, HEADS, DH).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    dO = datt.to(F64).view(nw, S_TOK, HEADS, DH).permute(0, 2, 1, 3)
    inv_q = 1.0 / q.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    inv_k = 1.0 / k.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    rs = torch.tensor(float(DH), dtype=F32, device=DEV).sqrt()
    G32 = (rs * rs * qg) * kg                                           # fp32, as the kernel forms it
    G = G32.to(F64).view(HEADS, 1, DH)
    GL = (G32 * torch.tensor(LOG2E, dtype=F32)).to(F64).view(HEADS, 1, DH)
    qh = (q * inv_q).to(BF16).to(F64)
    K2 = (k * inv_k * GL).to(BF16).to(F64)
    idx = _rel_pos_index(WIN, R_REG)
    bias = bt.to(F64)[idx].permute(2, 0, 1)                             # (heads, S, S)
    P = torch.softmax((qh @ K2.transpose(-1, -2)) / LOG2E + bias, dim=-1)
    Mk = 1.0 if pmask is None else pmask
    dPm = (dO @ v.transpose(-1, -2)) * Mk
    dS = P * (dPm - (P * dPm).sum(-1, keepdim=True))
    Pb = (P * Mk).to(BF16).to(F64)
    dSb = dS.to(BF16).to(F64)
    dv = Pb.transpose(-1, -2) @ dO
    att = Pb @ v
    dK2 = dSb.transpose(-1, -2) @ qh
    dQ2 = dSb @ K2
    dq = (dQ2 - qh * (dQ2 * qh).sum(-1, keepdim=True)) * inv_q / LOG2E
    uk = K2 / GL
    dk = (dK2 * G - uk * ((dK2 * K2).sum(-1, keepdim=True) / LOG2E)) * inv_k
    dG = (dK2 * uk).sum((0, 2))
    dbias = torch.zeros(bt.shape, dtype=F64, device=DEV)
    dbias.index_add_(0, idx.reshape(-1), dS.sum(0).permute(1, 2, 0).reshape(S_TOK * S_TOK, HEADS))
    return dq, dk, dv, att, dG, dbias


def _excess(got, ref):
    """(windows, heads, S, DH) -> (windows, heads): largest |got - ref| beyond half a bf16 ulp of the result, relative to the
    largest |ref| of the (window, head) block"""
    r16 = ref.to(BF16).to(F64)
    _, e = torch.frexp(torch.maximum(r16.abs(), got.abs()))
    half_ulp = torch.ldexp(torch.ones_like(ref), e - 9)
    ex = ((got - ref).abs() - half_ulp).clamp_min(0).amax((2, 3))
    return ex / ref.abs().amax((2, 3)).clamp_min(1e-300)


@pytest.mark.parametrize("case", list(ATTN_BWD_CASES))
def test_attn_core_bwd_tcgen05_per_window(case):
    """ops_train.attn_core_bwd in bf16 (attn_core_bwd_tc_kernel, mode 3) against the float64 backward that rounds where the
    kernel rounds, compared per (window, head) for dq / dk / dv / att and per head for the gamma and bias gradients: one bad
    window or item fails on its own.  Named on their own: the first and last window of the first and last field, and the
    last item of every persistent CTA (items are strided by the grid size)."""
    N, Hl, Wl, T = ATTN_BWD_CASES[case]
    nwin = (Hl // WIN) * (Wl // WIN)
    inner = HEADS * DH
    rows = N * nwin * S_TOK
    g = torch.Generator(device=DEV).manual_seed(41)
    qkv = torch.randn(rows, 3 * inner, device=DEV, generator=g).to(BF16)
    datt = torch.randn(rows, inner, device=DEV, generator=g).to(BF16)
    qg = 1 + 0.2 * torch.randn(inner, device=DEV, generator=g)
    kg = 1 + 0.2 * torch.randn(inner, device=DEV, generator=g)
    bt = 0.5 * torch.randn((2 * WIN - 1) ** 2 + 1, HEADS, device=DEV, generator=g)
    drop = (8642, 3, T)
    dqg, dkg, dbt = (torch.zeros_like(t) for t in (qg, kg, bt))
    dqkv, att = OT().attn_core_bwd(qkv, datt, qg, kg, bt, N, Hl, Wl, WIN, R_REG, HEADS, DH, dqg, dkg, dbt, want_att=True,
                                   drop=drop)
    torch.cuda.synchronize()
    assert not torch.isnan(dqkv.float()).any() and not torch.isnan(att.float()).any()
    tab = {k: torch.zeros(N, nwin, HEADS, dtype=F64, device=DEV) for k in ("dq", "dk", "dv", "att")}
    dG = torch.zeros(HEADS, DH, dtype=F64, device=DEV)
    dbias = torch.zeros(bt.shape, dtype=F64, device=DEV)
    pm = OT().dropout_masks(drop, N * nwin, HEADS, 128)[0] if T else None
    chunk = max(1, 16 * 30 // nwin)                                   # fields per reference chunk (about 480 windows)
    for f0 in range(0, N, chunk):
        f1 = min(N, f0 + chunk)
        r0, r1 = f0 * nwin * S_TOK, f1 * nwin * S_TOK
        pmask = None
        if T:
            pmask = pm[f0 * nwin:f1 * nwin, :, :S_TOK, :S_TOK].to(F64) * (256.0 / (256 - T))
        ref = _attn_bwd_ref(qkv[r0:r1], datt[r0:r1], qg, kg, bt, pmask)
        nw = (f1 - f0) * nwin
        got = dqkv[r0:r1].to(F64).view(nw, S_TOK, 3, HEADS, DH).permute(2, 0, 3, 1, 4)
        gatt = att[r0:r1].to(F64).view(nw, S_TOK, HEADS, DH).permute(0, 2, 1, 3)
        for name, gv, rv in (("dq", got[0], ref[0]), ("dk", got[1], ref[1]), ("dv", got[2], ref[2]), ("att", gatt, ref[3])):
            tab[name][f0:f1] = _excess(gv, rv).view(f1 - f0, nwin, HEADS)
        dG += ref[4]
        dbias += ref[5]
        del ref, got, gatt, pmask
    dh_ = float(DH)
    ref_dqg = (dh_ * kg.to(F64).view(HEADS, DH) * dG).reshape(-1)
    ref_dkg = (dh_ * qg.to(F64).view(HEADS, DH) * dG).reshape(-1)

    def per_head(got, ref, axis_heads):
        got, ref = got.to(F64), ref
        if axis_heads == 0:
            got, ref = got.view(HEADS, -1), ref.view(HEADS, -1)
        else:
            got, ref = got.t(), ref.t()
        return ((got - ref).abs().amax(1) / ref.abs().amax(1)).max().item()
    r = {k: v.max().item() / ATTN_BWD_TOL[k] for k, v in tab.items()}
    r["dq_gamma"] = per_head(dqg, ref_dqg, 0) / ATTN_BWD_TOL["dq_gamma"]
    r["dk_gamma"] = per_head(dkg, ref_dkg, 0) / ATTN_BWD_TOL["dk_gamma"]
    r["dbias"] = per_head(dbt, dbias, 1) / ATTN_BWD_TOL["dbias"]
    # the named blocks first: a failure says which window or item
    items = N * HEADS
    grid = min(items, _sms())
    for k, t in tab.items():
        for fn, wn in ((0, 0), (0, nwin - 1), (N - 1, 0), (N - 1, nwin - 1)):
            e = t[fn, wn].max().item()
            assert e <= ATTN_BWD_TOL[k], f"{k}: field {fn} window {wn}: {e:.3g}"
        for b in range(grid):
            last = b + (items - 1 - b) // grid * grid
            n, hd = divmod(last, HEADS)
            e = t[n, :, hd].max().item()
            assert e <= ATTN_BWD_TOL[k], f"{k}: last item {last} (field {n}, head {hd}) of CTA {b}: {e:.3g}"
    check_ratios(r)


# =========================================================================================== E. fused attention forward with dropout
def _attn_sd(dim, heads, dh, w, r, seed):
    from oracle import synth
    spec = {k[len("layers.0.1."):]: v for k, v in synth.maxvit_spec(dim, 1, 2, heads, dh, w, 4, 0.25, r).items()
            if k.startswith("layers.0.1.")}
    return synth.make_state_dict(spec, seed=seed)


@pytest.mark.parametrize("grid_mode", [False, True], ids=["block", "grid"])
def test_attention_fused_train_dropout(grid_mode):
    """ops.attn_fused with the training step's dropout (T = 26: p = 0.1 on the probabilities and after to_out) at 192 fields
    of 42x35 (5,760 windows), against the float64 attention of the oracle with the kernels' own masks (the test hook), per
    field: x_out, the attention term alone (x_out - x) and, in block mode, the register tokens within 4e-3 of their field's
    largest entry (fp16 QKV and X, bf16 P and V, as the inference kernel is held)"""
    from oracle import maxvit_oracle as mo
    o = O()
    N, H, W, C, heads, dh, w, R = 192, 42, 35, 128, HEADS, DH, WIN, R_REG
    S, nwin = R + w * w, (H // w) * (W // w)
    T = 26
    drop = (97531, 5 + int(grid_mode), T)
    scale = 256.0 / (256 - T)
    sd = _attn_sd(C, heads, dh, w, R, seed=19)
    x = rnd(N, H, W, C, seed=171)
    cond = rnd(N, 2, seed=172)
    reg = rnd(*((N, R, C) if grid_mode else (R, C)), seed=173)
    gamma, beta = mo.film(cond.cpu(), sd, "")
    film = torch.cat([gamma, beta], dim=1).to(DEV).contiguous()
    inner = heads * dh
    wq = sd["to_qkv.weight"]
    wqkv_h = torch.stack([wq[i * inner:(i + 1) * inner].reshape(heads, dh, C) for i in range(3)], dim=1).reshape(heads * 96, C)
    wout_h = sd["to_out.0.weight"].reshape(C, heads, dh).permute(1, 0, 2).contiguous()
    head_tab = o.pack_head_tables(sd["rel_pos_bias.weight"], sd["q_norm.gamma"], sd["k_norm.gamma"]).to(DEV)
    x_out, reg_out = o.attn_fused(x, reg, film, wqkv_h.contiguous().to(DEV), wout_h.to(DEV), head_tab, w, R, grid_mode,
                                  not grid_mode, heads, dh, drop=drop)
    torch.cuda.synchronize()
    sd64 = {k: (v.to(DEV, F64) if v.is_floating_point() else v.to(DEV)) for k, v in sd.items()}
    idx = (mo.grid_pixel_index if grid_mode else mo.block_pixel_index)(H, W, w).reshape(-1).to(DEV)
    pm, om = OT().dropout_masks(drop, N * nwin, heads, C)
    r = {"x": 0.0, "attn": 0.0, "reg": 0.0}
    rel = {"x_rel": 0.0, "attn_rel": 0.0, "reg_rel": 0.0}
    chunk = 16
    for f0 in range(0, N, chunk):
        f1 = min(N, f0 + chunk)
        n = f1 - f0
        flat = x[f0:f1].reshape(n, H * W, C).to(F64)
        tok = flat[:, idx].reshape(n * nwin, w * w, C)
        regs = reg[f0:f1].to(F64).repeat_interleave(nwin, 0) if grid_mode else reg.to(F64)[None].expand(n * nwin, R, C)
        seq = torch.cat([regs, tok], dim=1)
        wa, wb = f0 * nwin, f1 * nwin
        att = mo.attention(seq, cond[f0:f1].to(F64), sd64, "", heads=heads, window=w, num_reg=R,
                           prob_mask=pm[wa:wb, :, :S, :S].to(F64) * scale, out_mask=om[wa:wb, :S].to(F64) * scale)
        att_x = torch.empty_like(flat)
        att_x[:, idx] = att[:, R:].reshape(n, nwin * w * w, C)
        got = x_out[f0:f1].reshape(n, H * W, C)
        for key, g_, rf in (("x", got, flat + att_x), ("attn", got - x[f0:f1].reshape(n, H * W, C), att_x)):
            a, b_ = f32_ratio(g_, rf, tol=4e-3)
            r[key], rel[key + "_rel"] = max(r[key], a), max(rel[key + "_rel"], b_)
        if not grid_mode:
            a, b_ = f32_ratio(reg_out.view(N, nwin, R, C)[f0:f1], (seq[:, :R] + att[:, :R]).view(n, nwin, R, C), tol=4e-3)
            r["reg"], rel["reg_rel"] = max(r["reg"], a), max(rel["reg_rel"], b_)
        del flat, tok, seq, att, att_x
    check_ratios({**r, **rel})
