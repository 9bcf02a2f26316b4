"""Tensor-level wrappers over the C ABI (include/vitgrid.h).  PyTorch is used for device memory and streams
only; every computation below is a libvitgrid kernel launch on the caller's current stream."""
from __future__ import annotations

import ctypes

import torch

from . import _lib

DT_CODE = {torch.bfloat16: 0, torch.float32: 1, torch.float16: 3}


def _p(t):
    return None if t is None else t.data_ptr()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _gemm_code(dtype, tf32):
    """0 = bf16 tcgen05, 1 = fp32 SIMT, 2 = fp32 storage + tf32 tcgen05, 3 = fp16 tcgen05"""
    if dtype == torch.bfloat16:
        return 0
    if dtype == torch.float16:
        return 3
    return 2 if tf32 else 1


def _scratch(dtype, elems, device, tf32=False):
    """exact-fp32 (SIMT) GEMMs accumulate into a caller-provided scratch; the tcgen05 paths need none."""
    if dtype == torch.float32 and not tf32:
        t = torch.empty(int(elems), dtype=torch.float32, device=device)
        return t, t.data_ptr(), t.numel()
    return None, None, 0


def pg_pixels(N, HP, WP):
    return (N * (HP + 1) + 1) * (WP + 1)


def pg_empty(N, HP, WP, C, dtype, device):
    return torch.empty(pg_pixels(N, HP, WP), C, dtype=dtype, device=device)


def pg_from_nchw(x, dtype):
    """(N,C,H,W) -> PG buffer (test helper / standalone-module boundary; plain torch indexing)."""
    N, C, H, W = x.shape
    buf = torch.zeros(N * (H + 1) + 1, W + 1, C, dtype=dtype, device=x.device)
    buf[:N * (H + 1)].view(N, H + 1, W + 1, C)[:, 1:, 1:] = x.permute(0, 2, 3, 1).to(dtype)
    return buf.view(-1, C)


def pg_to_nchw(buf, N, H, W):
    C = buf.shape[1]
    v = buf.view(N * (H + 1) + 1, W + 1, C)[:N * (H + 1)].view(N, H + 1, W + 1, C)[:, 1:, 1:]
    return v.permute(0, 3, 1, 2).contiguous()


def prepare(x, cfg_pads, HP, WP, Cpad, mean, std, dtype, packed=False):
    """packed=True: x is a bf16 batch packed on the host (pipeline.pack_host), PM2.5 channels already standardised"""
    B, T, C, H, W = x.shape
    assert x.is_cuda and x.dtype == (torch.bfloat16 if packed else torch.float32)
    out = torch.empty(pg_pixels(B, HP, WP), Cpad, dtype=dtype, device=x.device)
    strides = (ctypes.c_longlong * 5)(*x.stride())
    pl, _, pt, _ = cfg_pads
    if packed:
        _lib.call("vg_prepare_packed_fwd", DT_CODE[dtype], x.data_ptr(), strides, B, T, C, H, W, pt, pl, HP, WP, Cpad,
                  out.data_ptr(), _st())
    else:
        _lib.call("vg_prepare_fwd", DT_CODE[dtype], x.data_ptr(), strides, B, T, C, H, W, pt, pl, HP, WP, Cpad,
                  float(mean), float(std), out.data_ptr(), _st())
    return out


def standardise_channel_(x, channel, mean, std):
    """x[:, :, channel] = (x[:, :, channel] - mean) / std in place (metnet3.py:701); x (B,T,C,H,W) fp32, any strides"""
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
    B, T, C, H, W = x.shape
    strides = (ctypes.c_longlong * 5)(*x.stride())
    _lib.call("vg_standardise_channel", x.data_ptr(), strides, B, T, C, H, W, int(channel), float(mean), float(std), _st())
    return x


def time_terms(ts, B, L, emb_lead, emb_m, emb_d, emb_h, w3, w1, c_data, Cout):
    le, te = emb_lead.shape[1], emb_m.shape[1]
    N = B * L
    dev = ts.device
    temb = torch.empty(N, le + 3 * te, dtype=torch.float32, device=dev)
    cond = torch.empty(N, le, dtype=torch.float32, device=dev)
    tt = torch.empty(N, 9, Cout, dtype=torch.float32, device=dev)
    tres = torch.empty(N, Cout, dtype=torch.float32, device=dev)
    assert ts.dtype == torch.float32 and ts.shape[1] > 6 and ts.shape[2] >= 4, "timestamps must be (B, >=7, 4) fp32"
    sB, sT, sF = ts.stride()
    _lib.call("vg_time_terms_fwd", ts.data_ptr(), sB, sT, sF, B, L, le, te, emb_lead.data_ptr(), emb_m.data_ptr(),
              emb_d.data_ptr(), emb_h.data_ptr(), w3.data_ptr(), _p(w1), w3.shape[1], c_data, Cout,
              temb.data_ptr(), cond.data_ptr(), tt.data_ptr(), tres.data_ptr(), _st())
    return temb, cond, tt, tres


def cond_mlp(cond, W0, b0, W1=None, b1=None, pre_relu=False):
    N, cd = cond.shape
    hid = W0.shape[0]
    od = W1.shape[0] if W1 is not None else hid
    out = torch.empty(N, od, dtype=torch.float32, device=cond.device)
    if W1 is not None and N <= 1024 and hid >= 1024:    # wide layers (configs[4])
        h = torch.empty(N, hid, dtype=torch.float32, device=cond.device)
        _lib.call("vg_dense_rows_fwd", cond.data_ptr(), N, cd, int(pre_relu), W0.data_ptr(), _p(b0), hid, 2, h.data_ptr(), _st())
        _lib.call("vg_dense_rows_fwd", h.data_ptr(), N, hid, 0, W1.data_ptr(), _p(b1), od, 0, out.data_ptr(), _st())
        return out
    _lib.call("vg_cond_mlp_fwd", cond.data_ptr(), N, cd, int(pre_relu), W0.data_ptr(), _p(b0), hid, _p(W1), _p(b1), od,
              out.data_ptr(), _st())
    return out


_X3_TAG = ""      # trace tag suffix of the GEMM issued by gemm(x3=True)


def split3_tf32(x, pattern):
    """fp32 [rows][K] -> fp32 [rows][3K]: (hi | hi | lo) for the left operand (pattern 0), (hi | lo | hi) for the [N][K] weights
    (pattern 1), hi = x truncated to tf32; one tf32 GEMM over 3K then computes hi*hi + hi*lo + lo*hi (include/vitgrid.h)"""
    rows, K = x.shape
    out = torch.empty(rows, 3 * K, dtype=torch.float32, device=x.device)
    _lib.call("vg_split3_tf32", x.data_ptr(), rows, K, out.data_ptr(), int(pattern), _st())
    return out


def gemm(A, Wt, *, ntaps=1, tap_shift=(0,), M=None, rows_per_batch=0, b_rows_per_batch=0, bias=None, scale=None,
         shift=None, act=0, res=None, out=None, out_f32=False, n_out=None, tf32=False, out_dtype=None, x3=False, Wt_x3=None):
    """out_dtype=torch.float16: fp16 output from any operand type (the MBConv hidden tensor).
    x3 (fp32 operands, no tf32): near-fp32 product (~1e-5, see include/vitgrid.h) on the tensor cores by the 3xTF32 operand split
    instead of the SIMT kernel; Wt_x3: the weights already split (split3_tf32(Wt, 1), cached by the caller)"""
    if x3 and not tf32 and A.dtype == torch.float32 and ntaps == 1 and A.is_contiguous() and Wt.is_contiguous() and A.shape[1] % 32 == 0:
        global _X3_TAG
        _X3_TAG = " 3xTF32"
        try:
            return gemm(split3_tf32(A, 0), Wt_x3 if Wt_x3 is not None else split3_tf32(Wt, 1), M=M, rows_per_batch=rows_per_batch, b_rows_per_batch=b_rows_per_batch,
                        bias=bias, scale=scale, shift=shift, act=act, res=res, out=out, out_f32=out_f32, n_out=n_out, tf32=True,
                        out_dtype=out_dtype)
        finally:
            _X3_TAG = ""
    dtype = A.dtype
    rowsA, Ca = A.shape
    M = rowsA if M is None else M
    Ntot = n_out if n_out is not None else (b_rows_per_batch if rows_per_batch else Wt.shape[0])
    if out is None:
        out = torch.empty(M, Ntot, dtype=out_dtype or (torch.float32 if out_f32 else dtype), device=A.device)
    shifts = (ctypes.c_int * ntaps)(*tap_shift)
    keep, sp, sn = _scratch(dtype, M * Ntot, A.device, tf32)
    _lib.TRACE_TAG = f"M={M} K={ntaps}x{Ca} N={Ntot} {'tf32' if tf32 else str(dtype)[6:]}{_X3_TAG}"
    res_f32 = int(res is not None and res.dtype == torch.float32)
    _lib.call("vg_gemm_fwd", _gemm_code(dtype, tf32), A.data_ptr(), rowsA, Ca, Wt.data_ptr(), Ntot, ntaps, shifts, M,
              rows_per_batch, b_rows_per_batch, _p(bias), _p(scale), _p(shift), act, _p(res),
              res.shape[1] if res is not None else 0, res_f32, out.data_ptr(), out.shape[1], _out_code(dtype, out.dtype, out_f32),
              sp, sn, _st())
    return out


def _out_code(in_dtype, out_dtype, out_f32):
    """EpiParams.out_f32: 0 = the operand dtype, 1 = fp32, 2 = bf16, 3 = fp16"""
    if out_dtype == torch.float16:
        return 3
    if out_dtype == torch.float32 and in_dtype != torch.float32:
        return 1
    if out_dtype == torch.bfloat16 and in_dtype != torch.bfloat16:
        return 2
    return int(out_f32)


def conv_tap_shifts(WP):
    P = WP + 1
    return tuple((ky - 1) * P + (kx - 1) for ky in range(3) for kx in range(3))


def conv3x3_ln(x, Wt, bias, ln_g, ln_b, eps, film, res, out, N, HP, WP, out_copy=None, head=None, tf32=False):
    """head = (w[C], b, std, mean, H, W, pads, out (N,H,W) fp32) fuses the 1x1 head / unpad / de-normalisation.
    tf32 (fp32 storage only): the contraction runs on tcgen05 kind::tf32 instead of the exact-fp32 SIMT kernel"""
    dtype = x.dtype
    C = x.shape[1]
    code = 2 if (tf32 and dtype == torch.float32) else DT_CODE[dtype]
    res_f32 = int(res is not None and res.dtype == torch.float32 and dtype != torch.float32)
    if head is None:
        hw, hb, hs, hm, H, W, pt, pl, ho = None, 0.0, 1.0, 0.0, 0, 0, 0, 0, None
    else:
        hw, hb, hs, hm, H, W, pads, ho = head
        pl, _, pt, _ = pads
    if C != 128:
        # other widths (256 / 384 / 512): plain shifted-row GEMM into an fp32 scratch + row-wise LN / FiLM / ReLU / residual
        scratch = torch.empty(x.shape[0] * C * (2 if dtype == torch.float32 else 1), dtype=torch.float32, device=x.device)
        _lib.call("vg_conv3x3_ln_wide_fwd", code, x.data_ptr(), C, Wt.data_ptr(), bias.data_ptr(), ln_g.data_ptr(),
                  ln_b.data_ptr(), float(eps), _p(film), _p(res), res_f32, _p(out), _p(out_copy), N, HP, WP, _p(hw), float(hb),
                  float(hs), float(hm), H, W, pt, pl, _p(ho), scratch.data_ptr(), scratch.numel(), _st())
        return out
    keep, sp, sn = _scratch(dtype, x.shape[0] * 128, x.device, tf32)
    _lib.TRACE_TAG = ("film" if film is not None else "plain") + ("+res" if res is not None else "") + \
        ("+copy" if out_copy is not None else "") + ("+head" if head is not None else "")
    _lib.call("vg_conv3x3_ln_fwd", code, x.data_ptr(), x.shape[1], Wt.data_ptr(), bias.data_ptr(),
              ln_g.data_ptr(), ln_b.data_ptr(), float(eps), _p(film), _p(res), res_f32, _p(out), _p(out_copy), N, HP, WP,
              _p(hw), float(hb), float(hs), float(hm), H, W, pt, pl, _p(ho), sp, sn, _st())
    return out


def stem_finish(raw3, rawres, bias3, bias1, tt, tres, ln_g, ln_b, eps, film, B, L, HP, WP, h1, res):
    C = h1.shape[1]
    if C != 128:
        _lib.call("vg_stem_finish_wide_fwd", DT_CODE[h1.dtype], raw3.data_ptr(), rawres.data_ptr(), bias3.data_ptr(),
                  bias1.data_ptr(), tt.data_ptr(), tres.data_ptr(), ln_g.data_ptr(), ln_b.data_ptr(), float(eps),
                  film.data_ptr(), B, L, HP, WP, C, h1.data_ptr(), res.data_ptr(), _st())
        return
    _lib.call("vg_stem_finish_fwd", DT_CODE[h1.dtype], raw3.data_ptr(), rawres.data_ptr(), bias3.data_ptr(),
              bias1.data_ptr(), tt.data_ptr(), tres.data_ptr(), ln_g.data_ptr(), ln_b.data_ptr(), float(eps),
              film.data_ptr(), B, L, HP, WP, h1.data_ptr(), res.data_ptr(), _st())


def pool2(x, N, HP, WP, out_dtype=None):
    C = x.shape[1]
    out_dtype = out_dtype or x.dtype
    out = torch.empty(N, HP // 2, WP // 2, C, dtype=out_dtype, device=x.device)
    assert out_dtype == x.dtype or (x.dtype == torch.bfloat16 and out_dtype == torch.float32)
    _lib.call("vg_pool2_fwd", DT_CODE[x.dtype], int(out_dtype != x.dtype), x.data_ptr(), out.data_ptr(), N, HP, WP, C, _st())
    return out


def dw3x3_bnact(x, w9, scale, shift, out=None):
    """depthwise 3x3 + folded BN + GELU (marching-stencil kernel); psum (N, strips, C) feeds the squeeze-excite mean"""
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    if C % 4 == 0 and 128 % (C // 4) == 0:
        strips = _lib.load().vg_dw_strips(W)
        psum = torch.empty(N, strips, C, dtype=torch.float32, device=x.device)
        _lib.call("vg_dw3x3_fwd", DT_CODE[x.dtype], x.data_ptr(), w9.data_ptr(), scale.data_ptr(), shift.data_ptr(), 1,
                  out.data_ptr(), psum.data_ptr(), N, H, W, C, _st())
        return out, psum
    psum = torch.empty(N, H, C, dtype=torch.float32, device=x.device)
    _lib.call("vg_dw3x3_bnact_fwd", DT_CODE[x.dtype], x.data_ptr(), w9.data_ptr(), scale.data_ptr(), shift.data_ptr(),
              out.data_ptr(), psum.data_ptr(), N, H, W, C, _st())
    return out, psum


def se_gate(psum, HW, W1, W2):
    """psum: (N, nparts, C) partial channel sums over the HW pixels of each field"""
    N, nparts, C = psum.shape
    gate = torch.empty(N, C, dtype=torch.float32, device=psum.device)
    mean = hid = None
    if N <= 1024 and C >= 1024:    # wide layers: the library runs the two layers as vg_dense_rows_fwd passes over (mean, hid)
        mean = torch.empty(N, C, dtype=torch.float32, device=psum.device)
        hid = torch.empty(N, W1.shape[0], dtype=torch.float32, device=psum.device)
    _lib.call("vg_se_gate_train_fwd", psum.data_ptr(), N, nparts, HW, W1.data_ptr(), W2.data_ptr(), C, W1.shape[0],
              gate.data_ptr(), _p(mean), _p(hid), _st())
    return gate


def se_fold_weights(W, gate, dtype=torch.float32):
    """(Cout, C) fp32 projection weights x (N, C) gates -> per-field weights (N*Cout, C) in fp32 or fp16"""
    Cout, C = W.shape
    N = gate.shape[0]
    out = torch.empty(N * Cout, C, dtype=dtype, device=W.device)
    _lib.call("vg_se_fold_weights", W.data_ptr(), gate.data_ptr(), out.data_ptr(), int(dtype == torch.float16), N, Cout, C, _st())
    return out


def se_scale_(x, gate):
    N, H, W, C = x.shape
    _lib.call("vg_se_scale_fwd", DT_CODE[x.dtype], x.data_ptr(), gate.data_ptr(), N, H * W, C, _st())
    return x


def attn_gather(x, reg, film, win, R, grid_mode, eps=1e-5, out=None, out_bf16=False):
    """out_bf16: bf16 tokens from an fp32 residual stream (16-bit attention backward chain of the training step)"""
    N, Hl, Wl, C = x.shape
    S = R + win * win
    rows = N * (Hl // win) * (Wl // win) * S
    if out is None:
        out = torch.empty(rows, C, dtype=torch.bfloat16 if out_bf16 else x.dtype, device=x.device)
    _lib.call("vg_attn_gather_fwd", DT_CODE[x.dtype], x.data_ptr(), reg.data_ptr(), int(reg.dim() == 3), film.data_ptr(),
              N, Hl, Wl, C, win, R, int(grid_mode), float(eps), out.data_ptr(), int(out.dtype == torch.bfloat16 and x.dtype != torch.bfloat16), _st())
    return out


def attn_core(qkv, q_gamma, k_gamma, bias_table, N, Hl, Wl, win, R, heads, dh, out=None, drop=(0, 0, 0), x3=False, tf32=False, split_out=False):
    """fp32 tensors: x3 = QK^T and PV as 3xTF32 split products on the tensor cores (dtype code 2), tf32 = single tf32 products (code 4),
    neither = exact-fp32 FMAs.  split_out (with x3, S <= 64): the output rows are written as [hi | hi | lo] (3 * heads * dh long), the left
    operand of the 3xTF32 out-projection, instead of a split3_tf32 pass over them (code 6)"""
    if split_out:
        assert x3 and qkv.dtype == torch.float32 and out is None and win * win + R <= 64 and not drop[2]
        out = torch.empty(qkv.shape[0], 3 * heads * dh, dtype=qkv.dtype, device=qkv.device)
    if out is None:
        out = torch.empty(qkv.shape[0], heads * dh, dtype=qkv.dtype, device=qkv.device)
    code = DT_CODE[qkv.dtype]
    if qkv.dtype == torch.float32 and (x3 or tf32):
        code = 4 if tf32 else (6 if split_out else 2)
    _lib.call("vg_attn_core_fwd", code, qkv.data_ptr(), q_gamma.data_ptr(), k_gamma.data_ptr(),
              bias_table.data_ptr(), N, Hl, Wl, win, R, heads, dh, out.data_ptr(), int(drop[0]), int(drop[1]), int(drop[2]), _st())
    return out


def attn_out(attn, Wt, x_in, reg_in, win, R, grid_mode, want_reg_out, x_out=None, tf32=False, drop=(0, 0, 0), x3=False, Wt_x3=None,
             attn_is_split=False):
    if attn_is_split:                                                                   # attn_core(split_out=True) wrote [hi | hi | lo] rows
        return attn_out(attn, Wt_x3 if Wt_x3 is not None else split3_tf32(Wt, 1), x_in, reg_in, win, R, grid_mode, want_reg_out, x_out=x_out,
                        tf32=True, drop=drop)
    if x3 and not tf32 and attn.dtype == torch.float32 and attn.shape[1] % 32 == 0:      # 3xTF32 (see gemm)
        return attn_out(split3_tf32(attn, 0), Wt_x3 if Wt_x3 is not None else split3_tf32(Wt, 1), x_in, reg_in, win, R, grid_mode, want_reg_out, x_out=x_out,
                        tf32=True, drop=drop)
    N, Hl, Wl, C = x_in.shape
    nwin = (Hl // win) * (Wl // win)
    if x_out is None:
        x_out = torch.empty_like(x_in)
    reg_out = torch.empty(N * nwin, R, C, dtype=torch.float32, device=x_in.device) if want_reg_out else None
    keep, sp, sn = _scratch(attn.dtype, attn.shape[0] * C, attn.device, tf32)
    _lib.call("vg_attn_out_fwd", _gemm_code(attn.dtype, tf32), attn.data_ptr(), attn.shape[1], Wt.data_ptr(), x_in.data_ptr(),
              reg_in.data_ptr(), int(reg_in.dim() == 3), _p(reg_out), x_out.data_ptr(), N, Hl, Wl, C, win, R,
              int(grid_mode), int(drop[0]), int(drop[1]), int(drop[2]), sp, sn, _st())
    return x_out, reg_out


TAB_SR, TAB_SB = 12, 180      # row / column-offset strides (floats) of the fused kernel's bias table: bank-conflict-free reads


def pack_head_tables(bias_table, q_gamma, k_gamma, win=7):
    """per-head table of the fused attention kernel: relative-position bias as `win` pre-shifted copies
    [bi][row 0..2w-2] with entry k (0..6) = table[row*(2w-1) + bi + (w-1) - k] (so that the 7 keys of one window row are two
    aligned 16-byte reads; row stride TAB_SR, bi stride TAB_SB floats, chosen so that a quarter-warp's reads hit different
    banks), then table[(2w-1)^2] x 8 (the register-token bias, maxvit.py:167, as a row of its own), dh * gamma_q * gamma_k [dh]
    (the two RMSNorm gains and the two sqrt(dh) factors of maxvit.py:26-30 folded into the key operand), dh unused.
    The bias entries are stored times log2(e): the kernel's softmax works in the exp2 domain.  bias_table: (nb, heads)."""
    assert win == 7, "the fused kernel is specialised for 7x7 windows"
    heads, w2 = bias_table.shape[1], 2 * win - 1
    bi = torch.arange(win).view(win, 1, 1)
    row = torch.arange(w2).view(1, w2, 1)
    k = torch.arange(8).view(1, 1, 8)
    idx = (row * w2 + bi + (win - 1) - k).clamp_(0, w2 * w2 - 1)                      # k = 7 is padding
    T = bias_table.t().float() * 1.4426950408889634                                  # (heads, nb), exp2 domain
    shifted = T[:, idx.reshape(-1).to(T.device)].reshape(heads, win, w2, 8)
    shifted[..., 7] = 0
    tab = torch.zeros(heads, win, TAB_SB, device=T.device)
    tab[:, :, :w2 * TAB_SR].view(heads, win, w2, TAB_SR)[..., :8] = shifted
    t_last = T[:, w2 * w2].reshape(heads, 1).expand(heads, 8)
    qg, kg = q_gamma.float().reshape(heads, -1), k_gamma.float().reshape(heads, -1)
    return torch.cat([tab.reshape(heads, -1), t_last, qg * kg * qg.shape[1], torch.zeros_like(kg)], dim=1).contiguous()


def attn_logit_bound(bias_table, q_gamma, k_gamma, dh):
    """bound of |logit + bias| in the exp2 domain for vg_attn_fused2_fwd: q-hat and k-hat are unit vectors times sqrt(dh) * gamma
    (maxvit.py:26-30), so |logit| <= dh * max|gamma_q gamma_k|; 2 % slack for the fp16 operands.  One host sync: call at pack time."""
    g = (q_gamma.float().reshape(-1, dh) * k_gamma.float().reshape(-1, dh)).abs().max()
    return float(1.02 * 1.4426950408889634 * (dh * g + bias_table.float().abs().max()).item())


def attn_fused(x, reg_in, film, wqkv_h, wout_h, head_tab, win, R, grid_mode, want_reg_out, heads, dh, eps=1e-5, drop=(0, 0, 0),
               inplace=False, logit_bound=0.0):
    """whole attention layer (+ residual) in one kernel; x CL (N,Hl,Wl,128) fp32.
    drop = (seed, salt, T): training dropout with probability T/256 on the probabilities and the to_out output.
    The kernel works in place on the residual stream (its TMA reduce-store performs the residual add): inplace=True lets it
    overwrite x (inference: x is a temporary), otherwise x is copied first (training keeps the input for backward).
    Needs heads even (the kernel's two compute groups alternate heads)."""
    N, Hl, Wl, C = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous()
    nwin = (Hl // win) * (Wl // win)
    reg_out = torch.empty(N * nwin, R, C, dtype=torch.float32, device=x.device) if want_reg_out else None
    if wqkv_h.dtype != torch.float16:                       # the kernel's QKV operand format (the modules pack it once)
        wqkv_h = wqkv_h.half()
    xio = x if inplace else x.clone()
    _lib.call("vg_attn_fused2_fwd", xio.data_ptr(), reg_in.data_ptr(), int(reg_in.dim() == 3), _p(reg_out), film.data_ptr(),
              wqkv_h.data_ptr(), wout_h.data_ptr(), head_tab.data_ptr(), N, Hl, Wl, C, win, R, int(grid_mode), heads, dh, float(eps),
              int(drop[0]), int(drop[1]), int(drop[2]), float(logit_bound), _st())
    return xio, reg_out


def reg_mean(reg_out, N, nwin):
    R, C = reg_out.shape[1], reg_out.shape[2]
    out = torch.empty(N, R, C, dtype=torch.float32, device=reg_out.device)
    _lib.call("vg_reg_mean_fwd", reg_out.data_ptr(), out.data_ptr(), N, nwin, R * C, _st())
    return out


def convT2(x, Wt, bias, out, tf32=False, out_copy=None):
    """x CL (N,Hl,Wl,C) -> out PG (N,2Hl,2Wl,C); `out` must already hold zeros at its pad positions.
    `out` may be bf16 while x is fp32 (mixed mode: tf32 MaxViT feeding the bf16 decoder convs)."""
    N, Hl, Wl, C = x.shape
    keep, sp, sn = _scratch(x.dtype, N * Hl * Wl * 4 * C, x.device, tf32)
    _lib.call("vg_convT2_fwd", _gemm_code(x.dtype, tf32), int(out.dtype == torch.bfloat16 and x.dtype != torch.bfloat16), x.data_ptr(), Wt.data_ptr(), bias.data_ptr(), out.data_ptr(), _p(out_copy), N, Hl, Wl,
              C, sp, sn, _st())
    return out


def head(h, w, bias, std, mean, N, HP, WP, H, W, pads, out=None):
    C = h.shape[1]
    if out is None:
        out = torch.empty(N, H, W, dtype=torch.float32, device=h.device)
    pl, _, pt, _ = pads
    _lib.call("vg_head_fwd", DT_CODE[h.dtype], h.data_ptr(), w.data_ptr(), float(bias), float(std), float(mean), N, HP, WP,
              C, H, W, pt, pl, out.data_ptr(), _st())
    return out


def focal_r_forward(pred, target, beta=0.2, gamma=1.0, mse=False):
    assert pred.dtype == torch.float32 and target.dtype == torch.float32 and pred.is_contiguous() and target.is_contiguous()
    n = pred.numel()
    nb = max(1, min(1024, (n + 1023) // 1024))
    partial = torch.empty(nb, dtype=torch.float32, device=pred.device)
    loss = torch.empty((), dtype=torch.float32, device=pred.device)
    _lib.call("vg_focal_r_fwd", pred.data_ptr(), target.data_ptr(), n, float(beta), float(gamma), int(mse),
              partial.data_ptr(), nb, loss.data_ptr(), _st())
    return loss


def focal_r_backward(pred, target, grad_out, beta=0.2, gamma=1.0, mse=False):
    n = pred.numel()
    grad = torch.empty_like(pred)
    _lib.call("vg_focal_r_bwd", pred.data_ptr(), target.data_ptr(), n, float(beta), float(gamma), int(mse),
              float(grad_out) / n, grad.data_ptr(), _st())
    return grad
