"""Tensor-level wrappers over the training entry points of the C ABI (include/vitgrid.h, "Training step").
PyTorch supplies device memory and streams; every computation is a libvitgrid kernel on the current stream."""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from .ops import DT_CODE, _gemm_code, _p, _st, pg_pixels


def _f32(n, dev):
    return torch.empty(int(n), dtype=torch.float32, device=dev)


def conv3x3_ln_train(x, Wt, bias, ln_g, ln_b, eps, film, res, out, N, HP, WP, out_copy=None):
    """forward Block that also returns the saved tensors (xhat, rstd, relu_mask) for backward"""
    dtype = x.dtype
    dev = x.device
    Q = x.shape[0]
    xhat = torch.empty(Q, 128, dtype=dtype, device=dev)
    rstd = _f32(Q, dev)
    mask = torch.empty(Q, 4, dtype=torch.int32, device=dev)
    scratch = _f32(Q * 128, dev) if dtype == torch.float32 else None
    res_f32 = int(res is not None and res.dtype == torch.float32 and dtype != torch.float32)
    _lib.call("vg_conv3x3_ln_train_fwd", DT_CODE[dtype], x.data_ptr(), x.shape[1], Wt.data_ptr(), bias.data_ptr(),
              ln_g.data_ptr(), ln_b.data_ptr(), float(eps), _p(film), _p(res), res_f32, out.data_ptr(), _p(out_copy),
              xhat.data_ptr(), rstd.data_ptr(), mask.data_ptr(), N, HP, WP, _p(scratch),
              scratch.numel() if scratch is not None else 0, _st())
    return out, (xhat, rstd, mask)


def stem_finish_train(raw3, rawres, bias3, bias1, tt, tres, ln_g, ln_b, eps, film, B, L, HP, WP, h1, res):
    Q = h1.shape[0]
    dev = h1.device
    xhat = torch.empty(Q, 128, dtype=h1.dtype, device=dev)
    rstd = _f32(Q, dev)
    mask = torch.empty(Q, 4, dtype=torch.int32, device=dev)
    _lib.call("vg_stem_finish_train_fwd", DT_CODE[h1.dtype], raw3.data_ptr(), rawres.data_ptr(), bias3.data_ptr(),
              bias1.data_ptr(), tt.data_ptr(), tres.data_ptr(), ln_g.data_ptr(), ln_b.data_ptr(), float(eps),
              film.data_ptr(), B, L, HP, WP, h1.data_ptr(), res.data_ptr(), xhat.data_ptr(), rstd.data_ptr(),
              mask.data_ptr(), _st())
    return xhat, rstd, mask


def conv_ln_bwd(dY, saved, ln_g, film, eps, N, HP, WP, out_dtype, want_border=False):
    """-> dconv (out_dtype, PG, zeros at pads), (sumA, sumB, sumD) (N,128) each, border (N,8,128) or None"""
    xhat, rstd, mask = saved
    dev = dY.device
    dconv = torch.empty(dY.shape[0], 128, dtype=out_dtype, device=dev)
    sums = torch.zeros(3, N, 128, dtype=torch.float32, device=dev)
    border = torch.zeros(N, 8, 128, dtype=torch.float32, device=dev) if want_border else None
    _lib.call("vg_conv_ln_bwd", DT_CODE[xhat.dtype], DT_CODE[out_dtype], dY.data_ptr(), xhat.data_ptr(), rstd.data_ptr(),
              mask.data_ptr(), ln_g.data_ptr(), _p(film), float(eps), dconv.data_ptr(), sums[0].data_ptr(),
              sums[1].data_ptr(), sums[2].data_ptr(), _p(border), N, HP, WP, _st())
    return dconv, sums, border


def conv_ln_param_grads(sums, N, ln_g, ln_b, film, dg, db, dbias, want_dfilm):
    dfilm = torch.empty(N, 256, dtype=torch.float32, device=sums.device) if want_dfilm else None
    _lib.call("vg_conv_ln_param_grads", sums[0].data_ptr(), sums[1].data_ptr(), sums[2].data_ptr(), N, ln_g.data_ptr(),
              ln_b.data_ptr(), _p(film), dg.data_ptr(), db.data_ptr(), dbias.data_ptr(), _p(dfilm), _st())
    return dfilm


def wgrad(dY, A, dW, *, ntaps=1, tap_shift=(0,), M=None, beta=1.0, tf32=False):
    """dW[n][tap*Ca + c] = beta*dW + sum_m dY[m][n] * A[m + shift(tap)][c]   (dW fp32 [Ntot][ntaps*Ca])"""
    assert dY.dtype == A.dtype and dW.dtype == torch.float32 and dW.is_contiguous()
    code = _gemm_code(dY.dtype, tf32)
    M = dY.shape[0] if M is None else M
    Ntot, Ca = dY.shape[1], A.shape[1]
    assert dW.numel() == Ntot * ntaps * Ca, (dW.shape, Ntot, ntaps, Ca)
    shifts = (ctypes.c_int * ntaps)(*tap_shift)
    need = _lib.load().vg_wgrad_workspace(code, M, Ntot, Ca, ntaps)
    work = _f32(need, dY.device)
    _lib.TRACE_TAG = f"wgrad M={M} N={Ntot} K={ntaps}x{Ca} {'tf32' if tf32 else str(dY.dtype)[6:]}"
    _lib.call("vg_wgrad", code, dY.data_ptr(), A.data_ptr(), A.shape[0], M, Ntot, Ca, ntaps, shifts, dW.data_ptr(),
              float(beta), work.data_ptr(), work.numel(), _st())
    return dW


def head_bwd(dpred, h, w, std, N, HP, WP, H, W, pads, dw, db):
    dH = torch.empty(pg_pixels(N, HP, WP), 128, dtype=torch.float32, device=h.device)
    pl, _, pt, _ = pads
    _lib.call("vg_head_bwd", DT_CODE[h.dtype], dpred.data_ptr(), h.data_ptr(), w.data_ptr(), float(std), N, HP, WP, H, W,
              pt, pl, dH.data_ptr(), dw.data_ptr(), db.data_ptr(), _st())
    return dH


def pool2_bwd(x, dlow, N, HP, WP):
    C = x.shape[1]
    dx = torch.empty(x.shape[0], C, dtype=torch.float32, device=x.device)
    _lib.call("vg_pool2_bwd", DT_CODE[x.dtype], x.data_ptr(), dlow.data_ptr(), dx.data_ptr(), N, HP, WP, C, _st())
    return dx


def convT2_bwd_gather(dUp, N, Hl, Wl, C, out_dtype, dbias):
    G = torch.empty(N * Hl * Wl, 4 * C, dtype=out_dtype, device=dUp.device)
    _lib.call("vg_convT2_bwd_gather", DT_CODE[out_dtype], dUp.data_ptr(), G.data_ptr(), dbias.data_ptr(), N, Hl, Wl, C, _st())
    return G


def lead_sum(x, B, L, HP, WP, out_dtype):
    out = torch.empty(pg_pixels(B, HP, WP), 128, dtype=out_dtype, device=x.device)
    _lib.call("vg_lead_sum", DT_CODE[x.dtype], DT_CODE[out_dtype], x.data_ptr(), out.data_ptr(), B, L, HP, WP, _st())
    return out


def pg_field_sum(x, N, HP, WP):
    out = torch.zeros(N, 128, dtype=torch.float32, device=x.device)
    _lib.call("vg_pg_field_sum", x.data_ptr(), out.data_ptr(), N, HP, WP, _st())
    return out


def time_terms_bwd(border, sumD, tres_sum, temb, w3, w1, c_data, dw3, dw1, db1):
    N, ntc = temb.shape
    Cout, c_in = w3.shape[0], w3.shape[1]
    dtemb = torch.empty(N, ntc, dtype=torch.float32, device=temb.device)
    _lib.call("vg_time_terms_bwd", border.data_ptr(), sumD.data_ptr(), tres_sum.data_ptr(), temb.data_ptr(), w3.data_ptr(),
              w1.data_ptr(), N, ntc, c_in, c_data, Cout, dw3.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dtemb.data_ptr(), _st())
    return dtemb


def time_embed_bwd(dtemb, dcond, ts, B, L, le, te, d_lead, d_m, d_d, d_h):
    sB, sT, sF = ts.stride()
    _lib.call("vg_time_embed_bwd", dtemb.data_ptr(), _p(dcond), ts.data_ptr(), sB, sT, sF, B, L, le, te, d_lead.data_ptr(),
              d_m.data_ptr(), d_d.data_ptr(), d_h.data_ptr(), _st())


def cond_mlp_bwd(cond, W0, b0, W1, dout, dW0, db0, dW1, db1, dcond, pre_relu=False):
    N, cd = cond.shape
    hid = W0.shape[0]
    od = W1.shape[0] if W1 is not None else hid
    work = _f32(N * (cd + 2 * hid), cond.device)
    _lib.call("vg_cond_mlp_bwd", cond.data_ptr(), N, cd, int(pre_relu), W0.data_ptr(), _p(b0), hid, _p(W1), od,
              dout.data_ptr(), dW0.data_ptr(), _p(db0), _p(dW1), _p(db1), dcond.data_ptr(), work.data_ptr(), work.numel(), _st())


def adamw_step(param, grad, m, v, lr, beta1, beta2, eps, wd, step, gscale=1.0):
    _lib.call("vg_adamw_step", param.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), param.numel(), float(lr),
              float(beta1), float(beta2), float(eps), float(wd), int(step), float(gscale), _st())


# ---------------------------------------------------------------------------------------------- MaxViT block
def bn_stats(x2d, gamma, beta, eps, momentum, run_mean, run_var):
    """-> (mean, rstd, scale, shift) of train-mode BatchNorm over the rows of x2d [M][C]; updates the running buffers"""
    M, C = x2d.shape
    dev = x2d.device
    st = torch.empty(4, C, dtype=torch.float32, device=dev)
    work = _f32(_lib.load().vg_bn_workspace(M, C), dev)
    _lib.call("vg_bn_stats", x2d.data_ptr(), M, C, gamma.data_ptr(), beta.data_ptr(), float(eps), float(momentum),
              _p(run_mean), _p(run_var), st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), st[3].data_ptr(),
              work.data_ptr(), work.numel(), _st())
    return st


def bn_act(raw, st, act, res=None, out=None):
    M, C = raw.shape
    out = torch.empty_like(raw) if out is None else out
    _lib.call("vg_bn_act", raw.data_ptr(), st[2].data_ptr(), st[3].data_ptr(), int(act), _p(res), out.data_ptr(), M, C, _st())
    return out


def bn_bwd(dOut, raw, st, gamma, act, dgamma, dbeta, fgate=None, fadd=None, rows_per_field=0, out=None):
    M, C = raw.shape
    dev = raw.device
    draw = torch.empty_like(raw) if out is None else out
    work = _f32(_lib.load().vg_bn_workspace(M, C) + 2 * C, dev)
    _lib.call("vg_bn_bwd", dOut.data_ptr(), raw.data_ptr(), st[2].data_ptr(), st[3].data_ptr(), st[0].data_ptr(),
              st[1].data_ptr(), gamma.data_ptr(), int(act), _p(fgate), _p(fadd), int(rows_per_field), M, C,
              dgamma.data_ptr(), dbeta.data_ptr(), draw.data_ptr(), work.data_ptr(), work.numel(), _st())
    return draw


def bn_frozen_stats(bn):
    """-> (mean, rstd, scale, shift) of an eval-mode BatchNorm: its running statistics, nothing updated"""
    st = torch.empty(4, bn.num_features, dtype=torch.float32, device=bn.running_mean.device)
    st[0] = bn.running_mean
    torch.rsqrt(bn.running_var.float() + bn.eps, out=st[1])
    torch.mul(bn.weight.detach(), st[1], out=st[2])
    torch.sub(bn.bias.detach(), st[0] * st[2], out=st[3])
    return st


def bn_bwd_frozen(dOut, raw, st, act, dgamma, dbeta, fgate=None, fadd=None, rows_per_field=0, out=None):
    """backward of bn_act with the running statistics of bn_frozen_stats: no batch-mean terms"""
    M, C = raw.shape
    draw = torch.empty_like(raw) if out is None else out
    work = _f32(_lib.load().vg_bn_workspace(M, C), raw.device)
    _lib.call("vg_bn_bwd_frozen", dOut.data_ptr(), raw.data_ptr(), st[2].data_ptr(), st[3].data_ptr(), st[0].data_ptr(),
              st[1].data_ptr(), int(act), _p(fgate), _p(fadd), int(rows_per_field), M, C, dgamma.data_ptr(), dbeta.data_ptr(),
              draw.data_ptr(), work.data_ptr(), work.numel(), _st())
    return draw


def prepare_bwd(g, B, T, C, H, W, pads, HP, WP, std, extra_channel=-1):
    """adjoint of ops.prepare: g fp32 PG [q][Cpad] over B frames -> dx (B,T,C,H,W) fp32, every element written"""
    assert g.dtype == torch.float32 and g.is_contiguous()
    dx = torch.empty(B, T, C, H, W, dtype=torch.float32, device=g.device)
    pl, _, pt, _ = pads
    _lib.call("vg_prepare_bwd", g.data_ptr(), B, T, C, H, W, pt, pl, HP, WP, g.shape[1], float(std), int(extra_channel),
              dx.data_ptr(), _st())
    return dx


def colsum(x2d, out):
    M, C = x2d.shape
    _lib.call("vg_colsum", x2d.data_ptr(), M, C, out.data_ptr(), _st())


def dw3x3(x, w9, scale, shift, act, want_psum=False, out=None):
    """marching-stencil depthwise 3x3 on CL (N,H,W,C): out = act(conv*scale + shift)"""
    N, H, W, C = x.shape
    out = torch.empty_like(x) if out is None else out
    strips = _lib.load().vg_dw_strips(W)
    psum = torch.empty(N, strips, C, dtype=torch.float32, device=x.device) if want_psum else None
    _lib.call("vg_dw3x3_fwd", DT_CODE[x.dtype], x.data_ptr(), w9.data_ptr(), scale.data_ptr(), shift.data_ptr(), int(act),
              out.data_ptr(), _p(psum), N, H, W, C, _st())
    return out, psum


def dw3x3_wgrad(x, dY, dw9, dbias):
    N, H, W, C = x.shape
    strips = _lib.load().vg_dw_strips(W)
    work = _f32((N * strips + 1) * 10 * C, x.device)
    _lib.call("vg_dw3x3_wgrad", x.data_ptr(), dY.data_ptr(), N, H, W, C, dw9.data_ptr(), dbias.data_ptr(), work.data_ptr(),
              work.numel(), _st())


def field_sum(x):
    """(N,H,W,C) fp32 -> (N, parts, C) deterministic partial per-field channel sums"""
    N, H, W, C = x.shape
    out = torch.empty(N, _lib.load().vg_field_parts(H * W), C, dtype=torch.float32, device=x.device)
    _lib.call("vg_field_dot", x.data_ptr(), None, out.data_ptr(), N, H * W, C, _st())
    return out


def se_gate_train(psum, HW, W1, W2):
    N, nparts, C = psum.shape
    se = W1.shape[0]
    dev = psum.device
    gate = torch.empty(N, C, dtype=torch.float32, device=dev)
    mean = torch.empty(N, C, dtype=torch.float32, device=dev)
    hid = torch.empty(N, se, dtype=torch.float32, device=dev)
    _lib.call("vg_se_gate_train_fwd", psum.data_ptr(), N, nparts, HW, W1.data_ptr(), W2.data_ptr(), C, se, gate.data_ptr(),
              mean.data_ptr(), hid.data_ptr(), _st())
    return gate, mean, hid


def se_scale_oop(x, gate):
    N, H, W, C = x.shape
    out = torch.empty_like(x)
    _lib.call("vg_se_scale_oop", x.data_ptr(), gate.data_ptr(), out.data_ptr(), N, H * W, C, _st())
    return out


def se_bwd(dh4, h3, gate, mean, hid, W1, W2, dW1, dW2):
    N, H, W, C = h3.shape
    se = W1.shape[0]
    dmean = torch.empty(N, C, dtype=torch.float32, device=h3.device)
    work = _f32(N * ((_lib.load().vg_field_parts(H * W) + 1) * C + se), h3.device)
    _lib.call("vg_se_bwd", dh4.data_ptr(), h3.data_ptr(), gate.data_ptr(), mean.data_ptr(), hid.data_ptr(), W1.data_ptr(),
              W2.data_ptr(), N, H * W, C, se, dW1.data_ptr(), dW2.data_ptr(), dmean.data_ptr(), work.data_ptr(), work.numel(), _st())
    return dmean


def dropout_masks(drop, n_windows, heads, C):
    """test hook: the (prob_mask [Nw][heads][64][64], out_mask [Nw][64][C]) uint8 masks the kernels derive from drop = (seed, salt, T)"""
    dev = torch.device("cuda")
    pm = torch.empty(n_windows, heads, 64, 64, dtype=torch.uint8, device=dev)
    om = torch.empty(n_windows, 64, C, dtype=torch.uint8, device=dev)
    _lib.call("vg_dropout_mask_debug", int(drop[0]), int(drop[1]), int(drop[2]), n_windows, heads, C, pm.data_ptr(), om.data_ptr(), _st())
    return pm, om


def attn_out_bwd_gather(dx_out, dreg, reg_scale, win, R, grid_mode, drop=(0, 0, 0), out_bf16=False):
    N, Hl, Wl, C = dx_out.shape
    rows = N * (Hl // win) * (Wl // win) * (R + win * win)
    dproj = torch.empty(rows, C, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=dx_out.device)
    _lib.call("vg_attn_out_bwd_gather", dx_out.data_ptr(), _p(dreg), float(reg_scale), N, Hl, Wl, C, win, R, int(grid_mode),
              dproj.data_ptr(), int(out_bf16), int(drop[0]), int(drop[1]), int(drop[2]), _st())
    return dproj


def attn_core_bwd(qkv, datt, q_gamma, k_gamma, bias_table, N, Hl, Wl, win, R, heads, dh, dq_gamma, dk_gamma, dbias_table,
                  tf32=False, want_att=False, drop=(0, 0, 0)):
    """-> dqkv (, att = softmax(.) V re-materialised by the tensor-core kernel when want_att)"""
    dqkv = torch.empty_like(qkv)
    att = torch.empty(qkv.shape[0], heads * dh, dtype=qkv.dtype, device=qkv.device) if want_att else None
    # 2 = bf16 mma + ldmatrix on fp32 tensors; 0 = exact-fp32 SIMT;
    # 3 = the tcgen05 kernel on bf16 tensors (qkv, datt -> dqkv, att), selected by the dtype of qkv
    mode = 2 if tf32 else 0
    if qkv.dtype == torch.bfloat16:
        assert datt.dtype == torch.bfloat16
        mode = 3
    _lib.call("vg_attn_core_bwd", qkv.data_ptr(), datt.data_ptr(), q_gamma.data_ptr(), k_gamma.data_ptr(),
              bias_table.data_ptr(), N, Hl, Wl, win, R, heads, dh, dqkv.data_ptr(), dq_gamma.data_ptr(), dk_gamma.data_ptr(),
              dbias_table.data_ptr(), mode, _p(att), int(drop[0]), int(drop[1]), int(drop[2]), _st())
    return (dqkv, att) if want_att else dqkv


def attn_gather_bwd(x, reg, film, dtok, dx_out, dreg_res, reg_scale, dreg_in, dfilm, win, R, grid_mode, eps=1e-5):
    N, Hl, Wl, C = x.shape
    dx_in = torch.empty_like(x)
    _lib.call("vg_attn_gather_bwd", x.data_ptr(), reg.data_ptr(), int(reg.dim() == 3), film.data_ptr(), dtok.data_ptr(),
              dx_out.data_ptr(), _p(dreg_res), float(reg_scale), dx_in.data_ptr(), dreg_in.data_ptr(), dfilm.data_ptr(),
              N, Hl, Wl, C, win, R, int(grid_mode), float(eps), _st())
    return dx_in
