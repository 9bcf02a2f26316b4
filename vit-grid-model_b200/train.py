"""Training step of MetNet3 / MaxViT on libvitgrid kernels: train-mode forward (batch-statistic BatchNorm, activations
saved for backward), hand-written backward, and the autograd / data-parallel plumbing around them.

The reference has no training code of its own beyond ``nn.Module`` autograd (metnet3.py:86-430, maxvit.py:33-341), so
parity is defined against autograd of the reference module in ``train()`` mode on identical weights and inputs
(tests/test_train_gpu.py; golden gradients generated from the real reference by tests/golden/make_golden.py).

Layout of the step (N = B*L fields):
  forward : prepare -> stem (per sample, lead-time dedup) -> stem finish -> conv blocks -> maxpool -> MaxViT -> convT
            -> conv blocks -> 1x1 head.  Every Block also stores xhat / rstd / ReLU mask (fused in the conv epilogue).
  backward: the exact transpose, section by section, writing parameter gradients into one flat fp32 buffer ordered
            by completion time (head, decoder, up, MaxViT, encoder, embeddings) so that a data-parallel run can start the
            NCCL all-reduce of a finished section on a side stream while the rest of backward is still running.
"""
from __future__ import annotations

from collections import OrderedDict

import torch

from . import _lib, ops, ops_train as ot
from .maxvit import MBConvResidual


# ------------------------------------------------------------------------------------------------ gradient buffer
class GradBuffer:
    """One flat fp32 buffer with a view per parameter, sections ordered by backward completion time."""

    SECTIONS = ("classifier_pm25.", "resnet2.", "up.", "vit.", "resnet1.", "condition_")
    ALIGN = 64                     # every view starts on a 256-byte boundary (kernels use 16-byte vector accesses)

    def __init__(self, model):
        named = list(model.named_parameters())
        order = []
        for sec in self.SECTIONS:
            order += [(n, p) for n, p in named if n.startswith(sec)]
        assert len(order) == len(named), "unexpected parameter outside the known sections"
        al = self.ALIGN
        total = sum((p.numel() + al - 1) // al * al for _, p in order)
        dev = order[0][1].device
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.views, self.bounds = OrderedDict(), []
        off = 0
        for sec in self.SECTIONS:
            start = off
            for n, p in order:
                if n.startswith(sec):
                    self.views[n] = self.flat[off:off + p.numel()].view(p.shape)
                    off += (p.numel() + al - 1) // al * al
            self.bounds.append((start, off))
        self.names = [n for n, _ in named]

    def zero_(self):
        self.flat.zero_()

    def views_of(self, flat):
        """the per-parameter views of another flat tensor with this buffer's layout"""
        return {n: flat[v.storage_offset():v.storage_offset() + v.numel()].view(v.shape) for n, v in self.views.items()}

    def snapshot(self):
        """copy of the flat buffer (one kernel) + its per-parameter views; remembered as `last_snapshot`"""
        self.last_snapshot = self.flat.clone()
        return self.views_of(self.last_snapshot)

    def flat_of(self, params):
        """If every ``p.grad`` of `params` ({name: parameter}) is a view, at this buffer's offsets, of ONE flat fp32 tensor,
        return that tensor (autograd accumulates later backward passes into the first snapshot in place, so it then holds
        the summed gradient); otherwise None."""
        base = None
        for n, v in self.views.items():
            g = params[n].grad
            if g is None or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != v.shape:
                return None
            start = g.data_ptr() - 4 * v.storage_offset()
            if base is None:
                base = start
            elif start != base:
                return None
        snap = getattr(self, "last_snapshot", None)
        for cand in (snap, self.flat):
            if cand is not None and cand.data_ptr() == base:
                return cand
        # p.grad lives in an older snapshot (gradient accumulation over several backward passes): rebuild the flat view
        g0 = params[next(iter(self.views))].grad
        st = g0.untyped_storage()
        off = (base - st.data_ptr()) // 4
        if off < 0 or (off + self.flat.numel()) * 4 > st.nbytes():
            return None
        return torch.empty(0, dtype=torch.float32, device=g0.device).set_(st, off, (self.flat.numel(),))

    def __getitem__(self, name):
        return self.views[name]

    def section(self, i):
        a, b = self.bounds[i]
        return self.flat[a:b]


class GradSync:
    """Sum all-reduce of finished gradient sections on a side stream (NCCL over NVLink), overlapped with the rest of
    backward; `finish()` makes the compute stream wait for every reduction.  world_size 1: no-op."""

    def __init__(self, process_group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        self.stream = None
        self.pending = []

    def section_done(self, tensor):
        if self.world == 1 or tensor.numel() == 0:
            return
        if tensor.is_cuda:
            if self.stream is None:
                self.stream = torch.cuda.Stream(device=tensor.device)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self.stream.wait_event(ev)
            with torch.cuda.stream(self.stream):
                self.dist.all_reduce(tensor, op=self.dist.ReduceOp.AVG, group=self.group)      # NCCL averages in flight
            done = torch.cuda.Event()
            done.record(self.stream)
            self.pending.append(done)
        else:                                    # gloo / CPU tensors (host-logic tests): gloo has no AVG
            self.dist.all_reduce(tensor, op=self.dist.ReduceOp.SUM, group=self.group)
            tensor.div_(self.world)

    def finish(self):
        for ev in self.pending:
            torch.cuda.current_stream().wait_event(ev)
        self.pending = []


# ------------------------------------------------------------------------------------------------ weight packing
def _pack_dgrad3x3(w, dtype):
    """(Cout,Cin,3,3) -> [Cin][9*Cout] with K index tap*Cout + co (dX = conv^T: negated tap shifts)"""
    co, ci = w.shape[:2]
    out = torch.empty(ci, 3, 3, co, dtype=dtype, device=w.device)
    out.copy_(w.permute(1, 2, 3, 0))                             # permutation and conversion in one pass
    return out.view(ci, 9 * co)


def _unpack_wgrad3x3(dWt, co, ci_pad, ci):
    """[Cout][9*ci_pad] tap-major -> (Cout, ci, 3, 3)"""
    return dWt.view(co, 3, 3, ci_pad)[..., :ci].permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------ MaxViT block
def _attention_train_fwd(vit, x, film, P, reg_in, grid_mode, want_reg_out, drop=(0, 0, 0)):
    """shapes vit.fused_attn_applies accepts (mixed precision): the fused one-kernel attention, nothing but its inputs is
    kept (backward re-materialises tokens / qkv / att on the tensor cores); fp32 mode and every other shape: un-fused path,
    intermediates saved (its core applies the same dropout masks as the fused kernel)."""
    N, H, W, C = x.shape
    w, R = vit.vit_window_size, vit.num_register_tokens
    if vit.fused_attn_applies(C):
        x_out, reg_out = ops.attn_fused(x, reg_in, film, P["wqkv_h"], P["wout_h"], P["head_tab"], w, R, grid_mode, want_reg_out,
                                        vit.heads, vit.dim_head, drop=drop)
        return x_out, reg_out, dict(x=x, film=film, reg_in=reg_in, grid_mode=grid_mode, drop=drop)
    tokens = ops.attn_gather(x, reg_in, film, w, R, grid_mode)
    qkv = ops.gemm(tokens, P["w_qkv"], tf32=vit.tf32)
    att = ops.attn_core(qkv, P["q_gamma"], P["k_gamma"], P["bias_table"], N, H, W, w, R, vit.heads, vit.dim_head, drop=drop)
    x_out, reg_out = ops.attn_out(att, P["w_out"], x, reg_in, w, R, grid_mode, want_reg_out, tf32=vit.tf32, drop=drop)
    return x_out, reg_out, dict(x=x, film=film, reg_in=reg_in, tokens=tokens, qkv=qkv, att=att, grid_mode=grid_mode, drop=drop)


def _attention_train_bwd(vit, sv, P, att_mod, pre, G, cond, dcond, dx_out, dreg_res, reg_scale, dreg_in):
    """-> dx_in.  dreg_in: accumulation target for the register-token input gradient ((R,C) param grad or (N,R,C)).
    Mixed precision (forward = the fused kernel): tokens, qkv, dproj, datt, dqkv and att -- everything between the fp32 residual
    stream and the fp32 gradients -- are re-materialised and kept in bf16 (kind::f16 GEMMs, half the HBM bytes)."""
    x = sv["x"]
    N, H, W, C = x.shape
    w, R = vit.vit_window_size, vit.num_register_tokens
    tf32 = vit.tf32
    gm = sv["grid_mode"]
    recompute = "qkv" not in sv
    lo = recompute and tf32                       # 16-bit backward chain
    if recompute:
        tokens = ops.attn_gather(x, sv["reg_in"], sv["film"], w, R, gm, out_bf16=lo)
        qkv = ops.gemm(tokens, P["w_qkv_bf16"] if lo else P["w_qkv"], tf32=tf32 and not lo)
    else:
        tokens, qkv = sv["tokens"], sv["qkv"]
    drop = sv["drop"]
    dproj = ot.attn_out_bwd_gather(dx_out, dreg_res, reg_scale, w, R, gm, drop=drop, out_bf16=lo)
    datt = ops.gemm(dproj, P["w_out_t_bf16"] if lo else P["w_out_t"], tf32=tf32 and not lo)
    res = ot.attn_core_bwd(qkv, datt, P["q_gamma"], P["k_gamma"], P["bias_table"], N, H, W, w, R, vit.heads, vit.dim_head,
                           G[pre + "q_norm.gamma"], G[pre + "k_norm.gamma"], G[pre + "rel_pos_bias.weight"], tf32=tf32,
                           want_att=recompute, drop=drop)
    dqkv, att = res if recompute else (res, sv["att"])
    del datt, qkv
    ot.wgrad(dproj, att, G[pre + "to_out.0.weight"], tf32=tf32 and not lo)
    del dproj, att
    ot.wgrad(dqkv, tokens, G[pre + "to_qkv.weight"], tf32=tf32 and not lo)
    dtok = ops.gemm(dqkv, P["w_qkv_t_bf16"] if lo else P["w_qkv_t"], tf32=tf32 and not lo, out_f32=True)
    del dqkv, tokens
    dfilm = torch.zeros(N, 2 * C, dtype=torch.float32, device=x.device)
    dx_in = ot.attn_gather_bwd(x, sv["reg_in"], sv["film"], dtok, dx_out, dreg_res, reg_scale, dreg_in, dfilm, w, R, gm)
    ot.cond_mlp_bwd(cond, P["film_w0"], P["film_b0"], P["film_w1"], dfilm, G[pre + "film.0.weight"], G[pre + "film.0.bias"],
                    G[pre + "film.2.weight"], G[pre + "film.2.bias"], dcond)
    return dx_in


def dropout_threshold(p: float) -> int:
    """drop probability -> mask-byte threshold T (p_eff = T/256)"""
    return max(0, min(255, int(round(p * 256))))


def _bn_stats(bn, raw, frozen):
    if frozen:
        return ot.bn_frozen_stats(bn)
    return ot.bn_stats(raw, bn.weight, bn.bias, bn.eps, bn.momentum, bn.running_mean, bn.running_var)


def _bn_bwd(dOut, raw, st, bn, act, dgamma, dbeta, frozen, **kw):
    if frozen:
        return ot.bn_bwd_frozen(dOut, raw, st, act, dgamma, dbeta, **kw)
    return ot.bn_bwd(dOut, raw, st, bn.weight, act, dgamma, dbeta, **kw)


def maxvit_train_forward(vit, x, cond, seed=0, frozen=False):
    """x CL (N,H,W,C) fp32, cond (N,cd) -> (y, saved).  seed: dropout seed of this step (ignored when dropout is 0).
    frozen: the eval-mode graph -- BatchNorm from its running statistics (nothing updated), no dropout.  The first layer of a
    stage of a tuple-depth MaxViT widens the map: its MBConv maps C_in -> C_out and everything after it runs at C_out."""
    N, H, W, _ = x.shape
    w = vit.vit_window_size
    nwin = (H // w) * (W // w)
    M = N * H * W
    tf32 = vit.tf32
    saved = []
    for li, (P, (conv, battn, gattn)) in enumerate(zip(vit.packed(x.dtype), vit.layers)):
        seq = conv.fn if isinstance(conv, MBConvResidual) else conv
        x2d = x.view(M, x.shape[3])
        bn1, bn2, bn3 = seq[1], seq[4], seq[8]
        h0 = ops.gemm(x2d, P["w_exp"], bias=P["b_exp"], tf32=tf32)
        hid = h0.shape[1]
        st1 = _bn_stats(bn1, h0, frozen)
        h1 = ot.bn_act(h0, st1, 1)
        h2, _ = ot.dw3x3(h1.view(N, H, W, hid), P["w_dw"], P["ones_hid"], P["b_dw"], 0)
        st2 = _bn_stats(bn2, h2.view(M, hid), frozen)
        h3 = ot.bn_act(h2.view(M, hid), st2, 1).view(N, H, W, hid)
        gate, mean, hidv = ot.se_gate_train(ot.field_sum(h3), H * W, P["se_w1"], P["se_w2"])
        h4 = ot.se_scale_oop(h3, gate)
        y0 = ops.gemm(h4.view(M, hid), P["w_proj"], bias=P["b_proj"], tf32=tf32)
        st3 = _bn_stats(bn3, y0, frozen)
        y = ot.bn_act(y0, st3, 0, res=x2d if P["residual"] else None).view(N, H, W, y0.shape[1])
        if not frozen:
            for bn in (bn1, bn2, bn3):
                bn.num_batches_tracked += 1
        sv = dict(x=x, h0=h0, st1=st1, h1=h1, h2=h2, st2=st2, h3=h3, gate=gate, mean=mean, hidv=hidv, h4=h4, y0=y0, st3=st3,
                  frozen=frozen)
        fb = P["block"]
        film_b = ops.cond_mlp(cond, fb["film_w0"], fb["film_b0"], fb["film_w1"], fb["film_b1"])
        T = 0 if frozen else dropout_threshold(battn.dropout_p)
        xb, reg_out, sv["battn"] = _attention_train_fwd(vit, y, film_b, fb, P["reg"], False, True, drop=(seed, 2 * li, T))
        reg = ops.reg_mean(reg_out, N, nwin)
        fg = P["grid"]
        film_g = ops.cond_mlp(cond, fg["film_w0"], fg["film_b0"], fg["film_w1"], fg["film_b1"])
        x, _, sv["gattn"] = _attention_train_fwd(vit, xb, film_g, fg, reg, True, False, drop=(seed, 2 * li + 1, T))
        saved.append(sv)
    return x, saved


def maxvit_train_backward(vit, saved, cond, dcond, dx, G, prefix):
    """dx: gradient wrt the MaxViT output, CL (N,H,W,C) fp32 -> gradient wrt its input"""
    packed = vit.packed(dx.dtype)
    w, R = vit.vit_window_size, vit.num_register_tokens
    tf32 = vit.tf32
    for li in reversed(range(len(vit.layers))):
        P, sv = packed[li], saved[li]
        conv, battn, gattn = vit.layers[li]
        seq = conv.fn if isinstance(conv, MBConvResidual) else conv
        pm = f"{prefix}layers.{li}.0." + ("fn." if isinstance(conv, MBConvResidual) else "")
        x = sv["x"]
        N, H, W, C = x.shape                              # MBConv input width; the attention runs at the output width C_out
        C_out = dx.shape[3]
        nwin = (H // w) * (W // w)
        M = N * H * W
        hid = sv["h0"].shape[1]
        # ---- grid attention, then block attention (register tokens link the two, maxvit.py:326)
        dreg_mean = torch.zeros(N, R, C_out, dtype=torch.float32, device=dx.device)
        dx = _attention_train_bwd(vit, sv["gattn"], P["grid"], gattn, f"{prefix}layers.{li}.2.", G, cond, dcond, dx, None, 0.0,
                                  dreg_mean)
        dx = _attention_train_bwd(vit, sv["battn"], P["block"], battn, f"{prefix}layers.{li}.1.", G, cond, dcond, dx, dreg_mean,
                                  1.0 / nwin, G[f"{prefix}register_tokens.{li}"])
        # ---- MBConv
        dy = dx.view(M, C_out)
        bn1, bn2, bn3 = seq[1], seq[4], seq[8]
        fz = sv["frozen"]
        dy0 = _bn_bwd(dy, sv["y0"], sv["st3"], bn3, 0, G[pm + "8.weight"], G[pm + "8.bias"], fz)
        ot.colsum(dy0, G[pm + "7.bias"])
        ot.wgrad(dy0, sv["h4"].view(M, hid), G[pm + "7.weight"], tf32=tf32)
        dh4 = ops.gemm(dy0, seq[7].weight.detach().flatten(1).t().contiguous(), tf32=tf32)
        del dy0
        dmean = ot.se_bwd(dh4, sv["h3"], sv["gate"], sv["mean"], sv["hidv"], P["se_w1"], P["se_w2"], G[pm + "6.gate.1.weight"],
                          G[pm + "6.gate.3.weight"])
        dh2 = _bn_bwd(dh4, sv["h2"].view(M, hid), sv["st2"], bn2, 1, G[pm + "4.weight"], G[pm + "4.bias"], fz,
                      fgate=sv["gate"], fadd=dmean, rows_per_field=H * W, out=dh4)
        dw9 = torch.zeros(9, hid, dtype=torch.float32, device=dx.device)
        ot.dw3x3_wgrad(sv["h1"].view(N, H, W, hid), dh2.view(N, H, W, hid), dw9, G[pm + "3.bias"])
        G[pm + "3.weight"].view(hid, 9).add_(dw9.t())
        dh1, _ = ot.dw3x3(dh2.view(N, H, W, hid), P["w_dw_flip"], P["ones_hid"], P["zeros_hid"], 0)
        del dh2, dh4
        dh0 = _bn_bwd(dh1.view(M, hid), sv["h0"], sv["st1"], bn1, 1, G[pm + "1.weight"], G[pm + "1.bias"], fz, out=dh1.view(M, hid))
        ot.colsum(dh0, G[pm + "0.bias"])
        ot.wgrad(dh0, x.view(M, C), G[pm + "0.weight"], tf32=tf32)
        dx = ops.gemm(dh0, seq[0].weight.detach().flatten(1).t().contiguous(), res=dy if P["residual"] else None,
                      tf32=tf32).view(N, H, W, C)
        del dh0, dh1
    return dx


class MaxViTTrainFn(torch.autograd.Function):
    """autograd node of a stand-alone ``MaxViT`` in train() mode (maxvit.py:289-341 under autograd): x CL (N,H,W,C) fp32,
    cond (N,cond_dim) -> y CL; backward returns the gradients of x, cond and every parameter.  frozen: the eval-mode graph
    (running-statistic BatchNorm, no dropout, the dropout seed not advanced)."""

    @staticmethod
    def forward(ctx, vit, x, cond, frozen, *params):
        y, saved = maxvit_train_forward(vit, x, cond, seed=0 if frozen else vit.next_dropout_seed(), frozen=frozen)
        ctx.vit, ctx.saved, ctx.cond = vit, saved, cond
        return y

    @staticmethod
    def backward(ctx, dy):
        vit = ctx.vit
        if ctx.saved is None:
            raise RuntimeError("MaxViT backward ran twice through the same forward (retain_graph is not supported)")
        named = list(vit.named_parameters())
        G = {n: torch.zeros(p.shape, dtype=torch.float32, device=p.device) for n, p in named}
        dcond = torch.zeros_like(ctx.cond)
        with torch.cuda.device(dy.device):
            dx = maxvit_train_backward(vit, ctx.saved, ctx.cond, dcond, dy.float().contiguous(), G, "")
        ctx.saved = None
        return (None, dx, dcond, None, *[G[n] for n, _ in named])


# ------------------------------------------------------------------------------------------------ MetNet3
def _resblock_train_fwd(x, skip, cond, d, N, HP, WP, mixed):
    """128->128 ResnetBlock.  x: conv input (compute dtype); skip: the same tensor as the residual operand (fp32 copy in
    mixed mode).  -> (out, out_fp32_copy or None, saved)"""
    dtype, dev = x.dtype, x.device
    film = ops.cond_mlp(cond, d["mlp_w"], d["mlp_b"], pre_relu=True)
    t1 = ops.pg_empty(N, HP, WP, 128, dtype, dev)
    _, sv1 = ot.conv3x3_ln_train(x, d["w1"], d["b1"], d["g1"], d["be1"], d["eps1"], film, None, t1, N, HP, WP)
    out = ops.pg_empty(N, HP, WP, 128, dtype, dev)
    copy = ops.pg_empty(N, HP, WP, 128, torch.float32, dev) if mixed else None
    _, sv2 = ot.conv3x3_ln_train(t1, d["w2"], d["b2"], d["g2"], d["be2"], d["eps2"], None, skip, out, N, HP, WP, out_copy=copy)
    return out, copy, dict(x=x, t1=t1, sv1=sv1, sv2=sv2, film=film)


def _block_bwd(dY, sv, conv_in, blk, d, which, film, G, pre, N, HP, WP, dtype, shifts, want_dfilm):
    """backward of one Block up to (and including) its weight gradient; returns dconv (GEMM dtype) and dfilm"""
    g, be, eps = d["g" + which], d["be" + which], d["eps" + which]
    dconv, sums, _ = ot.conv_ln_bwd(dY, sv, g, film, eps, N, HP, WP, dtype)
    name = pre + ("block1." if which == "1" else "block2.")
    dfilm = ot.conv_ln_param_grads(sums, N, g, be, film, G[name + "norm.g"].view(-1), G[name + "norm.b"].view(-1),
                                   G[name + "proj.bias"], want_dfilm)
    dWt = torch.empty(128, 9 * 128, dtype=torch.float32, device=dY.device)
    ot.wgrad(dconv, conv_in, dWt, ntaps=9, tap_shift=shifts, beta=0.0)
    G[name + "proj.weight"].add_(_unpack_wgrad3x3(dWt, 128, 128, 128))
    return dconv, dfilm


def _resblock_train_bwd(dOut, sv, blk, d, G, pre, cond, dcond, N, HP, WP, dtype, shifts, nshifts):
    dconv2, _ = _block_bwd(dOut, sv["sv2"], sv["t1"], blk, d, "2", None, G, pre, N, HP, WP, dtype, shifts, False)
    dt1 = ops.gemm(dconv2, _pack_dgrad3x3(blk.block2.proj.weight.detach(), dtype), ntaps=9, tap_shift=nshifts, out_f32=True)
    del dconv2
    dconv1, dfilm = _block_bwd(dt1, sv["sv1"], sv["x"], blk, d, "1", sv["film"], G, pre, N, HP, WP, dtype, shifts, True)
    del dt1
    dx = ops.gemm(dconv1, _pack_dgrad3x3(blk.block1.proj.weight.detach(), dtype), ntaps=9, tap_shift=nshifts, res=dOut, out_f32=True)
    ot.cond_mlp_bwd(cond, d["mlp_w"], None, None, dfilm, G[pre + "mlp.1.weight"], G[pre + "mlp.1.bias"], None, None, dcond,
                    pre_relu=True)
    return dx


def metnet3_train_forward(model, x, ts, frozen=False):
    """-> (pred (B,L,H,W) fp32, saved).  frozen: the eval-mode graph (MaxViT BatchNorm from its running statistics, nothing
    updated, no dropout, the dropout seed not advanced)"""
    B = x.shape[0]
    L, C = model.end_lead_time, model.n_start_channels
    N = B * L
    HP = model.input_height + (14 - model.input_height) % 14
    WP = model.input_width + (14 - model.input_width) % 14
    pads = model.pad_values()
    dtype = model.compute_dtype
    dev = x.device
    mixed = dtype != torch.float32
    P = model.packed(dtype)
    et = P["emb_time"]
    s0 = P["resnet1"][0]
    temb, cond, tt, tres = ops.time_terms(ts, B, L, P["emb_lead"], et[0], et[1], et[2], s0["w1_orig"], s0["wres_orig"],
                                          model.n_input_channels, C)
    S = dict(B=B, N=N, HP=HP, WP=WP, ts=ts, temb=temb, cond=cond)
    # ---- stem, once per sample
    xin = ops.prepare(x, pads, HP, WP, P["c_pad"], model.pm25_mean, model.pm25_std, dtype)
    raw3 = ops.gemm(xin, s0["w1"], ntaps=9, tap_shift=ops.conv_tap_shifts(WP), out_f32=True)
    rawres = ops.gemm(xin, s0["wres"], out_f32=True)
    film0 = ops.cond_mlp(cond, s0["mlp_w"], s0["mlp_b"], pre_relu=True)
    h1 = ops.pg_empty(N, HP, WP, C, dtype, dev)
    skip0 = ops.pg_empty(N, HP, WP, C, torch.float32, dev)
    sv_stem = ot.stem_finish_train(raw3, rawres, s0["b1"], s0["bres"], tt, tres, s0["g1"], s0["be1"], s0["eps1"], film0, B, L,
                                   HP, WP, h1, skip0)
    del raw3, rawres
    h = ops.pg_empty(N, HP, WP, C, dtype, dev)
    hs = ops.pg_empty(N, HP, WP, C, torch.float32, dev) if mixed else None
    _, sv_b2 = ot.conv3x3_ln_train(h1, s0["w2"], s0["b2"], s0["g2"], s0["be2"], s0["eps2"], None, skip0, h, N, HP, WP, out_copy=hs)
    del skip0
    S["stem"] = dict(xin=xin, film=film0, h1=h1, sv1=sv_stem, sv2=sv_b2)
    enc = []
    for d in P["resnet1"][1:]:
        h, hs, sv = _resblock_train_fwd(h, hs if mixed else h, cond, d, N, HP, WP, mixed)
        enc.append(sv)
    S["enc"], S["h_enc"] = enc, h
    # ---- MaxViT at half resolution
    low = ops.pool2(h, N, HP, WP, out_dtype=model.vit.compute_dtype)
    low, S["vit"] = maxvit_train_forward(model.vit, low, cond, seed=0 if frozen else model.next_dropout_seed(), frozen=frozen)
    S["low_out"] = low
    # ---- decoder
    up = torch.zeros(ops.pg_pixels(N, HP, WP), C, dtype=dtype, device=dev)
    ups = ops.pg_empty(N, HP, WP, C, torch.float32, dev) if mixed else None
    ops.convT2(low, P["w_up_vit"], P["b_up"], up, tf32=model.vit.tf32, out_copy=ups)
    h, hs = up, ups
    dec = []
    for d in P["resnet2"]:
        h, hs, sv = _resblock_train_fwd(h, hs if mixed else h, cond, d, N, HP, WP, mixed)
        dec.append(sv)
    S["dec"], S["h_last"] = dec, h
    pred = torch.empty(B, L, model.input_height, model.input_width, dtype=torch.float32, device=dev)
    ops.head(h, P["w_head"], P["b_head"], model.pm25_std, model.pm25_mean, N, HP, WP, model.input_height, model.input_width,
             pads, out=pred.view(N, model.input_height, model.input_width))
    return pred, S


def metnet3_train_backward(model, S, dpred, G: GradBuffer, sync: GradSync | None = None, want_dx=False):
    """dpred (B,L,H,W) fp32 -> fills G (parameter gradients, accumulated into the zeroed flat buffer); want_dx: also returns
    the gradient with respect to the input grids x (B,T,C,H,W) fp32 (else None)"""
    B, N, HP, WP = S["B"], S["N"], S["HP"], S["WP"]
    L, C = model.end_lead_time, model.n_start_channels
    dtype = model.compute_dtype
    vdt = model.vit.compute_dtype
    dev = dpred.device
    pads = model.pad_values()
    P = model.packed(dtype)
    cond = S["cond"]
    shifts = ops.conv_tap_shifts(WP)
    nshifts = tuple(-s for s in shifts)
    dcond = torch.zeros_like(cond)
    done = (lambda i: sync.section_done(G.section(i))) if sync is not None else (lambda i: None)

    # ---- head
    dH = ot.head_bwd(dpred.contiguous().view(N, model.input_height, model.input_width), S["h_last"], P["w_head"], model.pm25_std,
                     N, HP, WP, model.input_height, model.input_width, pads, G["classifier_pm25.weight"].view(-1),
                     G["classifier_pm25.bias"])
    done(0)
    # ---- decoder
    for k in reversed(range(len(model.resnet2.blocks))):
        dH = _resblock_train_bwd(dH, S["dec"][k], model.resnet2.blocks[k], P["resnet2"][k], G, f"resnet2.blocks.{k}.", cond, dcond,
                                 N, HP, WP, dtype, shifts, nshifts)
    done(1)
    # ---- ConvTranspose (metnet3.py:88-89)
    Hl, Wl = HP // 2, WP // 2
    Gm = ot.convT2_bwd_gather(dH, N, Hl, Wl, C, vdt, G["up.bias"])
    del dH
    low_out = S["low_out"].view(N * Hl * Wl, C)
    dWt = torch.empty(4 * C, C, dtype=torch.float32, device=dev)
    ot.wgrad(Gm, low_out, dWt, beta=0.0, tf32=model.vit.tf32)
    G["up.weight"].add_(dWt.view(2, 2, C, C).permute(3, 2, 0, 1))                 # [(di,dj,co)][ci] -> (ci, co, di, dj)
    dlow = ops.gemm(Gm, model.up.weight.detach().permute(0, 2, 3, 1).reshape(C, 4 * C).to(vdt).contiguous(), tf32=model.vit.tf32)
    del Gm
    done(2)
    # ---- MaxViT
    dlow = maxvit_train_backward(model.vit, S["vit"], cond, dcond, dlow.view(N, Hl, Wl, C), G, "vit.")
    done(3)
    # ---- encoder
    dH = ot.pool2_bwd(S["h_enc"], dlow, N, HP, WP)
    del dlow
    for k in reversed(range(1, len(model.resnet1.blocks))):
        dH = _resblock_train_bwd(dH, S["enc"][k - 1], model.resnet1.blocks[k], P["resnet1"][k], G, f"resnet1.blocks.{k}.", cond,
                                 dcond, N, HP, WP, dtype, shifts, nshifts)
    # ---- stem block (lead-time dedup): block2 is an ordinary Block, block1 / res_conv run per sample
    st, s0, blk0 = S["stem"], P["resnet1"][0], model.resnet1.blocks[0]
    pre = "resnet1.blocks.0."
    dconv2, _ = _block_bwd(dH, st["sv2"], st["h1"], blk0, s0, "2", None, G, pre, N, HP, WP, dtype, shifts, False)
    dh1 = ops.gemm(dconv2, _pack_dgrad3x3(blk0.block2.proj.weight.detach(), dtype), ntaps=9, tap_shift=nshifts, out_f32=True)
    del dconv2
    dconv1, sums, border = ot.conv_ln_bwd(dh1, st["sv1"], s0["g1"], st["film"], s0["eps1"], N, HP, WP, torch.float32, want_border=True)
    del dh1
    dfilm = ot.conv_ln_param_grads(sums, N, s0["g1"], s0["be1"], st["film"], G[pre + "block1.norm.g"].view(-1),
                                   G[pre + "block1.norm.b"].view(-1), G[pre + "block1.proj.bias"], True)
    ot.cond_mlp_bwd(cond, s0["mlp_w"], None, None, dfilm, G[pre + "mlp.1.weight"], G[pre + "mlp.1.bias"], None, None, dcond,
                    pre_relu=True)
    c_data, c_pad = model.n_input_channels, P["c_pad"]
    draw3 = ot.lead_sum(dconv1, B, L, HP, WP, dtype)
    del dconv1
    dWt = torch.empty(C, 9 * c_pad, dtype=torch.float32, device=dev)
    ot.wgrad(draw3, st["xin"], dWt, ntaps=9, tap_shift=shifts, beta=0.0)
    gw3 = G[pre + "block1.proj.weight"]
    gw3[:, :c_data].add_(_unpack_wgrad3x3(dWt, C, c_pad, c_data))
    del dWt
    if want_dx:
        # data gradient of the per-sample stem: 3x3 conv^T over the data channels (negated tap shifts), c_pad outputs
        w3t = torch.zeros(c_pad, 9 * C, dtype=dtype, device=dev)
        w3t[:c_data] = _pack_dgrad3x3(blk0.block1.proj.weight.detach()[:, :c_data], dtype)
        dxin = ops.gemm(draw3, w3t, ntaps=9, tap_shift=nshifts, out_f32=True)
        del w3t
    del draw3
    dres = ot.lead_sum(dH, B, L, HP, WP, dtype)
    dWr = torch.empty(C, c_pad, dtype=torch.float32, device=dev)
    ot.wgrad(dres, st["xin"], dWr, beta=0.0)
    dx = None
    if want_dx:
        # + res_conv^T, accumulated in the GEMM epilogue (each element is read and written by the same thread)
        wrt = torch.zeros(c_pad, C, dtype=dtype, device=dev)
        wrt[:c_data] = blk0.res_conv.weight.detach()[:, :c_data, 0, 0].t()
        ops.gemm(dres, wrt, res=dxin, out=dxin, out_f32=True)
        del wrt
        dx = ot.prepare_bwd(dxin, B, model.window_size, model.n_variables, model.input_height, model.input_width, pads, HP, WP,
                            model.pm25_std, model.standardised_extra_channel)
        del dxin
    gw1 = G[pre + "res_conv.weight"]
    gw1.view(C, -1)[:, :c_data].add_(dWr[:, :c_data])
    tres_sum = ot.pg_field_sum(dH, N, HP, WP)
    dtemb = ot.time_terms_bwd(border, sums[2], tres_sum, S["temb"], s0["w1_orig"], s0["wres_orig"], c_data, gw3, gw1,
                              G[pre + "res_conv.bias"])
    done(4)
    # ---- embeddings
    ot.time_embed_bwd(dtemb, dcond, S["ts"], B, L, model.lead_time_emb_dim, model.model_time_emb_dim,
                      G["condition_lead_time.weight"], G["condition_model_time.0.weight"], G["condition_model_time.1.weight"],
                      G["condition_model_time.2.weight"])
    done(5)
    if sync is not None:
        sync.finish()
    return dx


class MetNet3TrainFn(torch.autograd.Function):
    """autograd node of the whole network: forward = train-mode forward on libvitgrid kernels, backward = hand-written
    backward.  The backward kernels accumulate into the model's flat GradBuffer (all-reduced in place when the model is wrapped
    in `DataParallel`); what autograd receives are views of a SNAPSHOT of that buffer (one device copy of 13 MB), so that
    several applications of the model inside one graph -- two forwards summed into one loss, micro-batches sharing one
    backward -- accumulate correctly in ``p.grad`` instead of overwriting each other through the shared buffer.  The
    snapshot keeps GradBuffer's layout: ``FlatAdamW`` consumes ``p.grad`` in place when it is still such a view."""

    @staticmethod
    def forward(ctx, model, x, ts, frozen, *params):
        pred, S = metnet3_train_forward(model, x, ts, frozen=frozen)
        ctx.model, ctx.S = model, S
        return pred

    @staticmethod
    def backward(ctx, dpred):
        model = ctx.model
        if ctx.S is None:
            raise RuntimeError("MetNet3 backward ran twice through the same forward: the saved activations are released after "
                               "the first backward (retain_graph is not supported); call the model again")
        G = model.grad_buffer()
        G.zero_()
        with torch.cuda.device(dpred.device):
            dx = metnet3_train_backward(model, ctx.S, dpred.float(), G, model._grad_sync, want_dx=ctx.needs_input_grad[1])
        ctx.S = None
        snap = G.snapshot()
        return (None, dx, None, None, *[snap[n] for n in G.names])
