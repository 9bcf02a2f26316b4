"""MaxViT backbone with the reference's nn.Module API (/root/reference/src/maxvit.py:224-341) on libvitgrid kernels.

Same constructor arguments, parameter names and shapes as the reference ``MaxViT`` so reference state dicts load
unchanged.  The sub-modules below are *parameter holders* laid out to reproduce the reference's state-dict keys
(e.g. ``layers.0.0.3.weight`` = depthwise conv, ``layers.0.1.to_qkv.weight``); the computation is the fused
pipeline in ``MaxViT.forward_cl``:

  MBConv  : 1x1 GEMM + BN + GELU  ->  depthwise 3x3 + BN + GELU (+SE row sums)  ->  SE gate, scale  ->  1x1 GEMM + BN (+x)
  attention (block, then grid): gather+LN+FiLM -> QKV GEMM -> per-(window,head) core -> out-proj GEMM whose
            epilogue adds the residual and scatters through the inverse partition map.

This file holds the eval-mode forward (BatchNorm uses running statistics, dropout is identity); the train-mode
forward / backward (batch statistics, saved activations) is in train.py.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib, ops


class RMSNorm(nn.Module):
    """holder for q/k norm gamma (maxvit.py:18-30)"""

    def __init__(self, dim, *, heads):
        super().__init__()
        self.scale = dim ** 0.5
        self.gamma = nn.Parameter(torch.ones(heads, 1, dim))


class SqueezeExcitation(nn.Module):
    """holder: gate.1 = Linear(dim, hidden), gate.3 = Linear(hidden, dim) (maxvit.py:33-48)"""

    def __init__(self, dim, shrinkage_rate=0.25):
        super().__init__()
        hidden = int(dim * shrinkage_rate)
        self.gate = nn.Sequential(nn.Identity(), nn.Linear(dim, hidden, bias=False), nn.ReLU(),
                                  nn.Linear(hidden, dim, bias=False), nn.Sigmoid(), nn.Identity())


class MBConvResidual(nn.Module):
    """holder that reproduces the ``.fn.`` key level of residual MBConv blocks (maxvit.py:50-59)"""

    def __init__(self, fn):
        super().__init__()
        self.fn = fn


def MBConv(dim_in, dim_out, *, downsample, expansion_rate=4, shrinkage_rate=0.25):
    hidden = int(expansion_rate * dim_out)
    net = nn.Sequential(
        nn.Conv2d(dim_in, hidden, 1), nn.BatchNorm2d(hidden), nn.GELU(),
        nn.Conv2d(hidden, hidden, 3, padding=1, groups=hidden), nn.BatchNorm2d(hidden), nn.GELU(),
        SqueezeExcitation(hidden, shrinkage_rate=shrinkage_rate),
        nn.Conv2d(hidden, dim_out, 1), nn.BatchNorm2d(dim_out))
    # the first layer of a stage has no residual even though it never downsamples (maxvit.py:85,99-100,270)
    if dim_in == dim_out and not downsample:
        net = MBConvResidual(net)
    return net


def rel_pos_indices(window_size: int, num_registers: int) -> torch.Tensor:
    """closed form of maxvit.py:156-168 (bit-exact, tests/test_indices.py)"""
    w, r = window_size, num_registers
    s = r + w * w
    idx = torch.full((s, s), (2 * w - 1) ** 2, dtype=torch.int64)
    t = torch.arange(w * w)
    a, b = t // w, t % w
    idx[r:, r:] = (a[:, None] - a[None, :] + w - 1) * (2 * w - 1) + (b[:, None] - b[None, :] + w - 1)
    return idx


class Attention(nn.Module):
    """One window / grid attention (maxvit.py:106-219).  Inside ``MaxViT`` it is a parameter holder -- the partition, the
    register tokens and the residual are fused around it (``MaxViT.forward_cl``).  Called on its own it has the reference's
    ``forward(x, cond)``: x (Nw, num_registers + window_size^2, dim) token sequences -> to_out(attention(x)) without the
    residual; ``cond_dim=None`` gives the un-conditioned variant (LayerNorm with affine, no FiLM, maxvit.py:128-137)."""

    def __init__(self, dim, cond_dim=None, heads=32, dim_head=32, dropout=0., window_size=8, num_registers=1):
        super().__init__()
        assert num_registers > 0
        assert (dim % dim_head) == 0, 'dimension should be divisible by dimension per head'
        inner = dim_head * heads
        self.dim, self.heads, self.dim_head = dim, heads, dim_head
        self.window_size, self.num_registers, self.dropout_p = window_size, num_registers, dropout
        self.has_cond = cond_dim is not None
        self.film = None
        if self.has_cond:
            self.film = nn.Sequential(nn.Linear(cond_dim, dim * 2), nn.SiLU(), nn.Linear(dim * 2, dim * 2), nn.Identity())
        self.norm = nn.LayerNorm(dim, elementwise_affine=not self.has_cond)
        self.to_qkv = nn.Linear(dim, inner * 3, bias=False)
        self.q_norm = RMSNorm(dim_head, heads=heads)
        self.k_norm = RMSNorm(dim_head, heads=heads)
        self.to_out = nn.Sequential(nn.Linear(inner, dim, bias=False), nn.Dropout(dropout))
        self.rel_pos_bias = nn.Embedding((2 * window_size - 1) ** 2 + 1, heads)
        self.register_buffer('rel_pos_indices', rel_pos_indices(window_size, num_registers), persistent=False)

    @torch.no_grad()
    def forward(self, x, cond=None):
        """reference signature (maxvit.py:170): x (Nw, S, dim), cond (b, cond_dim) with Nw a multiple of b (window sequences
        field-major, as ``MaxViT`` packs them).  Inference only (eval mode, or dropout 0): the training path of the package is
        ``MetNet3`` / ``MaxViT`` in train() mode."""
        _lib.require_device()
        if not x.is_cuda:
            raise _lib.VitGridError("vit_grid_model_b200 runs on a CUDA (sm_100a) device only; there is no CPU fallback")
        if self.training and self.dropout_p > 0:
            raise NotImplementedError("stand-alone Attention.forward is the inference path; train through MaxViT / MetNet3")
        Nw, S, D = x.shape
        w, R = self.window_size, self.num_registers
        assert S == R + w * w and D == self.dim
        if D % 128 or D > 512:
            raise NotImplementedError("the attention kernels are built for dim = 128, 256, 384, 512")
        x = x.float().contiguous()
        if self.has_cond:
            assert cond is not None and Nw % cond.shape[0] == 0
            f = self.film
            gb = ops.cond_mlp(cond.float().contiguous(), f[0].weight.float().contiguous(), f[0].bias.float().contiguous(),
                              f[2].weight.float().contiguous(), f[2].bias.float().contiguous())
            film = gb.repeat_interleave(Nw // cond.shape[0], dim=0).contiguous()          # one FiLM row per window
        else:                                                    # LayerNorm affine == FiLM with (weight, bias) for every window
            film = torch.cat([self.norm.weight, self.norm.bias]).float().expand(Nw, 2 * D).contiguous()
        # every window sequence as a one-window "field": the gather kernel's block partition of a (w x w) map is the identity
        tokens = ops.attn_gather(x[:, R:].reshape(Nw, w, w, D).contiguous(), x[:, :R].contiguous(), film, w, R, False,
                                 eps=self.norm.eps)
        qkv = ops.gemm(tokens, self.to_qkv.weight.float().contiguous())
        att = ops.attn_core(qkv, self.q_norm.gamma.float().reshape(-1).contiguous(), self.k_norm.gamma.float().reshape(-1).contiguous(),
                            self.rel_pos_bias.weight.float().contiguous(), Nw, w, w, w, R, self.heads, self.dim_head)
        return ops.gemm(att, self.to_out[0].weight.float().contiguous()).view(Nw, S, D)


def _fold_bn(conv_bias, bn: nn.BatchNorm2d):
    """eval BatchNorm after a conv with bias -> per-channel (scale, shift) in fp32"""
    scale = bn.weight.float() / torch.sqrt(bn.running_var.float() + bn.eps)
    shift = bn.bias.float() - bn.running_mean.float() * scale + conv_bias.float() * scale
    return scale.contiguous(), shift.contiguous()


class MaxViT(nn.Module):
    def __init__(self, dim, depth, cond_dim=32, heads=32, dim_head=32, vit_window_size=8, mbconv_expansion_rate=4,
                 mbconv_shrinkage_rate=0.25, dropout=0.1, num_register_tokens=4):
        super().__init__()
        depth = (depth,) if isinstance(depth, int) else tuple(depth)
        assert num_register_tokens > 0
        self.cond_dim = cond_dim
        self.dim, self.heads, self.dim_head = dim, heads, dim_head
        self.vit_window_size = vit_window_size
        self.num_register_tokens = num_register_tokens
        self.layers = nn.ModuleList([])
        self.register_tokens = nn.ParameterList([])
        # Stage widths dim, 2 dim, 4 dim, ...: stage k maps width 2^k dim -> 2^(k+1) dim in its first layer.  The reference
        # pairs the (in, out) widths with `depth` through zip(), which drops the LAST depth entry: a tuple of n entries builds
        # n - 1 stages (maxvit.py:240-251, quirk Q9); an int builds one stage of constant width.
        widths = [dim * 2 ** i for i in range(len(depth))]
        stages = list(zip(widths[:-1], widths[1:])) if len(depth) > 1 else [(dim, dim)]
        for (w_in, w_out), n_layers in zip(stages, depth):
            for k in range(n_layers):
                conv = MBConv(w_in if k == 0 else w_out, w_out, downsample=(k == 0), expansion_rate=mbconv_expansion_rate,
                              shrinkage_rate=mbconv_shrinkage_rate)
                kw = dict(dim=w_out, cond_dim=cond_dim, heads=heads, dim_head=dim_head, dropout=dropout,
                          window_size=vit_window_size, num_registers=num_register_tokens)
                self.layers.append(nn.ModuleList([conv, Attention(**kw), Attention(**kw)]))
                self.register_tokens.append(nn.Parameter(torch.randn(num_register_tokens, w_out)))
        self.dim_out = stages[-1][1] if len(self.layers) else dim
        if cond_dim is None:
            raise NotImplementedError("MaxViT needs cond_dim: the reference's forward asserts cond.shape == (b, cond_dim) (maxvit.py:290)")
        self.set_precision("bf16")
        self._packed = None
        self._packed_key = None
        self._capture = None

    # ------------------------------------------------------------------ weights -> kernel layouts
    def set_precision(self, precision: str):
        """'bf16'     : fp32 storage, projections on tcgen05 kind::tf32 (the MaxViT block dominates the rounding error
                        of the network, see DESIGN.md, so it keeps 10-bit mantissas; the 3x3 convs around it are bf16)
           'bf16_all' : bf16 storage and kind::f16 MMA everywhere (faster, ~2x the error)
           'fp32'     : fp32 storage, exact-fp32 SIMT GEMMs
           'fp32_x3'  : fp32 storage, projections on the tensor cores by the 3xTF32 operand split (the MaxViT side of MetNet3's
                        'tf32_conv' mode: 3e-6 .. 3e-5 of the largest output per GEMM, bounded by the truncating fp32 accumulation
                        of the tensor core over 3K/8 instructions -- plain tf32 is 8e-4, the SIMT kernel 1e-6 -- and 9x faster
                        than the SIMT GEMM at 512 channels)"""
        self.compute_dtype, self.tf32 = {"bf16": (torch.float32, True), "bf16_all": (torch.bfloat16, False),
                                         "fp32": (torch.float32, False), "fp32_x3": (torch.float32, False)}[precision]
        self.fp32_x3 = precision == "fp32_x3"
        return self

    def _pack_key(self, dtype):
        # train() mode never reads the folded eval-BatchNorm constants (the only users of the buffers): keyed on the parameters
        # alone there, or the running-statistics update of every forward would force a second full pack in the backward pass
        return (dtype, self.fp32_x3, self.training, tuple((p.data_ptr(), p._version) for p in self.parameters()),
                () if self.training else tuple((b.data_ptr(), b._version) for b in self.buffers()))

    @torch.no_grad()
    def packed(self, dtype):
        key = self._pack_key(dtype)
        if self._packed_key == key:
            return self._packed
        layers = []
        for li, (conv, battn, gattn) in enumerate(self.layers):
            seq = conv.fn if isinstance(conv, MBConvResidual) else conv
            P = {"residual": isinstance(conv, MBConvResidual)}
            P["w_exp"] = seq[0].weight.flatten(1).to(dtype).contiguous()                     # (hidden, dim)
            P["s_exp"], P["t_exp"] = (None, None) if self.training else _fold_bn(seq[0].bias, seq[1])
            P["w_dw"] = seq[3].weight.float().reshape(seq[3].weight.shape[0], 9).t().contiguous()   # [9][hidden]
            P["s_dw"], P["t_dw"] = (None, None) if self.training else _fold_bn(seq[3].bias, seq[4])
            P["se_w1"] = seq[6].gate[1].weight.float().contiguous()
            P["se_w2"] = seq[6].gate[3].weight.float().contiguous()
            P["w_proj"] = seq[7].weight.flatten(1).to(dtype).contiguous()                    # (dim, hidden)
            P["s_proj"], P["t_proj"] = (None, None) if self.training else _fold_bn(seq[7].bias, seq[8])
            # training (batch-statistic BatchNorm: nothing is folded)
            P["b_exp"], P["b_dw"], P["b_proj"] = (seq[i].bias.float().contiguous() for i in (0, 3, 7))
            P["w_dw_flip"] = P["w_dw"].flip(0).contiguous()                                  # dgrad = correlation with flipped taps
            P["ones_hid"], P["zeros_hid"] = torch.ones_like(P["b_dw"]), torch.zeros_like(P["b_dw"])
            for name, att in (("block", battn), ("grid", gattn)):
                P[name] = dict(
                    film_w0=att.film[0].weight.float().contiguous(), film_b0=att.film[0].bias.float().contiguous(),
                    film_w1=att.film[2].weight.float().contiguous(), film_b1=att.film[2].bias.float().contiguous(),
                    w_qkv=att.to_qkv.weight.to(dtype).contiguous(),
                    q_gamma=att.q_norm.gamma.float().reshape(-1).contiguous(),
                    k_gamma=att.k_norm.gamma.float().reshape(-1).contiguous(),
                    w_out=att.to_out[0].weight.to(dtype).contiguous(),
                    # transposed / 16-bit copies for the backward GEMMs (packed once per weight version, not once per step)
                    w_out_t=att.to_out[0].weight.to(dtype).t().contiguous(),
                    w_qkv_t=att.to_qkv.weight.to(dtype).t().contiguous(),
                    w_qkv_bf16=att.to_qkv.weight.to(torch.bfloat16).contiguous(),
                    w_out_t_bf16=att.to_out[0].weight.to(torch.bfloat16).t().contiguous(),
                    w_qkv_t_bf16=att.to_qkv.weight.to(torch.bfloat16).t().contiguous(),
                    bias_table=att.rel_pos_bias.weight.float().contiguous())
                inner, dh, hd = att.heads * att.dim_head, att.dim_head, att.heads
                wq = att.to_qkv.weight.float()
                # per-head operand tiles of the fused kernel: [q_h | k_h | v_h] rows, and the head's to_out columns
                P[name]["wqkv_h"] = torch.stack([wq[i * inner:(i + 1) * inner].reshape(hd, dh, -1) for i in range(3)],
                                                dim=1).reshape(hd * 3 * dh, -1).half().contiguous()   # fp16 operand of the fused kernel
                P[name]["wout_h"] = att.to_out[0].weight.float().reshape(-1, hd, dh).permute(1, 0, 2).contiguous()
                if att.window_size == 7 and dh == 32:
                    P[name]["head_tab"] = ops.pack_head_tables(P[name]["bias_table"], P[name]["q_gamma"], P[name]["k_gamma"])
                    # inference packs once per weight version: one host read for the logit bound that lets the fused kernel skip the
                    # running maximum of its softmax (train() mode re-packs every step and keeps the maximum)
                    P[name]["logit_bound"] = 0.0 if self.training else ops.attn_logit_bound(P[name]["bias_table"], P[name]["q_gamma"],
                                                                                            P[name]["k_gamma"], dh)
            P["reg"] = self.register_tokens[li].float().contiguous()
            if self.fp32_x3 and dtype == torch.float32:              # 3xTF32 right operands [hi | lo | hi], split once per weight version
                P["w_exp_x3"] = ops.split3_tf32(P["w_exp"], 1)
                for name in ("block", "grid"):
                    P[name]["w_qkv_x3"], P[name]["w_out_x3"] = ops.split3_tf32(P[name]["w_qkv"], 1), ops.split3_tf32(P[name]["w_out"], 1)
            layers.append(P)
        self._packed, self._packed_key = layers, key
        return layers

    # ------------------------------------------------------------------ forward
    def fused_attn_applies(self, C):
        """whether an attention layer of width C runs as the one-kernel ops.attn_fused (inference and training); every
        other shape / precision takes the un-fused path (gather -> QKV GEMM -> attn_core -> attn_out)"""
        return (self.tf32 and C == 128 and self.dim_head == 32 and self.vit_window_size == 7 and self.num_register_tokens == 4
                and self.heads >= 4 and self.heads % 2 == 0)

    def _attention(self, x, film, P, reg_in, grid_mode, want_reg_out):
        """x: CL (N,H,W,C).  returns (x + attn(x), reg_out)"""
        N, H, W, C = x.shape
        w, R = self.vit_window_size, self.num_register_tokens
        if self.fused_attn_applies(C):
            # x is a temporary of forward_cl (MBConv output / the previous attention's result): updated in place
            return ops.attn_fused(x, reg_in, film, P["wqkv_h"], P["wout_h"], P["head_tab"], w, R, grid_mode, want_reg_out,
                                  self.heads, self.dim_head, inplace=True, logit_bound=P.get("logit_bound", 0.0))
        tokens = ops.attn_gather(x, reg_in, film, w, R, grid_mode)
        qkv = ops.gemm(tokens, P["w_qkv"], tf32=self.tf32, x3=self.fp32_x3, Wt_x3=P.get("w_qkv_x3"))
        del tokens
        split = self.fp32_x3 and qkv.dtype == torch.float32 and w * w + R <= 64 and self.dim_head in (32, 64)
        att = ops.attn_core(qkv, P["q_gamma"], P["k_gamma"], P["bias_table"], N, H, W, w, R, self.heads, self.dim_head, x3=self.fp32_x3, tf32=self.tf32,
                            split_out=split)
        del qkv
        return ops.attn_out(att, P["w_out"], x, reg_in, w, R, grid_mode, want_reg_out, tf32=self.tf32, x3=self.fp32_x3,
                            Wt_x3=P.get("w_out_x3"), attn_is_split=split)

    def forward_cl(self, x: torch.Tensor, cond: torch.Tensor) -> torch.Tensor:
        """channels-last entry used by MetNet3: x (N,H,W,dim) in the compute dtype, cond (N,cond_dim) fp32"""
        _lib.require_device()
        if self.training:
            raise NotImplementedError("MaxViT.forward_cl is the inference path; training goes through MetNet3 in train() mode "
                                      "(vit_grid_model_b200.train)")
        N, H, W, C = x.shape
        w = self.vit_window_size
        assert H % w == 0 and W % w == 0, "feature map must be divisible by the window size"
        assert cond.shape == (N, self.cond_dim)
        cond = cond.float().contiguous()
        nwin = (H // w) * (W // w)
        for P in self.packed(x.dtype):
            # mixed precision: the hidden tensor (4x the channels, written and read twice) is stored in fp16 -- the 10-bit mantissa a
            # tf32 MMA keeps of an fp32 operand anyway -- and the projection runs as kind::f16; exact-fp32 / bf16_all keep their dtype
            n_hid = P["w_exp"].shape[0]
            marching = n_hid % 4 == 0 and 128 % (n_hid // 4) == 0          # the fp16 depthwise kernel (hidden <= 512 channels)
            hid_dtype = torch.float16 if (self.tf32 and x.dtype == torch.float32 and marching) else None
            h = ops.gemm(x.view(N * H * W, C), P["w_exp"], scale=P["s_exp"], shift=P["t_exp"], act=1, tf32=self.tf32,
                         out_dtype=hid_dtype, x3=self.fp32_x3, Wt_x3=P.get("w_exp_x3"))
            hidden = h.shape[1]
            h2, psum = ops.dw3x3_bnact(h.view(N, H, W, hidden), P["w_dw"], P["s_dw"], P["t_dw"])
            del h
            gate = ops.se_gate(psum, H * W, P["se_w1"], P["se_w2"])
            if x.dtype == torch.float32:
                # the squeeze-excite scale rides on per-field projection weights (256 KB per field) instead of a
                # read-modify-write pass over the hidden activations
                wn = ops.se_fold_weights(P["w_proj"], gate, dtype=h2.dtype)
                y = ops.gemm(h2.view(N * H * W, hidden), wn, rows_per_batch=H * W, b_rows_per_batch=P["w_proj"].shape[0], scale=P["s_proj"],
                             shift=P["t_proj"], res=x.view(N * H * W, C) if P["residual"] else None, tf32=self.tf32, out_f32=True, x3=self.fp32_x3)
            else:
                ops.se_scale_(h2, gate)
                y = ops.gemm(h2.view(N * H * W, hidden), P["w_proj"], scale=P["s_proj"], shift=P["t_proj"],
                             res=x.view(N * H * W, C) if P["residual"] else None, tf32=self.tf32)
            del h2
            C = y.shape[1]                                       # the first layer of a stage of a tuple-depth MaxViT widens the map
            x = y.view(N, H, W, C)
            cap = self._capture
            if cap is not None:
                cap["mbconv"] = x.permute(0, 3, 1, 2).float()
            fb = P["block"]
            film = ops.cond_mlp(cond, fb["film_w0"], fb["film_b0"], fb["film_w1"], fb["film_b1"])
            x, reg_out = self._attention(x, film, fb, P["reg"], False, True)
            reg = ops.reg_mean(reg_out, N, nwin)
            if cap is not None:
                cap["block_attn"] = x.permute(0, 3, 1, 2).float()
            fg = P["grid"]
            film = ops.cond_mlp(cond, fg["film_w0"], fg["film_b0"], fg["film_w1"], fg["film_b1"])
            x, _ = self._attention(x, film, fg, reg, True, False)
        return x

    def next_dropout_seed(self) -> int:
        """32-bit seed of this step's dropout masks (see MetNet3.next_dropout_seed)"""
        if getattr(self, "_dropout_state", None) is None:
            self._dropout_state = torch.initial_seed() & 0x7FFFFFFF
        self._dropout_state = (self._dropout_state * 1103515245 + 12345) & 0x7FFFFFFF
        return self._dropout_state

    def forward(self, x: torch.Tensor, cond: torch.Tensor) -> torch.Tensor:
        """reference signature (maxvit.py:289): x (N,dim,H,W) -> (N,dim_out,H,W), same dtype as x.  In train() mode the module
        runs the training kernels (batch-statistic BatchNorm, dropout) and is differentiable with respect to x, cond and its
        parameters (train.MaxViTTrainFn), like the reference module under autograd.  In eval() mode the same holds when x
        requires grad and grad mode is on (BatchNorm from its running statistics, no dropout); every other eval() call is
        the inference path."""
        assert cond.shape == (x.shape[0], self.cond_dim)
        if not x.is_cuda:
            raise _lib.VitGridError("vit_grid_model_b200 runs on a CUDA (sm_100a) device only; there is no CPU fallback")
        with torch.cuda.device(x.device):
            x_cl = x.permute(0, 2, 3, 1).to(self.compute_dtype).contiguous()
            frozen = not self.training and torch.is_grad_enabled() and x.requires_grad
            if self.training or frozen:
                from .train import MaxViTTrainFn
                if self.compute_dtype != torch.float32:
                    raise NotImplementedError("MaxViT training and input gradients support set_precision('bf16') (mixed) and 'fp32'")
                y = MaxViTTrainFn.apply(self, x_cl, cond.float().contiguous(), frozen, *self.parameters())
            else:
                y = self.forward_cl(x_cl, cond)
            return y.permute(0, 3, 1, 2).to(x.dtype).contiguous()
