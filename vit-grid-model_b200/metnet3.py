"""MetNet3 encoder-decoder with the reference's nn.Module API (/root/reference/src/metnet3.py:191-430) on
libvitgrid kernels.

Constructor arguments, parameter/buffer names and shapes match the reference, so its checkpoints (with or without
the ``module.`` prefix that nn.DataParallel adds, evaluation_vit.py:107-109) load with ``strict=True``.

Data flow of ``forward`` (eval mode), N = B*L fields:
  prepare (PM2.5 standardise, pad, NHWC, bf16)                         per SAMPLE  (B frames, 600->608 channels)
  stem: 3x3 conv + 1x1 res_conv over the data channels                  per SAMPLE  (lead-time dedup, SURVEY H5)
  time terms: analytic contribution of the 5 constant time channels     per FIELD   (9 border cases)
  stem finish: +bias +time term, ChanLN, FiLM, ReLU                      per FIELD
  3 more 3x3 conv blocks (tcgen05 implicit GEMM, fused LN/FiLM/ReLU/residual epilogue) -> maxpool
  MaxViT (maxvit.py) -> ConvTranspose-as-GEMM -> 4 conv blocks -> 1x1 head + de-normalisation
"""
from __future__ import annotations

from typing import List

import torch
import torch.nn as nn

from . import _lib, ops
from .maxvit import MaxViT


class ChanLayerNorm(nn.Module):
    """holder for g, b (metnet3.py:94-104)"""

    def __init__(self, dim, eps=1e-5):
        super().__init__()
        self.eps = eps
        self.g = nn.Parameter(torch.ones(1, dim, 1, 1))
        self.b = nn.Parameter(torch.zeros(1, dim, 1, 1))


class Block(nn.Module):
    def __init__(self, dim, dim_out):
        super().__init__()
        self.proj = nn.Conv2d(dim, dim_out, 3, padding=1)
        self.norm = ChanLayerNorm(dim_out)


class ResnetBlock(nn.Module):
    def __init__(self, dim_in, dim_out, cond_dim=None):
        super().__init__()
        self.mlp = nn.Sequential(nn.ReLU(), nn.Linear(cond_dim, dim_out * 2)) if cond_dim is not None else None
        self.block1 = Block(dim_in, dim_out)
        self.block2 = Block(dim_out, dim_out)
        self.res_conv = nn.Conv2d(dim_in, dim_out, 1) if dim_in != dim_out else nn.Identity()


class ResnetBlocks(nn.Module):
    def __init__(self, dim_in, dim_out, depth=1, cond_dim=None):
        super().__init__()
        blocks, cur = [], dim_in
        for _ in range(depth):
            blocks.append(ResnetBlock(cur, dim_out, cond_dim=cond_dim))
            cur = dim_out
        self.blocks = nn.ModuleList(blocks)


def _pack_conv3x3(w, dtype, c_keep=None, c_pad=None):
    """(Cout,Cin,3,3) -> [Cout][9*Cp], K index = (ky*3+kx)*Cp + c (only the first c_keep input channels)"""
    co, ci = w.shape[:2]
    c_keep = ci if c_keep is None else c_keep
    c_pad = c_keep if c_pad is None else c_pad
    out = torch.zeros(co, 9, c_pad, dtype=dtype, device=w.device)
    out[:, :, :c_keep] = w[:, :c_keep].permute(0, 2, 3, 1).reshape(co, 9, c_keep).to(dtype)
    return out.reshape(co, 9 * c_pad).contiguous()


def _check_timestamps(ts):
    """month / day / hour of time index 6 (metnet3.py:405) must be valid rows of nn.Embedding(13 | 32 | 25)
    (metnet3.py:262-266); the reference raises IndexError from the lookup"""
    if ts.dim() != 3 or ts.shape[1] < 7 or ts.shape[2] < 4:
        raise ValueError("timestamps must be (B, >=7, 4) [year, month, day, hour]")
    t = ts[:, 6, 1:4].to(torch.float32)
    hi = torch.tensor([13.0, 32.0, 25.0])
    if not bool(((t > -1.0) & (t < hi)).all()):
        raise IndexError("timestamps[:, 6, 1:4] (month, day, hour) outside the embedding tables 13 / 32 / 25 (metnet3.py:392)")


class MetNet3(nn.Module):
    # variable standardised with the PM2.5 statistics next to {4,10,16,22} (-1: none; 24 in MetNet3_with_stn_imgs)
    standardised_extra_channel = -1

    def __init__(
        self,
        input_size_sample: tuple,      # window_size, n_variables, height, width
        n_start_channels: int,
        end_lead_time: int,
        pm25_boundaries: List[float],
        pm10_boundaries: List[float],
        pm25_mean: float,
        pm25_std: float,
        lead_time_emb_dim: int = 2,
        model_time_emb_dim: int = 1,
        concat_time_to_input: bool = True,
        pm25: bool = True,
        pm10: bool = False,
        resnet_block_depth: int = 2,
        direct_regional: bool = False,
        ignore_backbone: bool = False,
        vit_block_depth: int = 1,
        n_heads: int = 32,
        dim_head: int = 32,
        vit_window_size: int = 7,
        mbconv_expansion_rate=4,
        mbconv_shrinkage_rate=0.25,
        dropout=0.1,
        num_register_tokens: int = 4,
        normalization_method="Standard",
    ):
        super().__init__()
        window_size, n_variables, input_height, input_width = input_size_sample
        self.window_size, self.n_variables = window_size, n_variables
        self.input_height, self.input_width = input_height, input_width
        self.n_input_channels = window_size * n_variables
        self.n_start_channels = n_start_channels
        self.end_lead_time = end_lead_time
        self.concat_time_to_input = concat_time_to_input
        self.vit_window_size = vit_window_size
        self.pm25_mean, self.pm25_std = pm25_mean, pm25_std
        self.normalization_method = normalization_method
        self.lead_time_emb_dim, self.model_time_emb_dim = lead_time_emb_dim, model_time_emb_dim
        if not direct_regional:
            assert ignore_backbone == False
        # branches of the reference constructor that its own forward never reaches are not built
        if pm10 or direct_regional or not pm25:
            raise NotImplementedError("only the pm25=True, pm10=False, direct_regional=False path exists (metnet3.py:426-430)")
        if not concat_time_to_input:
            raise NotImplementedError("concat_time_to_input=False is not built")
        if normalization_method != "Standard":
            raise NotImplementedError("only normalization_method='Standard' is reachable in the reference forward (metnet3.py:369,428)")
        if pm25_boundaries is None:
            raise ValueError("pm25_boundaries must be provided")
        if n_variables < 23:
            raise ValueError("the PM2.5 channel indices {4,10,16,22} (metnet3.py:362) need n_variables >= 23")
        self.register_buffer('pm25_boundaries', torch.FloatTensor(pm25_boundaries))

        self.condition_lead_time = nn.Embedding(end_lead_time + 1, lead_time_emb_dim)
        self.condition_model_time = nn.ModuleList([
            nn.Embedding(12 + 1, model_time_emb_dim), nn.Embedding(31 + 1, model_time_emb_dim),
            nn.Embedding(24 + 1, model_time_emb_dim)])
        self.resnet1 = ResnetBlocks(dim_in=self.n_input_channels + lead_time_emb_dim + model_time_emb_dim * 3,
                                    dim_out=n_start_channels, cond_dim=lead_time_emb_dim, depth=resnet_block_depth)
        self.down = nn.MaxPool2d(kernel_size=2, stride=2)
        self.vit = MaxViT(dim=n_start_channels, depth=vit_block_depth, cond_dim=lead_time_emb_dim, heads=n_heads,
                          dim_head=dim_head, vit_window_size=vit_window_size,
                          mbconv_expansion_rate=mbconv_expansion_rate, mbconv_shrinkage_rate=mbconv_shrinkage_rate,
                          dropout=dropout, num_register_tokens=num_register_tokens)
        self.up = nn.ConvTranspose2d(n_start_channels, n_start_channels, kernel_size=2, stride=2)
        self.resnet2 = ResnetBlocks(dim_in=n_start_channels, dim_out=n_start_channels, cond_dim=lead_time_emb_dim,
                                    depth=resnet_block_depth)
        self.classifier_pm25 = nn.Conv2d(n_start_channels, 1, kernel_size=1)

        if n_start_channels not in (128, 256, 384, 512):
            # the fused conv+ChanLayerNorm epilogue keeps a 128-channel row per TMEM lane; 256 / 384 / 512 run the
            # GEMM + row-kernel path (inference); other widths have no kernels
            self._unsupported = f"n_start_channels={n_start_channels}: built for 128 (fused path), 256, 384 and 512 channels"
        else:
            self._unsupported = None
        self.compute_dtype, self.precision, self.conv_tf32 = torch.bfloat16, "bf16", False
        if n_start_channels > 128:
            self.compute_dtype, self.precision, self.conv_tf32 = torch.float32, "tf32_conv", True
            self.vit.set_precision("fp32_x3")
        self.max_fields = {torch.bfloat16: 768, torch.float32: 48}
        self._packed, self._packed_key = None, None
        self._capture = None          # debugging: set to a dict to collect stage outputs (NCHW copies)
        self._grad_buffer = None      # training: flat fp32 gradient buffer (train.GradBuffer)
        self._grad_sync = None        # training: data-parallel gradient all-reduce (set by parallel.DataParallel)
        self._dropout_state = None
        self.dropout = dropout

    # ------------------------------------------------------------------ helpers
    def set_precision(self, precision: str):
        """'bf16'     : bf16 storage + tcgen05 kind::f16 for the 3x3-conv encoder/decoder, fp32 storage + 16-bit / tf32 tensor-core
                        operands for the MaxViT block (default at 128 channels);
           'bf16_all' : bf16 everywhere;
           'tf32'     : fp32 storage, every contraction on tcgen05 kind::tf32;
           'tf32_conv': fp32 storage, tf32 convolutions, near-fp32 MaxViT block (its projections as 3xTF32 split products on the
                        tensor cores, ~1e-5 per GEMM; attention core exact fp32; default above 128 channels);
           'fp32'     : exact-fp32 SIMT path.
        Wide networks default to 'tf32_conv': on BASELINE configs[4] (512 channels, 32 x 64 heads, depth 4, random weights) the
        modes measure 3.6e-2 (bf16), 1.4e-2 (tf32), 4.3e-3 (tf32_conv) and 2e-5 (fp32) against the oracle -- four stacked MaxViT
        layers with un-scaled +-32 gamma^2 logits amplify operand rounding, and tf32_conv is the fastest mode inside the 1e-2
        tolerance (tests/test_parity_r2_gpu.py, tools/config5_parity.py)."""
        self.compute_dtype = {"bf16": torch.bfloat16, "bf16_all": torch.bfloat16, "fp32": torch.float32, "tf32": torch.float32,
                              "tf32_conv": torch.float32}[precision]
        self.conv_tf32 = precision in ("tf32", "tf32_conv")
        self.vit.set_precision({"tf32": "bf16", "tf32_conv": "fp32_x3"}.get(precision, precision))
        self.precision = precision
        self.invalidate_packed()
        return self

    def invalidate_packed(self):
        """Drop the kernel-layout copies of the weights (re-derived on the next forward).  The caches are keyed on
        (data_ptr, version) of every parameter, which in-place writes through ``.data`` -- broadcasts, EMA swaps, raw kernel
        updates such as FlatAdamW -- do not change: call this after any such write."""
        self._packed_key = None
        self.vit._packed_key = None

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        # checkpoints saved from nn.DataParallel carry a 'module.' prefix (evaluation_vit.py:107-109)
        if state_dict and all(k.startswith("module.") for k in state_dict):
            state_dict = {k[len("module."):]: v for k, v in state_dict.items()}
        self.invalidate_packed()
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def pad_values(self):
        """(left, right, top, bottom) of metnet3.py:324-333"""
        ph, pw = (14 - self.input_height) % 14, (14 - self.input_width) % 14
        return (pw // 2, pw - pw // 2, ph // 2, ph - ph // 2)

    @torch.no_grad()
    def packed(self, dtype):
        own = [p for n, p in self.named_parameters() if not n.startswith("vit.")]
        key = (dtype, self.vit.compute_dtype, tuple((p.data_ptr(), p._version) for p in own))
        if self._packed_key == key:
            return self._packed
        c_data = self.n_input_channels
        c_pad = (c_data + 63) // 64 * 64
        P = {"c_pad": c_pad}
        for name, rb in (("resnet1", self.resnet1), ("resnet2", self.resnet2)):
            blocks = []
            for bi, blk in enumerate(rb.blocks):
                d = dict(mlp_w=blk.mlp[1].weight.float().contiguous(), mlp_b=blk.mlp[1].bias.float().contiguous())
                stem = name == "resnet1" and bi == 0
                w1 = blk.block1.proj.weight
                if stem:
                    d["w1"] = _pack_conv3x3(w1, dtype, c_keep=c_data, c_pad=c_pad)
                    d["w1_orig"] = w1.float().contiguous()
                    wres = torch.zeros(w1.shape[0], c_pad, dtype=dtype, device=w1.device)
                    wres[:, :c_data] = blk.res_conv.weight[:, :c_data, 0, 0].to(dtype)
                    d["wres"], d["wres_orig"] = wres, blk.res_conv.weight.float().contiguous()
                    d["bres"] = blk.res_conv.bias.float().contiguous()
                else:
                    d["w1"] = _pack_conv3x3(w1, dtype)
                d["b1"] = blk.block1.proj.bias.float().contiguous()
                d["g1"], d["be1"] = blk.block1.norm.g.float().reshape(-1).contiguous(), blk.block1.norm.b.float().reshape(-1).contiguous()
                d["w2"] = _pack_conv3x3(blk.block2.proj.weight, dtype)
                d["b2"] = blk.block2.proj.bias.float().contiguous()
                d["g2"], d["be2"] = blk.block2.norm.g.float().reshape(-1).contiguous(), blk.block2.norm.b.float().reshape(-1).contiguous()
                d["eps1"], d["eps2"] = blk.block1.norm.eps, blk.block2.norm.eps
                blocks.append(d)
            P[name] = blocks
        C = self.n_start_channels
        P["w_up_vit"] = self.up.weight.permute(2, 3, 1, 0).reshape(4 * C, C).to(self.vit.compute_dtype).contiguous()
        P["b_up"] = self.up.bias.float().contiguous()
        P["w_head"] = self.classifier_pm25.weight.float().reshape(-1).contiguous()
        P["b_head"] = float(self.classifier_pm25.bias.float().item())
        P["emb_lead"] = self.condition_lead_time.weight.float().contiguous()
        P["emb_time"] = [e.weight.float().contiguous() for e in self.condition_model_time]
        self._packed, self._packed_key = P, key
        return P

    # ------------------------------------------------------------------ forward
    def _resblock(self, x, skip, cond, d, bufs, N, HP, WP, out_copy=None, head=None):
        """128->128 ResnetBlock on PG buffers (metnet3.py:149-162).  x: block input (compute dtype); skip: the same
        tensor as the residual operand (fp32 copy in bf16 mode).  Returns the buffer holding h + x (None when the head
        is fused into the last epilogue)."""
        film = ops.cond_mlp(cond, d["mlp_w"], d["mlp_b"], pre_relu=True)
        t1, t2 = [b for b in bufs if b is not x][:2]
        ops.conv3x3_ln(x, d["w1"], d["b1"], d["g1"], d["be1"], d["eps1"], film, None, t1, N, HP, WP, tf32=self.conv_tf32)
        ops.conv3x3_ln(t1, d["w2"], d["b2"], d["g2"], d["be2"], d["eps2"], None, skip, None if head else t2, N, HP, WP,
                       out_copy=out_copy, head=head, tf32=self.conv_tf32)
        return None if head else t2

    def _forward_chunk(self, x, b0, b1, terms, P, dtype, out, packed=False):
        """fields of samples [b0,b1) of x -> out[b0:b1]"""
        temb, cond_all, tt_all, tres_all = terms
        L, C = self.end_lead_time, self.n_start_channels
        B = b1 - b0
        N = B * L
        HP, WP = self.input_height + (14 - self.input_height) % 14, self.input_width + (14 - self.input_width) % 14
        pads = self.pad_values()
        dev = x.device
        cond = cond_all[b0 * L:b1 * L]
        tt, tres = tt_all[b0 * L:b1 * L], tres_all[b0 * L:b1 * L]
        mixed = dtype != torch.float32            # bf16 activations: skip connections travel as separate fp32 copies
        # ---- stem, once per sample
        s0 = P["resnet1"][0]
        xin = ops.prepare(x[b0:b1], pads, HP, WP, P["c_pad"], self.pm25_mean, self.pm25_std, dtype, packed=packed)
        raw3 = ops.gemm(xin, s0["w1"], ntaps=9, tap_shift=ops.conv_tap_shifts(WP), out_f32=True, tf32=self.conv_tf32)
        rawres = ops.gemm(xin, s0["wres"], out_f32=True, tf32=self.conv_tf32)
        del xin
        bufs = [ops.pg_empty(N, HP, WP, C, dtype, dev) for _ in range(3)]
        skips = [ops.pg_empty(N, HP, WP, C, torch.float32, dev) for _ in range(2)]
        film = ops.cond_mlp(cond, s0["mlp_w"], s0["mlp_b"], pre_relu=True)
        ops.stem_finish(raw3, rawres, s0["b1"], s0["bres"], tt, tres, s0["g1"], s0["be1"], s0["eps1"], film, B, L, HP, WP,
                        bufs[0], skips[0])
        del raw3, rawres
        blocks1, blocks2 = P["resnet1"][1:], P["resnet2"]
        # block output that a later ResnetBlock uses as its skip gets an fp32 copy (bf16 mode only)
        want_copy = mixed and len(blocks1) > 0
        ops.conv3x3_ln(bufs[0], s0["w2"], s0["b2"], s0["g2"], s0["be2"], s0["eps2"], None, skips[0], bufs[2], N, HP, WP,
                       out_copy=skips[1] if want_copy else None, tf32=self.conv_tf32)
        h, hs = bufs[2], (skips[1] if want_copy else bufs[2])
        cap = self._capture
        if cap is not None:
            cap["stem_h1"], cap["stem_res"] = ops.pg_to_nchw(bufs[0], N, HP, WP), ops.pg_to_nchw(skips[0], N, HP, WP)
            cap["resnet1.0"] = ops.pg_to_nchw(h, N, HP, WP)
        for k, d in enumerate(blocks1):
            nxt = [sk for sk in skips if sk is not hs][0]
            copy = nxt if (mixed and k + 1 < len(blocks1)) else None
            h = self._resblock(h, hs, cond, d, bufs, N, HP, WP, out_copy=copy)
            hs = copy if copy is not None else h
        # ---- MaxViT at half resolution
        low = ops.pool2(h, N, HP, WP, out_dtype=self.vit.compute_dtype)
        if cap is not None:
            cap["resnet1"] = ops.pg_to_nchw(h, N, HP, WP)
            self.vit._capture = cap
        low = self.vit.forward_cl(low, cond)
        if cap is not None:
            cap["vit"] = low.permute(0, 3, 1, 2).float()
        # ---- decoder
        up = [b for b in bufs if b is not h][0]       # pads of every PG buffer are already zero (written by conv/stem)
        ops.convT2(low, P["w_up_vit"], P["b_up"], up, tf32=self.vit.tf32 or self.conv_tf32, out_copy=skips[0] if mixed else None)
        del low
        h, hs = up, (skips[0] if mixed else up)
        if cap is not None:
            cap["up"] = ops.pg_to_nchw(h, N, HP, WP)
        head = (P["w_head"], P["b_head"], self.pm25_std, self.pm25_mean, self.input_height, self.input_width, pads,
                out[b0:b1].view(N, self.input_height, self.input_width))
        for k, d in enumerate(blocks2):
            last = k + 1 == len(blocks2)
            nxt = [sk for sk in skips if sk is not hs][0]
            copy = nxt if (mixed and not last) else None
            h = self._resblock(h, hs, cond, d, bufs, N, HP, WP, out_copy=copy, head=head if (last and cap is None) else None)
            hs = copy if copy is not None else h
        if cap is not None:
            cap["resnet2"] = ops.pg_to_nchw(h, N, HP, WP)
            ops.head(h, P["w_head"], P["b_head"], self.pm25_std, self.pm25_mean, N, HP, WP, self.input_height,
                     self.input_width, pads, out=out[b0:b1].view(N, self.input_height, self.input_width))

    # ------------------------------------------------------------------ training
    def grad_buffer(self):
        """flat fp32 gradient buffer the backward kernels accumulate into (one view per parameter)"""
        from .train import GradBuffer
        dev = next(self.parameters()).device
        if self._grad_buffer is None or self._grad_buffer.flat.device != dev:
            self._grad_buffer = GradBuffer(self)
        return self._grad_buffer

    def _forward_train(self, x, ts, frozen=False):
        """train() mode: batch-statistic BatchNorm, activations saved, hand-written backward (train.py).
        frozen (eval() mode with an input that requires grad): the same graph with BatchNorm from its running statistics and
        no dropout, so that x.grad and the parameter gradients are those of the reference module in eval() mode"""
        from .train import MetNet3TrainFn
        what = "input gradients in eval() mode" if frozen else "training"
        C = self.n_start_channels
        # 128 channels: the fused conv epilogues in every precision but bf16_all / tf32; wider networks: the shifted-row GEMM +
        # row kernels in fp32 storage with tf32 convolutions and the exact-fp32 MaxViT training kernels
        built = ("bf16", "fp32", "tf32_conv") if C == 128 else ("tf32_conv",)
        if self.precision not in built:
            raise NotImplementedError(f"{what} at n_start_channels={C} supports set_precision("
                                      f"{' | '.join(repr(p) for p in built)}), not {self.precision!r}")
        return MetNet3TrainFn.apply(self, x, ts, frozen, *self.parameters())

    def next_dropout_seed(self) -> int:
        """32-bit seed of this step's dropout masks: derived from torch's seed at the first training step (so that
        torch.manual_seed reproduces a run) and advanced by one per step; the masks themselves are a counter-based hash
        inside the kernels (vg_rng.cuh)"""
        if self._dropout_state is None:
            self._dropout_state = torch.initial_seed() & 0x7FFFFFFF
        self._dropout_state = (self._dropout_state * 1103515245 + 12345) & 0x7FFFFFFF
        return self._dropout_state

    def forward(self, x, labels_pm25=None, region_targets_pm25=None, labels_pm10=None, region_targets_pm10=None,
                timestamps: torch.Tensor = None, prev_vals: torch.Tensor = None):
        """x: (B,T,C,H,W) fp32; timestamps: (B, >=7, 4) [year, month, day, hour] -> (B, L, H, W) fp32 PM2.5"""
        _lib.require_device()
        if self._unsupported:
            raise NotImplementedError(self._unsupported)
        if timestamps is None:
            raise ValueError("timestamps is required (metnet3.py:405)")
        if not x.is_cuda:
            raise _lib.VitGridError("vit_grid_model_b200 runs on a CUDA (sm_100a) device only; there is no CPU fallback")
        _lib.raise_device_errors()                     # e.g. an out-of-range timestamp met by an earlier call's kernels
        if not timestamps.is_cuda:                      # host timestamps are validated for free, like nn.Embedding would
            _check_timestamps(timestamps)
        with torch.cuda.device(x.device):               # kernels launch on x's device and its current stream
            return self._forward_impl(x, timestamps)

    def forward_packed(self, x_packed, timestamps):
        """inference on a batch packed by ``pipeline.pack_host`` (bf16, PM2.5 channels standardised before the rounding):
        the same predictions, bit for bit, as ``forward`` on the fp32 tensor in the default 'bf16' precision"""
        _lib.require_device()
        if self._unsupported:
            raise NotImplementedError(self._unsupported)
        if self.training or self.compute_dtype != torch.bfloat16 or type(self) is not MetNet3:
            raise NotImplementedError("packed bf16 batches feed the bf16 inference path of MetNet3 only")
        if not x_packed.is_cuda or x_packed.dtype != torch.bfloat16:
            raise _lib.VitGridError("forward_packed takes a CUDA bf16 tensor produced by pipeline.pack_host")
        _lib.raise_device_errors()
        with torch.cuda.device(x_packed.device):
            return self._forward_impl(x_packed, timestamps, packed=True)

    def _forward_impl(self, x, timestamps, packed=False):
        B, T, Cv, H, W = x.shape
        assert (T, Cv, H, W) == (self.window_size, self.n_variables, self.input_height, self.input_width)
        pl, pr, pt, pb = self.pad_values()
        if 0 in (pr, pb):
            raise ValueError("the reference's unpad (metnet3.py:337) needs non-zero right/bottom pads")
        dtype = self.compute_dtype
        if not packed:
            x = x.float()
        ts = timestamps.to(device=x.device, dtype=torch.float32)
        if self.training:
            return self._forward_train(x, ts)
        if not packed and torch.is_grad_enabled() and x.requires_grad:
            # eval() mode under autograd with an input that requires grad (attribution, inverse problems): the frozen-BatchNorm
            # graph.  Every other eval() call -- parameters require grad by default -- stays on the inference path below.
            return self._forward_train(x, ts, frozen=True)
        P = self.packed(dtype)
        L = self.end_lead_time
        s0 = P["resnet1"][0]
        et = P["emb_time"]
        terms = ops.time_terms(ts, B, L, P["emb_lead"], et[0], et[1], et[2], s0["w1_orig"], s0["wres_orig"],
                               self.n_input_channels, self.n_start_channels)
        out = torch.empty(B, L, H, W, dtype=torch.float32, device=x.device)
        step = max(1, self.max_fields[dtype] // L)
        for b0 in range(0, B, step):
            self._forward_chunk(x, b0, min(B, b0 + step), terms, P, dtype, out, packed=packed)
        return out


class MetNet3_with_stn_imgs(MetNet3):
    """/root/reference/src/metnet3.py:518-759.  Same network and state dict as ``MetNet3`` with 25 input variables: variable
    24 is a station-observation image in raw ug/m3 that ``forward`` standardises with the PM2.5 statistics
    (metnet3.py:701) next to the four simulated-PM2.5 channels.

    Reference behaviour kept on purpose: the standardisation of variable 24 is written back into the CALLER's tensor
    (line 701 runs before the ``x.clone()`` of line 702), so calling ``forward`` twice on the same tensor normalises it
    twice.  ``tests/golden/metnet3_stn_small128.pt`` records that side effect.  Under autograd the write is the reference's
    in-place op: on a leaf that requires grad it raises as torch does, and the gradient of a non-leaf input carries the 1/std
    of the standardisation on variable 24."""

    standardised_extra_channel = 24

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        if self.n_variables < 25:
            raise ValueError("MetNet3_with_stn_imgs reads the station image from variable 24 (metnet3.py:701): n_variables >= 25")

    def forward(self, x, labels_pm25=None, region_targets_pm25=None, labels_pm10=None, region_targets_pm10=None,
                timestamps: torch.Tensor = None, prev_vals: torch.Tensor = None):
        _lib.require_device()
        if not x.is_cuda:
            raise _lib.VitGridError("vit_grid_model_b200 runs on a CUDA (sm_100a) device only; there is no CPU fallback")
        if self.normalization_method == "Standard":
            if x.dtype != torch.float32:
                raise _lib.VitGridError("MetNet3_with_stn_imgs takes the reference's fp32 input tensor")
            if torch.is_grad_enabled() and x.requires_grad:
                if x.is_leaf:
                    raise RuntimeError("a leaf Variable that requires grad is being used in an in-place operation.")
                torch.autograd.graph.increment_version(x)       # what the reference's in-place write does to x's version
            with torch.cuda.device(x.device):                   # the caller's tensor is updated, as in the reference (:701)
                ops.standardise_channel_(x, 24, self.pm25_mean, self.pm25_std)
        return super().forward(x, labels_pm25, region_targets_pm25, labels_pm10, region_targets_pm10, timestamps, prev_vals)
