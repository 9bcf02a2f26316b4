/* vitgrid.h -- C ABI of libvitgrid.so: the sm_100a (B200) kernels behind the MaxViT / MetNet3 hot path of
 * jhsk777/VIT-Grid-Model.
 *
 * The reference has no FFI layer (it is pure PyTorch); its boundary is the nn.Module API
 * (src/maxvit.py:224-341, src/metnet3.py:191-430).  These entry points are what a binding for that path
 * would call; each one names the reference lines it replaces.  The Python host side
 * (vit-grid-model_b200/{maxvit,metnet3}.py) binds them with ctypes and keeps the reference's nn.Module API.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless stated otherwise; `stream` is a cudaStream_t passed as void*
 *  - dtype: 0 = bf16 activations/weights (tcgen05 kind::f16), 1 = fp32 (SIMT FFMA path, "fp32 mode"),
 *    2 = fp32 storage with tcgen05 kind::tf32 MMA (GEMM entry points only; elsewhere 2 behaves as 1)
 *  - functions never allocate, never synchronise and never touch the default stream; workspaces are
 *    caller-provided; return 0 on success, non-zero on error (message via vg_last_error())
 *  - there is NO CPU fallback: on a device that is not sm_100 every launch fails loudly
 *
 * Layouts
 *  - "PG" (padded grid): a set of N frames of HP x WP pixels, channels-last, with one shared zero column
 *    between pixel rows and one shared zero row between frames:
 *        flat pixel q = (n*(HP+1) + h + 1)*(WP+1) + (w+1);   buffer = vg_pg_pixels(N,HP,WP) * C elements
 *    (a 3x3/pad-1 convolution becomes a GEMM over 9 row-shifted views of the same 2-D [q][C] tensor)
 *  - "CL" (channels-last): plain (N, H, W, C)
 */
#ifndef VITGRID_H_
#define VITGRID_H_

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VG_API __attribute__((visibility("default")))
#else
#define VG_API
#endif

#define VG_DTYPE_BF16 0
#define VG_DTYPE_FP32 1
/* fp16 storage: vg_gemm_fwd operands (dtype 3, plain store epilogue; out_f32 = 3 stores fp16) and vg_dw3x3_fwd -- the hidden
 * tensor of the MBConv block in mixed-precision inference (10-bit mantissa = what a tf32 MMA keeps of an fp32 operand) */
#define VG_DTYPE_FP16 3

VG_API int vg_version(void);
VG_API const char* vg_last_error(void);
/* number of kernels this library has launched in this process (bench.py reports the per-step delta) */
VG_API long long vg_launch_count(void);
/* 0 when the current CUDA device is compute capability 10.x; error otherwise */
VG_API int vg_device_check(void);
/* Sticky device-side error word: kernels that meet input the reference's PyTorch op would have raised on (today: a
 * timestamp whose month / day / hour falls outside nn.Embedding(13 | 32 | 25), metnet3.py:262-266,392 -> IndexError in
 * the reference) skip the access, poison the affected field's predictions with NaN and set bit 0 here.  Meaningful after
 * the stream has been synchronised; clear != 0 resets it.  Bit 0 (value 1) = timestamp out of range. */
VG_API int vg_device_error(int clear);
/* number of flat pixels (rows of the [q][C] matrix) of a PG buffer */
VG_API long long vg_pg_pixels(int N, int HP, int WP);

/* metnet3.py:356-387 -- PM2.5 standardisation of channels {4,10,16,22}, zero pad to the HPxWP frame, NCHW(T*C)
 * -> PG with Cpad channels (zeros above T*C).  x is fp32 (B,T,C,H,W) with element strides xstride[5] (HOST
 * array).  The L-fold lead-time replication (:383) is not materialised. */
VG_API int vg_prepare_fwd(int dtype, const float* x, const long long* xstride, int B, int T, int C, int H, int W,
                   int pad_top, int pad_left, int HP, int WP, int Cpad, float pm_mean, float pm_std, void* out,
                   void* stream);

/* Adjoint of vg_prepare_fwd (the gradient with respect to the input grids): g is the fp32 PG gradient [q][Cpad] of the B
 * sample frames (the stem's data gradient, summed over the lead times); dx is a fresh contiguous fp32 (B,T,C,H,W) tensor,
 * every element written.  Pad rows / columns and channels >= T*C are dropped; the PM2.5 channels {4,10,16,22} of every
 * time step, and extra_channel (-1 = none; 24 for MetNet3_with_stn_imgs, metnet3.py:701), are divided by pm_std.
 * HBM-bound: channel rows are read and (H,W) planes written coalesced through a shared-memory transpose. */
VG_API int vg_prepare_bwd(const float* g, int B, int T, int C, int H, int W, int pad_top, int pad_left, int HP, int WP, int Cpad,
                   float pm_std, int extra_channel, float* dx, void* stream);

/* metnet3.py:701 (MetNet3_with_stn_imgs) -- x[:, :, channel] = (x[:, :, channel] - pm_mean) / pm_std IN PLACE on the caller's
 * fp32 (B,T,C,H,W) tensor with element strides xstride[5] (HOST array): the reference normalises the station-image variable
 * through a view before it clones the input, so the caller's tensor changes; kept. */
VG_API int vg_standardise_channel(float* x, const long long* xstride, int B, int T, int C, int H, int W, int channel,
                           float pm_mean, float pm_std, void* stream);

/* Operand split for fp32-accurate products on the tf32 tensor cores ("3xTF32"): x = hi + lo with hi = x truncated to tf32's 10
 * mantissa bits.  in: fp32 [rows][K]; out: fp32 [rows][3K].  pattern 0 (left operand): [hi | hi | lo]; pattern 1 (right operand,
 * [N][K] weights): [hi | lo | hi] -- so that ONE tf32 GEMM over K' = 3K computes hi*hi + hi*lo + lo*hi with every epilogue of
 * vg_gemm_fwd intact (the dropped lo*lo term is ~2^-22 of the product; measured 3e-6 .. 3e-5 of the largest output for K = 128 ..
 * 2048, which is the truncating fp32 accumulation of the tensor core over 3K/8 instructions; plain tf32 measures 8e-4).  Used by the "tf32_conv" precision for the projections of
 * the MaxViT block (nn.Conv2d 1x1 / nn.Linear in maxvit.py:88-96, 139, 150), where exact fp32 is required but the SIMT GEMM is
 * 10x slower than the tensor cores. */
VG_API int vg_split3_tf32(const float* in, long long rows, int K, float* out, int pattern, void* stream);

/* Same as vg_prepare_fwd for a batch PACKED on the host (HostPipeline.pack_host: the data-loader side of
 * evaluation_vit.py:236-249): x is bf16 (B,T,C,H,W) whose PM2.5 channels were standardised in fp32 BEFORE the rounding
 * to bf16 -- exactly the values vg_prepare_fwd(VG_DTYPE_BF16) produces from the fp32 tensor, so the predictions are
 * bit-identical while the host->device copy moves half the bytes. */
VG_API int vg_prepare_packed_fwd(int dtype, const void* x_bf16, const long long* xstride, int B, int T, int C, int H, int W,
                          int pad_top, int pad_left, int HP, int WP, int Cpad, void* out, void* stream);

/* metnet3.py:389-416 -- lead-time / model-time embeddings (with the reference's dim-0 concat quirk and
 * hard-coded time index 6), and their analytic contribution to the first 3x3 conv (9 border cases) and to
 * res_conv: temb (N,le+3te), cond (N,le), tt (N,9,Cout), tres (N,Cout); N = B*L, all fp32.
 * ts: fp32 timestamps with element strides (ts_sB, ts_sT, ts_sF); w3/w1: the ORIGINAL fp32 conv weights
 * (Cout,c_in,3,3)/(Cout,c_in,1,1); c_data = T*C (index of the first time channel). */
VG_API int vg_time_terms_fwd(const float* ts, long long ts_sB, long long ts_sT, long long ts_sF, int B, int L, int le,
                      int te, const float* emb_lead, const float* emb_month, const float* emb_day,
                      const float* emb_hour, const float* w3, const float* w1, int c_in, int c_data, int Cout,
                      float* temb, float* cond, float* tt, float* tres, void* stream);

/* One nn.Linear over a few rows with wide weights: out (N,od) = act(W (od,in_dim) . relu?(in (N,in_dim)) + b), fp32; act 0 none,
 * 1 ReLU, 2 SiLU, 3 sigmoid.  The two layers of the FiLM MLP (maxvit.py:130-135) at BASELINE configs[4]'s widths (12 fields,
 * 512 -> 2048 -> 1024) are two calls of this instead of one vg_cond_mlp_fwd: a warp per weight row instead of a block per field. */
VG_API int vg_dense_rows_fwd(const float* in, int N, int in_dim, int pre_relu, const float* W, const float* b, int od, int act,
                             float* out, void* stream);

/* metnet3.py:140-143 (pre_relu=1, W1=NULL) and maxvit.py:130-135 (Linear->SiLU->Linear): per-field
 * conditioning vectors, fp32.  out (N,hid) if W1 is NULL else (N,od). */
VG_API int vg_cond_mlp_fwd(const float* cond, int N, int cond_dim, int pre_relu, const float* W0, const float* b0,
                    int hid, const float* W1, const float* b1, int od, float* out, void* stream);

/* Shifted-row GEMM with a plain epilogue: out[m][n] = act(acc*scale[n]+shift[n] | acc+bias[n]) (+res[m][n]),
 * acc = sum_tap sum_c A[m+shift[tap]][c] * Wt[n][tap*Ca+c].   Covers nn.Conv2d 1x1 + BatchNorm(eval) + GELU
 * (maxvit.py:88-90, 95-96), nn.Linear to_qkv (maxvit.py:139) and the raw 3x3 stem conv (ntaps=9).
 * A: [rowsA][Ca]; Wt: [Ntot*(batches)][ntaps*Ca]; tap_shift: HOST int[ntaps]; act: 0 none, 1 GELU, 2 ReLU.
 * rows_per_batch>0 selects per-batch weights (Wt rows advance by b_rows_per_batch every rows_per_batch rows).
 * out_f32: 0 = output in the activation dtype, 1 = fp32, 2 = bf16.  res_f32 = 1: the residual is fp32 whatever dtype is.
 * scratch (fp32, M*Ntot) is used by fp32 mode only.  The backward pass uses the same entry point for every dgrad
 * (3x3: negated tap shifts and [Cin][tap][Cout] weights). */
VG_API int vg_gemm_fwd(int dtype, const void* A, long long rowsA, int Ca, const void* Wt, int Ntot, int ntaps,
                const int* tap_shift, long long M, long long rows_per_batch, int b_rows_per_batch,
                const float* bias, const float* scale, const float* shift, int act, const void* res,
                long long ldres, int res_f32, void* out, long long ldo, int out_f32, float* scratch,
                long long scratch_elems, void* stream);

/* metnet3.py:110-126 Block = Conv2d 3x3 (pad 1) -> ChanLayerNorm (var.clamp(eps).rsqrt) -> optional FiLM
 * x*(scale+1)+shift -> ReLU, plus the ResnetBlock residual add (:162) when res != NULL.  x,out,res: PG
 * layout (N,HP,WP,C=128); Wt: [128][9*Ca] tap-major (ky,kx) then channel; film: (N,256) fp32 or NULL.
 * res_f32=1: the residual tensor is fp32 (skip connections are kept in full precision in bf16 mode);
 * out_f32_copy (or NULL): an additional fp32 copy of the block output for the next block's skip connection.
 * head_w != NULL fuses metnet3.py:424-430 (unpad, Conv2d 1x1 C->1, *std + mean) into the epilogue:
 * head_out (N,H,W) fp32 receives the predictions; `out` may then be NULL. */
VG_API int vg_conv3x3_ln_fwd(int dtype, const void* x, int Ca, const void* Wt, const float* bias, const float* ln_g,
                      const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, void* out,
                      float* out_f32_copy, int N, int HP, int WP, const float* head_w, float head_b, float head_std,
                      float head_mean, int H, int W, int pad_top, int pad_left, float* head_out, float* scratch,
                      long long scratch_elems, void* stream);

/* dedup'd first block (metnet3.py:383-418): raw3/rawres are the per-SAMPLE stem 3x3 / res_conv 1x1 GEMM
 * outputs (fp32, PG over B frames); per FIELD n=b*L+l adds bias + analytic time term, ChanLayerNorm, FiLM, ReLU
 * -> h1 (PG over N frames) and res = rawres + bias1 + tres (the ResnetBlock residual, always fp32). */
VG_API int vg_stem_finish_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                       const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                       const float* film, int B, int L, int HP, int WP, void* h1, float* res, void* stream);

/* Channel widths other than 128 (n_start_channels = 256 / 384 / 512; BASELINE configs[4]).  Same operators as
 * vg_conv3x3_ln_fwd (C -> C) and vg_stem_finish_fwd, built from a plain tcgen05 shifted-row GEMM into the fp32 scratch plus a
 * row-wise LayerNorm / FiLM / ReLU / residual kernel (inference only).  scratch: q*C floats (2*q*C in fp32 mode). */
VG_API int vg_conv3x3_ln_wide_fwd(int dtype, const void* x, int C, const void* Wt, const float* bias, const float* ln_g,
                           const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, void* out,
                           float* out_f32_copy, int N, int HP, int WP, const float* head_w, float head_b, float head_std,
                           float head_mean, int H, int W, int pad_top, int pad_left, float* head_out, float* scratch,
                           long long scratch_elems, void* stream);
VG_API int vg_stem_finish_wide_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                            const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                            const float* film, int B, int L, int HP, int WP, int C, void* h1, float* res, void* stream);

/* metnet3.py:86,419 -- MaxPool2d(2,2): PG (N,HP,WP,C) -> CL (N,HP/2,WP/2,C); out_f32=1: bf16 in, fp32 out */
VG_API int vg_pool2_fwd(int dtype, int out_f32, const void* in, void* out, int N, int HP, int WP, int C, void* stream);

/* maxvit.py:91-93 -- depthwise 3x3 + BatchNorm(eval, folded into scale/shift) + GELU on CL (N,H,W,C);
 * w9: fp32 [9][C]; psum: fp32 (N,H,C) per-row channel sums for the squeeze-excite mean. */
VG_API int vg_dw3x3_bnact_fwd(int dtype, const void* in, const float* w9, const float* scale, const float* shift,
                       void* out, float* psum, int N, int H, int W, int C, void* stream);

/* x *= gate (in place), CL (N,HW,C) */
VG_API int vg_se_scale_fwd(int dtype, void* x, const float* gate, int N, long long HW, int C, void* stream);

/* Test hook (bit-exact index parity, SURVEY 8a-7): the partition map every attention kernel of this library addresses
 * tokens through (attn_token_pixel), evaluated ON THE DEVICE for every token row: pixel_index[(n*nwin + wi)*S + tok] =
 * n*Hl*Wl + pixel of window token tok-R (maxvit.py:298 block / :322 grid), -1 for the R register-token rows. */
VG_API int vg_attn_partition_debug(int N, int Hl, int Wl, int win, int R, int grid_mode, long long* pixel_index, void* stream);

/* maxvit.py:298-308 / 322-332 + 176-187 -- partition (mode 0 block, 1 grid) folded into addressing, register
 * tokens prepended (reg: fp32 [R][C] shared or [N][R][C] per field), LayerNorm (no affine), FiLM (film: fp32
 * (N,2C) = gamma|beta)  ->  tokens [(N*nwin*S)][C] in x's dtype, or in bf16 from an fp32 x when tokens_bf16 != 0 (the
 * mixed-precision training backward re-materialises the tokens in 16-bit storage). */
VG_API int vg_attn_gather_fwd(int dtype, const void* x, const float* reg, int reg_per_field, const float* film, int N,
                       int Hl, int Wl, int C, int win, int R, int grid_mode, float ln_eps, void* tokens,
                       int tokens_bf16, void* stream);

/* maxvit.py:195-215 -- per (window, head): q,k RMSNorm (F.normalize * sqrt(d) * gamma), QK^T + rel-pos bias
 * (table (2w-1)^2+1 x heads, fp32), softmax, PV.  qkv [(Nw*S)][3*heads*dh] -> out [(Nw*S)][heads*dh].
 * dtype 0: bf16 tensors (tf32 mma products, fp32 softmax); 1: fp32 tensors, exact-fp32 FMAs; 2: fp32 tensors, QK^T and PV as 3xTF32
 * split products on the tensor cores (mma.sync; fp32-grade: 24 accumulation steps per score); 4: fp32 tensors, single tf32 products (the
 * mixed-precision modes); 6: as 2, with out [(Nw*S)][3*heads*dh] written as the split operand [hi | hi | lo] of vg_split3_tf32 (pattern 0).  Dropout and S > 64 run the SIMT kernel.
 * S <= 128, with or without dropout (drop_thresh > 0: nn.Dropout on the probabilities; at S > 64 the masks use 128 slots per
 * window and need heads <= 128, see vg_dropout_mask_debug).  S > 128 is an error. */
VG_API int vg_attn_core_fwd(int dtype, const void* qkv, const float* q_gamma, const float* k_gamma,
                     const float* bias_table, int N, int Hl, int Wl, int win, int R, int heads, int dh, void* out,
                     long long drop_seed, int drop_salt, int drop_thresh, void* stream);

/* maxvit.py:218-219 + 310/334 + 312-319/336-340 -- to_out projection, residual add and inverse partition:
 * window tokens are scattered back to CL x_out (N,Hl,Wl,C) = proj + x_in; register-token rows go to reg_out
 * (fp32 [Nw][R][C] = proj + reg_in) when reg_out != NULL (block attention) and are dropped otherwise. */
VG_API int vg_attn_out_fwd(int dtype, const void* attn, int inner, const void* Wt, const void* x_in, const float* reg_in,
                    int reg_per_field, float* reg_out, void* x_out, int N, int Hl, int Wl, int C, int win, int R,
                    int grid_mode, long long drop_seed, int drop_salt, int drop_thresh, float* scratch, long long scratch_elems,
                    void* stream);
/* (both: drop_thresh T in [1,255] = the training dropout of vg_attn_fused2_fwd -- same hash, same masks -- on the
 * probabilities / on the to_out output before the residual; 0 = none) */

/* maxvit.py:170-219 + 298-340 in ONE kernel, IN PLACE on the fp32 residual stream: xio += to_out(attn(xio)).
 * gather + register tokens + LayerNorm + FiLM -> per head {QKV, QK-RMSNorm, QK^T + rel-pos bias, softmax, PV,
 * out-projection accumulated over heads} -> + residual -> inverse partition.  xio: CL (N,Hl,Wl,128) fp32.
 * The window / grid partition (maxvit.py:298 / :322) is the TMA tensor map itself -- block: boxes (32 ch, 7, 7) of the view
 * (C, Wl, N*Hl); grid: boxes (32 ch, 1, 7, 1, 7) of the view (C, Y, 7, X, 7N) -- the token rows of the next tile are prefetched
 * by the TMA warp, and the result returns through the same maps with cp.reduce.async.bulk.tensor (.add), which performs the
 * residual add.  QKV projection, QK^T and PV run as tcgen05 kind::f16 (fp16 / bf16 operands), the out-projection as
 * kind::tf32 on the O_h accumulator read in place from TMEM; two compute groups of 8 warps alternate heads.
 * wqkv_h: fp16 [heads][96][128] (per head the 32 q rows, 32 k rows, 32 v rows of to_qkv.weight, rounded to fp16:
 * the QKV projection runs as kind::f16 on fp16 operands -- tf32's 10-bit mantissa at twice the rate);
 * wout_h: fp32 [heads][128][32] (per head the 32 columns of to_out.0.weight); head_tab: fp32 [heads][1332] =
 * per head the relative-position bias times log2(e) as 7 pre-shifted copies [bi][row 0..12] (bi stride 180 floats, row stride
 * 12 floats, entry k = 0..6 of a row = table[(row*13 + bi+6-k)]; the strides make the kernel's reads bank-conflict-free),
 * table[169]*log2(e) x 8, 32*gamma_q*gamma_k [32], 32 unused.  Needs C=128, dim_head=32, win=7, R=4, heads >= 4 and even.
 * Training: drop_thresh T in [1,255] enables nn.Dropout (maxvit.py:146,151) on the attention probabilities and on the
 * to_out output with drop probability T/256 (kept values scaled by 256/(256-T)); the masks are a counter-based hash of
 * (drop_seed, drop_salt = layer id, row, group) that the backward kernels regenerate.  T = 0: no dropout (eval).
 * A caller that needs the input afterwards (training) copies it first and passes the copy.
 * logit_bound: 0, or a bound of |logit + bias| * log2(e) over all heads that the caller derived from the weights (q-hat and k-hat are
 * unit vectors, maxvit.py:26-30: |logit| <= dh * max|gamma_q * gamma_k|); at most 115 lets the kernel skip the running maximum of the
 * softmax (2^-115 is a normal fp32 number, 53 * 2^115 is finite), the result is the same softmax. */
VG_API int vg_attn_fused2_fwd(float* xio, const float* reg_in, int reg_per_field, float* reg_out, const float* film,
                       const void* wqkv_h, const float* wout_h, const float* head_tab, int N, int Hl, int Wl, int C, int win,
                       int R, int grid_mode, int heads, int dh, float ln_eps, long long drop_seed, int drop_salt,
                       int drop_thresh, float logit_bound, void* stream);

/* maxvit.py:326 -- mean of the register tokens over windows: (N,nwin,R*C) -> (N,R*C), fp32 */
VG_API int vg_reg_mean_fwd(const float* in, float* out, int N, int nwin, int RC, void* stream);

/* metnet3.py:88-89,421 -- ConvTranspose2d(k=2,s=2) as GEMM + depth-to-space: CL (N,Hl,Wl,C) -> PG (N,2Hl,2Wl,C).
 * Wt: [4*C][C], row (di*2+dj)*C+co = weight[ci][co][di][dj].  out_bf16=1 writes bf16 whatever dtype is;
 * out_f32_copy (or NULL) receives an fp32 copy (skip connection of the next ResnetBlock). */
VG_API int vg_convT2_fwd(int dtype, int out_bf16, const void* x, const void* Wt, const float* bias, void* out,
                  float* out_f32_copy, int N, int Hl, int Wl, int C, float* scratch, long long scratch_elems, void* stream);

/* metnet3.py:424-430 -- unpad, Conv2d 1x1 C->1, *std + mean: PG (N,HP,WP,C) -> fp32 (N,H,W) */
VG_API int vg_head_fwd(int dtype, const void* h, const float* w, float bias, float pm_std, float pm_mean, int N, int HP,
                int WP, int C, int H, int W, int pad_top, int pad_left, float* out, void* stream);

/* Focal-R loss (README.md:16; no reference implementation): loss = mean(|e|*(2*sigmoid(beta|e|)-1)^gamma),
 * mse=1 uses e^2.  partial: fp32 workspace of nblocks floats.  bwd: grad[i] = gscale * d(sum_j term_j)/dpred_i
 * (pass gscale = upstream_grad / n for the mean). */
VG_API int vg_focal_r_fwd(const float* pred, const float* target, long long n, float beta, float gamma, int mse,
                   float* partial, int nblocks, float* loss, void* stream);
VG_API int vg_focal_r_bwd(const float* pred, const float* target, long long n, float beta, float gamma, int mse,
                   float gscale, float* grad, void* stream);

/* Fused evaluation statistics (replaces the ~200 host-synchronising reductions per batch of the reference's test loop,
 * /root/reference/src/evaluation_vit.py:239-455).  Four methods m are scored against the truth: 0 = the model's predictions,
 * 1 = persistence (last observation, (B,P), repeated over the leads), 2 = the 21 h CMAQ run, 3 = the mean of the four runs.
 * Class of a value: 0..3 by the boundaries b1 < b2 < b3 (assign_class, :31-32 with range_4class :194, default 0);
 * truth_class comes from the loader ((B,L,P), int32 or int64, -1 = no label).  One call ACCUMULATES a batch into
 *   counts  uint64 [4][L][4][5]   #{class(v_m) = a, truth class = t}, t index 0 <-> class -1
 *   sums    double [4][L][5][2]   sum |v_m - y| and (v_m - y)^2 per truth class
 *   glob    double [22]           over everything: [m][2] sum (v_m - y)/y, |(v_m - y)/y| over y > 0 (:311-326) | [m][3] sum v_m,
 *                                 v_m^2, v_m*y | sum y, y^2   (NMB / NME / Pearson r, :507-523, :572-576)
 *   nonzero uint64 [1]            #{y > 0};    loss_sum double [1] += MSE of this batch (criterion, :140 / :291)
 * from which every quantity of the reference's list is a linear combination (host side: eval_metrics.py).
 * clamp_preds != 0 also applies `preds[preds < 0] = 0` in place (:254).  work: vg_eval_metrics_workspace() doubles.
 * The floating-point sums are reduced in a fixed order (bit-reproducible); the integer tables are exact. */
VG_API long long vg_eval_metrics_workspace(int B, int L, int P);
VG_API int vg_eval_metrics(float* preds, const float* truth, const void* truth_class, int class_is_i64, const float* persist,
                    const float* sim_21h, const float* sim_avg, int B, int L, int P, float b1, float b2, float b3,
                    int clamp_preds, void* counts, double* sums, double* glob, void* nonzero, double* loss_sum,
                    double* work, long long work_elems, void* stream);

/* ================================================================================================================
 * Training step.  The reference has no hand-written backward: it is autograd over metnet3.py:86-430 and
 * maxvit.py:33-341 in train() mode (batch-statistic BatchNorm).  Gradients travel as fp32 tensors; dgrad GEMMs go
 * through vg_gemm_fwd; every dW below is ACCUMULATED (the caller zeroes the gradient buffer once per step).
 * ================================================================================================================ */

/* vg_conv3x3_ln_fwd that also saves what backward needs: xhat = normalised conv output (activation dtype, PG, zeros
 * at pads), rstd (fp32 [q]), relu_mask (4 x 32 bits per pixel: bit c%32 of word c/32 set where the ReLU input > 0). */
VG_API int vg_conv3x3_ln_train_fwd(int dtype, const void* x, int Ca, const void* Wt, const float* bias, const float* ln_g,
                            const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, void* out,
                            float* out_f32_copy, void* xhat, float* rstd, void* relu_mask, int N, int HP, int WP,
                            float* scratch, long long scratch_elems, void* stream);
/* vg_stem_finish_fwd with the same three saved tensors (per field) */
VG_API int vg_stem_finish_train_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                             const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                             const float* film, int B, int L, int HP, int WP, void* h1, float* res, void* xhat, float* rstd,
                             void* relu_mask, void* stream);
/* Training forward at C = 256 / 384 / 512 (also 128) in fp32 storage, the 'tf32_conv' precision: vg_conv3x3_ln_wide_fwd (no head)
 * that also saves xhat (fp32 [q][C]), rstd (fp32 [q]) and relu_mask (C/32 words per pixel: bit c%32 of word c/32 set where the
 * ReLU input > 0); pads of every output are zeros.  dtype 2: tf32 tensor cores, 1: exact-fp32 SIMT; bf16 is rejected.
 * scratch: q*C floats (2*q*C for dtype 1). */
VG_API int vg_conv3x3_ln_wide_train_fwd(int dtype, const void* x, int C, const void* Wt, const float* bias, const float* ln_g,
                                 const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, float* out,
                                 float* out_f32_copy, float* xhat, float* rstd, void* relu_mask, int N, int HP, int WP, float* scratch,
                                 long long scratch_elems, void* stream);
/* vg_stem_finish_wide_fwd with the same three saved tensors (fp32 storage: dtype 1 only) */
VG_API int vg_stem_finish_wide_train_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                                  const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                                  const float* film, int B, int L, int HP, int WP, int C, float* h1, float* res, float* xhat,
                                  float* rstd, void* relu_mask, void* stream);

/* Block backward (metnet3.py:110-126): dY fp32 PG -> dconv (odtype: 0 bf16, 1 fp32; zeros at pads) and per-field sums
 * sumA += dZ*xhat, sumB += dZ, sumD += dconv ((N,128) fp32, zeroed by the caller); border (or NULL): (N,8,128) sums of
 * dconv over first/last row, first/last column and the four corners (time-channel gradients of the stem). */
VG_API int vg_conv_ln_bwd(int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const void* relu_mask,
                   const float* ln_g, const float* film, float ln_eps, void* dconv, float* sumA, float* sumB, float* sumD,
                   float* border, int N, int HP, int WP, void* stream);
/* dg, db (ChanLayerNorm), dbias (conv) accumulated from the per-field sums; dfilm (N,256) written (or NULL) */
VG_API int vg_conv_ln_param_grads(const float* sumA, const float* sumB, const float* sumD, int N, const float* ln_g,
                           const float* ln_b, const float* film, float* dg, float* db, float* dbias, float* dfilm,
                           void* stream);
/* The same two operators at C = 128 / 256 / 384 / 512 on the saved tensors of vg_conv3x3_ln_wide_train_fwd (fp32 xhat, C/32
 * mask words per pixel): dconv fp32 (zeros at pads); sums (N,C); border (N,8,C) or NULL; dfilm (N,2C) written (or NULL). */
VG_API int vg_conv_ln_bwd_wide(int C, const float* dY, const float* xhat, const float* rstd, const void* relu_mask, const float* ln_g,
                        const float* film, float ln_eps, float* dconv, float* sumA, float* sumB, float* sumD, float* border, int N,
                        int HP, int WP, void* stream);
VG_API int vg_conv_ln_param_grads_wide(const float* sumA, const float* sumB, const float* sumD, int N, int C, const float* ln_g,
                                const float* ln_b, const float* film, float* dg, float* db, float* dbias, float* dfilm, void* stream);

/* Weight gradient of a shifted-row GEMM / 3x3 conv / linear layer:
 *   dW[n][tap*Ca + c] = beta*dW + sum_m dY[m][n] * A[m + tap_shift[tap]][c],   dW fp32 [Ntot][ntaps*Ca]
 * dtype 0: bf16 operands (tcgen05, MN-major operands straight from the row-major activations), 1: fp32 SIMT,
 * 2: fp32 operands as tf32 (tcgen05).  work: fp32 workspace of vg_wgrad_workspace() floats (split-K partials).
 * M = 0 sums no rows: dW = beta*dW (zeros for beta = 0), with no workspace; M < 0 is an error. */
VG_API long long vg_wgrad_workspace(int dtype, long long M, int Ntot, int Ca, int ntaps);
VG_API int vg_wgrad(int dtype, const void* dY, const void* A, long long rowsA, long long M, int Ntot, int Ca, int ntaps,
             const int* tap_shift, float* dW, float beta, float* work, long long work_elems, void* stream);

/* metnet3.py:424-430 backward: dH fp32 PG (every position written), dw[C] and db[1] accumulated */
VG_API int vg_head_bwd(int dtype, const float* dpred, const void* h, const float* w, float pm_std, int N, int HP, int WP, int H,
                int W, int pad_top, int pad_left, float* dH, float* dw, float* db, void* stream);
/* vg_head_bwd at C = 128 / 256 / 384 / 512 */
VG_API int vg_head_bwd_wide(int dtype, const float* dpred, const void* h, const float* w, float pm_std, int N, int HP, int WP, int C,
                     int H, int W, int pad_top, int pad_left, float* dH, float* dw, float* db, void* stream);
/* MaxPool2d(2,2) backward: gradient to the first maximum of each window; dx fp32 PG, every position written */
VG_API int vg_pool2_bwd(int dtype, const void* x, const float* dlow, float* dx, int N, int HP, int WP, int C, void* stream);
/* ConvTranspose2d(k2,s2) backward gather: dUp fp32 PG (N,2Hl,2Wl,C) -> G [N*Hl*Wl][4C] (odtype 0 bf16 / 1 fp32),
 * dbias[C] accumulated; dgrad / wgrad are then plain GEMMs on G.  C = 128, 256, 384 or 512. */
VG_API int vg_convT2_bwd_gather(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, void* stream);
/* transpose of the lead-time replication (metnet3.py:383): out[b] = sum_l in[b*L+l], PG over B frames */
VG_API int vg_lead_sum(int idtype, int odtype, const void* in, void* out, int B, int L, int HP, int WP, void* stream);
VG_API int vg_lead_sum_wide(int idtype, int odtype, const void* in, void* out, int B, int L, int HP, int WP, int C, void* stream);
/* out[n][c] += sum over the frame pixels of an fp32 PG tensor (C = 128; _wide: C = 128 / 256 / 384 / 512) */
VG_API int vg_pg_field_sum(const float* in, float* out, int N, int HP, int WP, void* stream);
VG_API int vg_pg_field_sum_wide(const float* in, float* out, int N, int HP, int WP, int C, void* stream);
/* transpose of vg_time_terms_fwd: time-channel slices of the stem conv / res_conv weight gradients (accumulated into
 * the ORIGINAL-layout gradients dw3 (Cout,c_in,3,3), dw1 (Cout,c_in,1,1)), db1 (Cout) and dtemb (N, le+3te) written */
VG_API int vg_time_terms_bwd(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                      const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                      float* dtemb, void* stream);
/* embedding gradients (accumulated): lead-time rows get dtemb[:, :le] + dcond, model-time rows follow the dim-0
 * concat quirk of metnet3.py:395-401 */
VG_API int vg_time_embed_bwd(const float* dtemb, const float* dcond, const float* ts, long long ts_sB, long long ts_sT,
                      long long ts_sF, int B, int L, int le, int te, float* d_lead, float* d_month, float* d_day,
                      float* d_hour, void* stream);
/* backward of vg_cond_mlp_fwd; dW*, db*, dcond (N,cond_dim) accumulated; work: N*(cond_dim + 2*hid) floats */
VG_API int vg_cond_mlp_bwd(const float* cond, int N, int cond_dim, int pre_relu, const float* W0, const float* b0, int hid,
                    const float* W1, int od, const float* dout, float* dW0, float* db0, float* dW1, float* db1,
                    float* dcond, float* work, long long work_elems, void* stream);
/* fused AdamW over a flat fp32 parameter buffer; gscale multiplies the gradient (1/world_size after a sum all-reduce) */
VG_API int vg_adamw_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, float gscale, void* stream);

/* BatchNorm2d in train() mode (maxvit.py:89,92,96) on a channels-last fp32 matrix [M][C]:
 * batch mean / rstd, folded affine (scale, shift), momentum update of the running buffers (NULL = no update).
 * work: vg_bn_workspace() floats. */
VG_API long long vg_bn_workspace(long long M, int C);
VG_API int vg_bn_stats(const float* x, long long M, int C, const float* gamma, const float* beta, float eps, float momentum,
                float* running_mean, float* running_var, float* mean, float* rstd, float* scale, float* shift,
                float* work, long long work_elems, void* stream);
/* out = act(raw*scale + shift) (+ res); act 0 none, 1 GELU(erf) */
VG_API int vg_bn_act(const float* raw, const float* scale, const float* shift, int act, const float* res, float* out,
              long long M, int C, void* stream);
/* BatchNorm (+ activation) backward; the upstream gradient is dOut*fgate[n] + fadd[n] (per-field vectors (N,C) or NULL,
 * n = row / rows_per_field: the squeeze-excite scale and mean paths).  dgamma, dbeta accumulated, draw [M][C] written.
 * C = 4*k with k | 256, or a multiple of 128 up to 2048.  work: vg_bn_workspace() + 2*C floats */
VG_API int vg_bn_bwd(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean,
              const float* rstd, const float* gamma, int act, const float* fgate, const float* fadd,
              long long rows_per_field, long long M, int C, float* dgamma, float* dbeta, float* draw, float* work,
              long long work_elems, void* stream);
/* BatchNorm with its running statistics (eval mode, frozen) (+ activation) backward, same upstream form as vg_bn_bwd
 * (g = dOut*fgate[n] + fadd[n]) and the same C limits: running_mean, running_rstd = 1/sqrt(running_var + eps), scale / shift
 * the affine folded from them.  draw = g*act'*scale written; dgamma += sum g*act'*(raw - running_mean)*running_rstd and
 * dbeta += sum g*act' accumulated (deterministic partial sums).  There are no batch-mean terms.  work: vg_bn_workspace() floats */
VG_API int vg_bn_bwd_frozen(const float* dOut, const float* raw, const float* scale, const float* shift, const float* running_mean,
                     const float* running_rstd, int act, const float* fgate, const float* fadd, long long rows_per_field,
                     long long M, int C, float* dgamma, float* dbeta, float* draw, float* work, long long work_elems,
                     void* stream);
/* out[c] += sum_m x[m][c] (bias gradients) */
VG_API int vg_colsum(const float* x, long long M, int C, float* out, void* stream);
/* depthwise 3x3 (marching stencil): out = act(conv(in, w9)*scale + shift); psum (or NULL): (N, vg_dw_strips(W), C)
 * partial channel sums of the outputs.  Training forward: scale = 1, shift = bias, act = 0; dgrad: flipped taps.
 * C = 4*k with k | 128, or (fp32 only) a multiple of 512 */
VG_API int vg_dw_strips(int W);
VG_API int vg_dw3x3_fwd(int dtype, const void* in, const float* w9, const float* scale, const float* shift, int act, void* out,
                 float* psum, int N, int H, int W, int C, void* stream);
/* depthwise weight / bias gradient (accumulated): dw9 [9][C], dbias [C]; C as vg_dw3x3_fwd; work: (N*strips + 1)*10*C floats */
VG_API int vg_dw3x3_wgrad(const float* x, const float* dY, int N, int H, int W, int C, float* dw9, float* dbias, float* work,
                   long long work_elems, void* stream);
/* squeeze-excite (maxvit.py:33-48) with saved intermediates, out-of-place scale, and backward (dW1, dW2 accumulated,
 * dmean (N,C) already divided by HW); work: N*((vg_field_parts(HW)+1)*C+se) floats */
VG_API int vg_se_gate_train_fwd(const float* psum, int N, int nparts, long long HW, const float* W1, const float* W2, int C,
                         int se, float* gate, float* mean, float* hid, void* stream);
/* out[n][k][c] = sum over chunk k of the HW positions of a[n][p][c] * b[n][p][c] (b = NULL: plain sums, the squeeze-excite
 * mean); k < vg_field_parts(HW); deterministic partial sums, no atomics */
VG_API int vg_field_parts(long long HW);
VG_API int vg_field_dot(const float* a, const float* b, float* out, int N, long long HW, int C, void* stream);
/* squeeze-excite scale folded into per-field weights of the following 1x1 projection: out[n][co][c] = W[co][c]*gate[n][c]
 * (fp32; consumed by vg_gemm_fwd with rows_per_batch = H*W, b_rows_per_batch = Cout) */
/* per-field projection weights out[n][co][c] = W[co][c] * gate[n][c] (the squeeze-excite scale folded into the 1x1 projection,
 * maxvit.py:38-48,95); out fp32, or fp16 when out_f16 != 0 (inference keeps the MBConv hidden tensor in fp16) */
VG_API int vg_se_fold_weights(const float* W, const float* gate, void* out, int out_f16, int N, int Cout, int C, void* stream);
VG_API int vg_se_scale_oop(const float* x, const float* gate, float* out, int N, long long HW, int C, void* stream);
VG_API int vg_se_bwd(const float* dh4, const float* h3, const float* gate, const float* mean, const float* hid, const float* W1,
              const float* W2, int N, long long HW, int C, int se, float* dW1, float* dW2, float* dmean, float* work,
              long long work_elems, void* stream);
/* attention backward: gradient at the out-projection output (inverse of the scatter + register rows); dproj fp32, or bf16
 * when dproj_bf16 != 0 */
VG_API int vg_attn_out_bwd_gather(const float* dx_out, const float* dreg, float reg_scale, int N, int Hl, int Wl, int C, int win,
                           int R, int grid_mode, void* dproj, int dproj_bf16, long long drop_seed, int drop_salt, int drop_thresh,
                           void* stream);
/* test hook: the dropout masks the kernels use, as bytes (1 = kept): prob_mask [n_windows][heads][slots][slots] (query slot,
 * key slot), out_mask [n_windows][slots][C].  slots = 64: the masks of windows of up to 64 tokens; slots = 128: those of windows
 * of 65 .. 128 tokens (un-fused path only; heads <= 128).  Any other slot count is an error. */
VG_API int vg_dropout_mask_debug(long long drop_seed, int drop_salt, int drop_thresh, long long n_windows, int heads, int C,
                          int slots, void* prob_mask, void* out_mask, void* stream);
/* per-(field, head) core backward: dqkv written; dq_gamma, dk_gamma, dbias_table accumulated.  dim_head 32 or 64 (mode 3: 32
 * only), S <= 128 (mode 3 and att_out: S <= 64; dropout at S > 64: heads <= 128).  Windows of 65 .. 128 tokens run kernels of
 * their own in modes 0 and 2.  use_tf32 = 2 / 3: tensor-core
 * kernel (2: bf16 mma + ldmatrix on fp32 tensors; 3: the tcgen05 kernel on bf16 tensors qkv, datt, dqkv and att_out, which
 * must be 16-byte aligned, S <= 64; fp32 accumulate), which can also re-materialise the forward output
 * att = softmax(.) V [rows][inner] (att_out, or NULL) for the to_out weight gradient when the forward pass was the fused
 * kernel; 0: exact-fp32 SIMT kernel.  Any other mode is an error.
 * drop_thresh > 0: the forward pass applied dropout to the probabilities with these parameters. */
VG_API int vg_attn_core_bwd(const void* qkv, const void* datt, const float* q_gamma, const float* k_gamma,
                     const float* bias_table, int N, int Hl, int Wl, int win, int R, int heads, int dh, void* dqkv,
                     float* dq_gamma, float* dk_gamma, float* dbias_table, int use_tf32, void* att_out, long long drop_seed,
                     int drop_salt, int drop_thresh, void* stream);
/* LayerNorm + FiLM backward with the inverse partition; dx_in written (= dx + dx_out), dreg_in and dfilm accumulated.
 * C = 128, 256, 384 or 512 */
VG_API int vg_attn_gather_bwd(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                       const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in,
                       float* dfilm, int N, int Hl, int Wl, int C, int win, int R, int grid_mode, float ln_eps,
                       void* stream);

/* Deterministic training backward (torch.use_deterministic_algorithms): the entry points above reduce with float atomics, whose
 * order changes from run to run.  Each _det variant computes the same quantities (same arguments, same accumulate / write
 * semantics) but stores per-warp or per-block partial sums into fixed slots of the caller's fp32 workspace `work` of
 * work_elems floats (size from the _workspace query) and reduces the slots in a fixed order, so two calls on the same inputs
 * and shapes give identical bits.  The result agrees with the atomic variant to fp32 reduction-order error. */
VG_API long long vg_conv_ln_bwd_det_workspace(int C, int N, int HP, int WP);
/* vg_conv_ln_bwd / vg_conv_ln_bwd_wide; border (or NULL) needs an fp32 dconv (odtype 1) */
VG_API int vg_conv_ln_bwd_det(int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const void* relu_mask,
                       const float* ln_g, const float* film, float ln_eps, void* dconv, float* sumA, float* sumB, float* sumD,
                       float* border, int N, int HP, int WP, float* work, long long work_elems, void* stream);
VG_API int vg_conv_ln_bwd_wide_det(int C, const float* dY, const float* xhat, const float* rstd, const void* relu_mask,
                            const float* ln_g, const float* film, float ln_eps, float* dconv, float* sumA, float* sumB,
                            float* sumD, float* border, int N, int HP, int WP, float* work, long long work_elems, void* stream);
VG_API long long vg_head_bwd_det_workspace(int N, int HP, int WP, int C);
VG_API int vg_head_bwd_det(int dtype, const float* dpred, const void* h, const float* w, float pm_std, int N, int HP, int WP, int C,
                    int H, int W, int pad_top, int pad_left, float* dH, float* dw, float* db, float* work, long long work_elems,
                    void* stream);
VG_API long long vg_convT2_bwd_gather_det_workspace(int N, int Hl, int Wl, int C);
VG_API int vg_convT2_bwd_gather_det(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, float* work,
                             long long work_elems, void* stream);
VG_API long long vg_pg_field_sum_det_workspace(int N, int HP, int WP, int C);
VG_API int vg_pg_field_sum_det(const float* in, float* out, int N, int HP, int WP, int C, float* work, long long work_elems,
                        void* stream);
VG_API long long vg_time_terms_bwd_det_workspace(int N, int Cout);
VG_API int vg_time_terms_bwd_det(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                          const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                          float* dtemb, float* work, long long work_elems, void* stream);
/* one thread per embedding-table element gathers its contributions in field order: no workspace (the query returns 0) */
VG_API long long vg_time_embed_bwd_det_workspace(int B, int L, int le, int te);
VG_API int vg_time_embed_bwd_det(const float* dtemb, const float* dcond, const float* ts, long long ts_sB, long long ts_sT,
                          long long ts_sF, int B, int L, int le, int te, float* d_lead, float* d_month, float* d_day,
                          float* d_hour, float* work, long long work_elems, void* stream);
VG_API long long vg_colsum_det_workspace(long long M, int C);
VG_API int vg_colsum_det(const float* x, long long M, int C, float* out, float* work, long long work_elems, void* stream);
/* vg_attn_core_bwd in every mode and window it accepts (modes 0, 2 and 3; S <= 128, mode 3 S <= 64): the bias-table gradient of a
 * block is gathered from dS (or its per-pair sums over the windows) in a fixed order, the gamma partials of its warps are summed
 * in warp order, and each (field, head) block / tcgen05 item stores its bias-table and gamma gradients into [field][...] slots
 * that are reduced over the fields in a fixed order. */
VG_API long long vg_attn_core_bwd_det_workspace(int N, int Hl, int Wl, int win, int R, int heads, int dh);
VG_API int vg_attn_core_bwd_det(const void* qkv, const void* datt, const float* q_gamma, const float* k_gamma,
                         const float* bias_table, int N, int Hl, int Wl, int win, int R, int heads, int dh, void* dqkv,
                         float* dq_gamma, float* dk_gamma, float* dbias_table, int use_tf32, void* att_out, long long drop_seed,
                         int drop_salt, int drop_thresh, float* work, long long work_elems, void* stream);
VG_API long long vg_attn_gather_bwd_det_workspace(int N, int Hl, int Wl, int C, int win, int R, int reg_per_field);
VG_API int vg_attn_gather_bwd_det(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                           const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in,
                           float* dfilm, int N, int Hl, int Wl, int C, int win, int R, int grid_mode, float ln_eps,
                           float* work, long long work_elems, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VITGRID_H_ */
