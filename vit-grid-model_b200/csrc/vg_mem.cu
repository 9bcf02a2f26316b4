// Bandwidth-bound kernels of the MetNet3 / MaxViT path (judged by achieved HBM GB/s):
// input preparation, time-channel terms, stem finish (LN+FiLM+ReLU per lead time), max-pool, depthwise 3x3 +
// BN + GELU (+ squeeze-excite partial sums), SE gate / scale, conditioning MLPs, register-token mean,
// 1x1 head + de-normalisation, Focal-R loss.
// All kernels are templated on the activation dtype T (bf16 mode / fp32 mode) and use channels-last layouts.
#include "vg_common.cuh"
#include "vg_host.h"

namespace vg {

// 4 consecutive activations <-> float4 (8-byte vector for bf16)
template <typename T> struct Ld4;
template <> struct Ld4<float> {
  static __device__ __forceinline__ float4 ld(const float* p) { return *reinterpret_cast<const float4*>(p); }
  static __device__ __forceinline__ void st(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
};
template <> struct Ld4<bf16> {
  static __device__ __forceinline__ float4 ld(const bf16* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  static __device__ __forceinline__ void st(bf16* p, float4 v) {
    uint2 u;
    *reinterpret_cast<__nv_bfloat162*>(&u.x) = __floats2bfloat162_rn(v.x, v.y);
    *reinterpret_cast<__nv_bfloat162*>(&u.y) = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = u;
  }
};

// ================================================================================================
// prepare: x (B,T,C,H,W) fp32, arbitrary strides -> PG layout [q][Cpad] with PM2.5 channels standardised
// (metnet3.py:361-380), spatially zero-padded into the HPxWP frame (metnet3.py:384), channel padded with zeros.
// The L-fold replication (metnet3.py:383) is NOT materialised: the stem convolution runs once per sample.
// The output buffer is zero-filled first (pads, channel padding); this kernel writes frame pixels with a source.
// ================================================================================================

__device__ __forceinline__ float ld_in(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_in(const bf16* p) { return __bfloat162float(*p); }

// TIn = float: the reference's input tensor; TIn = bf16: a batch packed on the host by HostPipeline.pack_host (PM2.5 channels
// already standardised in fp32, then everything rounded to bf16 -- p.prestd = 1)
template <typename T, typename TIn>
__global__ void __launch_bounds__(256) prepare_kernel(const PrepParams p, T* __restrict__ out) {
  __shared__ float tile[64][33];
  const int w0 = blockIdx.x * 32;
  const int h = blockIdx.y;
  const int cblocks = p.Cpad / 64;
  const int b = blockIdx.z / cblocks, ch0 = (blockIdx.z - b * cblocks) * 64;
  const int TC = p.T * p.C;
  const TIn* xb = reinterpret_cast<const TIn*>(p.x) + (long long)b * p.sB + (long long)h * p.sH;
  for (int i = threadIdx.x; i < 64 * 32; i += 256) {
    int cl, wl;
    if (p.w_fast) { wl = i & 31; cl = i >> 5; } else { cl = i & 63; wl = i >> 6; }
    const int ch = ch0 + cl, w = w0 + wl;
    float v = 0.f;
    if (ch < TC && w < p.W) {
      const int t = ch / p.C, c = ch - t * p.C;
      v = ld_in(xb + (long long)t * p.sT + (long long)c * p.sC + (long long)w * p.sW);
      if (!p.prestd && (c == 4 || c == 10 || c == 16 || c == 22)) v = (v - p.mean) / p.stdv;     // metnet3.py:362,370
    }
    tile[cl][wl] = v;
  }
  __syncthreads();
  const int wl = threadIdx.x >> 3, c8 = (threadIdx.x & 7) * 8;
  const int w = w0 + wl;
  if (w < p.W) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = tile[c8 + j][wl];
    st8(out + p.pg.q(b, h + p.pad_top, w + p.pad_left) * p.Cpad + ch0 + c8, v);
  }
}

// prepare for inputs whose (H, W) planes are contiguous (the layout the reference's loader produces after its permute,
// evaluation_vit.py:248-249): tiles run over the FLAT pixel index h*W + w, so a 67-wide row does not waste a third of
// every 32-column tile, and each thread has its eight loads in flight before the transposing store.
template <typename T, typename TIn>
__global__ void __launch_bounds__(256) prepare_flat_kernel(const PrepParams p, T* __restrict__ out) {
  // (round 2: ncu showed this kernel instruction-bound -- 76 % issue utilisation, 32 instructions per element, two thirds of them
  //  integer: a channel -> (t, c) division per thread and channel, a pixel -> (h, w) division per thread and tile, predicates and
  //  64-bit address arithmetic around every load.  The channel offsets and the output rows of the block's 64 channels / 128 pixels
  //  are now computed once into shared memory, and interior blocks load without predicates.)
  constexpr int PT = 4;                                            // 32-pixel tiles per block: 32 loads in flight per thread
  __shared__ float tile[PT][64][33];
  __shared__ long long s_off[64];                                  // element offset of channel ch0 + i inside the sample, -1 = padding channel
  __shared__ long long s_row[PT * 32];                             // output row (PG pixel index) of pixel px0 + i, -1 = outside the field
  __shared__ int s_pm[64];
  const int HW = p.H * p.W;
  const int px0 = blockIdx.x * 32 * PT;
  const int cblocks = p.Cpad / 64;
  const int b = blockIdx.y / cblocks, ch0 = (blockIdx.y - b * cblocks) * 64;
  const int TC = p.T * p.C;
  if (threadIdx.x < 64) {
    const int ch = ch0 + threadIdx.x;
    const int t = ch / p.C, c = ch - t * p.C;
    s_off[threadIdx.x] = ch < TC ? (long long)t * p.sT + (long long)c * p.sC : -1;
    s_pm[threadIdx.x] = (!p.prestd && ch < TC && (c == 4 || c == 10 || c == 16 || c == 22)) ? 1 : 0;       // metnet3.py:362,370
  } else if (threadIdx.x < 64 + PT * 32) {
    const int i = threadIdx.x - 64, px = px0 + i;
    long long q = -1;
    if (px < HW) { const int h = px / p.W, w = px - h * p.W; q = p.pg.q(b, h + p.pad_top, w + p.pad_left); }
    s_row[i] = q;
  }
  __syncthreads();
  const TIn* xb = reinterpret_cast<const TIn*>(p.x) + (long long)b * p.sB + px0;
  const int pl = threadIdx.x & 31, cl0 = threadIdx.x >> 5;         // lane = pixel (coalesced 128-byte rows), warp = channel
  const bool interior = px0 + 32 * PT <= HW;                       // block-uniform
  float v[PT][8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const long long off = s_off[cl0 + 8 * k];                      // warp-uniform
    if (off >= 0) {
      const TIn* xc = xb + off + pl;
      if (interior) {
#pragma unroll
        for (int u = 0; u < PT; ++u) v[u][k] = ld_in(xc + u * 32);
      } else {
#pragma unroll
        for (int u = 0; u < PT; ++u) v[u][k] = (px0 + u * 32 + pl < HW) ? ld_in(xc + u * 32) : 0.f;
      }
      if (s_pm[cl0 + 8 * k]) {
#pragma unroll
        for (int u = 0; u < PT; ++u) v[u][k] = (v[u][k] - p.mean) / p.stdv;
      }
    } else {
#pragma unroll
      for (int u = 0; u < PT; ++u) v[u][k] = 0.f;
    }
  }
#pragma unroll
  for (int u = 0; u < PT; ++u)
#pragma unroll
    for (int k = 0; k < 8; ++k) tile[u][cl0 + 8 * k][pl] = v[u][k];
  __syncthreads();
  const int wl = threadIdx.x >> 3, c8 = (threadIdx.x & 7) * 8;
#pragma unroll
  for (int u = 0; u < PT; ++u) {
    const long long q = s_row[u * 32 + wl];
    if (q >= 0) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = tile[u][c8 + j][wl];
      st8(out + q * p.Cpad + ch0 + c8, o);
    }
  }
}

// adjoint of prepare (the input gradient): g fp32 PG [q][Cpad] over B frames -> dx fp32 (B, T*C, H*W) contiguous, every element
// written.  Pad rows / columns and channels >= T*C are dropped; the PM2.5 channels (and `extra`, the station image of
// MetNet3_with_stn_imgs, metnet3.py:701) are divided by std, the derivative of their standardisation.  The tiling of
// prepare_flat_kernel in reverse: 64 channels x 128 pixels per block, read as 256-byte channel rows, written as 128-byte
// plane rows through a shared-memory transpose.
__global__ void __launch_bounds__(256) prepare_bwd_kernel(const float* __restrict__ g, int TC, int C, int HW, int W, int pad_top,
                                                          int pad_left, int Cpad, PGeom pg, float stdv, int extra,
                                                          float* __restrict__ dx) {
  constexpr int PT = 4;                                            // 32-pixel tiles per block
  __shared__ float tile[PT][64][33];
  __shared__ long long s_row[PT * 32];                             // PG row of pixel px0 + i, -1 = outside the field
  __shared__ int s_pm[64];
  const int px0 = blockIdx.x * 32 * PT;
  const int cblocks = (TC + 63) / 64;
  const int b = blockIdx.y / cblocks, ch0 = (blockIdx.y - b * cblocks) * 64;
  if (threadIdx.x < 64) {
    const int c = (ch0 + threadIdx.x) % C;
    s_pm[threadIdx.x] = c == 4 || c == 10 || c == 16 || c == 22 || c == extra;
  } else if (threadIdx.x < 64 + PT * 32) {
    const int i = threadIdx.x - 64, px = px0 + i;
    long long q = -1;
    if (px < HW) { const int h = px / W, w = px - h * W; q = pg.q(b, h + pad_top, w + pad_left); }
    s_row[i] = q;
  }
  __syncthreads();
  const int wl = threadIdx.x >> 3, c8 = (threadIdx.x & 7) * 8;
#pragma unroll
  for (int u = 0; u < PT; ++u) {
    const long long q = s_row[u * 32 + wl];
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (q >= 0) ld8(g + q * Cpad + ch0 + c8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) tile[u][c8 + j][wl] = v[j];
  }
  __syncthreads();
  const int pl = threadIdx.x & 31, cl0 = threadIdx.x >> 5;         // lane = pixel (coalesced plane rows), warp = channel
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int cl = cl0 + 8 * k, ch = ch0 + cl;
    if (ch >= TC) break;                                           // warp-uniform
    float* o = dx + ((long long)b * TC + ch) * HW + px0 + pl;
    const bool pm = s_pm[cl];
#pragma unroll
    for (int u = 0; u < PT; ++u) {
      if (px0 + u * 32 + pl < HW) {
        const float v = tile[u][cl][pl];
        o[u * 32] = pm ? v / stdv : v;
      }
    }
  }
}

// MetNet3_with_stn_imgs (metnet3.py:701): x[:, :, ch] = (x[:, :, ch] - mean) / std, written back into the CALLER's tensor
// (the reference normalises the view before its clone).  x (B,T,C,H,W) fp32 with arbitrary element strides.
__global__ void __launch_bounds__(256) standardise_channel_kernel(float* __restrict__ x, long long sB, long long sT, long long sC, long long sH,
                                                                  long long sW, int B, int T, int H, int W, int ch, float mean, float stdv) {
  const long long total = (long long)B * T * H * W;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(i % W);
    long long r = i / W;
    const int h = (int)(r % H); r /= H;
    const int t = (int)(r % T);
    const long long b = r / T;
    float* p = x + b * sB + t * sT + ch * sC + h * sH + w * sW;
    *p = (*p - mean) / stdv;
  }
}

// ================================================================================================
// time terms.  Field n = b*L + l.  temb[n] = [lead_emb(l+1) | scrambled model-time embedding] (metnet3.py:389-402,
// quirk Q1: the three (N,te) embeddings are concatenated on dim 0 and re-viewed as (N,3te)); cond[n] = lead_emb.
// The time channels are spatially constant over the whole HPxWP frame, so their contribution to the first 3x3
// convolution is a per-(field, border case, out-channel) constant tt[n][case][co] (case = 3*ry+rx; r=0 first
// row/col: tap 0 falls outside, r=2 last row/col: tap 2 outside, r=1 interior) and to the 1x1 res_conv tres[n][co].
// ================================================================================================

__global__ void time_embed_kernel(const TimeParams p) {
  const int N = p.B * p.L, ntc = p.le + 3 * p.te;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * ntc) return;
  const int n = i / ntc, c = i - n * ntc;
  float v;
  if (c < p.le) {
    v = p.emb_lead[((n % p.L) + 1) * p.le + c];
    p.cond[n * p.le + c] = v;
  } else {
    const int f = n * 3 * p.te + (c - p.le);          // flat index into the (3N, te) concatenation
    const int r = f / p.te, col = f - r * p.te;
    const int which = r / N, idx = r - which * N;     // which embedding, which field's timestamp
    const int b = idx / p.L;
    const float tv = p.ts[(long long)b * p.ts_sB + 6 * p.ts_sT + (long long)(1 + which) * p.ts_sF];   // time index 6 (Q2)
    const int k = (int)tv;                            // .int() truncation (metnet3.py:392)
    const float* e = which == 0 ? p.emb_m : (which == 1 ? p.emb_d : p.emb_h);
    const int rows = which == 0 ? 13 : (which == 1 ? 32 : 25);      // nn.Embedding(12+1 | 31+1 | 24+1) (metnet3.py:262-266)
    // nn.Embedding raises IndexError on an out-of-range row; a kernel cannot: the lookup is skipped, the field is poisoned
    // with NaN (visible in its predictions, evaluation_vit.py:256) and the sticky device flag is raised (vg_device_error)
    if (!(tv > -1.0f && tv < (float)rows)) { v = __int_as_float(0x7fc00000); if (p.err) atomicOr(p.err, VG_DEVERR_TIMESTAMP); }
    else v = e[k * p.te + col];
  }
  p.temb[i] = v;
}

__global__ void time_terms_kernel(const TimeParams p) {
  const int N = p.B * p.L, ntc = p.le + 3 * p.te;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * 10 * p.Cout) return;
  const int co = i % p.Cout, cs = (i / p.Cout) % 10, n = i / (p.Cout * 10);
  const float* te = p.temb + n * ntc;
  float acc = 0.f;
  if (cs == 9) {
    for (int c = 0; c < ntc; ++c) acc += p.w1[(long long)co * p.c_in + p.c_data + c] * te[c];
    p.tres[n * p.Cout + co] = acc;
  } else {
    const int ry = cs / 3, rx = cs - ry * 3;
    for (int ky = 0; ky < 3; ++ky) {
      if ((ry == 0 && ky == 0) || (ry == 2 && ky == 2)) continue;
      for (int kx = 0; kx < 3; ++kx) {
        if ((rx == 0 && kx == 0) || (rx == 2 && kx == 2)) continue;
        for (int c = 0; c < ntc; ++c)
          acc += p.w3[(((long long)co * p.c_in + p.c_data + c) * 3 + ky) * 3 + kx] * te[c];
      }
    }
    p.tt[(n * 9 + cs) * p.Cout + co] = acc;
  }
}

// ================================================================================================
// conditioning MLPs (tiny): out = W1 * mid(W0 * pre(cond) + b0) + b1   or   out = W0 * pre(cond) + b0
// resnet cond (metnet3.py:140-143): pre = ReLU, single layer.  FiLM (maxvit.py:130-135): Linear -> SiLU -> Linear.
// ================================================================================================
__global__ void cond_mlp_kernel(const float* __restrict__ cond, int cd, int pre_relu, const float* __restrict__ W0,
                                const float* __restrict__ b0, int hid, const float* __restrict__ W1,
                                const float* __restrict__ b1, int od, float* __restrict__ out) {
  extern __shared__ float sh[];      // cd + hid
  float* sc = sh; float* shid = sh + cd;
  const int n = blockIdx.x;
  for (int i = threadIdx.x; i < cd; i += blockDim.x) { float v = cond[n * cd + i]; sc[i] = pre_relu ? fmaxf(v, 0.f) : v; }
  __syncthreads();
  for (int j = threadIdx.x; j < hid; j += blockDim.x) {
    float a = b0 ? b0[j] : 0.f;
    for (int i = 0; i < cd; ++i) a += W0[j * cd + i] * sc[i];
    if (W1) { a = a / (1.0f + expf(-a)); shid[j] = a; }          // SiLU
    else out[(long long)n * hid + j] = a;
  }
  if (!W1) return;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int o = warp; o < od; o += nw) {
    float a = 0.f;
    for (int j = lane; j < hid; j += 32) a += W1[(long long)o * hid + j] * shid[j];
    a = warp_sum(a);
    if (lane == 0) out[(long long)n * od + o] = a + (b1 ? b1[o] : 0.f);
  }
}

// One dense layer over a FEW rows (fields) with wide weights (configs[4]: 12 fields through 512 -> 2048 -> 1024 FiLM layers and the
// 2048 -> 512 -> 2048 squeeze-excite): the weights are the traffic, so a warp owns one output row of W, reads it once with
// coalesced 16-byte loads and dots it with NF fields' inputs at a time (the inputs stay in L1).  grid (od / 8, fields / NF).
// act: 0 none, 1 ReLU, 2 SiLU, 3 sigmoid.  (The block-per-field kernels above walk each W row with one thread or one rolled
// loop: 0.4 ms / 1.0 ms per call at these widths, a chain of dependent L2 round trips.)
template <int NF>
__global__ void __launch_bounds__(256) dense_rows_kernel(const float* __restrict__ in, int N, int cd, int pre_relu,
                                                         const float* __restrict__ W, const float* __restrict__ b, int od, int act,
                                                         float* __restrict__ out, int vec) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int o = blockIdx.x * 8 + warp, n0 = blockIdx.y * NF;
  if (o >= od) return;
  float acc[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) acc[f] = 0.f;
  const float4* w4 = reinterpret_cast<const float4*>(W + (long long)o * cd);
  const float4* x4 = reinterpret_cast<const float4*>(in + (long long)n0 * cd);
  const int q = vec ? cd >> 2 : 0;
  if (!vec) {                                                  // narrow / odd input widths (the 2-wide condition of maxvit.py:130)
    for (int j = lane; j < cd; j += 32) {
      const float w = W[(long long)o * cd + j];
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        if (n0 + f < N) { const float x = in[(long long)(n0 + f) * cd + j]; acc[f] = fmaf(w, pre_relu ? fmaxf(x, 0.f) : x, acc[f]); }
      }
    }
  }
#pragma unroll 4
  for (int j = lane; j < q; j += 32) {
    const float4 w = __ldg(w4 + j);
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      if (n0 + f < N) {
        float4 x = __ldg(x4 + (long long)f * q + j);
        if (pre_relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
        acc[f] = fmaf(w.x, x.x, fmaf(w.y, x.y, fmaf(w.z, x.z, fmaf(w.w, x.w, acc[f]))));
      }
    }
  }
  const float bo = b ? b[o] : 0.f;
#pragma unroll
  for (int f = 0; f < NF; ++f) {
    float a = warp_sum(acc[f]) + bo;
    if (act == 1) a = fmaxf(a, 0.f);
    else if (act == 2) a = a / (1.0f + expf(-a));
    else if (act == 3) a = 1.0f / (1.0f + expf(-a));
    if (lane == 0 && n0 + f < N) out[(long long)(n0 + f) * od + o] = a;
  }
}

// ================================================================================================
// stem finish: per field n = b*L + l and frame pixel: v = raw3[b] + bias + tt[n][case]; ChanLayerNorm; FiLM
// (scale+1, shift); ReLU -> h1[n].  Also the per-field residual  res[n] = rawres[b] + res_bias + tres[n].
// One warp per output flat pixel q (C = 128: 4 channels per lane).  Pads are written as zeros.
// ================================================================================================

template <typename T, bool TRAIN>
__global__ void __launch_bounds__(256) stem_finish_kernel(const StemParams p, T* __restrict__ h1, float* __restrict__ res) {
  // One block per (sample b, PG row r): the L fields of a sample share raw3 / rawres, so each pixel's two rows are loaded
  // ONCE and finished for all L lead times (L2 reads / L); the per-lead constants of the row (FiLM scale / shift, the
  // residual's time term, the three border cases of the conv's time term) sit in shared memory.  Each warp walks the
  // row's pixels.  (History: pixel-per-warp with per-pixel index divisions and six table loads, 1.81 ms at 768 fields;
  // row-per-field blocks, 1.45 ms, bound by re-reading raw3 / rawres from L2 for each of the 12 leads.)
  constexpr int C = 128, LS = 6 * C;                         // per lead: film scale | film shift | tres | tt[rx = 0, 1, 2]
  extern __shared__ float s_lead[];
  const int R = p.pgN.R, P = p.pgN.P, L = p.L;
  const int b = blockIdx.x / R, r = blockIdx.x - b * R;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  T* xhat = reinterpret_cast<T*>(p.xhat);
  const int h = r - 1;
  const bool pad_row = r < 1;
  if (!pad_row) {
    const int ry = h == 0 ? 0 : (h == p.pgN.HP - 1 ? 2 : 1);
    // (round 2: the LayerNorm affine is folded into the FiLM rows here -- y = xhat G + B with G = g (scale + 1), B = b (scale + 1) + shift --
    //  two instructions per element less in a loop that ncu showed instruction-bound at 28 instructions per element)
    for (int i = threadIdx.x; i < L * LS / 4; i += 256) {
      const int l = i / (LS / 4), k = (i - l * (LS / 4)) * 4, n = b * L + l;
      float4 v4;
      if (k < 2 * C) {
        const int c = k < C ? k : k - C;
        const float4 sc = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + c);
        if (k < C) {
          const float4 g = *reinterpret_cast<const float4*>(p.ln_g + c);
          v4 = make_float4(g.x * (sc.x + 1.0f), g.y * (sc.y + 1.0f), g.z * (sc.z + 1.0f), g.w * (sc.w + 1.0f));
        } else {
          const float4 be = *reinterpret_cast<const float4*>(p.ln_b + c), sh = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + C + c);
          v4 = make_float4(fmaf(be.x, sc.x + 1.0f, sh.x), fmaf(be.y, sc.y + 1.0f, sh.y), fmaf(be.z, sc.z + 1.0f, sh.z), fmaf(be.w, sc.w + 1.0f, sh.w));
        }
      } else {
        const float* src = k < 3 * C ? p.tres + (long long)n * C + (k - 2 * C) : p.tt + ((long long)n * 9 + ry * 3) * C + (k - 3 * C);
        v4 = *reinterpret_cast<const float4*>(src);
      }
      *reinterpret_cast<float4*>(s_lead + l * LS + k) = v4;
    }
  }
  __syncthreads();
  const float4 bb = *reinterpret_cast<const float4*>(p.bias3 + c0), rb = *reinterpret_cast<const float4*>(p.bias1 + c0);
  const long long qb_row = ((long long)b * R + r) * P;       // this row in the B-image geometry (same R, P)
  for (int col = warp; col < P; col += 8) {
    const bool pad = pad_row || col < 1;
    float4 a = z, ra = z;
    if (!pad) {
      a = *reinterpret_cast<const float4*>(p.raw3 + (qb_row + col) * C + c0);
      ra = *reinterpret_cast<const float4*>(p.rawres + (qb_row + col) * C + c0);
      a.x += bb.x; a.y += bb.y; a.z += bb.z; a.w += bb.w;
      ra.x += rb.x; ra.y += rb.y; ra.z += rb.z; ra.w += rb.w;
    }
    const int w = col - 1;
    const int rx = w == 0 ? 0 : (w == p.pgN.WP - 1 ? 2 : 1);
    if (pad) {                                                // pad pixels: zeros for every lead (no branch in the main loop below)
      for (int l = 0; l < L; ++l) {
        const long long q = (((long long)(b * L + l)) * R + r) * P + col;
        Ld4<T>::st(h1 + q * C + c0, z);
        *reinterpret_cast<float4*>(res + q * C + c0) = z;
        if (xhat) {
          Ld4<T>::st(xhat + q * C + c0, z);
          if ((lane & 7) == 0) p.mask[q * 4 + (lane >> 3)] = 0u;
          if (lane == 0) p.rstd[q] = 0.f;
        }
      }
      continue;
    }
    // four leads in flight: the two warp reductions per (pixel, lead) are chains of five dependent shuffles
#pragma unroll 4
    for (int l = 0; l < L; ++l) {
      const long long q = (((long long)(b * L + l)) * R + r) * P + col;
      float y[4], rr[4], xh[4];
      unsigned nib = 0u;
      const float* sl = s_lead + l * LS + c0;
      const float4 f0 = *reinterpret_cast<const float4*>(sl), f1 = *reinterpret_cast<const float4*>(sl + C);
      const float4 rt = *reinterpret_cast<const float4*>(sl + 2 * C), tt = *reinterpret_cast<const float4*>(sl + (3 + rx) * C);
      float v[4] = {a.x + tt.x, a.y + tt.y, a.z + tt.z, a.w + tt.w};
      const float mean = warp_sum(v[0] + v[1] + v[2] + v[3]) * (1.0f / C);
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) { v[i] -= mean; ss += v[i] * v[i]; }
      const float rstd = rsqrtf(fmaxf(warp_sum(ss) * (1.0f / C), p.eps));
      const float sc[4] = {f0.x, f0.y, f0.z, f0.w}, t[4] = {f1.x, f1.y, f1.z, f1.w};       // folded affine: G, B
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        xh[i] = v[i] * rstd;
        const float zz = fmaf(xh[i], sc[i], t[i]);
        if (TRAIN && zz > 0.f) nib |= 1u << i;
        y[i] = fmaxf(zz, 0.f);
      }
      rr[0] = ra.x + rt.x; rr[1] = ra.y + rt.y; rr[2] = ra.z + rt.z; rr[3] = ra.w + rt.w;
      Ld4<T>::st(h1 + q * C + c0, make_float4(y[0], y[1], y[2], y[3]));
      *reinterpret_cast<float4*>(res + q * C + c0) = make_float4(rr[0], rr[1], rr[2], rr[3]);
      if (TRAIN && xhat) {                            // training: what the backward pass needs
        Ld4<T>::st(xhat + q * C + c0, make_float4(xh[0], xh[1], xh[2], xh[3]));
        unsigned wbits = nib << ((lane & 7) * 4);
        wbits |= __shfl_xor_sync(0xffffffffu, wbits, 1);
        wbits |= __shfl_xor_sync(0xffffffffu, wbits, 2);
        wbits |= __shfl_xor_sync(0xffffffffu, wbits, 4);
        if ((lane & 7) == 0) p.mask[q * 4 + (lane >> 3)] = wbits;
        if (lane == 0) p.rstd[q] = rstd;
      }
    }
  }
  // the single extra pad row that closes the PG buffer (row index N*R)
  if (blockIdx.x == gridDim.x - 1) {
    const long long rowl = (long long)p.pgN.N * R;
    for (int col = warp; col < P; col += 8) {
      const long long q = rowl * P + col;
      Ld4<T>::st(h1 + q * C + c0, z);
      *reinterpret_cast<float4*>(res + q * C + c0) = z;
      if (xhat) {
        Ld4<T>::st(xhat + q * C + c0, z);
        if ((lane & 7) == 0) p.mask[q * 4 + (lane >> 3)] = 0u;
        if (lane == 0) p.rstd[q] = 0.f;
      }
    }
  }
}

// ================================================================================================
// 3xTF32 operand split (see vg_split3_tf32 in include/vitgrid.h): one float4 of the input -> three float4s of the output row
// ================================================================================================
__global__ void __launch_bounds__(256) split3_tf32_kernel(const float* __restrict__ in, long long rows, int K, float* __restrict__ out, int pattern) {
  const int k4 = K >> 2;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * k4) return;
  const long long r = i / k4;
  const int c = (int)(i - r * k4) * 4;
  const float4 x = *reinterpret_cast<const float4*>(in + r * K + c);
  float4 hi, lo;
  hi.x = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u); hi.y = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
  hi.z = __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u); hi.w = __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
  lo.x = x.x - hi.x; lo.y = x.y - hi.y; lo.z = x.z - hi.z; lo.w = x.w - hi.w;      // exact in fp32
  float* o = out + r * 3 * K + c;
  *reinterpret_cast<float4*>(o) = hi;
  *reinterpret_cast<float4*>(o + K) = pattern ? lo : hi;
  *reinterpret_cast<float4*>(o + 2 * K) = pattern ? hi : lo;
}

int split3_tf32_run(const float* in, long long rows, int K, float* out, int pattern, cudaStream_t st) {
  if (K % 4 || (((uintptr_t)in | (uintptr_t)out) & 15)) return set_error("split3_tf32: K = %d must be a multiple of 4 and both pointers 16-byte aligned", K);
  if (pattern != 0 && pattern != 1) return set_error("split3_tf32: pattern %d (0 = [hi|hi|lo], 1 = [hi|lo|hi])", pattern);
  if (rows <= 0) return 0;
  const long long total = rows * (K / 4);
  split3_tf32_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, rows, K, out, pattern);
  return check_launch("split3_tf32_kernel");
}

// ================================================================================================
// 2x2 max-pool: PG layout (N,HP,WP,C) -> plain channels-last (N,HP/2,WP/2,C)   (metnet3.py:86,419)
// ================================================================================================
template <typename T, typename TO>
__global__ void __launch_bounds__(256) maxpool2_kernel(const T* __restrict__ in, TO* __restrict__ out, PGeom pg, int C) {
  const int Ho = pg.HP / 2, Wo = pg.WP / 2, cv = C / 8;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)pg.N * Ho * Wo * cv;
  if (i >= total) return;
  const int c8 = (int)(i % cv) * 8;
  long long p = i / cv;
  const int wo = (int)(p % Wo); p /= Wo;
  const int ho = (int)(p % Ho); const int n = (int)(p / Ho);
  float m[8], v[8];
  ld8(in + pg.q(n, 2 * ho, 2 * wo) * C + c8, m);
#pragma unroll
  for (int k = 1; k < 4; ++k) {
    ld8(in + pg.q(n, 2 * ho + (k >> 1), 2 * wo + (k & 1)) * C + c8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], v[j]);
  }
  st8(out + (((long long)n * Ho + ho) * Wo + wo) * C + c8, m);
}

// ================================================================================================
// depthwise 3x3 (pad 1) + folded BatchNorm + GELU(erf) on plain channels-last (N,H,W,C); also emits per-(n,row)
// channel sums for the squeeze-excite mean (deterministic two-stage reduction, no atomics).  maxvit.py:91-93,39
// block = one (n, row): C/8 channel groups x WL w-lanes.
// ================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) dwconv3x3_kernel(const T* __restrict__ in, const float* __restrict__ w9,
                                                        const float* __restrict__ scale, const float* __restrict__ shift,
                                                        T* __restrict__ out, float* __restrict__ psum, int H, int W, int C) {
  extern __shared__ float red[];               // [WL][C]
  const int cg = C / 8, WL = blockDim.x / cg;
  const int g = threadIdx.x % cg, wl = threadIdx.x / cg, c8 = g * 8;
  const int h = blockIdx.x % H, n = blockIdx.x / H;
  float wk[9][8], sc[8], sh[8], acc_sum[8];
#pragma unroll
  for (int k = 0; k < 9; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) wk[k][j] = w9[k * C + c8 + j];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = scale[c8 + j]; sh[j] = shift[c8 + j]; acc_sum[j] = 0.f; }
  const T* base = in + (long long)n * H * W * C;
  if (wl < WL) {
    for (int w = wl; w < W; w += WL) {
      float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, v[8];
#pragma unroll
      for (int dy = -1; dy <= 1; ++dy) {
        const int hh = h + dy;
        if (hh < 0 || hh >= H) continue;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
          const int ww = w + dx;
          if (ww < 0 || ww >= W) continue;
          ld8(base + ((long long)hh * W + ww) * C + c8, v);
#pragma unroll
          for (int j = 0; j < 8; ++j) a[j] = fmaf(v[j], wk[(dy + 1) * 3 + dx + 1][j], a[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        const float2 g = gelu_erf2(f2_fma(make_float2(a[j], a[j + 1]), make_float2(sc[j], sc[j + 1]), make_float2(sh[j], sh[j + 1])));
        a[j] = g.x; a[j + 1] = g.y;
      }
      st8(out + (((long long)n * H + h) * W + w) * C + c8, a);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc_sum[j] += a[j];               // SE mean over the fp32 values
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[wl * C + c8 + j] = acc_sum[j];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int l = 0; l < WL; ++l) s += red[l * C + c];
    psum[((long long)n * H + h) * C + c] = s;
  }
}

// x[n][p][c] *= gate[n][c]   (in place)
template <typename T>
__global__ void __launch_bounds__(256) se_scale_kernel(T* __restrict__ x, const float* __restrict__ gate, long long HW, int C, long long total_vec) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_vec) return;
  const int cv = C / 8;
  const int c8 = (int)(i % cv) * 8;
  const long long n = (i / cv) / HW;
  float v[8];
  ld8(x + i * 8, v);
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] *= gate[n * C + c8 + j];
  st8(x + i * 8, v);
}

// register-token mean over windows (maxvit.py:326): (N, nwin, R*C) -> (N, R*C), fp32
__global__ void reg_mean_kernel(const float* __restrict__ in, float* __restrict__ out, int nwin, int RC, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / RC; const int k = (int)(i - n * RC);
  float s = 0.f;
  for (int w = 0; w < nwin; ++w) s += in[(n * nwin + w) * RC + k];
  out[i] = s / (float)nwin;
}

// ================================================================================================
// head (metnet3.py:424-430): unpad, 1x1 conv C->1, *std + mean.  One warp per output pixel.
// ================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) head_kernel(const T* __restrict__ h, const float* __restrict__ w, float bias, float stdv,
                                                   float mean, PGeom pg, int C, int H, int W, int pad_top, int pad_left,
                                                   float* __restrict__ out, long long total) {
  const long long i = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= total) return;
  const int lane = threadIdx.x & 31;
  int x, y, n;
  if (total < (1ll << 31)) {                                 // 32-bit divisions (the 64-bit ones are software routines)
    const unsigned iu = (unsigned)i, t = iu / (unsigned)W;
    x = (int)(iu - t * (unsigned)W); n = (int)(t / (unsigned)H); y = (int)(t - (unsigned)n * (unsigned)H);
  } else {
    x = (int)(i % W); const long long t = i / W;
    y = (int)(t % H); n = (int)(t / H);
  }
  const T* p = h + pg.q(n, y + pad_top, x + pad_left) * C;
  float a = 0.f;
  if ((C & 127) == 0) {                                      // four channels per lane and 128-channel block: one vector load each
    for (int c = lane * 4; c < C; c += 128) {
      float v[4];
      if constexpr (sizeof(T) == 4) { const float4 f = *reinterpret_cast<const float4*>(p + c); v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w; }
      else {
        const uint2 u = *reinterpret_cast<const uint2*>(p + c);
        const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x)), hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
      }
      const float4 w4 = *reinterpret_cast<const float4*>(w + c);
      a = fmaf(v[0], w4.x, a); a = fmaf(v[1], w4.y, a); a = fmaf(v[2], w4.z, a); a = fmaf(v[3], w4.w, a);
    }
  } else {
    for (int c = lane; c < C; c += 32) a += Act<T>::ld(p + c) * w[c];
  }
  a = warp_sum(a);
  if (lane == 0) out[i] = (a + bias) * stdv + mean;
}

// ================================================================================================
// Channel widths other than 128 (n_start_channels = 256 / 384 / 512, BASELINE configs[4]).  The fused conv kernels keep
// one 128-channel row per TMEM lane; wider networks run the 3x3 convolution as a plain tcgen05 shifted-row GEMM into an
// fp32 scratch [q][C] and finish with the row kernels below (HBM-bound: one warp per pixel, lane owns channels
// i*128 + lane*4 .. +3, statistics by warp shuffles).  Same math as epi_conv_ln / stem_finish_kernel.
// ================================================================================================
struct WideRowParams {
  const float* acc;                          // [q][C] GEMM result (no bias)
  const float* bias; const float* ln_g; const float* ln_b; float eps;
  const float* film;                         // (N, 2C) or null
  const void* res; int res_f32;              // residual [q][C] (fp32 or T) or null
  void* out; float* out2;                    // [q][C] in T (or null) / fp32 copy (or null)
  const float* head_w; float* head_out; float head_b, head_std, head_mean; int head_H, head_W, head_pt, head_pl;
  int C;
  PGeom pg;
};

template <typename T>
__global__ void __launch_bounds__(256) conv_ln_rows_kernel(const WideRowParams p) {
  const long long q = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (q >= p.pg.pixels()) return;
  const int lane = threadIdx.x & 31, C = p.C, nv = C >> 7;
  int n = 0, h = 0, w = 0;
  const bool valid = p.pg.decode(q, n, h, w);
  float4 y[4];
  float head = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) y[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) {
        const int c = i * 128 + lane * 4;
        const float4 a = *reinterpret_cast<const float4*>(p.acc + q * C + c), b = *reinterpret_cast<const float4*>(p.bias + c);
        y[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
        s += (y[i].x + y[i].y) + (y[i].z + y[i].w);
      }
    const float mean = warp_sum(s) / (float)C;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) {
        y[i].x -= mean; y[i].y -= mean; y[i].z -= mean; y[i].w -= mean;
        ss += y[i].x * y[i].x + y[i].y * y[i].y + y[i].z * y[i].z + y[i].w * y[i].w;
      }
    const float rstd = rsqrtf(fmaxf(warp_sum(ss) / (float)C, p.eps));       // var.clamp(min=eps).rsqrt()  (metnet3.py:104)
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) {
        const int c = i * 128 + lane * 4;
        const float4 g = *reinterpret_cast<const float4*>(p.ln_g + c), b = *reinterpret_cast<const float4*>(p.ln_b + c);
        float z[4] = {y[i].x * rstd * g.x + b.x, y[i].y * rstd * g.y + b.y, y[i].z * rstd * g.z + b.z, y[i].w * rstd * g.w + b.w};
        if (p.film) {
          const float4 sc = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + c);
          const float4 sh = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + C + c);
          z[0] = z[0] * (sc.x + 1.0f) + sh.x; z[1] = z[1] * (sc.y + 1.0f) + sh.y;
          z[2] = z[2] * (sc.z + 1.0f) + sh.z; z[3] = z[3] * (sc.w + 1.0f) + sh.w;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) z[k] = fmaxf(z[k], 0.f);
        if (p.res) {
          const float4 r = p.res_f32 ? *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.res) + q * C + c)
                                     : Ld4<T>::ld(reinterpret_cast<const T*>(p.res) + q * C + c);
          z[0] += r.x; z[1] += r.y; z[2] += r.z; z[3] += r.w;
        }
        y[i] = make_float4(z[0], z[1], z[2], z[3]);
        if (p.head_w) {
          const float4 hw = *reinterpret_cast<const float4*>(p.head_w + c);
          head += z[0] * hw.x + z[1] * hw.y + z[2] * hw.z + z[3] * hw.w;
        }
      }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (i < nv) {
      const int c = i * 128 + lane * 4;
      if (p.out) Ld4<T>::st(reinterpret_cast<T*>(p.out) + q * C + c, y[i]);
      if (p.out2) *reinterpret_cast<float4*>(p.out2 + q * C + c) = y[i];
    }
  if (p.head_w && valid) {
    head = warp_sum(head);
    const int hh = h - p.head_pt, ww = w - p.head_pl;
    if (lane == 0 && hh >= 0 && hh < p.head_H && ww >= 0 && ww < p.head_W)
      p.head_out[((long long)n * p.head_H + hh) * p.head_W + ww] = (head + p.head_b) * p.head_std + p.head_mean;
  }
}

// stem_finish_kernel for C = 128 * nv (inference only)
template <typename T>
__global__ void __launch_bounds__(256) stem_finish_wide_kernel(const StemParams p, int C, T* __restrict__ h1, float* __restrict__ res) {
  const long long q = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (q >= p.pgN.pixels()) return;
  const int lane = threadIdx.x & 31, nv = C >> 7;
  int n = 0, h = 0, w = 0;
  const bool valid = p.pgN.decode(q, n, h, w);
  float4 y[4], r[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) y[i] = r[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) {
    const int b = n / p.L;
    const long long qb = p.pgB.q(b, h, w);
    const int ry = h == 0 ? 0 : (h == p.pgN.HP - 1 ? 2 : 1), rx = w == 0 ? 0 : (w == p.pgN.WP - 1 ? 2 : 1);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) {
        const int c = i * 128 + lane * 4;
        const float4 a = *reinterpret_cast<const float4*>(p.raw3 + qb * C + c), bb = *reinterpret_cast<const float4*>(p.bias3 + c);
        const float4 tt = *reinterpret_cast<const float4*>(p.tt + ((long long)n * 9 + ry * 3 + rx) * C + c);
        y[i] = make_float4(a.x + bb.x + tt.x, a.y + bb.y + tt.y, a.z + bb.z + tt.z, a.w + bb.w + tt.w);
        s += (y[i].x + y[i].y) + (y[i].z + y[i].w);
        const float4 ra = *reinterpret_cast<const float4*>(p.rawres + qb * C + c), rb = *reinterpret_cast<const float4*>(p.bias1 + c);
        const float4 rt = *reinterpret_cast<const float4*>(p.tres + (long long)n * C + c);
        r[i] = make_float4(ra.x + rb.x + rt.x, ra.y + rb.y + rt.y, ra.z + rb.z + rt.z, ra.w + rb.w + rt.w);
      }
    const float mean = warp_sum(s) / (float)C;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) {
        y[i].x -= mean; y[i].y -= mean; y[i].z -= mean; y[i].w -= mean;
        ss += y[i].x * y[i].x + y[i].y * y[i].y + y[i].z * y[i].z + y[i].w * y[i].w;
      }
    const float rstd = rsqrtf(fmaxf(warp_sum(ss) / (float)C, p.eps));
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) {
        const int c = i * 128 + lane * 4;
        const float4 g = *reinterpret_cast<const float4*>(p.ln_g + c), be = *reinterpret_cast<const float4*>(p.ln_b + c);
        const float4 sc = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + c);
        const float4 sh = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + C + c);
        y[i].x = fmaxf((y[i].x * rstd * g.x + be.x) * (sc.x + 1.0f) + sh.x, 0.f);
        y[i].y = fmaxf((y[i].y * rstd * g.y + be.y) * (sc.y + 1.0f) + sh.y, 0.f);
        y[i].z = fmaxf((y[i].z * rstd * g.z + be.z) * (sc.z + 1.0f) + sh.z, 0.f);
        y[i].w = fmaxf((y[i].w * rstd * g.w + be.w) * (sc.w + 1.0f) + sh.w, 0.f);
      }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (i < nv) {
      const int c = i * 128 + lane * 4;
      Ld4<T>::st(h1 + q * C + c, y[i]);
      *reinterpret_cast<float4*>(res + q * C + c) = r[i];
    }
}

// ================================================================================================
// Focal-R loss (not in the reference; README.md:16): loss = mean(|e| * (2*sigmoid(beta*|e|)-1)^gamma)
// ================================================================================================
__device__ __forceinline__ float focal_term(float e, float beta, float gamma, int mse, float* dterm) {
  const float ae = fabsf(e);
  const float s = 1.0f / (1.0f + expf(-beta * ae));
  const float wgt = 2.0f * s - 1.0f;
  const float wg = gamma == 1.0f ? wgt : powf(wgt, gamma);
  const float base = mse ? ae * ae : ae;
  if (dterm) {
    const float dw = 2.0f * beta * s * (1.0f - s);
    const float wgm1 = gamma == 1.0f ? 1.0f : (wgt > 0.f ? powf(wgt, gamma - 1.0f) : 0.f);
    const float dbase = mse ? 2.0f * ae : 1.0f;
    const float d = dbase * wg + base * gamma * wgm1 * dw;
    *dterm = e > 0.f ? d : (e < 0.f ? -d : 0.f);
  }
  return base * wg;
}

__global__ void __launch_bounds__(256) focal_r_partial_kernel(const float* __restrict__ pred, const float* __restrict__ tgt,
                                                              long long n, float beta, float gamma, int mse, float* __restrict__ partial) {
  __shared__ float sw[8];
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc += focal_term(pred[i] - tgt[i], beta, gamma, mse, nullptr);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) { float s = 0.f; for (int i = 0; i < 8; ++i) s += sw[i]; partial[blockIdx.x] = s; }
}
__global__ void focal_r_final_kernel(const float* __restrict__ partial, int nb, float inv_n, float* __restrict__ loss) {
  __shared__ float sw[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) acc += partial[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) { float s = 0.f; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += sw[i]; *loss = s * inv_n; }
}
__global__ void __launch_bounds__(256) focal_r_bwd_kernel(const float* __restrict__ pred, const float* __restrict__ tgt, long long n,
                                                          float beta, float gamma, int mse, float gscale, float* __restrict__ grad) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float d; focal_term(pred[i] - tgt[i], beta, gamma, mse, &d);
    grad[i] = d * gscale;
  }
}

// ================================================================================================
// host launchers (called from vg_api.cu)
// ================================================================================================
static inline unsigned nblk(long long total, int per) { return (unsigned)((total + per - 1) / per); }

int prepare_run(int dtype, const void* x, int x_bf16, int prestd, const long long* xs, int B, int T, int C, int H, int W, int pad_top,
                int pad_left, int HP, int WP, int Cpad, float mean, float stdv, void* out, cudaStream_t st) {
  if (Cpad % 64 || Cpad < T * C) return set_error("prepare: Cpad=%d must be a multiple of 64 and >= T*C=%d", Cpad, T * C);
  PrepParams p;
  p.x = x; p.sB = xs[0]; p.sT = xs[1]; p.sC = xs[2]; p.sH = xs[3]; p.sW = xs[4];
  p.B = B; p.T = T; p.C = C; p.H = H; p.W = W; p.pad_top = pad_top; p.pad_left = pad_left; p.Cpad = Cpad;
  p.mean = mean; p.stdv = stdv; p.prestd = prestd; p.pg = make_pgeom(B, HP, WP); p.w_fast = (xs[4] == 1);
  const size_t esz = dtype == 0 ? 2 : 4;
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)p.pg.pixels() * Cpad * esz, st);
  if (e != cudaSuccess) return set_error("prepare memset: %s", cudaGetErrorString(e));
  const bool flat = xs[4] == 1 && xs[3] == W;                  // contiguous (H, W) planes
  dim3 gridf((unsigned)((H * W + 127) / 128), (unsigned)(B * (Cpad / 64)));
  dim3 grid((W + 31) / 32, H, B * (Cpad / 64));
#define VG_PREP(TO, TI)                                                                                             \
  do {                                                                                                              \
    if (flat) prepare_flat_kernel<TO, TI><<<gridf, 256, 0, st>>>(p, reinterpret_cast<TO*>(out));                    \
    else prepare_kernel<TO, TI><<<grid, 256, 0, st>>>(p, reinterpret_cast<TO*>(out));                               \
  } while (0)
  if (dtype == 0) { if (x_bf16) VG_PREP(bf16, bf16); else VG_PREP(bf16, float); }
  else { if (x_bf16) VG_PREP(float, bf16); else VG_PREP(float, float); }
#undef VG_PREP
  return check_launch(flat ? "prepare_flat_kernel" : "prepare_kernel");
}

int prepare_bwd_run(const float* g, int B, int T, int C, int H, int W, int pad_top, int pad_left, int HP, int WP, int Cpad,
                    float stdv, int extra, float* dx, cudaStream_t st) {
  if (Cpad % 64 || Cpad < T * C) return set_error("prepare_bwd: Cpad=%d must be a multiple of 64 and >= T*C=%d", Cpad, T * C);
  if (extra < -1 || extra >= C) return set_error("prepare_bwd: extra channel %d outside [-1, %d)", extra, C);
  if (pad_top < 0 || pad_left < 0 || H + pad_top > HP || W + pad_left > WP)
    return set_error("prepare_bwd: the %dx%d field at (%d, %d) does not fit the %dx%d frame", H, W, pad_top, pad_left, HP, WP);
  if (B <= 0 || T * C <= 0 || H * W <= 0) return 0;
  dim3 grid((unsigned)((H * W + 127) / 128), (unsigned)(B * ((T * C + 63) / 64)));
  prepare_bwd_kernel<<<grid, 256, 0, st>>>(g, T * C, C, H * W, W, pad_top, pad_left, Cpad, make_pgeom(B, HP, WP), stdv, extra, dx);
  return check_launch("prepare_bwd_kernel");
}

int standardise_channel_run(float* x, const long long* xs, int B, int T, int C, int H, int W, int ch, float mean, float stdv, cudaStream_t st) {
  if (ch < 0 || ch >= C) return set_error("standardise_channel: channel %d outside [0, %d)", ch, C);
  const long long total = (long long)B * T * H * W;
  if (total <= 0) return 0;
  const unsigned grid = (unsigned)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  standardise_channel_kernel<<<grid, 256, 0, st>>>(x, xs[0], xs[1], xs[2], xs[3], xs[4], B, T, H, W, ch, mean, stdv);
  return check_launch("standardise_channel_kernel");
}

int time_terms_run(const TimeParams& p, cudaStream_t st) {
  const int N = p.B * p.L, ntc = p.le + 3 * p.te;
  time_embed_kernel<<<nblk((long long)N * ntc, 128), 128, 0, st>>>(p);
  int rc = check_launch("time_embed_kernel");
  if (rc) return rc;
  time_terms_kernel<<<nblk((long long)N * 10 * p.Cout, 256), 256, 0, st>>>(p);
  return check_launch("time_terms_kernel");
}

int cond_mlp_run(const float* cond, int N, int cd, int pre_relu, const float* W0, const float* b0, int hid,
                 const float* W1, const float* b1, int od, float* out, cudaStream_t st) {
  cond_mlp_kernel<<<N, 256, (cd + hid) * sizeof(float), st>>>(cond, cd, pre_relu, W0, b0, hid, W1, b1, od, out);
  return check_launch("cond_mlp_kernel");
}

int dense_rows_run(const float* in, int N, int cd, int pre_relu, const float* W, const float* b, int od, int act, float* out,
                   cudaStream_t st) {
  if (act < 0 || act > 3) return set_error("dense_rows: activation code %d (0 none, 1 ReLU, 2 SiLU, 3 sigmoid)", act);
  const int vec = cd % 4 == 0 && (((uintptr_t)in | (uintptr_t)W) & 15) == 0;
  if (N <= 0 || od <= 0) return 0;
  constexpr int NF = 4;
  dense_rows_kernel<NF><<<dim3(nblk(od, 8), nblk(N, NF)), 256, 0, st>>>(in, N, cd, pre_relu, W, b, od, act, out, vec);
  return check_launch("dense_rows_kernel");
}

int stem_finish_run(int dtype, const StemParams& p, void* h1, float* res, cudaStream_t st) {
  const unsigned g = (unsigned)(p.pgB.N * p.pgB.R);          // one block per (sample, PG row)
  const size_t smem = (size_t)p.L * 6 * 128 * sizeof(float);
  if (smem > 200 * 1024) return set_error("stem_finish: %d lead times need %zu bytes of shared memory", p.L, smem);
  static PerDeviceSize attr_pd;
  size_t& attr_cur = attr_pd.cur();
  if (smem > attr_cur) {
    cudaError_t e = cudaFuncSetAttribute(stem_finish_kernel<bf16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(stem_finish_kernel<bf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(stem_finish_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(stem_finish_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error("stem_finish smem attr: %s", cudaGetErrorString(e));
    attr_cur = smem;
  }
  const bool train = p.xhat != nullptr;
  if (dtype == 0) { if (train) stem_finish_kernel<bf16, true><<<g, 256, smem, st>>>(p, reinterpret_cast<bf16*>(h1), res); else stem_finish_kernel<bf16, false><<<g, 256, smem, st>>>(p, reinterpret_cast<bf16*>(h1), res); }
  else { if (train) stem_finish_kernel<float, true><<<g, 256, smem, st>>>(p, reinterpret_cast<float*>(h1), res); else stem_finish_kernel<float, false><<<g, 256, smem, st>>>(p, reinterpret_cast<float*>(h1), res); }
  return check_launch("stem_finish_kernel");
}

int stem_finish_wide_run(int dtype, const StemParams& p, int C, void* h1, float* res, cudaStream_t st) {
  if (C % 128 || C < 128 || C > 512) return set_error("stem_finish_wide: C=%d must be 128, 256, 384 or 512", C);
  const unsigned g = nblk(p.pgN.pixels(), 8);
  if (dtype == 0) stem_finish_wide_kernel<bf16><<<g, 256, 0, st>>>(p, C, reinterpret_cast<bf16*>(h1), res);
  else stem_finish_wide_kernel<float><<<g, 256, 0, st>>>(p, C, reinterpret_cast<float*>(h1), res);
  return check_launch("stem_finish_wide_kernel");
}

int conv_ln_rows_run(int dtype, const float* acc, int C, const float* bias, const float* ln_g, const float* ln_b, float eps,
                     const float* film, const void* res, int res_f32, void* out, float* out2, const PGeom& pg,
                     const float* head_w, float head_b, float head_std, float head_mean, int H, int W, int pad_top,
                     int pad_left, float* head_out, cudaStream_t st) {
  if (C % 128 || C < 128 || C > 512) return set_error("conv_ln_rows: C=%d must be 128, 256, 384 or 512", C);
  WideRowParams p;
  p.acc = acc; p.bias = bias; p.ln_g = ln_g; p.ln_b = ln_b; p.eps = eps; p.film = film; p.res = res; p.res_f32 = res_f32;
  p.out = out; p.out2 = out2; p.head_w = head_w; p.head_out = head_out; p.head_b = head_b; p.head_std = head_std;
  p.head_mean = head_mean; p.head_H = H; p.head_W = W; p.head_pt = pad_top; p.head_pl = pad_left; p.C = C; p.pg = pg;
  const unsigned g = nblk(pg.pixels(), 8);
  if (dtype == 0) conv_ln_rows_kernel<bf16><<<g, 256, 0, st>>>(p);
  else conv_ln_rows_kernel<float><<<g, 256, 0, st>>>(p);
  return check_launch("conv_ln_rows_kernel");
}

int maxpool2_run(int dtype, int out_f32, const void* in, void* out, int N, int HP, int WP, int C, cudaStream_t st) {
  if (C % 8 || HP % 2 || WP % 2) return set_error("maxpool2: bad shape");
  PGeom pg = make_pgeom(N, HP, WP);
  const long long total = (long long)N * (HP / 2) * (WP / 2) * (C / 8);
  if (dtype == 0 && out_f32) maxpool2_kernel<bf16, float><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<const bf16*>(in), reinterpret_cast<float*>(out), pg, C);
  else if (dtype == 0) maxpool2_kernel<bf16, bf16><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<const bf16*>(in), reinterpret_cast<bf16*>(out), pg, C);
  else maxpool2_kernel<float, float><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<const float*>(in), reinterpret_cast<float*>(out), pg, C);
  return check_launch("maxpool2_kernel");
}

int dwconv_run(int dtype, const void* in, const float* w9, const float* scale, const float* shift, void* out, float* psum,
               int N, int H, int W, int C, cudaStream_t st) {
  if (C % 8) return set_error("dwconv: C %% 8 != 0");
  const int cg = C / 8;
  int threads = 256;
  if (cg > 256) return set_error("dwconv: C=%d too large", C);
  const int WL = threads / cg;
  threads = WL * cg;
  const size_t smem = (size_t)WL * C * sizeof(float);
  if (dtype == 0) dwconv3x3_kernel<bf16><<<N * H, threads, smem, st>>>(reinterpret_cast<const bf16*>(in), w9, scale, shift, reinterpret_cast<bf16*>(out), psum, H, W, C);
  else dwconv3x3_kernel<float><<<N * H, threads, smem, st>>>(reinterpret_cast<const float*>(in), w9, scale, shift, reinterpret_cast<float*>(out), psum, H, W, C);
  return check_launch("dwconv3x3_kernel");
}

int se_scale_run(int dtype, void* x, const float* gate, int N, long long HW, int C, cudaStream_t st) {
  const long long total = (long long)N * HW * (C / 8);
  if (dtype == 0) se_scale_kernel<bf16><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<bf16*>(x), gate, HW, C, total);
  else se_scale_kernel<float><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<float*>(x), gate, HW, C, total);
  return check_launch("se_scale_kernel");
}

int reg_mean_run(const float* in, float* out, int N, int nwin, int RC, cudaStream_t st) {
  const long long total = (long long)N * RC;
  reg_mean_kernel<<<nblk(total, 256), 256, 0, st>>>(in, out, nwin, RC, total);
  return check_launch("reg_mean_kernel");
}

int head_run(int dtype, const void* h, const float* w, float bias, float stdv, float mean, int N, int HP, int WP, int C,
             int H, int W, int pad_top, int pad_left, float* out, cudaStream_t st) {
  PGeom pg = make_pgeom(N, HP, WP);
  const long long total = (long long)N * H * W;
  if (dtype == 0) head_kernel<bf16><<<nblk(total, 8), 256, 0, st>>>(reinterpret_cast<const bf16*>(h), w, bias, stdv, mean, pg, C, H, W, pad_top, pad_left, out, total);
  else head_kernel<float><<<nblk(total, 8), 256, 0, st>>>(reinterpret_cast<const float*>(h), w, bias, stdv, mean, pg, C, H, W, pad_top, pad_left, out, total);
  return check_launch("head_kernel");
}

int focal_r_fwd_run(const float* pred, const float* tgt, long long n, float beta, float gamma, int mse, float* partial,
                    int nb, float* loss, cudaStream_t st) {
  focal_r_partial_kernel<<<nb, 256, 0, st>>>(pred, tgt, n, beta, gamma, mse, partial);
  int rc = check_launch("focal_r_partial_kernel");
  if (rc) return rc;
  focal_r_final_kernel<<<1, 256, 0, st>>>(partial, nb, 1.0f / (float)n, loss);
  return check_launch("focal_r_final_kernel");
}

int focal_r_bwd_run(const float* pred, const float* tgt, long long n, float beta, float gamma, int mse, float gscale,
                    float* grad, cudaStream_t st) {
  focal_r_bwd_kernel<<<nblk(n, 256 * 4) < 4096 ? nblk(n, 256 * 4) : 4096, 256, 0, st>>>(pred, tgt, n, beta, gamma, mse, gscale, grad);
  return check_launch("focal_r_bwd_kernel");
}

}  // namespace vg
