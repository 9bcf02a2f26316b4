// Training kernels of the MaxViT block (maxvit.py:33-102 MBConv with batch-statistic BatchNorm, :170-219 attention):
// column statistics, BatchNorm apply / backward, depthwise 3x3 (marching stencil, also the inference kernel),
// squeeze-excite backward, and the attention backward (out-projection gather, per-(field, head) core backward with the
// relative-position-bias gradient accumulated in shared memory, LayerNorm + FiLM backward with the inverse partition).
// The dense projections' dgrad / wgrad run on the tcgen05 GEMMs (vg_gemm.cu, vg_wgrad.cu).
#include "vg_common.cuh"
#include "vg_host.h"
#include "vg_rng.cuh"

namespace vg {

static inline unsigned nblk(long long total, int per) { return (unsigned)((total + per - 1) / per); }

__device__ __forceinline__ float gelu_grad(float u) {
  const float cdf = 0.5f * (1.0f + erf_as(u * 0.70710678118654752440f));
  return cdf + u * 0.3989422804014327f * __expf(-0.5f * u * u);
}

// ================================================================================================
// column statistics of X fp32 [M][C]: partial (sum, sum of squares) per 256-row block, combined in double.
// ================================================================================================
constexpr int STAT_ROWS = 256;

__global__ void __launch_bounds__(256) colstats_kernel(const float* __restrict__ X, long long M, int C, float* __restrict__ part) {
  const long long r0 = (long long)blockIdx.x * STAT_ROWS;
  long long r1 = r0 + STAT_ROWS;
  if (r1 > M) r1 = M;
  for (int c = threadIdx.x; c < C; c += 256) {
    float s = 0.f, s2 = 0.f;
    for (long long r = r0; r < r1; ++r) { const float v = X[r * C + c]; s += v; s2 = fmaf(v, v, s2); }
    part[((long long)blockIdx.x * 2) * C + c] = s;
    part[((long long)blockIdx.x * 2 + 1) * C + c] = s2;
  }
}

// Sum of the per-block partials part[p][2][C] over p for channel c, by the 8 slices (threadIdx.x >> 5) of a 256-thread block that
// covers 32 channels: the single-thread loop over ~1000-2000 partials was a chain of dependent L2 round trips (170 us per
// launch for a kernel that moves 4 MB).  Returns the totals to every thread of the channel.
__device__ __forceinline__ void sum_parts2(const float* __restrict__ part, int nparts, int C, int c, double& s1, double& s2) {
  __shared__ double red[2][8][32];
  const int slice = threadIdx.x >> 5, l = threadIdx.x & 31;
  double a = 0.0, b = 0.0;
  if (c < C) {
    int p = slice;
    for (; p + 24 < nparts; p += 32) {
      const float a0 = part[((long long)p * 2) * C + c], b0 = part[((long long)p * 2 + 1) * C + c];
      const float a1 = part[((long long)(p + 8) * 2) * C + c], b1 = part[((long long)(p + 8) * 2 + 1) * C + c];
      const float a2 = part[((long long)(p + 16) * 2) * C + c], b2 = part[((long long)(p + 16) * 2 + 1) * C + c];
      const float a3 = part[((long long)(p + 24) * 2) * C + c], b3 = part[((long long)(p + 24) * 2 + 1) * C + c];
      a += ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
      b += ((double)b0 + (double)b1) + ((double)b2 + (double)b3);
    }
    for (; p < nparts; p += 8) { a += part[((long long)p * 2) * C + c]; b += part[((long long)p * 2 + 1) * C + c]; }
  }
  red[0][slice][l] = a; red[1][slice][l] = b;
  __syncthreads();
  s1 = 0.0; s2 = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) { s1 += red[0][k][l]; s2 += red[1][k][l]; }
}

// BatchNorm2d training statistics (maxvit.py:89,92,96) of channel c from its fp64 sums s = Σx, s2 = Σx² over M rows: biased
// variance for normalisation, unbiased for the running estimate, momentum update of the running buffers, and the folded
// per-channel affine  y = raw*scale + shift.  Shared by the one-GPU and the synchronised (all ranks' rows) statistics.
__device__ __forceinline__ void bn_finalize_channel(double s, double s2, long long M, int c, const float* __restrict__ gamma,
                                                    const float* __restrict__ beta, float eps, float momentum,
                                                    float* __restrict__ run_mean, float* __restrict__ run_var, float* __restrict__ mean,
                                                    float* __restrict__ rstd, float* __restrict__ scale, float* __restrict__ shift) {
  const double m = s / (double)M;
  double var = s2 / (double)M - m * m;
  if (var < 0.0) var = 0.0;
  const float r = (float)(1.0 / sqrt(var + (double)eps));
  mean[c] = (float)m; rstd[c] = r;
  const float sc = gamma[c] * r;
  scale[c] = sc; shift[c] = beta[c] - (float)m * sc;
  if (run_mean) {
    const double unb = M > 1 ? var * (double)M / (double)(M - 1) : var;
    run_mean[c] = (1.0f - momentum) * run_mean[c] + momentum * (float)m;
    run_var[c] = (1.0f - momentum) * run_var[c] + momentum * (float)unb;
  }
}

__global__ void bn_finalize_kernel(const float* __restrict__ part, int nparts, long long M, int C, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, float* __restrict__ run_mean,
                                   float* __restrict__ run_var, float* __restrict__ mean, float* __restrict__ rstd,
                                   float* __restrict__ scale, float* __restrict__ shift) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);       // 256 threads: 32 channels x 8 slices of the partials
  double s = 0.0, s2 = 0.0;
  sum_parts2(part, nparts, C, c, s, s2);
  if (c >= C || threadIdx.x >= 32) return;
  bn_finalize_channel(s, s2, M, c, gamma, beta, eps, momentum, run_mean, run_var, mean, rstd, scale, shift);
}

// ---- synchronised (cross-rank) statistics.  A rank's contribution is one fp64 row [Σx (C) | Σx² (C) | M]; the rows of all
// ranks, gathered in rank order, are summed in that order by every rank, so every rank finalizes the same bits.
__global__ void bn_stats_local_kernel(const float* __restrict__ part, int nparts, long long M, int C, double* __restrict__ row) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);       // 256 threads: 32 channels x 8 slices of the partials
  double s = 0.0, s2 = 0.0;
  sum_parts2(part, nparts, C, c, s, s2);
  if (blockIdx.x == 0 && threadIdx.x == 0) row[2 * C] = (double)M;
  if (c >= C || threadIdx.x >= 32) return;
  row[c] = s; row[C + c] = s2;
}

__global__ void __launch_bounds__(256) bn_stats_global_kernel(const double* __restrict__ rows, int world, int C,
                                                              const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                                              float momentum, float* __restrict__ run_mean, float* __restrict__ run_var,
                                                              float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ scale,
                                                              float* __restrict__ shift, double* __restrict__ count) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const long long stride = 2LL * C + 1;
  double s = 0.0, s2 = 0.0, m = 0.0;
  for (int r = 0; r < world; ++r) { s += rows[r * stride + c]; s2 += rows[r * stride + C + c]; m += rows[r * stride + 2 * C]; }
  if (c == 0 && count) *count = m;
  bn_finalize_channel(s, s2, (long long)m, c, gamma, beta, eps, momentum, run_mean, run_var, mean, rstd, scale, shift);
}

// out = act(raw*scale + shift) (+ res)     act: 0 none, 1 GELU(erf)
__global__ void __launch_bounds__(256) bn_act_kernel(const float* __restrict__ raw, const float* __restrict__ scale,
                                                     const float* __restrict__ shift, int act, const float* __restrict__ res,
                                                     float* __restrict__ out, long long total4, int C) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c = (int)((i * 4) % C);
  const float4 v = *reinterpret_cast<const float4*>(raw + i * 4);
  const float4 sc = *reinterpret_cast<const float4*>(scale + c), sh = *reinterpret_cast<const float4*>(shift + c);
  float o[4] = {fmaf(v.x, sc.x, sh.x), fmaf(v.y, sc.y, sh.y), fmaf(v.z, sc.z, sh.z), fmaf(v.w, sc.w, sh.w)};
  if (act == 1) {
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = gelu_erf(o[j]);
  }
  if (res) { const float4 r = *reinterpret_cast<const float4*>(res + i * 4); o[0] += r.x; o[1] += r.y; o[2] += r.z; o[3] += r.w; }
  *reinterpret_cast<float4*>(out + i * 4) = make_float4(o[0], o[1], o[2], o[3]);
}

// ---- BatchNorm (+activation) backward.  Upstream gradient wrt the activation output:
//        g = dOut * fgate[n][c] + fadd[n][c]        (squeeze-excite scale / mean paths; both optional, n = row / rows_per_field)
//      dpre = g * act'(raw*scale+shift);  xhat = (raw-mean)*rstd;  S1 = sum dpre, S2 = sum dpre*xhat
//      draw = gamma*rstd*(dpre - S1/M - xhat*S2/M);  dgamma += S2;  dbeta += S1
struct BnBwdParams {
  const float* dOut; const float* raw;
  const float* scale; const float* shift; const float* mean; const float* rstd; const float* gamma;
  const float* fgate; const float* fadd; long long rows_per_field;
  int act, C;
  long long M;
};

// 4 consecutive channels of one row
__device__ __forceinline__ float4 bn_dpre4(const BnBwdParams& p, long long r, int c, const float4 rawv) {
  float4 g = *reinterpret_cast<const float4*>(p.dOut + r * p.C + c);
  if (p.fgate) {
    const long long n = r / p.rows_per_field;
    const float4 fg = *reinterpret_cast<const float4*>(p.fgate + n * p.C + c);
    g.x *= fg.x; g.y *= fg.y; g.z *= fg.z; g.w *= fg.w;
    if (p.fadd) { const float4 fa = *reinterpret_cast<const float4*>(p.fadd + n * p.C + c); g.x += fa.x; g.y += fa.y; g.z += fa.z; g.w += fa.w; }
  }
  if (p.act == 1) {
    const float4 sc = *reinterpret_cast<const float4*>(p.scale + c), sh = *reinterpret_cast<const float4*>(p.shift + c);
    g.x *= gelu_grad(fmaf(rawv.x, sc.x, sh.x)); g.y *= gelu_grad(fmaf(rawv.y, sc.y, sh.y));
    g.z *= gelu_grad(fmaf(rawv.z, sc.z, sh.z)); g.w *= gelu_grad(fmaf(rawv.w, sc.w, sh.w));
  }
  return g;
}

// block = 256 threads = (C/4 channel quads) x (256 / (C/4) row lanes) over STAT_ROWS rows; partial (S1, S2) per block.
// WIDE (C > 1024, more quads than threads): a thread per quad of the block's 1024-channel slice blockIdx.y, over all STAT_ROWS rows.
template <bool WIDE>
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const BnBwdParams p, float* __restrict__ part) {
  if constexpr (WIDE) {
    const int c = (blockIdx.y * 256 + threadIdx.x) * 4;
    if (c >= p.C) return;
    const long long r0 = (long long)blockIdx.x * STAT_ROWS;
    long long r1 = r0 + STAT_ROWS;
    if (r1 > p.M) r1 = p.M;
    float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
    const float4 m = *reinterpret_cast<const float4*>(p.mean + c), rs = *reinterpret_cast<const float4*>(p.rstd + c);
#pragma unroll 2
    for (long long r = r0; r < r1; ++r) {
      const float4 rawv = *reinterpret_cast<const float4*>(p.raw + r * p.C + c);
      const float4 d = bn_dpre4(p, r, c, rawv);
      s1.x += d.x; s1.y += d.y; s1.z += d.z; s1.w += d.w;
      s2.x = fmaf(d.x, (rawv.x - m.x) * rs.x, s2.x); s2.y = fmaf(d.y, (rawv.y - m.y) * rs.y, s2.y);
      s2.z = fmaf(d.z, (rawv.z - m.z) * rs.z, s2.z); s2.w = fmaf(d.w, (rawv.w - m.w) * rs.w, s2.w);
    }
    *reinterpret_cast<float4*>(part + ((long long)blockIdx.x * 2) * p.C + c) = s1;
    *reinterpret_cast<float4*>(part + ((long long)blockIdx.x * 2 + 1) * p.C + c) = s2;
    return;
  }
  __shared__ float4 red[2][256];
  const int quads = p.C / 4, nrl = 256 / quads;
  const int q = threadIdx.x % quads, rl = threadIdx.x / quads, c = q * 4;
  const long long r0 = (long long)blockIdx.x * STAT_ROWS;
  long long r1 = r0 + STAT_ROWS;
  if (r1 > p.M) r1 = p.M;
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
  if (rl < nrl) {
    const float4 m = *reinterpret_cast<const float4*>(p.mean + c), rs = *reinterpret_cast<const float4*>(p.rstd + c);
#pragma unroll 2
    for (long long r = r0 + rl; r < r1; r += nrl) {
      const float4 rawv = *reinterpret_cast<const float4*>(p.raw + r * p.C + c);
      const float4 d = bn_dpre4(p, r, c, rawv);
      s1.x += d.x; s1.y += d.y; s1.z += d.z; s1.w += d.w;
      s2.x = fmaf(d.x, (rawv.x - m.x) * rs.x, s2.x); s2.y = fmaf(d.y, (rawv.y - m.y) * rs.y, s2.y);
      s2.z = fmaf(d.z, (rawv.z - m.z) * rs.z, s2.z); s2.w = fmaf(d.w, (rawv.w - m.w) * rs.w, s2.w);
    }
  }
  red[0][threadIdx.x] = s1; red[1][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.x < quads) {
    for (int k = 1; k < nrl; ++k) {
      const float4 a = red[0][k * quads + q], b = red[1][k * quads + q];
      s1.x += a.x; s1.y += a.y; s1.z += a.z; s1.w += a.w; s2.x += b.x; s2.y += b.y; s2.z += b.z; s2.w += b.w;
    }
    *reinterpret_cast<float4*>(part + ((long long)blockIdx.x * 2) * p.C + c) = s1;
    *reinterpret_cast<float4*>(part + ((long long)blockIdx.x * 2 + 1) * p.C + c) = s2;
  }
}

__global__ void bn_bwd_finalize_kernel(const float* __restrict__ part, int nparts, long long M, int C, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta, float* __restrict__ k1, float* __restrict__ k2) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);       // 256 threads: 32 channels x 8 slices of the partials
  double s1 = 0.0, s2 = 0.0;
  sum_parts2(part, nparts, C, c, s1, s2);
  if (c >= C || threadIdx.x >= 32) return;
  dbeta[c] += (float)s1; dgamma[c] += (float)s2;
  if (k1) { k1[c] = (float)(s1 / (double)M); k2[c] = (float)(s2 / (double)M); }
}

// synchronised backward: this rank's fp64 row [S1 (C) | S2 (C)]; dgamma / dbeta accumulate the local sums
__global__ void bn_bwd_local_kernel(const float* __restrict__ part, int nparts, int C, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta, double* __restrict__ row) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);       // 256 threads: 32 channels x 8 slices of the partials
  double s1 = 0.0, s2 = 0.0;
  sum_parts2(part, nparts, C, c, s1, s2);
  if (c >= C || threadIdx.x >= 32) return;
  dbeta[c] += (float)s1; dgamma[c] += (float)s2;
  row[c] = s1; row[C + c] = s2;
}

// k1 = ΣS1 / M_global, k2 = ΣS2 / M_global over the gathered rows [world][2C], summed in rank order
__global__ void __launch_bounds__(256) bn_bwd_global_kernel(const double* __restrict__ rows, int world, int C,
                                                            const double* __restrict__ count, float* __restrict__ k1, float* __restrict__ k2) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (int r = 0; r < world; ++r) { s1 += rows[2LL * r * C + c]; s2 += rows[2LL * r * C + C + c]; }
  const double M = *count;
  k1[c] = (float)(s1 / M); k2[c] = (float)(s2 / M);
}

// BatchNorm with running statistics (eval mode, frozen): no batch-mean terms, draw = dpre * scale
__global__ void __launch_bounds__(256) bn_bwd_frozen_apply_kernel(const BnBwdParams p, float* __restrict__ draw) {
  const int quads = p.C / 4;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.M * quads) return;
  const long long r = i / quads;
  const int c = (int)(i - r * quads) * 4;
  const float4 rawv = *reinterpret_cast<const float4*>(p.raw + r * p.C + c);
  const float4 d = bn_dpre4(p, r, c, rawv);
  const float4 sc = *reinterpret_cast<const float4*>(p.scale + c);
  *reinterpret_cast<float4*>(draw + r * p.C + c) = make_float4(d.x * sc.x, d.y * sc.y, d.z * sc.z, d.w * sc.w);
}

__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const BnBwdParams p, const float* __restrict__ k1, const float* __restrict__ k2,
                                                           float* __restrict__ draw) {
  const int quads = p.C / 4;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.M * quads) return;
  const long long r = i / quads;
  const int c = (int)(i - r * quads) * 4;
  const float4 rawv = *reinterpret_cast<const float4*>(p.raw + r * p.C + c);
  const float4 d = bn_dpre4(p, r, c, rawv);
  const float4 m = *reinterpret_cast<const float4*>(p.mean + c), rs = *reinterpret_cast<const float4*>(p.rstd + c);
  const float4 g = *reinterpret_cast<const float4*>(p.gamma + c);
  const float4 a1 = *reinterpret_cast<const float4*>(k1 + c), a2 = *reinterpret_cast<const float4*>(k2 + c);
  float4 o;
  o.x = g.x * rs.x * (d.x - a1.x - (rawv.x - m.x) * rs.x * a2.x); o.y = g.y * rs.y * (d.y - a1.y - (rawv.y - m.y) * rs.y * a2.y);
  o.z = g.z * rs.z * (d.z - a1.z - (rawv.z - m.z) * rs.z * a2.z); o.w = g.w * rs.w * (d.w - a1.w - (rawv.w - m.w) * rs.w * a2.w);
  *reinterpret_cast<float4*>(draw + r * p.C + c) = o;
}

// out[j] (+)= sum_p part[p][j]: 32 outputs x 8 slices of the partials per block
__global__ void __launch_bounds__(256) partial_sum_kernel(const float* __restrict__ part, int nparts, long long n, float beta, float* __restrict__ out) {
  __shared__ float red[8][32];
  const int l = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const long long j = (long long)blockIdx.x * 32 + l;
  float s0 = 0.f, s1 = 0.f;
  if (j < n) {
    int p = slice;
    for (; p + 8 < nparts; p += 16) { s0 += part[(long long)p * n + j]; s1 += part[(long long)(p + 8) * n + j]; }
    if (p < nparts) s0 += part[(long long)p * n + j];
  }
  red[slice][l] = s0 + s1;
  __syncthreads();
  if (slice == 0 && j < n) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][l];
    out[j] = (beta != 0.f ? beta * out[j] : 0.f) + s;
  }
}

// column sums of X fp32 [M][C] accumulated into out[C] (bias gradients); DET: block b stores its sums into row b of out
template <bool DET = false>
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ X, long long M, int C, float* __restrict__ out) {
  const long long r0 = (long long)blockIdx.x * STAT_ROWS;
  long long r1 = r0 + STAT_ROWS;
  if (r1 > M) r1 = M;
  for (int c = threadIdx.x; c < C; c += 256) {
    float s = 0.f;
    for (long long r = r0; r < r1; ++r) s += X[r * C + c];
    if constexpr (DET) out[(long long)blockIdx.x * C + c] = s;
    else atomicAdd(out + c, s);
  }
}

// ================================================================================================
// depthwise 3x3 (pad 1) on channels-last (N,H,W,C): marching stencil.  One thread owns 4 channels x a strip of SW
// columns and walks down the rows keeping a 3-row register window, so every input element is loaded once per strip
// (plus the one-column halo) instead of nine times.   out = act(conv*scale + shift)   (act: 0 none, 1 GELU)
// psum (optional): (N, strips, C) per-strip channel sums of the outputs (squeeze-excite mean).
// Used for: inference (folded BN + GELU), training forward (scale = 1, shift = bias), dgrad (flipped taps).
// ================================================================================================
constexpr int DW_SW = 5;

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

template <> struct Ld4<__half> {
  static __device__ __forceinline__ float4 ld(const __half* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  static __device__ __forceinline__ void st(__half* p, float4 v) {
    uint2 u;
    *reinterpret_cast<__half2*>(&u.x) = __floats2half2_rn(v.x, v.y);
    *reinterpret_cast<__half2*>(&u.y) = __floats2half2_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = u;
  }
};

// (round 2, from ncu's executed-instruction mix of the fp16 instantiation -- 41 instructions per element at 60 % issue utilisation,
//  i.e. instruction-bound: the row rotation r0 = r1, r1 = r2 was 4.9 MOVs per element -> the row loop is unrolled by three with the
//  three row buffers changing roles; the nine taps were 9 scalar FFMAs per element -> 4.5 packed FFMA2; GELU see gelu_erf2)
struct F22 { float2 lo, hi; };
__device__ __forceinline__ F22 f22(float4 v) { F22 r; r.lo = make_float2(v.x, v.y); r.hi = make_float2(v.z, v.w); return r; }

// SLICED (C a multiple of 512 above 512, fp32: the training forward and data gradient): a block covers one strip of the 512-channel
// slice blockIdx.y.  At three blocks per SM its register cap spilled; two keep everything in registers.
template <typename T, bool SLICED = false>
__global__ void __launch_bounds__(128, SLICED ? 2 : 3) dwconv_march_kernel(const T* __restrict__ in, const float* __restrict__ w9,
                                                           const float* __restrict__ scale, const float* __restrict__ shift, int act,
                                                           T* __restrict__ out, float* __restrict__ psum, int H, int W, int C, int strips) {
  const int quads = SLICED ? 128 : C / 4;
  const int spb = SLICED ? 1 : (128 / quads > 0 ? 128 / quads : 1);             // strips per block
  const int quad = SLICED ? threadIdx.x : threadIdx.x % quads, sub = SLICED ? 0 : threadIdx.x / quads;
  const int sblocks = (strips + spb - 1) / spb;
  const int n = blockIdx.x / sblocks, strip = (blockIdx.x - n * sblocks) * spb + sub;
  if (sub >= spb || strip >= strips) return;
  if constexpr (SLICED) {                                          // the slice's channels: offset every channel-indexed pointer once
    const int cs = blockIdx.y * 512;
    in += cs; w9 += cs; scale += cs; shift += cs; out += cs;
    if (psum) psum += cs;
  }
  const int c0 = quad * 4, w0 = strip * DW_SW;
  F22 wk[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) wk[k] = f22(*reinterpret_cast<const float4*>(w9 + k * C + c0));
  const F22 sc = f22(*reinterpret_cast<const float4*>(scale + c0)), sh = f22(*reinterpret_cast<const float4*>(shift + c0));
  const T* base = in + (long long)n * H * W * C + c0;
  T* obase = out + (long long)n * H * W * C + c0;
  const float2 z2 = make_float2(0.f, 0.f);
  F22 r0[DW_SW + 2], r1[DW_SW + 2], r2[DW_SW + 2];
  bool colok[DW_SW + 2];
#pragma unroll
  for (int j = 0; j < DW_SW + 2; ++j) {
    const int w = w0 - 1 + j;
    colok[j] = w >= 0 && w < W;
    r0[j].lo = r0[j].hi = z2;
    r1[j] = r0[j];
    if (colok[j]) r1[j] = f22(Ld4<T>::ld(base + (long long)w * C));
  }
  float2 sum_lo = z2, sum_hi = z2;
  // one output row: ra / rb / rc hold input rows h-1 / h / h+1 (rc is loaded here)
  auto step = [&](int h, F22 (&ra)[DW_SW + 2], F22 (&rb)[DW_SW + 2], F22 (&rc)[DW_SW + 2]) {
    const T* nxt = base + ((long long)(h + 1) * W + (w0 - 1)) * C;
    const bool more = h + 1 < H;
#pragma unroll
    for (int j = 0; j < DW_SW + 2; ++j) {
      rc[j].lo = rc[j].hi = z2;
      if (more && colok[j]) rc[j] = f22(Ld4<T>::ld(nxt + (long long)j * C));
    }
    T* orow = obase + ((long long)h * W + w0) * C;
#pragma unroll
    for (int j = 0; j < DW_SW; ++j) {
      if (colok[j + 1]) {
        float2 lo = z2, hi = z2;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          lo = f2_fma(ra[j + dx].lo, wk[dx].lo, lo); hi = f2_fma(ra[j + dx].hi, wk[dx].hi, hi);
          lo = f2_fma(rb[j + dx].lo, wk[3 + dx].lo, lo); hi = f2_fma(rb[j + dx].hi, wk[3 + dx].hi, hi);
          lo = f2_fma(rc[j + dx].lo, wk[6 + dx].lo, lo); hi = f2_fma(rc[j + dx].hi, wk[6 + dx].hi, hi);
        }
        lo = f2_fma(lo, sc.lo, sh.lo); hi = f2_fma(hi, sc.hi, sh.hi);
        if (act == 1) { lo = gelu_erf2(lo); hi = gelu_erf2(hi); }
        Ld4<T>::st(orow + (long long)j * C, make_float4(lo.x, lo.y, hi.x, hi.y));
        sum_lo.x += lo.x; sum_lo.y += lo.y; sum_hi.x += hi.x; sum_hi.y += hi.y;
      }
    }
  };
  for (int h = 0; h < H; h += 3) {
    step(h, r0, r1, r2);
    if (h + 1 < H) step(h + 1, r1, r2, r0);
    if (h + 2 < H) step(h + 2, r2, r0, r1);
  }
  if (psum) *reinterpret_cast<float4*>(psum + ((long long)n * strips + strip) * C + c0) = make_float4(sum_lo.x, sum_lo.y, sum_hi.x, sum_hi.y);
}

// depthwise weight gradient: part[(n,strip)][k][c] = sum_{h, w in strip} dY[n,h,w,c] * X[n,h+dy,w+dx,c]  (k = 3*(dy+1)+dx+1),
// k = 9: sum dY (bias gradient).  fp32 only.
// SLICED as in dwconv_march_kernel
template <bool SLICED = false>
__global__ void __launch_bounds__(128) dw_wgrad_kernel(const float* __restrict__ X, const float* __restrict__ dY, float* __restrict__ part,
                                                       int H, int W, int C, int strips) {
  const int quads = SLICED ? 128 : C / 4;
  const int spb = SLICED ? 1 : (128 / quads > 0 ? 128 / quads : 1);
  const int quad = SLICED ? threadIdx.x : threadIdx.x % quads, sub = SLICED ? 0 : threadIdx.x / quads;
  const int sblocks = (strips + spb - 1) / spb;
  const int n = blockIdx.x / sblocks, strip = (blockIdx.x - n * sblocks) * spb + sub;
  if (sub >= spb || strip >= strips) return;
  if constexpr (SLICED) { const int cs = blockIdx.y * 512; X += cs; dY += cs; part += cs; }
  const int c0 = quad * 4, w0 = strip * DW_SW;
  const float* xb = X + (long long)n * H * W * C + c0;
  const float* gb = dY + (long long)n * H * W * C + c0;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 acc[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] = z;
  for (int h = 0; h < H; ++h) {
    float4 g[DW_SW];
#pragma unroll
    for (int j = 0; j < DW_SW; ++j) {
      g[j] = (w0 + j < W) ? *reinterpret_cast<const float4*>(gb + ((long long)h * W + w0 + j) * C) : z;
      acc[9].x += g[j].x; acc[9].y += g[j].y; acc[9].z += g[j].z; acc[9].w += g[j].w;
    }
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      const int hh = h + dy - 1;
      if (hh < 0 || hh >= H) continue;
      float4 x[DW_SW + 2];
#pragma unroll
      for (int j = 0; j < DW_SW + 2; ++j) {
        const int w = w0 - 1 + j;
        x[j] = (w >= 0 && w < W) ? *reinterpret_cast<const float4*>(xb + ((long long)hh * W + w) * C) : z;
      }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx)
#pragma unroll
        for (int j = 0; j < DW_SW; ++j) {
          float4& a = acc[dy * 3 + dx];
          a.x = fmaf(g[j].x, x[j + dx].x, a.x); a.y = fmaf(g[j].y, x[j + dx].y, a.y);
          a.z = fmaf(g[j].z, x[j + dx].z, a.z); a.w = fmaf(g[j].w, x[j + dx].w, a.w);
        }
    }
  }
#pragma unroll
  for (int k = 0; k < 10; ++k) *reinterpret_cast<float4*>(part + (((long long)n * strips + strip) * 10 + k) * C + c0) = acc[k];
}

// ================================================================================================
// squeeze-excite (maxvit.py:33-48)
// ================================================================================================
// gate with the intermediates the backward pass needs (mean (N,C), hid (N,se)); psum: (N, nparts, C) partial sums
__global__ void __launch_bounds__(256) se_gate_train_kernel(const float* __restrict__ psum, int nparts, float inv_count,
                                                            const float* __restrict__ W1, const float* __restrict__ W2, int C, int se,
                                                            float* __restrict__ gate, float* __restrict__ mean_out, float* __restrict__ hid_out) {
  extern __shared__ float sh[];
  float* mean = sh; float* hid = sh + C;
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int h = 0; h < nparts; ++h) s += psum[((long long)n * nparts + h) * C + c];
    mean[c] = s * inv_count;
    if (mean_out) mean_out[(long long)n * C + c] = mean[c];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int j = warp; j < se; j += nw) {
    float a = 0.f;
    for (int c = lane; c < C; c += 32) a += W1[(long long)j * C + c] * mean[c];
    a = warp_sum(a);
    if (lane == 0) { hid[j] = fmaxf(a, 0.f); if (hid_out) hid_out[(long long)n * se + j] = hid[j]; }
  }
  __syncthreads();
  for (int c = warp; c < C; c += nw) {
    float a = 0.f;
    for (int j = lane; j < se; j += 32) a += W2[(long long)c * se + j] * hid[j];
    a = warp_sum(a);
    if (lane == 0) gate[(long long)n * C + c] = 1.0f / (1.0f + expf(-a));
  }
}

__global__ void __launch_bounds__(256) field_mean_kernel(const float* __restrict__ psum, int nparts, float inv_count, int C,
                                                         long long total, float* __restrict__ mean) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / C;
  const int c = (int)(i - n * C);
  float s = 0.f;
  for (int h = 0; h < nparts; ++h) s += psum[(n * nparts + h) * C + c];
  mean[i] = s * inv_count;
}

// squeeze-excite scale folded into the per-field weights of the 1x1 projection that follows (maxvit.py:47 + :95):
//   Wn[n][co][c] = W[co][c] * gate[n][c]    -- 256 KB per field instead of a read-modify-write pass over the activations
template <typename TO>
__global__ void __launch_bounds__(256) se_fold_kernel(const float* __restrict__ W, const float* __restrict__ gate, TO* __restrict__ out,
                                                      int Cout, int C, long long total4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const long long e = i * 4;
  const int c = (int)(e % C);
  const long long r = e / C;
  const int co = (int)(r % Cout);
  const long long n = r / Cout;
  const float4 w = *reinterpret_cast<const float4*>(W + (long long)co * C + c), g = *reinterpret_cast<const float4*>(gate + n * C + c);
  if constexpr (sizeof(TO) == 4) {
    *reinterpret_cast<float4*>(out + e) = make_float4(w.x * g.x, w.y * g.y, w.z * g.z, w.w * g.w);
  } else {                                                    // fp16 per-field weights (the hidden tensor of the MBConv is fp16)
    uint2 u;
    *reinterpret_cast<__half2*>(&u.x) = __floats2half2_rn(w.x * g.x, w.y * g.y);
    *reinterpret_cast<__half2*>(&u.y) = __floats2half2_rn(w.z * g.z, w.w * g.w);
    *reinterpret_cast<uint2*>(out + e) = u;
  }
}

// out[n][p][c] = x[n][p][c] * gate[n][c]   (out of place: training keeps the pre-gate activations)
__global__ void __launch_bounds__(256) se_scale_oop_kernel(const float* __restrict__ x, const float* __restrict__ gate, float* __restrict__ out,
                                                           long long HW, int C, long long total4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const long long e = i * 4;
  const int c = (int)(e % C);
  const long long n = (e / C) / HW;
  const float4 v = *reinterpret_cast<const float4*>(x + e), g = *reinterpret_cast<const float4*>(gate + n * C + c);
  *reinterpret_cast<float4*>(out + e) = make_float4(v.x * g.x, v.y * g.y, v.z * g.z, v.w * g.w);
}

// out[n][chunk][c] = sum over the chunk's positions p of a[n][p][c] * b[n][p][c]  (b = NULL: plain sums)   grid (chunks, N)
// Deterministic: per-chunk partial sums, no atomics (the squeeze-excite mean feeds the forward pass; run-to-run bit
// differences there are amplified to tf32-rounding level by the layers that follow).
__global__ void __launch_bounds__(256) field_dot_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                                                        long long HW, int C) {
  const int n = blockIdx.y;
  const long long rows_per = (HW + gridDim.x - 1) / gridDim.x;
  const long long p0 = blockIdx.x * rows_per;
  long long p1 = p0 + rows_per;
  if (p1 > HW) p1 = HW;
  for (int c = threadIdx.x; c < C; c += 256) {
    float s = 0.f;
    for (long long p = p0; p < p1; ++p) { const long long i = ((long long)n * HW + p) * C + c; s = b ? fmaf(a[i], b[i], s) : s + a[i]; }
    out[((long long)n * gridDim.x + blockIdx.x) * C + c] = s;
  }
}

// per field: dpre2 = dgate*gate*(1-gate); dhid = relu'(hid) * W2^T dpre2; dmean = W1^T dhid  (scaled by 1/HW for the apply)
__global__ void __launch_bounds__(256) se_bwd_kernel(const float* __restrict__ dgate_parts, int nparts, const float* __restrict__ gate,
                                                     const float* __restrict__ hid, const float* __restrict__ W1, const float* __restrict__ W2,
                                                     int C, int se, float inv_count, float* __restrict__ dpre2, float* __restrict__ dhid,
                                                     float* __restrict__ dmean) {
  extern __shared__ float sh[];
  float* sp = sh; float* sd = sh + C;
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float g = gate[(long long)n * C + c];
    float dg = 0.f;
    for (int k = 0; k < nparts; ++k) dg += dgate_parts[((long long)n * nparts + k) * C + c];
    const float v = dg * g * (1.0f - g);
    sp[c] = v; dpre2[(long long)n * C + c] = v;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < se; j += blockDim.x) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;         // four chains: the loads of a single one waited for each other
    int c = 0;
    for (; c + 3 < C; c += 4) {
      a0 = fmaf(W2[(long long)c * se + j], sp[c], a0); a1 = fmaf(W2[(long long)(c + 1) * se + j], sp[c + 1], a1);
      a2 = fmaf(W2[(long long)(c + 2) * se + j], sp[c + 2], a2); a3 = fmaf(W2[(long long)(c + 3) * se + j], sp[c + 3], a3);
    }
    for (; c < C; ++c) a0 = fmaf(W2[(long long)c * se + j], sp[c], a0);
    float a = (a0 + a1) + (a2 + a3);
    if (hid[(long long)n * se + j] <= 0.f) a = 0.f;
    sd[j] = a; dhid[(long long)n * se + j] = a;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int j = 0;
    for (; j + 3 < se; j += 4) {
      a0 = fmaf(W1[(long long)j * C + c], sd[j], a0); a1 = fmaf(W1[(long long)(j + 1) * C + c], sd[j + 1], a1);
      a2 = fmaf(W1[(long long)(j + 2) * C + c], sd[j + 2], a2); a3 = fmaf(W1[(long long)(j + 3) * C + c], sd[j + 3], a3);
    }
    for (; j < se; ++j) a0 = fmaf(W1[(long long)j * C + c], sd[j], a0);
    dmean[(long long)n * C + c] = ((a0 + a1) + (a2 + a3)) * inv_count;
  }
}

// ================================================================================================
// attention backward
// ================================================================================================
// gradient wrt the out-projection output (maxvit.py:218-219, 310-319): window rows gather dX_out through the partition
// map, register rows take dreg (N,R,C) * reg_scale (the mean over windows, maxvit.py:326) or zero.
template <typename TO>
__global__ void __launch_bounds__(256) attn_out_bwd_gather_kernel(const float* __restrict__ dx_out, const float* __restrict__ dreg, float reg_scale,
                                                                  const AttnGeom g, TO* __restrict__ dproj, long long rows, const DropCfg drop) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31, C = g.C, S = g.S(), nwin = g.nwin();
  const long long wdx = r / S;
  const int tok = (int)(r - wdx * S);
  const int n = (int)(wdx / nwin), wi = (int)(wdx - (long long)n * nwin);
  for (int c = lane * 4; c < C; c += 128) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tok < g.R) {
      if (dreg) { v = *reinterpret_cast<const float4*>(dreg + ((long long)n * g.R + tok) * C + c); v.x *= reg_scale; v.y *= reg_scale; v.z *= reg_scale; v.w *= reg_scale; }
    } else {
      v = *reinterpret_cast<const float4*>(dx_out + ((long long)n * g.Hl * g.Wl + attn_token_pixel(g, wi, tok - g.R)) * C + c);
    }
    if (drop.thresh) {                                       // the to_out dropout mask of the forward pass (maxvit.py:151)
      const uint32_t hsh = drop_hash(drop.seed, drop_row(wdx, tok, drop_slots(S)), drop_group_out(drop.salt, c >> 2));
      v.x *= (int)(hsh & 255u) >= drop.thresh ? drop.scale : 0.f;
      v.y *= (int)((hsh >> 8) & 255u) >= drop.thresh ? drop.scale : 0.f;
      v.z *= (int)((hsh >> 16) & 255u) >= drop.thresh ? drop.scale : 0.f;
      v.w *= (int)((hsh >> 24) & 255u) >= drop.thresh ? drop.scale : 0.f;
    }
    if constexpr (sizeof(TO) == 4) {
      *reinterpret_cast<float4*>(dproj + r * C + c) = v;
    } else {
      uint2 u;
      *reinterpret_cast<__nv_bfloat162*>(&u.x) = __floats2bfloat162_rn(v.x, v.y);
      *reinterpret_cast<__nv_bfloat162*>(&u.y) = __floats2bfloat162_rn(v.z, v.w);
      *reinterpret_cast<uint2*>(dproj + r * C + c) = u;
    }
  }
}

// Core backward (maxvit.py:195-215), one block per (field, head), looping over the field's windows so that the
// relative-position-bias and q/k-gamma gradients accumulate in shared memory / registers and reach global memory
// once per block.  fp32, DH = 32 or 64, S <= 64.
struct AttnCoreBwdParams {
  const float* qkv;        // [rows][3*inner]
  const float* datt;       // [rows][inner]
  const float* qgamma; const float* kgamma;   // [heads*DH]
  const float* bias_table; // [nb][heads]
  float* dqkv;             // [rows][3*inner]
  float* dqgamma; float* dkgamma; float* dbias_table;
  AttnGeom g;
  int heads;
};


// Deterministic bias-table gradient of one window (the DET kernels): dbias[b] += sum of dS[i][j] over the (i, j) pairs of
// relative-position index b, in (i, j) order.  Index b < nb-1 is the offset (ai - aj, bi - bj) of two window tokens; nb-1 is
// every pair with a register token.  dS: [S][ld] in shared memory; thread tid of nthreads.
// Query rows i0 .. i0+ni-1 only (dS row i - i0 holds query i): the long-window kernels hold dS one block of query rows at a time.
__device__ __forceinline__ void dbias_gather(const float* dS, int ld, const AttnGeom& g, int nb, float* dbias, int tid, int nthreads,
                                             int i0 = 0, int ni = 1 << 30) {
  const int S = g.S(), w = g.win, W2 = 2 * w - 1, R = g.R, i1 = min(S, i0 + ni);
  for (int b = tid; b < nb; b += nthreads) {
    float acc = 0.f;
    if (b < nb - 1) {
      const int da = b / W2 - (w - 1), db = b % W2 - (w - 1);
      for (int ai = max(0, da); ai < min(w, w + da); ++ai)
        for (int bi = max(0, db); bi < min(w, w + db); ++bi) {
          const int i = R + ai * w + bi;
          if (i >= i0 && i < i1) acc += dS[(i - i0) * ld + R + (ai - da) * w + (bi - db)];
        }
    } else {
      for (int i = i0; i < i1; ++i)
        for (int j = 0; j < (i < R ? S : R); ++j) acc += dS[(i - i0) * ld + j];
    }
    dbias[b] += acc;
  }
}

// the block's bias-table gradient into its field's slots (DET kernels)
__device__ __forceinline__ void det_flush_bias(const AttnDetSlots& det, const float* dbias, int n, int nb, int heads, int hd, int tid,
                                               int nthreads) {
  for (int i = tid; i < nb; i += nthreads) det.bias[((long long)n * nb + i) * heads + hd] = dbias[i];
}

// sum_k a[k] b[k] of one lane's values
template <int K>
__device__ __forceinline__ float lane_dot(const float (&a)[K], const float (&b)[K]) {
  float r = a[0] * b[0];
#pragma unroll
  for (int k = 1; k < K; ++k) r = fmaf(a[k], b[k], r);
  return r;
}

// DET: the bias-table gradient of a window is gathered from dS in a fixed order (dbias_gather) and the block's gamma / bias
// gradients go to its field's slots (det_gamma, det_bias) instead of global atomics
template <int DH, bool DET = false>
__global__ void __launch_bounds__(256) attn_core_bwd_kernel(const AttnCoreBwdParams p, const DropCfg drop, const AttnDetSlots det) {
  constexpr int LD = DH + 1, SM = 64, DPL = DH / 32;        // DPL head dims per lane: d = lane + 32*k
  extern __shared__ float sm[];
  const AttnGeom g = p.g;
  const int S = g.S(), nwin = g.nwin(), W2 = 2 * g.win - 1, nb = W2 * W2 + 1;
  float* qh = sm;                 // [SM][LD] normalised * gamma
  float* kh = qh + SM * LD;
  float* vv = kh + SM * LD;
  float* dO = vv + SM * LD;
  float* qu = dO + SM * LD;       // unit vectors
  float* ku = qu + SM * LD;
  float* dqh = ku + SM * LD;
  float* dkh = dqh + SM * LD;
  float* P = dkh + SM * LD;       // [SM][SM+1]
  float* sbias = P + SM * (SM + 1);   // [nb]
  float* dbias = sbias + nb;          // [nb]
  float* inq = dbias + nb;            // [SM] 1/|q|
  float* ink = inq + SM;
  float* gred = ink + SM;             // [8][2][DH]
  float* MK = gred + 8 * 2 * DH;      // [SM][SM+1] dropout mask * scale of the probabilities (allocated when dropout is on)
  const int n = blockIdx.x / p.heads, hd = blockIdx.x - n * p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = p.heads * DH;
  const float rs = sqrtf((float)DH);
  for (int i = threadIdx.x; i < nb; i += 256) { sbias[i] = p.bias_table[i * p.heads + hd]; dbias[i] = 0.f; }
  float gq[DPL], gk[DPL], dgq[DPL], dgk[DPL];
#pragma unroll
  for (int k = 0; k < DPL; ++k) {
    gq[k] = p.qgamma[hd * DH + lane + 32 * k]; gk[k] = p.kgamma[hd * DH + lane + 32 * k];
    dgq[k] = 0.f; dgk[k] = 0.f;
  }
  __syncthreads();

  for (int wi = 0; wi < nwin; ++wi) {
    const long long row0 = ((long long)n * nwin + wi) * S;
    // ---- load + normalise: warp per row, lane = d
    for (int i = warp; i < S; i += 8) {
      const float* src = p.qkv + (row0 + i) * 3 * inner + hd * DH + lane;
      float q[DPL], k[DPL], v[DPL];
#pragma unroll
      for (int j = 0; j < DPL; ++j) { q[j] = src[32 * j]; k[j] = src[inner + 32 * j]; v[j] = src[2 * inner + 32 * j]; }
      const float nq = fmaxf(sqrtf(warp_sum(lane_dot<DPL>(q, q))), 1e-12f), nk = fmaxf(sqrtf(warp_sum(lane_dot<DPL>(k, k))), 1e-12f);
#pragma unroll
      for (int j = 0; j < DPL; ++j) {
        const int d = lane + 32 * j;
        const float uq = q[j] / nq, uk = k[j] / nk;
        qu[i * LD + d] = uq; ku[i * LD + d] = uk;
        qh[i * LD + d] = uq * rs * gq[j]; kh[i * LD + d] = uk * rs * gk[j];
        vv[i * LD + d] = v[j];
        dO[i * LD + d] = p.datt[(row0 + i) * inner + hd * DH + d];
      }
      if (lane == 0) { inq[i] = 1.0f / nq; ink[i] = 1.0f / nk; }
    }
    __syncthreads();
    // ---- P = softmax(qh kh^T + bias): warp per row, lanes over keys j, j+32
    for (int i = warp; i < S; i += 8) {
      float s[2];
      const int ti = i - g.R, ai = ti / g.win, bi = ti - ai * g.win;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = lane + 32 * t;
        float a = -INFINITY;
        if (j < S) {
          a = 0.f;
#pragma unroll
          for (int d = 0; d < DH; ++d) a = fmaf(qh[i * LD + d], kh[j * LD + d], a);
          int bidx = nb - 1;
          if (i >= g.R && j >= g.R) { const int tj = j - g.R, aj = tj / g.win, bj = tj - aj * g.win; bidx = (ai - aj + g.win - 1) * W2 + (bi - bj + g.win - 1); }
          a += sbias[bidx];
        }
        s[t] = a;
      }
      const float m = warp_max(fmaxf(s[0], s[1]));
      const float e0 = lane < S ? __expf(s[0] - m) : 0.f, e1 = lane + 32 < S ? __expf(s[1] - m) : 0.f;
      const float inv = 1.0f / warp_sum(e0 + e1);
      P[i * (SM + 1) + lane] = e0 * inv;
      P[i * (SM + 1) + lane + 32] = e1 * inv;
      if (drop.thresh) {                                     // the forward pass's mask on the probabilities (maxvit.py:146)
        const uint32_t rid = drop_row((long long)n * nwin + wi, i);
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const int j = lane + 32 * t;
          const uint32_t hsh = drop_hash(drop.seed, rid, drop_group_prob(drop.salt, hd, j >> 2));
          MK[i * (SM + 1) + j] = (int)((hsh >> (8 * (j & 3))) & 255u) >= drop.thresh ? drop.scale : 0.f;
        }
      }
    }
    __syncthreads();
    // ---- dV[j][d] = sum_i P'[i][j] dO[i][d] (P' = P * mask): warp per j, lane = d
    for (int j = warp; j < S; j += 8) {
      float a[DPL];
#pragma unroll
      for (int k = 0; k < DPL; ++k) a[k] = 0.f;
      if (drop.thresh) {
        for (int i = 0; i < S; ++i) {
          const float pm = P[i * (SM + 1) + j] * MK[i * (SM + 1) + j];
#pragma unroll
          for (int k = 0; k < DPL; ++k) a[k] = fmaf(pm, dO[i * LD + lane + 32 * k], a[k]);
        }
      } else {
        for (int i = 0; i < S; ++i)
#pragma unroll
          for (int k = 0; k < DPL; ++k) a[k] = fmaf(P[i * (SM + 1) + j], dO[i * LD + lane + 32 * k], a[k]);
      }
#pragma unroll
      for (int k = 0; k < DPL; ++k) p.dqkv[(row0 + j) * 3 * inner + 2 * inner + hd * DH + lane + 32 * k] = a[k];
    }
    __syncthreads();
    // ---- dS = P * (dP - sum_j P dP), dP[i][j] = dO[i] . v[j]; overwrite P with dS; bias-table gradient
    for (int i = warp; i < S; i += 8) {
      float dp[2], pr[2];
      const int ti = i - g.R, ai = ti / g.win, bi = ti - ai * g.win;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = lane + 32 * t;
        float a = 0.f;
        if (j < S) {
#pragma unroll
          for (int d = 0; d < DH; ++d) a = fmaf(dO[i * LD + d], vv[j * LD + d], a);
          if (drop.thresh) a *= MK[i * (SM + 1) + j];         // d(att)/dP passes through the mask
        }
        dp[t] = a; pr[t] = j < S ? P[i * (SM + 1) + j] : 0.f;
      }
      const float dot = warp_sum(pr[0] * dp[0] + pr[1] * dp[1]);
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = lane + 32 * t;
        if (j < S) {
          const float ds = pr[t] * (dp[t] - dot);
          P[i * (SM + 1) + j] = ds;
          if constexpr (!DET) {
            int bidx = nb - 1;
            if (i >= g.R && j >= g.R) { const int tj = j - g.R, aj = tj / g.win, bj = tj - aj * g.win; bidx = (ai - aj + g.win - 1) * W2 + (bi - bj + g.win - 1); }
            atomicAdd(&dbias[bidx], ds);
          }
        }
      }
    }
    __syncthreads();
    if constexpr (DET) dbias_gather(P, SM + 1, g, nb, dbias, threadIdx.x, 256);
    // ---- dqh[i][d] = sum_j dS[i][j] kh[j][d];  dkh[j][d] = sum_i dS[i][j] qh[i][d]
    for (int i = warp; i < S; i += 8) {
      float a[DPL], b[DPL];
#pragma unroll
      for (int k = 0; k < DPL; ++k) a[k] = b[k] = 0.f;
      for (int j = 0; j < S; ++j) {
#pragma unroll
        for (int k = 0; k < DPL; ++k) {
          a[k] = fmaf(P[i * (SM + 1) + j], kh[j * LD + lane + 32 * k], a[k]);
          b[k] = fmaf(P[j * (SM + 1) + i], qh[j * LD + lane + 32 * k], b[k]);
        }
      }
#pragma unroll
      for (int k = 0; k < DPL; ++k) { dqh[i * LD + lane + 32 * k] = a[k]; dkh[i * LD + lane + 32 * k] = b[k]; }
    }
    __syncthreads();
    // ---- RMSNorm backward (maxvit.py:30): xh = u * rs * gamma, u = x/|x|
    for (int i = warp; i < S; i += 8) {
      float uq[DPL], uk[DPL], g1[DPL], g2[DPL];
#pragma unroll
      for (int k = 0; k < DPL; ++k) {
        const float aq = dqh[i * LD + lane + 32 * k], ak = dkh[i * LD + lane + 32 * k];
        uq[k] = qu[i * LD + lane + 32 * k]; uk[k] = ku[i * LD + lane + 32 * k];
        dgq[k] = fmaf(aq, uq[k] * rs, dgq[k]); dgk[k] = fmaf(ak, uk[k] * rs, dgk[k]);
        g1[k] = aq * rs * gq[k]; g2[k] = ak * rs * gk[k];
      }
      const float d1 = warp_sum(lane_dot<DPL>(g1, uq)), d2 = warp_sum(lane_dot<DPL>(g2, uk));
      float* dst = p.dqkv + (row0 + i) * 3 * inner + hd * DH + lane;
#pragma unroll
      for (int k = 0; k < DPL; ++k) {
        dst[32 * k] = inq[i] * (g1[k] - uq[k] * d1);
        dst[inner + 32 * k] = ink[i] * (g2[k] - uk[k] * d2);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < DPL; ++k) { gred[(warp * 2) * DH + lane + 32 * k] = dgq[k]; gred[(warp * 2 + 1) * DH + lane + 32 * k] = dgk[k]; }
  __syncthreads();
  if (threadIdx.x < 2 * DH) {
    const int which = threadIdx.x / DH, d = threadIdx.x % DH;
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += gred[(w * 2 + which) * DH + d];
    if constexpr (DET) det.gamma[((long long)n * 2 + which) * inner + hd * DH + d] = s;
    else atomicAdd((which ? p.dkgamma : p.dqgamma) + hd * DH + d, s);
  }
  if constexpr (DET) {
    for (int i = threadIdx.x; i < nb; i += 256) det.bias[((long long)n * nb + i) * p.heads + hd] = dbias[i];
  } else {
    for (int i = threadIdx.x; i < nb; i += 256) atomicAdd(p.dbias_table + i * p.heads + hd, dbias[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// Tensor-core version of the core backward on fp32 tensors (mode 2, the un-fused mixed-precision path): bf16 mma.sync
// m16n8k16 (fp32 accumulate) with ldmatrix operand fetch (transposed operands come for free from ldmatrix.trans).
// Block = (field, head), 4 warps, looping over the field's windows (3 blocks per SM hide each other's load latency);
// each warp owns 16 rows of the window:
//   phase 1  load q,k,v,dO rows, RMSNorm -> Qh, Kh, V, dO in shared memory (row stride 80 B: conflict-free ldmatrix)
//   phase 2  S = Qh Kh^T (+bias), row softmax in registers -> P (smem);  [att = P V, optional output]
//            dP = dO V^T, dS = P*(dP - rowdot) -> dS (smem), bias-table gradient
//   phase 3  dV = P^T dO, dKh = dS^T Qh (rows = keys), dQh = dS Kh (rows = queries); RMSNorm backward on the
//            accumulator fragments (raw q,k re-read from global) -> dqkv
// The 53 valid tokens are padded to 64 with zero rows; padded keys are masked to -inf before the softmax.  The
// relative-position-bias gradient of a thread's 32 fixed (query, key) pairs is accumulated in registers over the field's windows.
// ------------------------------------------------------------------------------------------------
template <int DH_>
struct cbh {
  static constexpr int DH = DH_, SM = 64;
  static constexpr int LDQ = DH + 8;   // bf16 elements per Q/K/V/dO row (80 / 144 B: ldmatrix rows hit distinct banks)
  static constexpr int LDP = 72;       // bf16 elements per P/dS row (144 B)
  static constexpr int BYTES = 4 * SM * LDQ * 2 + 2 * SM * LDP * 2 + 2 * SM * 4;
  static constexpr int LPR = DH / 8;   // phase 1: lanes per row (8 consecutive head dims each), rows per pass 32 / LPR
  static constexpr int PASSES = 16 / (32 / LPR);
};

__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t* r) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm4t(uint32_t addr, uint32_t* r) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// C[16 x 8*NT] += A * B over K (multiple of 16).  a_/b_ are shared-memory byte addresses of the operand matrices.
//   A normal : element (r, k) at a_ + (r*lda + k)*2          A transposed: element (r, k) stored at (k*lda + r)
//   B "NT"   : element (k, n) stored at (n*ldb + k)           B "NN"      : element (k, n) stored at (k*ldb + n)
template <int NT, int K, bool TRANS_A, bool NN>
__device__ __forceinline__ void warp_mma_bf16(float (*acc)[4], uint32_t a_, int lda, int a_r0, uint32_t b_, int ldb, int lane) {
  const int l7 = lane & 7, l3 = (lane >> 3) & 1, l4 = lane >> 4;
#pragma unroll
  for (int ks = 0; ks < K / 16; ++ks) {
    const int k0 = ks * 16;
    uint32_t af[4];
    if (!TRANS_A) ldsm4(a_ + (uint32_t)(((a_r0 + l7 + 8 * l3) * lda + k0 + 8 * l4) * 2), af);
    else ldsm4t(a_ + (uint32_t)(((k0 + l7 + 8 * l4) * lda + a_r0 + 8 * l3) * 2), af);
#pragma unroll
    for (int np = 0; np < NT / 2; ++np) {
      uint32_t bf[4];
      if (!NN) ldsm4(b_ + (uint32_t)(((np * 16 + l7 + 8 * l4) * ldb + k0 + 8 * l3) * 2), bf);
      else ldsm4t(b_ + (uint32_t)(((k0 + l7 + 8 * l3) * ldb + np * 16 + 8 * l4) * 2), bf);
      mma_bf16_16816(acc[2 * np], af, bf[0], bf[1]);
      mma_bf16_16816(acc[2 * np + 1], af, bf[2], bf[3]);
    }
  }
}
__device__ __forceinline__ uint32_t pack2bf(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// DH 64: two blocks per SM (the 64-wide accumulators do not fit the three-block register cap; at 255 registers 20 bytes still spill)
// DET (dynamic shared memory grows by 8*DH + 64*65 floats after sgam): the four warps' gamma partials go to per-warp rows gw
// summed in warp order, and each thread's per-pair bias gradients to a [64][65] pair table that dbias_gather reduces
template <int DH_, bool DET = false>
__global__ void __launch_bounds__(128, DH_ == 32 ? 3 : 2) attn_core_bwd_bf16_kernel(const AttnCoreBwdParams p, float* __restrict__ att_out, const DropCfg drop,
                                                                                    const AttnDetSlots det) {
  using K = cbh<DH_>;
  constexpr int DH = K::DH, SM = K::SM, LDQ = K::LDQ, LDP = K::LDP, LPR = K::LPR, PASSES = K::PASSES;
  extern __shared__ __align__(16) uint8_t smraw[];
  const AttnGeom g_ = p.g;
  const int S = g_.S(), nwin = g_.nwin(), W2 = 2 * g_.win - 1, nb = W2 * W2 + 1, R = g_.R, win = g_.win;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  bf16* sQ = reinterpret_cast<bf16*>(smraw); bf16* sK = sQ + SM * LDQ; bf16* sV = sK + SM * LDQ; bf16* sdO = sV + SM * LDQ;
  bf16* sP = sdO + SM * LDQ; bf16* sDS = sP + SM * LDP;
  float* inq = reinterpret_cast<float*>(sDS + SM * LDP); float* ink = inq + SM;
  float* sbias = ink + SM; float* dbias = sbias + nb; float* gred = dbias + nb;
  float* sgam = gred + 2 * DH;             // [4][DH]: rs*gq, 1/(rs*gq), rs*gk, 1/(rs*gk)   (1/. = 0 where gamma = 0)
  const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV), adO = smem_u32(sdO), aP = smem_u32(sP), aDS = smem_u32(sDS);
  const int n = blockIdx.x / p.heads, hd = blockIdx.x - n * p.heads;
  const int inner = p.heads * DH;
  const float rs = sqrtf((float)DH);
  for (int i = threadIdx.x; i < nb; i += 128) { sbias[i] = p.bias_table[i * p.heads + hd]; dbias[i] = 0.f; }
  if (threadIdx.x < 2 * DH) gred[threadIdx.x] = 0.f;
  if (threadIdx.x < DH) {
    const float a = rs * p.qgamma[hd * DH + threadIdx.x], b = rs * p.kgamma[hd * DH + threadIdx.x];
    sgam[threadIdx.x] = a; sgam[DH + threadIdx.x] = a != 0.f ? 1.0f / a : 0.f;
    sgam[2 * DH + threadIdx.x] = b; sgam[3 * DH + threadIdx.x] = b != 0.f ? 1.0f / b : 0.f;
  }
  // phase-1 mapping: LPR lanes per row (32 / LPR rows per pass), each lane 8 consecutive head dims
  const int prow = lane / LPR, pd0 = (lane % LPR) * 8;
  float dgq[DH / 4], dgk[DH / 4];         // DH 32 only (DH 64 sums them in gred once per window)
#pragma unroll
  for (int k = 0; k < DH / 4; ++k) dgq[k] = dgk[k] = 0.f;
  const int r0 = warp * 16;
  const int ia = r0 + g, ib = r0 + g + 8;
  // relative-position-bias index of (query i, key j) = base(i) - off(j); nb-1 when either token is a register token
  int base_a = -1, base_b = -1;
  if (ia >= R && ia < S) { const int ti = ia - R, a = ti / win, b = ti - a * win; base_a = (a + win - 1) * W2 + (b + win - 1); }
  if (ib >= R && ib < S) { const int ti = ib - R, a = ti / win, b = ti - a * win; base_b = (a + win - 1) * W2 + (b + win - 1); }
  float bsa[16], bsb[16];                 // bias of this thread's 32 fixed (query, key) pairs (head-specific, window-independent)
  float dba[16], dbb[16];                 // and its gradient, summed over the windows
  float* gw = sgam + 4 * DH;              // DET: [4 warps][2][DH]
  if constexpr (DET)
    for (int i = threadIdx.x; i < 8 * DH; i += 128) gw[i] = 0.f;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int j = (k >> 1) * 8 + 2 * t + (k & 1);
    int oj = -1;
    if (j >= R && j < S) { const int tj = j - R, a = tj / win, b = tj - a * win; oj = a * W2 + b; }
    bsa[k] = sbias[(oj >= 0 && base_a >= 0) ? base_a - oj : nb - 1];
    bsb[k] = sbias[(oj >= 0 && base_b >= 0) ? base_b - oj : nb - 1];
    dba[k] = dbb[k] = 0.f;
  }

  for (int wi = 0; wi < nwin; ++wi) {
    const long long row0 = ((long long)n * nwin + wi) * S;
    // ---------------- phase 1: rows r0..r0+15; LPR lanes per row, 16-byte loads, two passes' loads issued before the first use
#pragma unroll
    for (int pg = 0; pg < PASSES; pg += 2) {
      float4 ld[2][4][2];                                   // [pass][q,k,v,dO][half]
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        const int i = r0 + (pg + ps) * (32 / LPR) + prow;
#pragma unroll
        for (int m = 0; m < 4; ++m) { ld[ps][m][0] = make_float4(0.f, 0.f, 0.f, 0.f); ld[ps][m][1] = ld[ps][m][0]; }
        if (i < S) {
          const float* src = p.qkv + (row0 + i) * 3 * inner + hd * DH + pd0;
          const float* sdo = p.datt + (row0 + i) * inner + hd * DH + pd0;
#pragma unroll
          for (int m = 0; m < 3; ++m) {
            ld[ps][m][0] = __ldg(reinterpret_cast<const float4*>(src + m * inner));
            ld[ps][m][1] = __ldg(reinterpret_cast<const float4*>(src + m * inner + 4));
          }
          ld[ps][3][0] = __ldg(reinterpret_cast<const float4*>(sdo));
          ld[ps][3][1] = __ldg(reinterpret_cast<const float4*>(sdo + 4));
        }
      }
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        const int i = r0 + (pg + ps) * (32 / LPR) + prow;
        float x[4][8];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          x[m][0] = ld[ps][m][0].x; x[m][1] = ld[ps][m][0].y; x[m][2] = ld[ps][m][0].z; x[m][3] = ld[ps][m][0].w;
          x[m][4] = ld[ps][m][1].x; x[m][5] = ld[ps][m][1].y; x[m][6] = ld[ps][m][1].z; x[m][7] = ld[ps][m][1].w;
        }
        float nq = 0.f, nk = 0.f;
#pragma unroll
        for (int d = 0; d < 8; ++d) { nq = fmaf(x[0][d], x[0][d], nq); nk = fmaf(x[1][d], x[1][d], nk); }
#pragma unroll
        for (int o = 1; o < LPR; o <<= 1) nq += __shfl_xor_sync(0xffffffffu, nq, o);
#pragma unroll
        for (int o = 1; o < LPR; o <<= 1) nk += __shfl_xor_sync(0xffffffffu, nk, o);
        const float iq = 1.0f / fmaxf(sqrtf(nq), 1e-12f), ik = 1.0f / fmaxf(sqrtf(nk), 1e-12f);    // F.normalize eps (maxvit.py:30)
        float gq8[8], gk8[8];
        *reinterpret_cast<float4*>(gq8) = *reinterpret_cast<const float4*>(sgam + pd0);
        *reinterpret_cast<float4*>(gq8 + 4) = *reinterpret_cast<const float4*>(sgam + pd0 + 4);
        *reinterpret_cast<float4*>(gk8) = *reinterpret_cast<const float4*>(sgam + 2 * DH + pd0);
        *reinterpret_cast<float4*>(gk8 + 4) = *reinterpret_cast<const float4*>(sgam + 2 * DH + pd0 + 4);
        uint4 uq, uk, uv, ud;
        uq.x = pack2bf(x[0][0] * iq * gq8[0], x[0][1] * iq * gq8[1]); uq.y = pack2bf(x[0][2] * iq * gq8[2], x[0][3] * iq * gq8[3]);
        uq.z = pack2bf(x[0][4] * iq * gq8[4], x[0][5] * iq * gq8[5]); uq.w = pack2bf(x[0][6] * iq * gq8[6], x[0][7] * iq * gq8[7]);
        uk.x = pack2bf(x[1][0] * ik * gk8[0], x[1][1] * ik * gk8[1]); uk.y = pack2bf(x[1][2] * ik * gk8[2], x[1][3] * ik * gk8[3]);
        uk.z = pack2bf(x[1][4] * ik * gk8[4], x[1][5] * ik * gk8[5]); uk.w = pack2bf(x[1][6] * ik * gk8[6], x[1][7] * ik * gk8[7]);
        uv.x = pack2bf(x[2][0], x[2][1]); uv.y = pack2bf(x[2][2], x[2][3]); uv.z = pack2bf(x[2][4], x[2][5]); uv.w = pack2bf(x[2][6], x[2][7]);
        ud.x = pack2bf(x[3][0], x[3][1]); ud.y = pack2bf(x[3][2], x[3][3]); ud.z = pack2bf(x[3][4], x[3][5]); ud.w = pack2bf(x[3][6], x[3][7]);
        *reinterpret_cast<uint4*>(sQ + i * LDQ + pd0) = uq; *reinterpret_cast<uint4*>(sK + i * LDQ + pd0) = uk;
        *reinterpret_cast<uint4*>(sV + i * LDQ + pd0) = uv; *reinterpret_cast<uint4*>(sdO + i * LDQ + pd0) = ud;
        if (lane % LPR == 0) { inq[i] = iq; ink[i] = ik; }
      }
    }
    __syncthreads();
    // ---------------- phase 2: my 16 query rows x 64 keys
    {
      float pr[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) pr[nt][0] = pr[nt][1] = pr[nt][2] = pr[nt][3] = 0.f;
      warp_mma_bf16<8, DH, false, false>(pr, aQ, LDQ, r0, aK, LDQ, lane);
      float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = nt * 8 + 2 * t + e;
          if (j < S) {
            pr[nt][e] += bsa[nt * 2 + e]; pr[nt][2 + e] += bsb[nt * 2 + e];
            ma = fmaxf(ma, pr[nt][e]); mb = fmaxf(mb, pr[nt][2 + e]);
          } else { pr[nt][e] = -INFINITY; pr[nt][2 + e] = -INFINITY; }
        }
      ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, 1)); ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, 2));
      mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, 1)); mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, 2));
      float sa = 0.f, sb = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          pr[nt][e] = __expf(pr[nt][e] - ma); pr[nt][2 + e] = __expf(pr[nt][2 + e] - mb);
          sa += pr[nt][e]; sb += pr[nt][2 + e];
        }
      sa += __shfl_xor_sync(0xffffffffu, sa, 1); sa += __shfl_xor_sync(0xffffffffu, sa, 2);
      sb += __shfl_xor_sync(0xffffffffu, sb, 1); sb += __shfl_xor_sync(0xffffffffu, sb, 2);
      const float ia_ = ia < S ? 1.0f / sa : 0.f, ib_ = ib < S ? 1.0f / sb : 0.f;      // padded query rows: P = 0
      // dropout on the probabilities (maxvit.py:146): mk = mask * scale per element; smem holds P' = P*mk (used by att and dV),
      // the registers keep P (the softmax Jacobian needs the undropped probabilities)
      float mk[8][4];
      const long long wdx = (long long)n * nwin + wi;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        pr[nt][0] *= ia_; pr[nt][1] *= ia_; pr[nt][2] *= ib_; pr[nt][3] *= ib_;
        mk[nt][0] = mk[nt][1] = mk[nt][2] = mk[nt][3] = 1.0f;
        if (drop.thresh) {
          const int grp = nt * 2 + (t >> 1), sh = 16 * (t & 1);          // keys 4*grp .. 4*grp+3; this thread: bytes 2(t&1), 2(t&1)+1
          const uint32_t ha = drop_hash(drop.seed, drop_row(wdx, ia), drop_group_prob(drop.salt, hd, grp)) >> sh;
          const uint32_t hb = drop_hash(drop.seed, drop_row(wdx, ib), drop_group_prob(drop.salt, hd, grp)) >> sh;
          mk[nt][0] = (int)(ha & 255u) >= drop.thresh ? drop.scale : 0.f; mk[nt][1] = (int)((ha >> 8) & 255u) >= drop.thresh ? drop.scale : 0.f;
          mk[nt][2] = (int)(hb & 255u) >= drop.thresh ? drop.scale : 0.f; mk[nt][3] = (int)((hb >> 8) & 255u) >= drop.thresh ? drop.scale : 0.f;
        }
        *reinterpret_cast<uint32_t*>(sP + ia * LDP + nt * 8 + 2 * t) = pack2bf(pr[nt][0] * mk[nt][0], pr[nt][1] * mk[nt][1]);
        *reinterpret_cast<uint32_t*>(sP + ib * LDP + nt * 8 + 2 * t) = pack2bf(pr[nt][2] * mk[nt][2], pr[nt][3] * mk[nt][3]);
      }
      __syncwarp();
      if (att_out) {                                                // att = P V (re-materialised forward output)
        float av[DH / 8][4];
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) av[nt][0] = av[nt][1] = av[nt][2] = av[nt][3] = 0.f;
        warp_mma_bf16<DH / 8, SM, false, true>(av, aP, LDP, r0, aV, LDQ, lane);
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) {
          if (ia < S) *reinterpret_cast<float2*>(att_out + ((row0 + ia) * inner + hd * DH + nt * 8 + 2 * t)) = make_float2(av[nt][0], av[nt][1]);
          if (ib < S) *reinterpret_cast<float2*>(att_out + ((row0 + ib) * inner + hd * DH + nt * 8 + 2 * t)) = make_float2(av[nt][2], av[nt][3]);
        }
      }
      float dp[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
      warp_mma_bf16<8, DH, false, false>(dp, adO, LDQ, r0, aV, LDQ, lane);
      if (drop.thresh) {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) { dp[nt][0] *= mk[nt][0]; dp[nt][1] *= mk[nt][1]; dp[nt][2] *= mk[nt][2]; dp[nt][3] *= mk[nt][3]; }
      }
      float da = 0.f, db = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) { da += pr[nt][0] * dp[nt][0] + pr[nt][1] * dp[nt][1]; db += pr[nt][2] * dp[nt][2] + pr[nt][3] * dp[nt][3]; }
      da += __shfl_xor_sync(0xffffffffu, da, 1); da += __shfl_xor_sync(0xffffffffu, da, 2);
      db += __shfl_xor_sync(0xffffffffu, db, 1); db += __shfl_xor_sync(0xffffffffu, db, 2);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float dsa = pr[nt][e] * (dp[nt][e] - da), dsb = pr[nt][2 + e] * (dp[nt][2 + e] - db);
          dp[nt][e] = dsa; dp[nt][2 + e] = dsb;
          dba[nt * 2 + e] += dsa; dbb[nt * 2 + e] += dsb;          // zero for padded rows / keys (P = 0 there)
        }
        *reinterpret_cast<uint32_t*>(sDS + ia * LDP + nt * 8 + 2 * t) = pack2bf(dp[nt][0], dp[nt][1]);
        *reinterpret_cast<uint32_t*>(sDS + ib * LDP + nt * 8 + 2 * t) = pack2bf(dp[nt][2], dp[nt][3]);
      }
    }
    __syncthreads();
    // ---------------- phase 3: rows r0..r0+15 as keys (dV, dKh) and as queries (dQh)
    {
      float acc[DH / 8][4];
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
      warp_mma_bf16<DH / 8, SM, true, true>(acc, aP, LDP, r0, adO, LDQ, lane);                 // dV[j][d] = sum_i P[i][j] dO[i][d]
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt) {
        if (ia < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ia) * 3 * inner + 2 * inner + hd * DH + nt * 8 + 2 * t)) = make_float2(acc[nt][0], acc[nt][1]);
        if (ib < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ib) * 3 * inner + 2 * inner + hd * DH + nt * 8 + 2 * t)) = make_float2(acc[nt][2], acc[nt][3]);
      }
#pragma unroll
      for (int which = 0; which < 2; ++which) {
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        if (which == 0) warp_mma_bf16<DH / 8, SM, false, true>(acc, aDS, LDP, r0, aK, LDQ, lane);   // dQh = dS Kh
        else warp_mma_bf16<DH / 8, SM, true, true>(acc, aDS, LDP, r0, aQ, LDQ, lane);               // dKh = dS^T Qh
        const float* inv = which == 0 ? inq : ink;
        const bf16* sX = which == 0 ? sQ : sK;               // xh = u * rs * gamma (bf16): u = xh / (rs * gamma)
        const float* gtab = sgam + which * 2 * DH;
        float* dg = which == 0 ? dgq : dgk;
        float ua[DH / 4], ub[DH / 4], ga[DH / 4], gb[DH / 4], dota = 0.f, dotb = 0.f;
        const float inva = inv[ia], invb = inv[ib];
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) {
          const int d = nt * 8 + 2 * t;
          const float2 xa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sX + ia * LDQ + d));
          const float2 xb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sX + ib * LDQ + d));
          const float2 gg = *reinterpret_cast<const float2*>(gtab + d), ig = *reinterpret_cast<const float2*>(gtab + DH + d);
          ua[2 * nt] = xa.x * ig.x; ua[2 * nt + 1] = xa.y * ig.y; ub[2 * nt] = xb.x * ig.x; ub[2 * nt + 1] = xb.y * ig.y;
          if constexpr (DH == 32) {
            dg[2 * nt] += (acc[nt][0] * ua[2 * nt] + acc[nt][2] * ub[2 * nt]) * rs;
            dg[2 * nt + 1] += (acc[nt][1] * ua[2 * nt + 1] + acc[nt][3] * ub[2 * nt + 1]) * rs;
          } else {                                         // DH 64: the window's gamma partials go to shared memory (register cap)
            float a0 = (acc[nt][0] * ua[2 * nt] + acc[nt][2] * ub[2 * nt]) * rs, a1 = (acc[nt][1] * ua[2 * nt + 1] + acc[nt][3] * ub[2 * nt + 1]) * rs;
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
            if (g == 0) {
              if constexpr (DET) { gw[warp * 2 * DH + which * DH + d] += a0; gw[warp * 2 * DH + which * DH + d + 1] += a1; }
              else { atomicAdd(&gred[which * DH + d], a0); atomicAdd(&gred[which * DH + d + 1], a1); }
            }
          }
          ga[2 * nt] = acc[nt][0] * gg.x; ga[2 * nt + 1] = acc[nt][1] * gg.y;
          gb[2 * nt] = acc[nt][2] * gg.x; gb[2 * nt + 1] = acc[nt][3] * gg.y;
          dota += ga[2 * nt] * ua[2 * nt] + ga[2 * nt + 1] * ua[2 * nt + 1];
          dotb += gb[2 * nt] * ub[2 * nt] + gb[2 * nt + 1] * ub[2 * nt + 1];
        }
        dota += __shfl_xor_sync(0xffffffffu, dota, 1); dota += __shfl_xor_sync(0xffffffffu, dota, 2);
        dotb += __shfl_xor_sync(0xffffffffu, dotb, 1); dotb += __shfl_xor_sync(0xffffffffu, dotb, 2);
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) {
          const int d = nt * 8 + 2 * t;
          if (ia < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ia) * 3 * inner + which * inner + hd * DH + d)) =
                            make_float2(inva * (ga[2 * nt] - ua[2 * nt] * dota), inva * (ga[2 * nt + 1] - ua[2 * nt + 1] * dota));
          if (ib < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ib) * 3 * inner + which * inner + hd * DH + d)) =
                            make_float2(invb * (gb[2 * nt] - ub[2 * nt] * dotb), invb * (gb[2 * nt + 1] - ub[2 * nt + 1] * dotb));
        }
      }
    }
    __syncthreads();
  }
  // relative-position-bias gradient: one shared-memory atomic per (thread, pair) per BLOCK, then one global atomic per entry
  float* pairs = gw + 8 * DH;             // DET: [64][65] per-pair sums over the windows
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int j = (k >> 1) * 8 + 2 * t + (k & 1);
    if (j < S) {
      if constexpr (DET) {
        if (ia < S) pairs[ia * 65 + j] = dba[k];
        if (ib < S) pairs[ib * 65 + j] = dbb[k];
      } else {
        int oj = -1;
        if (j >= R) { const int tj = j - R, a = tj / win, b = tj - a * win; oj = a * W2 + b; }
        if (ia < S) atomicAdd(&dbias[(oj >= 0 && base_a >= 0) ? base_a - oj : nb - 1], dba[k]);
        if (ib < S) atomicAdd(&dbias[(oj >= 0 && base_b >= 0) ? base_b - oj : nb - 1], dbb[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < (DH == 32 ? DH / 4 : 0); ++k) {
    float a = dgq[k], b = dgk[k];
    a += __shfl_xor_sync(0xffffffffu, a, 4); a += __shfl_xor_sync(0xffffffffu, a, 8); a += __shfl_xor_sync(0xffffffffu, a, 16);
    b += __shfl_xor_sync(0xffffffffu, b, 4); b += __shfl_xor_sync(0xffffffffu, b, 8); b += __shfl_xor_sync(0xffffffffu, b, 16);
    if (g == 0) {
      const int d = (k >> 1) * 8 + 2 * t + (k & 1);
      if constexpr (DET) { gw[warp * 2 * DH + d] += a; gw[warp * 2 * DH + DH + d] += b; }
      else { atomicAdd(&gred[d], a); atomicAdd(&gred[DH + d], b); }
    }
  }
  __syncthreads();
  if constexpr (DET) {
    dbias_gather(pairs, 65, g_, nb, dbias, threadIdx.x, 128);
    if (threadIdx.x < 2 * DH) {
      const int which = threadIdx.x / DH, d = threadIdx.x % DH;
      det.gamma[((long long)n * 2 + which) * inner + hd * DH + d] =
          (gw[threadIdx.x] + gw[2 * DH + threadIdx.x]) + (gw[4 * DH + threadIdx.x] + gw[6 * DH + threadIdx.x]);
    }
    det_flush_bias(det, dbias, n, nb, p.heads, hd, threadIdx.x, 128);
  } else {
    if (threadIdx.x < 2 * DH) {
      const int which = threadIdx.x / DH, d = threadIdx.x % DH;
      atomicAdd((which ? p.dkgamma : p.dqgamma) + hd * DH + d, gred[threadIdx.x]);
    }
    for (int i = threadIdx.x; i < nb; i += 128) atomicAdd(p.dbias_table + i * p.heads + hd, dbias[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// Core backward for windows of 65 .. 128 tokens (the reference default, window 8 with four register tokens, has 68).
// The kernels above keep every row tile of a window in shared memory; at 128 slots those tiles do not fit (mode 0: 266 KB of
// [128][DH+1] tiles at DH 64), so these are kernels of their own, launched only when S > 64.  Their dropout masks use the
// 128-slot ids of vg_rng.cuh.
// ------------------------------------------------------------------------------------------------
// Mode 0 (exact fp32, SIMT): K-hat, V and the key-side accumulators dK-hat, dV stay resident ([128][DH+1] each); the query rows
// stream through in blocks of QB: per block Q-hat, the unit q, dO, P (overwritten by dS) and the dropout mask; dQ of a query row
// is finished inside its block.  The key-side RMSNorm backward runs after the last block, with the unit k re-derived from k in
// global memory.  Same arithmetic as attn_core_bwd_kernel per element; DH 64: 199 KB of shared memory (window 11).
template <int DH>
struct cbs_long {
  static constexpr int SK = 128, QB = 32, LD = DH + 1, LP = SK + 1;
  static size_t bytes(int nb) { return (size_t)(4 * SK * LD + 3 * QB * LD + 2 * QB * LP + 2 * nb + SK + QB + 8 * 2 * DH) * sizeof(float); }
};

// DET: as attn_core_bwd_kernel, the bias-table gradient gathered per block of query rows (dbias_gather over rows q0 ..)
template <int DH, bool DET = false>
__global__ void __launch_bounds__(256, 1) attn_core_bwd_long_kernel(const AttnCoreBwdParams p, const DropCfg drop, const AttnDetSlots det) {
  using L = cbs_long<DH>;
  constexpr int SK = L::SK, QB = L::QB, LD = L::LD, LP = L::LP, DPL = DH / 32;
  extern __shared__ float sm[];
  const AttnGeom g = p.g;
  const int S = g.S(), nwin = g.nwin(), W2 = 2 * g.win - 1, nb = W2 * W2 + 1;
  float* kh = sm;                  // [SK][LD] normalised * gamma
  float* vv = kh + SK * LD;
  float* dkh = vv + SK * LD;       // accumulated over the query blocks of a window
  float* dv = dkh + SK * LD;
  float* qh = dv + SK * LD;        // [QB][LD]
  float* qu = qh + QB * LD;        // unit vectors
  float* dO = qu + QB * LD;
  float* P = dO + QB * LD;         // [QB][LP]: P, then dS
  float* MK = P + QB * LP;         // [QB][LP] dropout mask * scale
  float* sbias = MK + QB * LP;     // [nb]
  float* dbias = sbias + nb;       // [nb]
  float* nrk = dbias + nb;         // [SK] |k|
  float* inq = nrk + SK;           // [QB] 1/|q|
  float* gred = inq + QB;          // [8][2][DH]
  const int n = blockIdx.x / p.heads, hd = blockIdx.x - n * p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = p.heads * DH;
  const float rs = sqrtf((float)DH);
  for (int i = threadIdx.x; i < nb; i += 256) { sbias[i] = p.bias_table[i * p.heads + hd]; dbias[i] = 0.f; }
  float gq[DPL], gk[DPL], dgq[DPL], dgk[DPL];
#pragma unroll
  for (int k = 0; k < DPL; ++k) {
    gq[k] = p.qgamma[hd * DH + lane + 32 * k]; gk[k] = p.kgamma[hd * DH + lane + 32 * k];
    dgq[k] = 0.f; dgk[k] = 0.f;
  }
  __syncthreads();

  for (int wi = 0; wi < nwin; ++wi) {
    const long long wdx = (long long)n * nwin + wi, row0 = wdx * S;
    // ---- keys: K-hat, V; dK-hat and dV start at zero.  Warp per row, lane = d
    for (int j = warp; j < S; j += 8) {
      const float* src = p.qkv + (row0 + j) * 3 * inner + hd * DH + lane;
      float k[DPL], v[DPL];
#pragma unroll
      for (int c = 0; c < DPL; ++c) { k[c] = src[inner + 32 * c]; v[c] = src[2 * inner + 32 * c]; }
      const float nk = fmaxf(sqrtf(warp_sum(lane_dot<DPL>(k, k))), 1e-12f);
#pragma unroll
      for (int c = 0; c < DPL; ++c) {
        const int d = lane + 32 * c;
        kh[j * LD + d] = k[c] / nk * rs * gk[c]; vv[j * LD + d] = v[c];
        dkh[j * LD + d] = 0.f; dv[j * LD + d] = 0.f;
      }
      if (lane == 0) nrk[j] = nk;
    }
    for (int q0 = 0; q0 < S; q0 += QB) {
      const int nq = min(QB, S - q0);
      // ---- query rows q0 .. q0 + nq - 1
      for (int r = warp; r < nq; r += 8) {
        const float* src = p.qkv + (row0 + q0 + r) * 3 * inner + hd * DH + lane;
        float q[DPL];
#pragma unroll
        for (int c = 0; c < DPL; ++c) q[c] = src[32 * c];
        const float nq_ = fmaxf(sqrtf(warp_sum(lane_dot<DPL>(q, q))), 1e-12f);
#pragma unroll
        for (int c = 0; c < DPL; ++c) {
          const int d = lane + 32 * c;
          const float uq = q[c] / nq_;
          qu[r * LD + d] = uq; qh[r * LD + d] = uq * rs * gq[c];
          dO[r * LD + d] = p.datt[(row0 + q0 + r) * inner + hd * DH + d];
        }
        if (lane == 0) inq[r] = 1.0f / nq_;
      }
      __syncthreads();
      // ---- P = softmax(qh kh^T + bias): warp per query row, lanes over keys j = lane + 32t
      for (int r = warp; r < nq; r += 8) {
        const int i = q0 + r;
        const int ti = i - g.R, ai = ti / g.win, bi = ti - ai * g.win;
        float s[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int j = lane + 32 * t;
          float a = -INFINITY;
          if (j < S) {
            a = 0.f;
#pragma unroll
            for (int d = 0; d < DH; ++d) a = fmaf(qh[r * LD + d], kh[j * LD + d], a);
            int bidx = nb - 1;
            if (i >= g.R && j >= g.R) { const int tj = j - g.R, aj = tj / g.win, bj = tj - aj * g.win; bidx = (ai - aj + g.win - 1) * W2 + (bi - bj + g.win - 1); }
            a += sbias[bidx];
          }
          s[t] = a;
        }
        const float m = warp_max(fmaxf(fmaxf(s[0], s[1]), fmaxf(s[2], s[3])));
        float e[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) e[t] = lane + 32 * t < S ? __expf(s[t] - m) : 0.f;
        const float inv = 1.0f / warp_sum((e[0] + e[1]) + (e[2] + e[3]));
#pragma unroll
        for (int t = 0; t < 4; ++t) P[r * LP + lane + 32 * t] = e[t] * inv;
        if (drop.thresh) {                                   // the forward pass's mask on the probabilities (maxvit.py:146)
          const uint32_t rid = drop_row(wdx, i, SK);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int j = lane + 32 * t;
            const uint32_t hsh = drop_hash(drop.seed, rid, drop_group_prob(drop.salt, hd, j >> 2, SK));
            MK[r * LP + j] = (int)((hsh >> (8 * (j & 3))) & 255u) >= drop.thresh ? drop.scale : 0.f;
          }
        }
      }
      __syncthreads();
      // ---- dV[j][d] += sum_i P'[i][j] dO[i][d] (P' = P * mask): warp per key, lane = d
      for (int j = warp; j < S; j += 8) {
        float a[DPL];
#pragma unroll
        for (int c = 0; c < DPL; ++c) a[c] = dv[j * LD + lane + 32 * c];
        for (int r = 0; r < nq; ++r) {
          const float pm = drop.thresh ? P[r * LP + j] * MK[r * LP + j] : P[r * LP + j];
#pragma unroll
          for (int c = 0; c < DPL; ++c) a[c] = fmaf(pm, dO[r * LD + lane + 32 * c], a[c]);
        }
#pragma unroll
        for (int c = 0; c < DPL; ++c) dv[j * LD + lane + 32 * c] = a[c];
      }
      __syncthreads();
      // ---- dS = P * (dP - sum_j P dP), dP[i][j] = dO[i] . v[j] (* mask); overwrite P with dS; bias-table gradient
      for (int r = warp; r < nq; r += 8) {
        const int i = q0 + r;
        const int ti = i - g.R, ai = ti / g.win, bi = ti - ai * g.win;
        float dp[4], pr[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int j = lane + 32 * t;
          float a = 0.f;
          if (j < S) {
#pragma unroll
            for (int d = 0; d < DH; ++d) a = fmaf(dO[r * LD + d], vv[j * LD + d], a);
            if (drop.thresh) a *= MK[r * LP + j];
          }
          dp[t] = a; pr[t] = j < S ? P[r * LP + j] : 0.f;
        }
        const float dot = warp_sum((pr[0] * dp[0] + pr[1] * dp[1]) + (pr[2] * dp[2] + pr[3] * dp[3]));
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int j = lane + 32 * t;
          if (j < S) {
            const float ds = pr[t] * (dp[t] - dot);
            P[r * LP + j] = ds;
            if constexpr (!DET) {
              int bidx = nb - 1;
              if (i >= g.R && j >= g.R) { const int tj = j - g.R, aj = tj / g.win, bj = tj - aj * g.win; bidx = (ai - aj + g.win - 1) * W2 + (bi - bj + g.win - 1); }
              atomicAdd(&dbias[bidx], ds);
            }
          }
        }
      }
      __syncthreads();
      if constexpr (DET) dbias_gather(P, LP, g, nb, dbias, threadIdx.x, 256, q0, nq);
      // ---- dK-hat[j] += sum_i dS[i][j] qh[i] (warp per key); dQ-hat[i] = sum_j dS[i][j] kh[j] (warp per query row), then the
      // RMSNorm backward of q (maxvit.py:30): qh = u * rs * gamma, u = q/|q|
      for (int j = warp; j < S; j += 8) {
        float b[DPL];
#pragma unroll
        for (int c = 0; c < DPL; ++c) b[c] = dkh[j * LD + lane + 32 * c];
        for (int r = 0; r < nq; ++r)
#pragma unroll
          for (int c = 0; c < DPL; ++c) b[c] = fmaf(P[r * LP + j], qh[r * LD + lane + 32 * c], b[c]);
#pragma unroll
        for (int c = 0; c < DPL; ++c) dkh[j * LD + lane + 32 * c] = b[c];
      }
      for (int r = warp; r < nq; r += 8) {
        float a[DPL], uq[DPL], g1[DPL];
#pragma unroll
        for (int c = 0; c < DPL; ++c) a[c] = 0.f;
        for (int j = 0; j < S; ++j)
#pragma unroll
          for (int c = 0; c < DPL; ++c) a[c] = fmaf(P[r * LP + j], kh[j * LD + lane + 32 * c], a[c]);
#pragma unroll
        for (int c = 0; c < DPL; ++c) {
          uq[c] = qu[r * LD + lane + 32 * c];
          dgq[c] = fmaf(a[c], uq[c] * rs, dgq[c]);
          g1[c] = a[c] * rs * gq[c];
        }
        const float d1 = warp_sum(lane_dot<DPL>(g1, uq));
        float* dst = p.dqkv + (row0 + q0 + r) * 3 * inner + hd * DH + lane;
#pragma unroll
        for (int c = 0; c < DPL; ++c) dst[32 * c] = inq[r] * (g1[c] - uq[c] * d1);
      }
      __syncthreads();
    }
    // ---- keys: dV out, and the RMSNorm backward of k with u = k/|k| from global memory
    for (int j = warp; j < S; j += 8) {
      const float* src = p.qkv + (row0 + j) * 3 * inner + inner + hd * DH + lane;
      const float nk = nrk[j];
      float uk[DPL], g2[DPL];
#pragma unroll
      for (int c = 0; c < DPL; ++c) {
        const float ak = dkh[j * LD + lane + 32 * c];
        uk[c] = src[32 * c] / nk;
        dgk[c] = fmaf(ak, uk[c] * rs, dgk[c]);
        g2[c] = ak * rs * gk[c];
      }
      const float d2 = warp_sum(lane_dot<DPL>(g2, uk));
      float* dst = p.dqkv + (row0 + j) * 3 * inner + hd * DH + lane;
#pragma unroll
      for (int c = 0; c < DPL; ++c) {
        dst[inner + 32 * c] = (1.0f / nk) * (g2[c] - uk[c] * d2);
        dst[2 * inner + 32 * c] = dv[j * LD + lane + 32 * c];
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < DPL; ++k) { gred[(warp * 2) * DH + lane + 32 * k] = dgq[k]; gred[(warp * 2 + 1) * DH + lane + 32 * k] = dgk[k]; }
  __syncthreads();
  if (threadIdx.x < 2 * DH) {
    const int which = threadIdx.x / DH, d = threadIdx.x % DH;
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += gred[(w * 2 + which) * DH + d];
    if constexpr (DET) det.gamma[((long long)n * 2 + which) * inner + hd * DH + d] = s;
    else atomicAdd((which ? p.dkgamma : p.dqgamma) + hd * DH + d, s);
  }
  if constexpr (DET) det_flush_bias(det, dbias, n, nb, p.heads, hd, threadIdx.x, 256);
  else
    for (int i = threadIdx.x; i < nb; i += 256) atomicAdd(p.dbias_table + i * p.heads + hd, dbias[i]);
}

// Mode 2 (bf16 mma.sync on fp32 tensors): the layout of attn_core_bwd_bf16_kernel at 128 slots, 8 warps of 16 query rows, one
// block per SM (DH 64: 214 KB of shared memory at window 11).  Registers are the limit -- the 64-key kernel already needs 255 at
// DH 64 -- so the score and dP fragments are taken in two 64-key halves: pass 1 finds the row max and the sum of exp over both
// halves, pass 2 writes P' = P * mask and forms the row dot sum_j P dP', pass 3 recomputes the scores and dP' of each half for
// dS.  The bias of a (query, key) pair is read from the table in shared memory, and the bias gradient sums dS per pair over the
// field's windows in an fp32 [128][136] shared tile (the 64-key kernel keeps both in registers).  No att_out.
template <int DH_>
struct cbh_long {
  static constexpr int DH = DH_, SM = 128;
  static constexpr int LDQ = DH + 8;   // as cbh
  static constexpr int LDP = SM + 8;   // bf16 elements per P/dS row (272 B: ldmatrix rows hit distinct banks)
  static constexpr int LDS = SM + 8;   // floats per row of the dS sum (float2 stores of a warp hit distinct banks)
  static constexpr int BYTES = 4 * SM * LDQ * 2 + 2 * SM * LDP * 2 + SM * LDS * 4 + 2 * SM * 4;
  static constexpr int LPR = DH / 8;
  static constexpr int PASSES = 16 / (32 / LPR);
};

// DET (dynamic shared memory grows by 16*DH floats after sgam): per-warp gamma rows gw summed in warp order, the bias table
// gathered from dsum by dbias_gather
template <int DH_, bool DET = false>
__global__ void __launch_bounds__(256, 1) attn_core_bwd_bf16_long_kernel(const AttnCoreBwdParams p, const DropCfg drop, const AttnDetSlots det) {
  using K = cbh_long<DH_>;
  constexpr int DH = K::DH, SM = K::SM, LDQ = K::LDQ, LDP = K::LDP, LDS = K::LDS, LPR = K::LPR, PASSES = K::PASSES;
  extern __shared__ __align__(16) uint8_t smraw[];
  const AttnGeom g_ = p.g;
  const int S = g_.S(), nwin = g_.nwin(), W2 = 2 * g_.win - 1, nb = W2 * W2 + 1, R = g_.R, win = g_.win;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  bf16* sQ = reinterpret_cast<bf16*>(smraw); bf16* sK = sQ + SM * LDQ; bf16* sV = sK + SM * LDQ; bf16* sdO = sV + SM * LDQ;
  bf16* sP = sdO + SM * LDQ; bf16* sDS = sP + SM * LDP;
  float* dsum = reinterpret_cast<float*>(sDS + SM * LDP);     // [SM][LDS] dS of each (query, key) pair summed over the windows
  float* inq = dsum + SM * LDS; float* ink = inq + SM;
  float* sbias = ink + SM; float* dbias = sbias + nb; float* gred = dbias + nb;
  float* sgam = gred + 2 * DH;             // [4][DH]: rs*gq, 1/(rs*gq), rs*gk, 1/(rs*gk)   (1/. = 0 where gamma = 0)
  const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV), adO = smem_u32(sdO), aP = smem_u32(sP), aDS = smem_u32(sDS);
  const int n = blockIdx.x / p.heads, hd = blockIdx.x - n * p.heads;
  const int inner = p.heads * DH;
  const float rs = sqrtf((float)DH);
  for (int i = threadIdx.x; i < nb; i += 256) { sbias[i] = p.bias_table[i * p.heads + hd]; dbias[i] = 0.f; }
  for (int i = threadIdx.x; i < SM * LDS; i += 256) dsum[i] = 0.f;
  if (threadIdx.x < 2 * DH) gred[threadIdx.x] = 0.f;
  if (threadIdx.x < DH) {
    const float a = rs * p.qgamma[hd * DH + threadIdx.x], b = rs * p.kgamma[hd * DH + threadIdx.x];
    sgam[threadIdx.x] = a; sgam[DH + threadIdx.x] = a != 0.f ? 1.0f / a : 0.f;
    sgam[2 * DH + threadIdx.x] = b; sgam[3 * DH + threadIdx.x] = b != 0.f ? 1.0f / b : 0.f;
  }
  const int prow = lane / LPR, pd0 = (lane % LPR) * 8;
  const int r0 = warp * 16;
  const int ia = r0 + g, ib = r0 + g + 8;
  // relative-position-bias index of (query i, key j) = base(i) - off(j); nb-1 when either token is a register token
  int base_a = -1, base_b = -1;
  if (ia >= R && ia < S) { const int ti = ia - R, a = ti / win, b = ti - a * win; base_a = (a + win - 1) * W2 + (b + win - 1); }
  if (ib >= R && ib < S) { const int ti = ib - R, a = ti / win, b = ti - a * win; base_b = (a + win - 1) * W2 + (b + win - 1); }
  float* gw = sgam + 4 * DH;              // DET: [8 warps][2][DH]
  if constexpr (DET)
    for (int i = threadIdx.x; i < 16 * DH; i += 256) gw[i] = 0.f;
  __syncthreads();

  for (int wi = 0; wi < nwin; ++wi) {
    const long long wdx = (long long)n * nwin + wi, row0 = wdx * S;
    // ---------------- phase 1 (as attn_core_bwd_bf16_kernel): rows r0..r0+15, rows >= S zero
#pragma unroll
    for (int pg = 0; pg < PASSES; pg += 2) {
      float4 ld[2][4][2];
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        const int i = r0 + (pg + ps) * (32 / LPR) + prow;
#pragma unroll
        for (int m = 0; m < 4; ++m) { ld[ps][m][0] = make_float4(0.f, 0.f, 0.f, 0.f); ld[ps][m][1] = ld[ps][m][0]; }
        if (i < S) {
          const float* src = p.qkv + (row0 + i) * 3 * inner + hd * DH + pd0;
          const float* sdo = p.datt + (row0 + i) * inner + hd * DH + pd0;
#pragma unroll
          for (int m = 0; m < 3; ++m) {
            ld[ps][m][0] = __ldg(reinterpret_cast<const float4*>(src + m * inner));
            ld[ps][m][1] = __ldg(reinterpret_cast<const float4*>(src + m * inner + 4));
          }
          ld[ps][3][0] = __ldg(reinterpret_cast<const float4*>(sdo));
          ld[ps][3][1] = __ldg(reinterpret_cast<const float4*>(sdo + 4));
        }
      }
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        const int i = r0 + (pg + ps) * (32 / LPR) + prow;
        float x[4][8];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          x[m][0] = ld[ps][m][0].x; x[m][1] = ld[ps][m][0].y; x[m][2] = ld[ps][m][0].z; x[m][3] = ld[ps][m][0].w;
          x[m][4] = ld[ps][m][1].x; x[m][5] = ld[ps][m][1].y; x[m][6] = ld[ps][m][1].z; x[m][7] = ld[ps][m][1].w;
        }
        float nq = 0.f, nk = 0.f;
#pragma unroll
        for (int d = 0; d < 8; ++d) { nq = fmaf(x[0][d], x[0][d], nq); nk = fmaf(x[1][d], x[1][d], nk); }
#pragma unroll
        for (int o = 1; o < LPR; o <<= 1) nq += __shfl_xor_sync(0xffffffffu, nq, o);
#pragma unroll
        for (int o = 1; o < LPR; o <<= 1) nk += __shfl_xor_sync(0xffffffffu, nk, o);
        const float iq = 1.0f / fmaxf(sqrtf(nq), 1e-12f), ik = 1.0f / fmaxf(sqrtf(nk), 1e-12f);    // F.normalize eps (maxvit.py:30)
        float gq8[8], gk8[8];
        *reinterpret_cast<float4*>(gq8) = *reinterpret_cast<const float4*>(sgam + pd0);
        *reinterpret_cast<float4*>(gq8 + 4) = *reinterpret_cast<const float4*>(sgam + pd0 + 4);
        *reinterpret_cast<float4*>(gk8) = *reinterpret_cast<const float4*>(sgam + 2 * DH + pd0);
        *reinterpret_cast<float4*>(gk8 + 4) = *reinterpret_cast<const float4*>(sgam + 2 * DH + pd0 + 4);
        uint4 uq, uk, uv, ud;
        uq.x = pack2bf(x[0][0] * iq * gq8[0], x[0][1] * iq * gq8[1]); uq.y = pack2bf(x[0][2] * iq * gq8[2], x[0][3] * iq * gq8[3]);
        uq.z = pack2bf(x[0][4] * iq * gq8[4], x[0][5] * iq * gq8[5]); uq.w = pack2bf(x[0][6] * iq * gq8[6], x[0][7] * iq * gq8[7]);
        uk.x = pack2bf(x[1][0] * ik * gk8[0], x[1][1] * ik * gk8[1]); uk.y = pack2bf(x[1][2] * ik * gk8[2], x[1][3] * ik * gk8[3]);
        uk.z = pack2bf(x[1][4] * ik * gk8[4], x[1][5] * ik * gk8[5]); uk.w = pack2bf(x[1][6] * ik * gk8[6], x[1][7] * ik * gk8[7]);
        uv.x = pack2bf(x[2][0], x[2][1]); uv.y = pack2bf(x[2][2], x[2][3]); uv.z = pack2bf(x[2][4], x[2][5]); uv.w = pack2bf(x[2][6], x[2][7]);
        ud.x = pack2bf(x[3][0], x[3][1]); ud.y = pack2bf(x[3][2], x[3][3]); ud.z = pack2bf(x[3][4], x[3][5]); ud.w = pack2bf(x[3][6], x[3][7]);
        *reinterpret_cast<uint4*>(sQ + i * LDQ + pd0) = uq; *reinterpret_cast<uint4*>(sK + i * LDQ + pd0) = uk;
        *reinterpret_cast<uint4*>(sV + i * LDQ + pd0) = uv; *reinterpret_cast<uint4*>(sdO + i * LDQ + pd0) = ud;
        if (lane % LPR == 0) { inq[i] = iq; ink[i] = ik; }
      }
    }
    __syncthreads();
    // ---------------- phase 2: my 16 query rows x 128 keys, in two halves of 64 keys
    {
      // scores of half h (keys 64h + 8nt + 2t + e) with the relative-position bias; pad keys -inf
      auto scores = [&](float (&pr)[8][4], int h) {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) pr[nt][0] = pr[nt][1] = pr[nt][2] = pr[nt][3] = 0.f;
        warp_mma_bf16<8, DH, false, false>(pr, aQ, LDQ, r0, aK + (uint32_t)(h * 64 * LDQ * 2), LDQ, lane);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = h * 64 + nt * 8 + 2 * t + e;
            if (j < S) {
              int oj = -1;
              if (j >= R) { const int tj = j - R, a = tj / win, b = tj - a * win; oj = a * W2 + b; }
              pr[nt][e] += sbias[(oj >= 0 && base_a >= 0) ? base_a - oj : nb - 1];
              pr[nt][2 + e] += sbias[(oj >= 0 && base_b >= 0) ? base_b - oj : nb - 1];
            } else { pr[nt][e] = -INFINITY; pr[nt][2 + e] = -INFINITY; }
          }
      };
      // dropout mask * scale of key tile nt of half h: (ia, 2t), (ia, 2t+1), (ib, 2t), (ib, 2t+1)
      auto masks = [&](float (&mk)[4], int h, int nt) {
        mk[0] = mk[1] = mk[2] = mk[3] = 1.0f;
        if (drop.thresh) {
          const int grp = h * 16 + nt * 2 + (t >> 1), sh = 16 * (t & 1);
          const uint32_t ha = drop_hash(drop.seed, drop_row(wdx, ia, SM), drop_group_prob(drop.salt, hd, grp, SM)) >> sh;
          const uint32_t hb = drop_hash(drop.seed, drop_row(wdx, ib, SM), drop_group_prob(drop.salt, hd, grp, SM)) >> sh;
          mk[0] = (int)(ha & 255u) >= drop.thresh ? drop.scale : 0.f; mk[1] = (int)((ha >> 8) & 255u) >= drop.thresh ? drop.scale : 0.f;
          mk[2] = (int)(hb & 255u) >= drop.thresh ? drop.scale : 0.f; mk[3] = (int)((hb >> 8) & 255u) >= drop.thresh ? drop.scale : 0.f;
        }
      };
      // pass 1: row max and sum of exp (online over the halves; the first half is all valid keys since S > 64)
      float ma = -INFINITY, mb = -INFINITY, la = 0.f, lb = 0.f;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        float pr[8][4];
        scores(pr, h);
        float xa = -INFINITY, xb = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) { xa = fmaxf(xa, fmaxf(pr[nt][0], pr[nt][1])); xb = fmaxf(xb, fmaxf(pr[nt][2], pr[nt][3])); }
        xa = fmaxf(xa, __shfl_xor_sync(0xffffffffu, xa, 1)); xa = fmaxf(xa, __shfl_xor_sync(0xffffffffu, xa, 2));
        xb = fmaxf(xb, __shfl_xor_sync(0xffffffffu, xb, 1)); xb = fmaxf(xb, __shfl_xor_sync(0xffffffffu, xb, 2));
        xa = fmaxf(ma, xa); xb = fmaxf(mb, xb);
        float sa = 0.f, sb = 0.f;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) { sa += __expf(pr[nt][e] - xa); sb += __expf(pr[nt][2 + e] - xb); }
        sa += __shfl_xor_sync(0xffffffffu, sa, 1); sa += __shfl_xor_sync(0xffffffffu, sa, 2);
        sb += __shfl_xor_sync(0xffffffffu, sb, 1); sb += __shfl_xor_sync(0xffffffffu, sb, 2);
        la = la * __expf(ma - xa) + sa; lb = lb * __expf(mb - xb) + sb;
        ma = xa; mb = xb;
      }
      const float ia_ = ia < S ? 1.0f / la : 0.f, ib_ = ib < S ? 1.0f / lb : 0.f;      // padded query rows: P = 0
      // pass 2: P' = P * mask -> shared memory (att and dV use it), row dot sum_j P dP' with dP' = (dO V^T) * mask
      float da = 0.f, db = 0.f;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        float pr[8][4], dp[8][4];
        scores(pr, h);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
        warp_mma_bf16<8, DH, false, false>(dp, adO, LDQ, r0, aV + (uint32_t)(h * 64 * LDQ * 2), LDQ, lane);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float mk[4];
          masks(mk, h, nt);
          const float p0 = __expf(pr[nt][0] - ma) * ia_, p1 = __expf(pr[nt][1] - ma) * ia_;
          const float p2 = __expf(pr[nt][2] - mb) * ib_, p3 = __expf(pr[nt][3] - mb) * ib_;
          da += p0 * (dp[nt][0] * mk[0]) + p1 * (dp[nt][1] * mk[1]); db += p2 * (dp[nt][2] * mk[2]) + p3 * (dp[nt][3] * mk[3]);
          *reinterpret_cast<uint32_t*>(sP + ia * LDP + h * 64 + nt * 8 + 2 * t) = pack2bf(p0 * mk[0], p1 * mk[1]);
          *reinterpret_cast<uint32_t*>(sP + ib * LDP + h * 64 + nt * 8 + 2 * t) = pack2bf(p2 * mk[2], p3 * mk[3]);
        }
      }
      da += __shfl_xor_sync(0xffffffffu, da, 1); da += __shfl_xor_sync(0xffffffffu, da, 2);
      db += __shfl_xor_sync(0xffffffffu, db, 1); db += __shfl_xor_sync(0xffffffffu, db, 2);
      // pass 3: dS = P * (dP' - rowdot) -> shared memory (bf16) and the per-pair sum (fp32)
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        float pr[8][4], dp[8][4];
        scores(pr, h);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
        warp_mma_bf16<8, DH, false, false>(dp, adO, LDQ, r0, aV + (uint32_t)(h * 64 * LDQ * 2), LDQ, lane);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float mk[4];
          masks(mk, h, nt);
          const float p0 = __expf(pr[nt][0] - ma) * ia_, p1 = __expf(pr[nt][1] - ma) * ia_;
          const float p2 = __expf(pr[nt][2] - mb) * ib_, p3 = __expf(pr[nt][3] - mb) * ib_;
          const float s0 = p0 * (dp[nt][0] * mk[0] - da), s1 = p1 * (dp[nt][1] * mk[1] - da);
          const float s2 = p2 * (dp[nt][2] * mk[2] - db), s3 = p3 * (dp[nt][3] * mk[3] - db);
          const int j = h * 64 + nt * 8 + 2 * t;
          *reinterpret_cast<uint32_t*>(sDS + ia * LDP + j) = pack2bf(s0, s1);
          *reinterpret_cast<uint32_t*>(sDS + ib * LDP + j) = pack2bf(s2, s3);
          float2* qa = reinterpret_cast<float2*>(dsum + ia * LDS + j);
          float2* qb = reinterpret_cast<float2*>(dsum + ib * LDS + j);
          const float2 va = *qa, vb = *qb;                     // zero for padded rows / keys (P = 0 there)
          *qa = make_float2(va.x + s0, va.y + s1); *qb = make_float2(vb.x + s2, vb.y + s3);
        }
      }
    }
    __syncthreads();
    // ---------------- phase 3: rows r0..r0+15 as keys (dV, dKh) and as queries (dQh), contractions over 128 slots
    {
      float acc[DH / 8][4];
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
      warp_mma_bf16<DH / 8, SM, true, true>(acc, aP, LDP, r0, adO, LDQ, lane);                 // dV[j][d] = sum_i P'[i][j] dO[i][d]
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt) {
        if (ia < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ia) * 3 * inner + 2 * inner + hd * DH + nt * 8 + 2 * t)) = make_float2(acc[nt][0], acc[nt][1]);
        if (ib < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ib) * 3 * inner + 2 * inner + hd * DH + nt * 8 + 2 * t)) = make_float2(acc[nt][2], acc[nt][3]);
      }
#pragma unroll 1
      for (int which = 0; which < 2; ++which) {
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        if (which == 0) warp_mma_bf16<DH / 8, SM, false, true>(acc, aDS, LDP, r0, aK, LDQ, lane);   // dQh = dS Kh
        else warp_mma_bf16<DH / 8, SM, true, true>(acc, aDS, LDP, r0, aQ, LDQ, lane);               // dKh = dS^T Qh
        const float* inv = which == 0 ? inq : ink;
        const bf16* sX = which == 0 ? sQ : sK;               // xh = u * rs * gamma (bf16): u = xh / (rs * gamma)
        const float* gtab = sgam + which * 2 * DH;
        float ua[DH / 4], ub[DH / 4], ga[DH / 4], gb[DH / 4], dota = 0.f, dotb = 0.f;
        const float inva = inv[ia], invb = inv[ib];
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) {
          const int d = nt * 8 + 2 * t;
          const float2 xa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sX + ia * LDQ + d));
          const float2 xb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sX + ib * LDQ + d));
          const float2 gg = *reinterpret_cast<const float2*>(gtab + d), ig = *reinterpret_cast<const float2*>(gtab + DH + d);
          ua[2 * nt] = xa.x * ig.x; ua[2 * nt + 1] = xa.y * ig.y; ub[2 * nt] = xb.x * ig.x; ub[2 * nt + 1] = xb.y * ig.y;
          float a0 = (acc[nt][0] * ua[2 * nt] + acc[nt][2] * ub[2 * nt]) * rs, a1 = (acc[nt][1] * ua[2 * nt + 1] + acc[nt][3] * ub[2 * nt + 1]) * rs;
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
          if (g == 0) {
            if constexpr (DET) { gw[warp * 2 * DH + which * DH + d] += a0; gw[warp * 2 * DH + which * DH + d + 1] += a1; }
            else { atomicAdd(&gred[which * DH + d], a0); atomicAdd(&gred[which * DH + d + 1], a1); }
          }
          ga[2 * nt] = acc[nt][0] * gg.x; ga[2 * nt + 1] = acc[nt][1] * gg.y;
          gb[2 * nt] = acc[nt][2] * gg.x; gb[2 * nt + 1] = acc[nt][3] * gg.y;
          dota += ga[2 * nt] * ua[2 * nt] + ga[2 * nt + 1] * ua[2 * nt + 1];
          dotb += gb[2 * nt] * ub[2 * nt] + gb[2 * nt + 1] * ub[2 * nt + 1];
        }
        dota += __shfl_xor_sync(0xffffffffu, dota, 1); dota += __shfl_xor_sync(0xffffffffu, dota, 2);
        dotb += __shfl_xor_sync(0xffffffffu, dotb, 1); dotb += __shfl_xor_sync(0xffffffffu, dotb, 2);
#pragma unroll
        for (int nt = 0; nt < DH / 8; ++nt) {
          const int d = nt * 8 + 2 * t;
          if (ia < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ia) * 3 * inner + which * inner + hd * DH + d)) =
                            make_float2(inva * (ga[2 * nt] - ua[2 * nt] * dota), inva * (ga[2 * nt + 1] - ua[2 * nt + 1] * dota));
          if (ib < S) *reinterpret_cast<float2*>(p.dqkv + ((row0 + ib) * 3 * inner + which * inner + hd * DH + d)) =
                            make_float2(invb * (gb[2 * nt] - ub[2 * nt] * dotb), invb * (gb[2 * nt + 1] - ub[2 * nt + 1] * dotb));
        }
      }
    }
    __syncthreads();
  }
  // relative-position-bias gradient: the per-pair sums into the table (shared atomics once per block), then one global atomic
  // per entry
  if constexpr (DET) {
    dbias_gather(dsum, LDS, g_, nb, dbias, threadIdx.x, 256);
    if (threadIdx.x < 2 * DH) {
      const int which = threadIdx.x / DH, d = threadIdx.x % DH;
      float s = 0.f;
      for (int w = 0; w < 8; ++w) s += gw[w * 2 * DH + threadIdx.x];
      det.gamma[((long long)n * 2 + which) * inner + hd * DH + d] = s;
    }
    det_flush_bias(det, dbias, n, nb, p.heads, hd, threadIdx.x, 256);
  } else {
    for (int e = threadIdx.x; e < S * S; e += 256) {
      const int i = e / S, j = e - i * S;
      int bidx = nb - 1;
      if (i >= R && j >= R) {
        const int ti = i - R, ai = ti / win, bi = ti - ai * win, tj = j - R, aj = tj / win, bj = tj - aj * win;
        bidx = (ai - aj + win - 1) * W2 + (bi - bj + win - 1);
      }
      atomicAdd(&dbias[bidx], dsum[i * LDS + j]);
    }
    __syncthreads();
    if (threadIdx.x < 2 * DH) {
      const int which = threadIdx.x / DH, d = threadIdx.x % DH;
      atomicAdd((which ? p.dkgamma : p.dqgamma) + hd * DH + d, gred[threadIdx.x]);
    }
    for (int i = threadIdx.x; i < nb; i += 256) atomicAdd(p.dbias_table + i * p.heads + hd, dbias[i]);
  }
}

// LayerNorm (no affine) + FiLM backward with the inverse partition (maxvit.py:176-187, 298-308, 322-332), C = 128 .. 512.
//   tok = xhat*gamma[n] + beta[n];  dgamma[n][c] += dtok*xhat;  dbeta[n][c] += dtok;  dxhat = dtok*gamma
//   dx = rstd*(dxhat - mean(dxhat) - xhat*mean(dxhat*xhat)) + dres   (dres = gradient of the residual path)
// window rows write dx_in[pix] = dx + dx_out[pix]; register rows accumulate into dreg_in ([R][C] or [N][R][C]) with
// the residual gradient dreg_res (N,R,C)*reg_scale (or none).  A warp per row; lane owns channels [lane*4 + 128*k, +4).
struct AttnGatherBwdParams {
  const float* x; const float* reg; int reg_per_field; const float* film;
  const float* dtok; const float* dx_out; const float* dreg_res; float reg_scale;
  float* dx_in; float* dreg_in; float* dfilm;     // dfilm (N, 2C) accumulated
  AttnGeom g; float eps;
};

// DET: dfilm partials go to slot (n, warp - first warp of field n) of det_film, register rows to their window's row of det_reg
template <int C, bool DET = false>
__global__ void __launch_bounds__(256) attn_gather_bwd_kernel(const AttnGatherBwdParams p, long long rows, const AttnDetSlots det) {
  constexpr int RPW = 16, NV = C / 128, NE = 4 * NV;
  const AttnGeom g = p.g;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  const int S = g.S(), nwin = g.nwin();
  float ag[NE], ab[NE];
#pragma unroll
  for (int i = 0; i < NE; ++i) ag[i] = ab[i] = 0.f;
  int n_cur = -1;
  auto flush = [&]() {
    if (n_cur < 0) return;
    if constexpr (DET) {
      const long long rf = (long long)nwin * S;                        // rows per field
      const int j = (int)(((long long)blockIdx.x * 8 + warp) - ((long long)n_cur * rf) / RPW);
      float* d = det.film + ((long long)n_cur * det.K + j) * 2 * C + c0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        *reinterpret_cast<float4*>(d + 128 * k) = make_float4(ag[4 * k], ag[4 * k + 1], ag[4 * k + 2], ag[4 * k + 3]);
        *reinterpret_cast<float4*>(d + C + 128 * k) = make_float4(ab[4 * k], ab[4 * k + 1], ab[4 * k + 2], ab[4 * k + 3]);
      }
#pragma unroll
      for (int i = 0; i < NE; ++i) ag[i] = ab[i] = 0.f;
    } else {
#pragma unroll
      for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          atomicAdd(p.dfilm + (long long)n_cur * 2 * C + 128 * k + c0 + i, ag[4 * k + i]);
          atomicAdd(p.dfilm + (long long)n_cur * 2 * C + C + 128 * k + c0 + i, ab[4 * k + i]);
          ag[4 * k + i] = ab[4 * k + i] = 0.f;
        }
    }
  };
  const long long r0 = ((long long)blockIdx.x * 8 + warp) * RPW;
  // (window, token) of the warp's first row by division, then incrementally: four 64- / 32-bit divisions per row were most of the
  // kernel's instructions
  long long wdx0 = r0 / S;
  int tok = (int)(r0 - wdx0 * S);
  int n = (int)(wdx0 / nwin), wi = (int)(wdx0 - (long long)n * nwin);
  int wx = wi / g.Y, wy = wi - wx * g.Y;                    // window coordinates (attn_token_pixel: wi = x*Y + y)
  int ta = tok >= g.R ? (tok - g.R) / g.win : 0, tb = tok >= g.R ? (tok - g.R) - ta * g.win : 0;   // token row / column inside the window
  for (int k = 0; k < RPW; ++k) {
    const long long r = r0 + k;
    if (r >= rows) break;
    if (n != n_cur) { flush(); n_cur = n; }
    const float* src; long long pix = -1;
    if (tok < g.R) src = p.reg + (p.reg_per_field ? (long long)n * g.R * C : 0) + (long long)tok * C;
    else {
      const int ph = g.grid_mode ? ta * g.X + wx : wx * g.win + ta, pw = g.grid_mode ? tb * g.Y + wy : wy * g.win + tb;      // == attn_token_pixel(g, wi, tok - R)
      pix = (long long)n * g.Hl * g.Wl + (long long)ph * g.Wl + pw;
      src = p.x + pix * C;
    }
    float v[NE];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const float4 xv = *reinterpret_cast<const float4*>(src + 128 * j + c0);
      v[4 * j] = xv.x; v[4 * j + 1] = xv.y; v[4 * j + 2] = xv.z; v[4 * j + 3] = xv.w;
    }
    float sum = v[0] + v[1] + v[2] + v[3];
#pragma unroll
    for (int j = 1; j < NV; ++j) sum += v[4 * j] + v[4 * j + 1] + v[4 * j + 2] + v[4 * j + 3];
    const float mean = warp_sum(sum) * (1.0f / C);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < NE; ++i) { v[i] -= mean; ss += v[i] * v[i]; }
    const float rstd = rsqrtf(warp_sum(ss) * (1.0f / C) + p.eps);
    float gmv[NE], dtv[NE];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const float4 gm = *reinterpret_cast<const float4*>(p.film + (long long)n * 2 * C + 128 * j + c0);
      const float4 dt = *reinterpret_cast<const float4*>(p.dtok + r * C + 128 * j + c0);
      gmv[4 * j] = gm.x; gmv[4 * j + 1] = gm.y; gmv[4 * j + 2] = gm.z; gmv[4 * j + 3] = gm.w;
      dtv[4 * j] = dt.x; dtv[4 * j + 1] = dt.y; dtv[4 * j + 2] = dt.z; dtv[4 * j + 3] = dt.w;
    }
    float dx[NE], s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NE; ++i) {
      v[i] *= rstd;                                            // xhat
      ag[i] = fmaf(dtv[i], v[i], ag[i]); ab[i] += dtv[i];
      dx[i] = dtv[i] * gmv[i]; s1 += dx[i]; s2 = fmaf(dx[i], v[i], s2);
    }
    s1 = warp_sum(s1) * (1.0f / C); s2 = warp_sum(s2) * (1.0f / C);
#pragma unroll
    for (int i = 0; i < NE; ++i) dx[i] = rstd * (dx[i] - s1 - v[i] * s2);
    if (DET && tok < g.R) {
      float* d = det.reg + (((long long)n * nwin + wi) * g.R + tok) * C + c0;
      const float* rr = p.dreg_res ? p.dreg_res + ((long long)n * g.R + tok) * C + c0 : nullptr;
#pragma unroll
      for (int j = 0; j < NV; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) d[128 * j + i] = dx[4 * j + i] + (rr ? rr[128 * j + i] * p.reg_scale : 0.f);
    } else if (tok < g.R) {
      float* d = p.dreg_in + (p.reg_per_field ? (long long)n * g.R * C : 0) + (long long)tok * C + c0;
      const float* rr = p.dreg_res ? p.dreg_res + ((long long)n * g.R + tok) * C + c0 : nullptr;
#pragma unroll
      for (int j = 0; j < NV; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) atomicAdd(d + 128 * j + i, dx[4 * j + i] + (rr ? rr[128 * j + i] * p.reg_scale : 0.f));
    } else {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const float4 ro = *reinterpret_cast<const float4*>(p.dx_out + pix * C + 128 * j + c0);
        *reinterpret_cast<float4*>(p.dx_in + pix * C + 128 * j + c0) =
            make_float4(dx[4 * j] + ro.x, dx[4 * j + 1] + ro.y, dx[4 * j + 2] + ro.z, dx[4 * j + 3] + ro.w);
      }
    }
    // next row
    if (tok >= g.R) { if (++tb == g.win) { tb = 0; ++ta; } }
    if (++tok == S) {
      tok = 0; ta = 0; tb = 0;
      if (++wy == g.Y) { wy = 0; ++wx; }
      if (++wi == nwin) { wi = 0; wx = 0; wy = 0; ++n; }
    }
  }
  flush();
}

// ================================================================================================
// host launchers
// ================================================================================================
long long bn_workspace_elems(long long M, int C) { return ((M + STAT_ROWS - 1) / STAT_ROWS) * 2 * C; }

int bn_stats_run(const float* X, long long M, int C, const float* gamma, const float* beta, float eps, float momentum,
                 float* run_mean, float* run_var, float* mean, float* rstd, float* scale, float* shift, float* work,
                 long long work_elems, cudaStream_t st) {
  const int nparts = (int)((M + STAT_ROWS - 1) / STAT_ROWS);
  if (work_elems < (long long)nparts * 2 * C) return set_error("bn_stats: workspace too small");
  colstats_kernel<<<nparts, 256, 0, st>>>(X, M, C, work);
  int rc = check_launch("colstats_kernel");
  if (rc) return rc;
  bn_finalize_kernel<<<nblk(C, 32), 256, 0, st>>>(work, nparts, M, C, gamma, beta, eps, momentum, run_mean, run_var, mean, rstd, scale, shift);
  return check_launch("bn_finalize_kernel");
}

int bn_stats_local_run(const float* X, long long M, int C, double* row, float* work, long long work_elems, cudaStream_t st) {
  const int nparts = (int)((M + STAT_ROWS - 1) / STAT_ROWS);
  if (work_elems < (long long)nparts * 2 * C) return set_error("bn_stats_local: workspace too small");
  if (nparts > 0) {
    colstats_kernel<<<nparts, 256, 0, st>>>(X, M, C, work);
    int rc = check_launch("colstats_kernel");
    if (rc) return rc;
  }
  bn_stats_local_kernel<<<nblk(C, 32), 256, 0, st>>>(work, nparts, M, C, row);
  return check_launch("bn_stats_local_kernel");
}

int bn_stats_global_run(const double* rows, int world, int C, const float* gamma, const float* beta, float eps, float momentum,
                        float* run_mean, float* run_var, float* mean, float* rstd, float* scale, float* shift, double* count,
                        cudaStream_t st) {
  if (world < 1) return set_error("bn_stats_global: world=%d", world);
  bn_stats_global_kernel<<<nblk(C, 256), 256, 0, st>>>(rows, world, C, gamma, beta, eps, momentum, run_mean, run_var, mean, rstd,
                                                       scale, shift, count);
  return check_launch("bn_stats_global_kernel");
}

int bn_act_run(const float* raw, const float* scale, const float* shift, int act, const float* res, float* out, long long M, int C,
               cudaStream_t st) {
  if (C % 4) return set_error("bn_act: C %% 4 != 0");
  const long long total4 = M * C / 4;
  bn_act_kernel<<<nblk(total4, 256), 256, 0, st>>>(raw, scale, shift, act, res, out, total4, C);
  return check_launch("bn_act_kernel");
}

static bool bn_bwd_width_ok(int C) { return C > 0 && ((C % 4 == 0 && 256 % (C / 4) == 0) || (C % 128 == 0 && C <= 2048)); }

// partial (S1, S2) per STAT_ROWS rows into work[nparts][2][C]
static int bn_bwd_reduce_launch(const BnBwdParams& p, int nparts, float* work, cudaStream_t st) {
  if (p.C <= 1024) bn_bwd_reduce_kernel<false><<<nparts, 256, 0, st>>>(p, work);
  else bn_bwd_reduce_kernel<true><<<dim3(nparts, (p.C + 1023) / 1024), 256, 0, st>>>(p, work);
  return check_launch("bn_bwd_reduce_kernel");
}

static BnBwdParams bn_bwd_params(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean,
                                 const float* rstd, const float* gamma, int act, const float* fgate, const float* fadd,
                                 long long rows_per_field, long long M, int C) {
  BnBwdParams p;
  p.dOut = dOut; p.raw = raw; p.scale = scale; p.shift = shift; p.mean = mean; p.rstd = rstd; p.gamma = gamma;
  p.fgate = fgate; p.fadd = fadd; p.rows_per_field = rows_per_field > 0 ? rows_per_field : 1; p.act = act; p.C = C; p.M = M;
  return p;
}

int bn_bwd_run(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean, const float* rstd,
               const float* gamma, int act, const float* fgate, const float* fadd, long long rows_per_field, long long M, int C,
               float* dgamma, float* dbeta, float* draw, float* work, long long work_elems, cudaStream_t st) {
  const int nparts = (int)((M + STAT_ROWS - 1) / STAT_ROWS);
  if (!bn_bwd_width_ok(C)) return set_error("bn_bwd: C=%d must be 4*k with k | 256, or a multiple of 128 up to 2048", C);
  if (work_elems < (long long)nparts * 2 * C + 2 * C) return set_error("bn_bwd: workspace too small");
  const BnBwdParams p = bn_bwd_params(dOut, raw, scale, shift, mean, rstd, gamma, act, fgate, fadd, rows_per_field, M, C);
  float* k1 = work + (long long)nparts * 2 * C; float* k2 = k1 + C;
  int rc = bn_bwd_reduce_launch(p, nparts, work, st);
  if (rc) return rc;
  bn_bwd_finalize_kernel<<<nblk(C, 32), 256, 0, st>>>(work, nparts, M, C, dgamma, dbeta, k1, k2);
  rc = check_launch("bn_bwd_finalize_kernel");
  if (rc) return rc;
  bn_bwd_apply_kernel<<<nblk(M * (C / 4), 256), 256, 0, st>>>(p, k1, k2, draw);
  return check_launch("bn_bwd_apply_kernel");
}

int bn_bwd_local_run(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean, const float* rstd,
                     int act, const float* fgate, const float* fadd, long long rows_per_field, long long M, int C, float* dgamma,
                     float* dbeta, double* row, float* work, long long work_elems, cudaStream_t st) {
  const int nparts = (int)((M + STAT_ROWS - 1) / STAT_ROWS);
  if (!bn_bwd_width_ok(C)) return set_error("bn_bwd_local: C=%d must be 4*k with k | 256, or a multiple of 128 up to 2048", C);
  if (work_elems < (long long)nparts * 2 * C) return set_error("bn_bwd_local: workspace too small");
  if (nparts > 0) {
    const BnBwdParams p = bn_bwd_params(dOut, raw, scale, shift, mean, rstd, nullptr, act, fgate, fadd, rows_per_field, M, C);
    int rc = bn_bwd_reduce_launch(p, nparts, work, st);
    if (rc) return rc;
  }
  bn_bwd_local_kernel<<<nblk(C, 32), 256, 0, st>>>(work, nparts, C, dgamma, dbeta, row);
  return check_launch("bn_bwd_local_kernel");
}

int bn_bwd_global_run(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean, const float* rstd,
                      const float* gamma, int act, const float* fgate, const float* fadd, long long rows_per_field, long long M, int C,
                      const double* rows, int world, const double* count, float* draw, float* work, long long work_elems,
                      cudaStream_t st) {
  if (!bn_bwd_width_ok(C)) return set_error("bn_bwd_global: C=%d must be 4*k with k | 256, or a multiple of 128 up to 2048", C);
  if (world < 1) return set_error("bn_bwd_global: world=%d", world);
  if (work_elems < 2LL * C) return set_error("bn_bwd_global: workspace too small");
  float* k1 = work; float* k2 = work + C;
  bn_bwd_global_kernel<<<nblk(C, 256), 256, 0, st>>>(rows, world, C, count, k1, k2);
  int rc = check_launch("bn_bwd_global_kernel");
  if (rc || M <= 0) return rc;
  const BnBwdParams p = bn_bwd_params(dOut, raw, scale, shift, mean, rstd, gamma, act, fgate, fadd, rows_per_field, M, C);
  bn_bwd_apply_kernel<<<nblk(M * (C / 4), 256), 256, 0, st>>>(p, k1, k2, draw);
  return check_launch("bn_bwd_apply_kernel");
}

// mean / rstd: the running mean and 1/sqrt(running_var + eps); scale / shift: the affine folded from them
int bn_bwd_frozen_run(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean, const float* rstd,
                      int act, const float* fgate, const float* fadd, long long rows_per_field, long long M, int C, float* dgamma,
                      float* dbeta, float* draw, float* work, long long work_elems, cudaStream_t st) {
  const int nparts = (int)((M + STAT_ROWS - 1) / STAT_ROWS);
  if (!bn_bwd_width_ok(C)) return set_error("bn_bwd_frozen: C=%d must be 4*k with k | 256, or a multiple of 128 up to 2048", C);
  if (work_elems < (long long)nparts * 2 * C) return set_error("bn_bwd_frozen: workspace too small");
  if (M <= 0) return 0;
  const BnBwdParams p = bn_bwd_params(dOut, raw, scale, shift, mean, rstd, nullptr, act, fgate, fadd, rows_per_field, M, C);
  int rc = bn_bwd_reduce_launch(p, nparts, work, st);
  if (rc) return rc;
  bn_bwd_finalize_kernel<<<nblk(C, 32), 256, 0, st>>>(work, nparts, M, C, dgamma, dbeta, nullptr, nullptr);
  rc = check_launch("bn_bwd_finalize_kernel");
  if (rc) return rc;
  bn_bwd_frozen_apply_kernel<<<nblk(M * (C / 4), 256), 256, 0, st>>>(p, draw);
  return check_launch("bn_bwd_frozen_apply_kernel");
}

int colsum_run(const float* X, long long M, int C, float* out, cudaStream_t st) {
  colsum_kernel<<<nblk(M, STAT_ROWS), 256, 0, st>>>(X, M, C, out);
  return check_launch("colsum_kernel");
}

int dwconv_march_run(int dtype, const void* in, const float* w9, const float* scale, const float* shift, int act, void* out,
                     float* psum, int N, int H, int W, int C, cudaStream_t st) {
  const bool sliced = C > 512 && C % 512 == 0;
  if (!sliced && (C % 4 || C / 4 > 128 || (128 % (C / 4)))) return set_error("dwconv: C=%d must be 4*k with k | 128, or a multiple of 512", C);
  const int strips = (W + DW_SW - 1) / DW_SW;
  if (sliced) {
    if (dtype != 1) return set_error("dwconv: C=%d > 512 is built for fp32 only", C);
    dwconv_march_kernel<float, true><<<dim3(N * strips, C / 512), 128, 0, st>>>(reinterpret_cast<const float*>(in), w9, scale, shift, act,
                                                                               reinterpret_cast<float*>(out), psum, H, W, C, strips);
    return check_launch("dwconv_march_kernel");
  }
  const int spb = 128 / (C / 4);
  const int sblocks = (strips + spb - 1) / spb;
  if (dtype == 0) dwconv_march_kernel<bf16><<<N * sblocks, 128, 0, st>>>(reinterpret_cast<const bf16*>(in), w9, scale, shift, act, reinterpret_cast<bf16*>(out), psum, H, W, C, strips);
  else if (dtype == 3) dwconv_march_kernel<__half><<<N * sblocks, 128, 0, st>>>(reinterpret_cast<const __half*>(in), w9, scale, shift, act, reinterpret_cast<__half*>(out), psum, H, W, C, strips);
  else dwconv_march_kernel<float><<<N * sblocks, 128, 0, st>>>(reinterpret_cast<const float*>(in), w9, scale, shift, act, reinterpret_cast<float*>(out), psum, H, W, C, strips);
  return check_launch("dwconv_march_kernel");
}
int dwconv_strips(int W) { return (W + DW_SW - 1) / DW_SW; }

int dw_wgrad_run(const float* X, const float* dY, int N, int H, int W, int C, float* dw9, float* dbias, float* work,
                 long long work_elems, cudaStream_t st) {
  const bool sliced = C > 512 && C % 512 == 0;
  if (!sliced && (C % 4 || C / 4 > 128 || (128 % (C / 4)))) return set_error("dw_wgrad: C=%d must be 4*k with k | 128, or a multiple of 512", C);
  const int strips = (W + DW_SW - 1) / DW_SW;
  const long long nparts = (long long)N * strips;
  if (work_elems < nparts * 10 * C + 10 * C) return set_error("dw_wgrad: workspace too small");
  if (sliced) {
    dw_wgrad_kernel<true><<<dim3(N * strips, C / 512), 128, 0, st>>>(X, dY, work, H, W, C, strips);
  } else {
    const int spb = 128 / (C / 4);
    const int sblocks = (strips + spb - 1) / spb;
    dw_wgrad_kernel<<<N * sblocks, 128, 0, st>>>(X, dY, work, H, W, C, strips);
  }
  int rc = check_launch("dw_wgrad_kernel");
  if (rc) return rc;
  float* tot = work + nparts * 10 * C;
  partial_sum_kernel<<<nblk(10LL * C, 32), 256, 0, st>>>(work, (int)nparts, 10LL * C, 0.f, tot);
  rc = check_launch("partial_sum_kernel");
  if (rc) return rc;
  // dw9 [9][C] += tot[0..9), dbias[C] += tot[9]
  partial_sum_kernel<<<nblk(9LL * C, 32), 256, 0, st>>>(tot, 1, 9LL * C, 1.f, dw9);
  rc = check_launch("partial_sum_kernel");
  if (rc) return rc;
  partial_sum_kernel<<<nblk(C, 32), 256, 0, st>>>(tot + 9LL * C, 1, C, 1.f, dbias);
  return check_launch("partial_sum_kernel");
}

int se_gate_train_run(const float* psum, int N, int nparts, long long HW, const float* W1, const float* W2, int C, int se,
                      float* gate, float* mean, float* hid, cudaStream_t st) {
  if (N <= 1024 && C >= 1024 && C % 4 == 0 && se % 4 == 0 && mean && hid) {      // few fields, wide layers: a warp per weight row (vg_mem.cu)
    field_mean_kernel<<<nblk((long long)N * C, 256), 256, 0, st>>>(psum, nparts, 1.0f / (float)HW, C, (long long)N * C, mean);
    int rc = check_launch("field_mean_kernel");
    if (rc == 0) rc = dense_rows_run(mean, N, C, 0, W1, nullptr, se, 1, hid, st);
    if (rc == 0) rc = dense_rows_run(hid, N, se, 0, W2, nullptr, C, 3, gate, st);
    return rc;
  }
  se_gate_train_kernel<<<N, 256, (C + se) * sizeof(float), st>>>(psum, nparts, 1.0f / (float)HW, W1, W2, C, se, gate, mean, hid);
  return check_launch("se_gate_train_kernel");
}

int field_parts(long long HW) {
  int chunks = (int)((HW + 127) / 128);
  return chunks > 16 ? 16 : (chunks < 1 ? 1 : chunks);
}

int field_dot_run(const float* a, const float* b, float* out, int N, long long HW, int C, cudaStream_t st) {
  field_dot_kernel<<<dim3(field_parts(HW), N), 256, 0, st>>>(a, b, out, HW, C);
  return check_launch("field_dot_kernel");
}

int se_fold_run(const float* W, const float* gate, void* out, int out_f16, int N, int Cout, int C, cudaStream_t st) {
  if (C % 4) return set_error("se_fold: C %% 4 != 0");
  const long long total4 = (long long)N * Cout * C / 4;
  if (out_f16) se_fold_kernel<__half><<<nblk(total4, 256), 256, 0, st>>>(W, gate, reinterpret_cast<__half*>(out), Cout, C, total4);
  else se_fold_kernel<float><<<nblk(total4, 256), 256, 0, st>>>(W, gate, reinterpret_cast<float*>(out), Cout, C, total4);
  return check_launch("se_fold_kernel");
}

int se_scale_oop_run(const float* x, const float* gate, float* out, int N, long long HW, int C, cudaStream_t st) {
  const long long total4 = (long long)N * HW * C / 4;
  se_scale_oop_kernel<<<nblk(total4, 256), 256, 0, st>>>(x, gate, out, HW, C, total4);
  return check_launch("se_scale_oop_kernel");
}

int se_bwd_run(const float* dh4, const float* h3, const float* gate, const float* mean, const float* hid, const float* W1,
               const float* W2, int N, long long HW, int C, int se, float* dW1, float* dW2, float* dmean, float* work,
               long long work_elems, cudaStream_t st) {
  const int nparts = field_parts(HW);
  const long long need = (long long)N * ((nparts + 1) * C + se);
  if (work_elems < need) return set_error("se_bwd: workspace too small");
  float* dgate = work; float* dpre2 = dgate + (long long)N * nparts * C; float* dhid = dpre2 + (long long)N * C;
  field_dot_kernel<<<dim3(nparts, N), 256, 0, st>>>(dh4, h3, dgate, HW, C);
  int rc = check_launch("field_dot_kernel");
  if (rc) return rc;
  se_bwd_kernel<<<N, 256, (C + se) * sizeof(float), st>>>(dgate, nparts, gate, hid, W1, W2, C, se, 1.0f / (float)HW, dpre2, dhid, dmean);
  rc = check_launch("se_bwd_kernel");
  if (rc) return rc;
  rc = outer_sum_run(dpre2, hid, N, C, se, dW2, nullptr, st);       // dW2[c][j] += sum_n dpre2[n][c] hid[n][j]
  if (rc) return rc;
  return outer_sum_run(dhid, mean, N, se, C, dW1, nullptr, st);     // dW1[j][c] += sum_n dhid[n][j] mean[n][c]
}

static DropCfg make_drop(unsigned seed, unsigned salt, int thresh) {
  DropCfg d;
  d.seed = seed; d.salt = salt; d.thresh = thresh; d.scale = 256.0f / (256.0f - (float)thresh);
  return d;
}

int attn_out_bwd_gather_run(const float* dx_out, const float* dreg, float reg_scale, const AttnGeom& g, void* dproj, int out_bf16,
                            unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st) {
  if (g.C % 128) return set_error("attn_out_bwd_gather: C %% 128 != 0");
  if (drop_thresh < 0 || drop_thresh > 255) return set_error("attn_out_bwd_gather: dropout threshold %d outside [0, 255]", drop_thresh);
  const long long rows = (long long)g.N * g.nwin() * g.S();
  if (out_bf16) attn_out_bwd_gather_kernel<bf16><<<nblk(rows, 8), 256, 0, st>>>(dx_out, dreg, reg_scale, g, reinterpret_cast<bf16*>(dproj), rows, make_drop(seed, salt, drop_thresh));
  else attn_out_bwd_gather_kernel<float><<<nblk(rows, 8), 256, 0, st>>>(dx_out, dreg, reg_scale, g, reinterpret_cast<float*>(dproj), rows, make_drop(seed, salt, drop_thresh));
  return check_launch("attn_out_bwd_gather_kernel");
}

// test hook: the masks as bytes, for windows of `slots` (64 or 128) token slots
__global__ void dropout_mask_debug_kernel(DropCfg drop, long long n_windows, int heads, int C, int slots, unsigned char* __restrict__ prob_mask,
                                          unsigned char* __restrict__ out_mask) {
  const int ng = slots / 4;
  const long long total_p = n_windows * heads * slots * ng, total_o = n_windows * slots * (C / 4);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total_p + total_o; idx += (long long)gridDim.x * blockDim.x) {
    if (idx < total_p) {
      const int g = (int)(idx % ng); long long r = idx / ng;
      const int i = (int)(r % slots); r /= slots;
      const int h = (int)(r % heads); const long long wdx = r / heads;
      const uint32_t hsh = drop_hash(drop.seed, drop_row(wdx, i, slots), drop_group_prob(drop.salt, h, g, slots));
      for (int k = 0; k < 4; ++k) prob_mask[((wdx * heads + h) * slots + i) * slots + g * 4 + k] = (int)((hsh >> (8 * k)) & 255u) >= drop.thresh;
    } else {
      const long long j = idx - total_p;
      const int g = (int)(j % (C / 4)); long long r = j / (C / 4);
      const int i = (int)(r % slots); const long long wdx = r / slots;
      const uint32_t hsh = drop_hash(drop.seed, drop_row(wdx, i, slots), drop_group_out(drop.salt, g));
      for (int k = 0; k < 4; ++k) out_mask[(wdx * slots + i) * C + g * 4 + k] = (int)((hsh >> (8 * k)) & 255u) >= drop.thresh;
    }
  }
}

int dropout_mask_debug_run(unsigned seed, unsigned salt, int drop_thresh, long long n_windows, int heads, int C, int slots, unsigned char* prob_mask,
                           unsigned char* out_mask, cudaStream_t st) {
  if (slots != 64 && slots != 128) return set_error("dropout_mask_debug: %d slots (64 or 128)", slots);
  if (slots == 128 && heads > DROP_MAX_HEADS_LONG) return set_error("dropout_mask_debug: %d heads with 128 slots (at most %d)", heads, DROP_MAX_HEADS_LONG);
  dropout_mask_debug_kernel<<<1024, 256, 0, st>>>(make_drop(seed, salt, drop_thresh), n_windows, heads, C, slots, prob_mask, out_mask);
  return check_launch("dropout_mask_debug_kernel");
}

int attn_core_bwd_tc_run(const void* qkv, const void* datt, const float* qgamma, const float* kgamma, const float* bias_table,
                         const AttnGeom& g, int heads, void* dqkv, float* dqgamma, float* dkgamma, float* dbias_table,
                         void* att_out, unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st, const AttnDetSlots* det);

// exact-fp32 SIMT core backward: 8 [64][DH+1] row tiles, P (and the dropout mask) [64][65], bias-table rows, 1/|q|, 1/|k| and the
// per-warp gamma partials (DH 64 with dropout: 172 KB)
template <int DH>
static int core_bwd_simt_launch(const AttnCoreBwdParams& p, int nb, const DropCfg& drop, cudaStream_t st) {
  const size_t smem = (size_t)(8 * 64 * (DH + 1) + 64 * 65 + 2 * nb + 128 + 8 * 2 * DH + (drop.thresh ? 64 * 65 : 0)) * sizeof(float);
  static PerDeviceSize attr_pd;                  // depends on the window size: raise the limit when it grows
  size_t& attr = attr_pd.cur();
  if (smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_bwd_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error("attn_core_bwd smem attr: %s", cudaGetErrorString(e));
    attr = smem;
  }
  attn_core_bwd_kernel<DH><<<p.g.N * p.heads, 256, smem, st>>>(p, drop, AttnDetSlots{});
  return check_launch("attn_core_bwd_kernel");
}

template <int DH>
static int core_bwd_bf16_launch(const AttnCoreBwdParams& q, int nb, float* att_out, const DropCfg& drop, cudaStream_t st) {
  const size_t smem3 = (size_t)cbh<DH>::BYTES + (size_t)(2 * nb + 6 * DH) * sizeof(float);
  static PerDeviceSize attr3_pd;                  // depends on the window size: raise the limit when it grows
  size_t& attr3 = attr3_pd.cur();
  if (smem3 > attr3) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_bwd_bf16_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3);
    if (e != cudaSuccess) return set_error("attn_core_bwd_bf16 smem attr: %s", cudaGetErrorString(e));
    attr3 = smem3;
  }
  attn_core_bwd_bf16_kernel<DH><<<q.g.N * q.heads, 128, smem3, st>>>(q, att_out, drop, AttnDetSlots{});
  return check_launch("attn_core_bwd_bf16_kernel");
}

// windows of 65 .. 128 tokens: one block per (field, head) and SM
template <int DH>
static int core_bwd_simt_long_launch(const AttnCoreBwdParams& p, int nb, const DropCfg& drop, cudaStream_t st) {
  const size_t smem = cbs_long<DH>::bytes(nb);
  static PerDeviceSize attr_pd;                  // depends on the window size: raise the limit when it grows
  size_t& attr = attr_pd.cur();
  if (smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_bwd_long_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error("attn_core_bwd (S > 64) smem attr: %s", cudaGetErrorString(e));
    attr = smem;
  }
  attn_core_bwd_long_kernel<DH><<<p.g.N * p.heads, 256, smem, st>>>(p, drop, AttnDetSlots{});
  return check_launch("attn_core_bwd_long_kernel");
}

template <int DH>
static int core_bwd_bf16_long_launch(const AttnCoreBwdParams& q, int nb, const DropCfg& drop, cudaStream_t st) {
  const size_t smem = (size_t)cbh_long<DH>::BYTES + (size_t)(2 * nb + 6 * DH) * sizeof(float);
  static PerDeviceSize attr_pd;                  // depends on the window size: raise the limit when it grows
  size_t& attr = attr_pd.cur();
  if (smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_bwd_bf16_long_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error("attn_core_bwd_bf16 (S > 64) smem attr: %s", cudaGetErrorString(e));
    attr = smem;
  }
  attn_core_bwd_bf16_long_kernel<DH><<<q.g.N * q.heads, 256, smem, st>>>(q, drop, AttnDetSlots{});
  return check_launch("attn_core_bwd_bf16_long_kernel");
}

// use_tf32: 0 exact-fp32 SIMT, 2 bf16 mma.sync on fp32 tensors, 3 bf16 tensors (qkv, datt, dqkv, att_out): the
// tcgen05 kernel (vg_attn_bwd_tc.cu).  S > 64 (modes 0 and 2 only) runs the long-window kernels.
int attn_core_bwd_run(const float* qkv, const float* datt, const float* qgamma, const float* kgamma, const float* bias_table,
                      const AttnGeom& g, int heads, int dh, float* dqkv, float* dqgamma, float* dkgamma, float* dbias_table,
                      int use_tf32, float* att_out, unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st) {
  if (drop_thresh < 0 || drop_thresh > 255) return set_error("attn_core_bwd: dropout threshold %d outside [0, 255]", drop_thresh);
  if (use_tf32 != 0 && use_tf32 != 2 && use_tf32 != 3) return set_error("attn_core_bwd: mode %d (0 exact fp32, 2 bf16 mma on fp32 tensors, 3 bf16 tensors)", use_tf32);
  if ((use_tf32 == 3 && dh != 32) || (dh != 32 && dh != 64)) return set_error("attn_core_bwd: dim_head must be 32 (got %d)", dh);
  const int max_s = use_tf32 == 3 ? 64 : 128;
  if (g.S() > max_s) return set_error("attn_core_bwd: sequence %d > %d", g.S(), max_s);
  const bool long_win = g.S() > 64;
  if (long_win && att_out) return set_error("attn_core_bwd: att_out needs S <= 64 (got %d)", g.S());
  if (long_win && drop_thresh && heads > DROP_MAX_HEADS_LONG)
    return set_error("attn_core_bwd: dropout with %d heads at sequence %d > 64 (at most %d heads)", heads, g.S(), DROP_MAX_HEADS_LONG);
  const int nb = (2 * g.win - 1) * (2 * g.win - 1) + 1;
  if (use_tf32 == 3)
    return attn_core_bwd_tc_run(qkv, datt, qgamma, kgamma, bias_table, g, heads, dqkv, dqgamma, dkgamma, dbias_table, att_out, seed, salt,
                                drop_thresh, st, nullptr);
  if (use_tf32 == 2) {
    AttnCoreBwdParams q;
    q.qkv = qkv; q.datt = datt; q.qgamma = qgamma; q.kgamma = kgamma; q.bias_table = bias_table; q.dqkv = dqkv;
    q.dqgamma = dqgamma; q.dkgamma = dkgamma; q.dbias_table = dbias_table; q.g = g; q.heads = heads;
    if (long_win)
      return dh == 32 ? core_bwd_bf16_long_launch<32>(q, nb, make_drop(seed, salt, drop_thresh), st)
                      : core_bwd_bf16_long_launch<64>(q, nb, make_drop(seed, salt, drop_thresh), st);
    return dh == 32 ? core_bwd_bf16_launch<32>(q, nb, att_out, make_drop(seed, salt, drop_thresh), st)
                    : core_bwd_bf16_launch<64>(q, nb, att_out, make_drop(seed, salt, drop_thresh), st);
  }
  if (att_out) return set_error("attn_core_bwd: att_out is only produced by the tensor-core kernels (modes 2, 3)");
  AttnCoreBwdParams p;
  p.qkv = qkv; p.datt = datt; p.qgamma = qgamma; p.kgamma = kgamma; p.bias_table = bias_table; p.dqkv = dqkv;
  p.dqgamma = dqgamma; p.dkgamma = dkgamma; p.dbias_table = dbias_table; p.g = g; p.heads = heads;
  if (long_win)
    return dh == 32 ? core_bwd_simt_long_launch<32>(p, nb, make_drop(seed, salt, drop_thresh), st)
                    : core_bwd_simt_long_launch<64>(p, nb, make_drop(seed, salt, drop_thresh), st);
  return dh == 32 ? core_bwd_simt_launch<32>(p, nb, make_drop(seed, salt, drop_thresh), st)
                  : core_bwd_simt_launch<64>(p, nb, make_drop(seed, salt, drop_thresh), st);
}

// ------------------------------------------------------------------------------------------------
// deterministic variants (fixed-order slot reductions, det_sum_run in vg_bwd.cu)
// ------------------------------------------------------------------------------------------------
static int det_work_check(const char* what, long long need, float* work, long long work_elems) {
  if (need > 0 && (!work || work_elems < need)) return set_error("%s: workspace too small (%lld < %lld floats)", what, work_elems, need);
  return 0;
}

long long colsum_det_workspace_elems(long long M, int C) {
  const long long S = (M + STAT_ROWS - 1) / STAT_ROWS;
  return S * C + det_sum_tmp_elems(1, S, C);
}

int colsum_det_run(const float* X, long long M, int C, float* out, float* work, long long work_elems, cudaStream_t st) {
  if (det_work_check("colsum_det", colsum_det_workspace_elems(M, C), work, work_elems)) return 1;
  const long long S = (M + STAT_ROWS - 1) / STAT_ROWS;
  if (S == 0) return 0;
  colsum_kernel<true><<<(unsigned)S, 256, 0, st>>>(X, M, C, work);
  int rc = check_launch("colsum_kernel (det)");
  return rc ? rc : det_sum_run(work, 1, S, C, C, out, C, work + S * C, st);
}

long long attn_core_bwd_det_workspace_elems(const AttnGeom& g, int heads, int dh) {
  const int nb = (2 * g.win - 1) * (2 * g.win - 1) + 1, inner = heads * dh;
  const long long a = (long long)g.N * 2 * inner, b = (long long)g.N * nb * heads;
  const long long t1 = det_sum_tmp_elems(1, g.N, inner), t2 = det_sum_tmp_elems(1, g.N, nb * heads);
  return a + b + (t1 > t2 ? t1 : t2);
}

template <typename KernelFn>
static int det_smem_attr(KernelFn fn, size_t smem, size_t& attr, const char* what) {
  if (smem <= attr) return 0;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return set_error("%s smem attr: %s", what, cudaGetErrorString(e));
  attr = smem;
  return 0;
}

// the DET instantiations of the five core-backward kernels (the modes and limits of attn_core_bwd_run)
template <int DH>
static int core_bwd_det_launch(const AttnCoreBwdParams& p, int nb, int mode, float* att_out, const DropCfg& drop, const AttnDetSlots& det,
                               cudaStream_t st) {
  const bool long_win = p.g.S() > 64;
  const unsigned grid = (unsigned)(p.g.N * p.heads);
  if (mode == 0 && !long_win) {
    const size_t smem = (size_t)(8 * 64 * (DH + 1) + 64 * 65 + 2 * nb + 128 + 8 * 2 * DH + (drop.thresh ? 64 * 65 : 0)) * sizeof(float);
    static PerDeviceSize a_pd;
    if (det_smem_attr(attn_core_bwd_kernel<DH, true>, smem, a_pd.cur(), "attn_core_bwd_det")) return 1;
    attn_core_bwd_kernel<DH, true><<<grid, 256, smem, st>>>(p, drop, det);
  } else if (mode == 0) {
    const size_t smem = cbs_long<DH>::bytes(nb);
    static PerDeviceSize a_pd;
    if (det_smem_attr(attn_core_bwd_long_kernel<DH, true>, smem, a_pd.cur(), "attn_core_bwd_det (S > 64)")) return 1;
    attn_core_bwd_long_kernel<DH, true><<<grid, 256, smem, st>>>(p, drop, det);
  } else if (!long_win) {
    const size_t smem = (size_t)cbh<DH>::BYTES + (size_t)(2 * nb + 6 * DH + 8 * DH + 64 * 65) * sizeof(float);
    static PerDeviceSize a_pd;
    if (det_smem_attr(attn_core_bwd_bf16_kernel<DH, true>, smem, a_pd.cur(), "attn_core_bwd_bf16_det")) return 1;
    attn_core_bwd_bf16_kernel<DH, true><<<grid, 128, smem, st>>>(p, att_out, drop, det);
  } else {
    const size_t smem = (size_t)cbh_long<DH>::BYTES + (size_t)(2 * nb + 6 * DH + 16 * DH) * sizeof(float);
    static PerDeviceSize a_pd;
    if (det_smem_attr(attn_core_bwd_bf16_long_kernel<DH, true>, smem, a_pd.cur(), "attn_core_bwd_bf16_det (S > 64)")) return 1;
    attn_core_bwd_bf16_long_kernel<DH, true><<<grid, 256, smem, st>>>(p, drop, det);
  }
  return check_launch("attn_core_bwd (det)");
}

int attn_core_bwd_det_run(const float* qkv, const float* datt, const float* qgamma, const float* kgamma, const float* bias_table,
                          const AttnGeom& g, int heads, int dh, float* dqkv, float* dqgamma, float* dkgamma, float* dbias_table,
                          int use_tf32, float* att_out, unsigned seed, unsigned salt, int drop_thresh, float* work,
                          long long work_elems, cudaStream_t st) {
  // the checks of attn_core_bwd_run: every mode and window it accepts has a deterministic kernel
  if (drop_thresh < 0 || drop_thresh > 255) return set_error("attn_core_bwd_det: dropout threshold %d outside [0, 255]", drop_thresh);
  if (use_tf32 != 0 && use_tf32 != 2 && use_tf32 != 3) return set_error("attn_core_bwd_det: mode %d (0 exact fp32, 2 bf16 mma on fp32 tensors, 3 bf16 tensors)", use_tf32);
  if ((use_tf32 == 3 && dh != 32) || (dh != 32 && dh != 64)) return set_error("attn_core_bwd_det: dim_head must be 32 (got %d)", dh);
  const int max_s = use_tf32 == 3 ? 64 : 128;
  if (g.S() > max_s) return set_error("attn_core_bwd_det: sequence %d > %d", g.S(), max_s);
  const bool long_win = g.S() > 64;
  if (long_win && att_out) return set_error("attn_core_bwd_det: att_out needs S <= 64 (got %d)", g.S());
  if (long_win && drop_thresh && heads > DROP_MAX_HEADS_LONG)
    return set_error("attn_core_bwd_det: dropout with %d heads at sequence %d > 64 (at most %d heads)", heads, g.S(), DROP_MAX_HEADS_LONG);
  if (use_tf32 == 0 && att_out) return set_error("attn_core_bwd_det: att_out is only produced by the tensor-core kernels (modes 2, 3)");
  if (det_work_check("attn_core_bwd_det", attn_core_bwd_det_workspace_elems(g, heads, dh), work, work_elems)) return 1;
  const int nb = (2 * g.win - 1) * (2 * g.win - 1) + 1, inner = heads * dh;
  AttnDetSlots det{};
  det.gamma = work; det.bias = work + (long long)g.N * 2 * inner;
  float* tmp = det.bias + (long long)g.N * nb * heads;
  int rc;
  if (use_tf32 == 3) {
    rc = attn_core_bwd_tc_run(qkv, datt, qgamma, kgamma, bias_table, g, heads, dqkv, dqgamma, dkgamma, dbias_table, att_out, seed, salt,
                              drop_thresh, st, &det);
  } else {
    AttnCoreBwdParams p;
    p.qkv = qkv; p.datt = datt; p.qgamma = qgamma; p.kgamma = kgamma; p.bias_table = bias_table; p.dqkv = dqkv;
    p.dqgamma = dqgamma; p.dkgamma = dkgamma; p.dbias_table = dbias_table; p.g = g; p.heads = heads;
    const DropCfg drop = make_drop(seed, salt, drop_thresh);
    rc = dh == 32 ? core_bwd_det_launch<32>(p, nb, use_tf32, att_out, drop, det, st)
                  : core_bwd_det_launch<64>(p, nb, use_tf32, att_out, drop, det, st);
  }
  if (!rc) rc = det_sum_run(det.gamma, 1, g.N, inner, 2LL * inner, dqgamma, inner, tmp, st);
  if (!rc) rc = det_sum_run(det.gamma + inner, 1, g.N, inner, 2LL * inner, dkgamma, inner, tmp, st);
  if (!rc) rc = det_sum_run(det.bias, 1, g.N, nb * heads, (long long)nb * heads, dbias_table, (long long)nb * heads, tmp, st);
  return rc;
}

static int gather_bwd_slots(const AttnGeom& g) { return (int)(((long long)g.nwin() * g.S() + 15) / 16) + 1; }

long long attn_gather_bwd_det_workspace_elems(const AttnGeom& g, int reg_per_field) {
  const int K = gather_bwd_slots(g);
  const long long film = (long long)g.N * K * 2 * g.C, reg = (long long)g.N * g.nwin() * g.R * g.C;
  const long long t1 = det_sum_tmp_elems(g.N, K, 2 * g.C);
  const long long t2 = reg_per_field ? det_sum_tmp_elems(g.N, g.nwin(), g.R * g.C) : det_sum_tmp_elems(1, (long long)g.N * g.nwin(), g.R * g.C);
  return film + reg + (t1 > t2 ? t1 : t2);
}

int attn_gather_bwd_det_run(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                            const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in, float* dfilm,
                            const AttnGeom& g, float eps, float* work, long long work_elems, cudaStream_t st) {
  if (g.C != 128 && g.C != 256 && g.C != 384 && g.C != 512) return set_error("attn_gather_bwd_det: C=%d must be 128, 256, 384 or 512", g.C);
  if (det_work_check("attn_gather_bwd_det", attn_gather_bwd_det_workspace_elems(g, reg_per_field), work, work_elems)) return 1;
  AttnGatherBwdParams p;
  p.x = x; p.reg = reg; p.reg_per_field = reg_per_field; p.film = film; p.dtok = dtok; p.dx_out = dx_out; p.dreg_res = dreg_res;
  p.reg_scale = reg_scale; p.dx_in = dx_in; p.dreg_in = dreg_in; p.dfilm = dfilm; p.g = g; p.eps = eps;
  AttnDetSlots det{};
  det.K = gather_bwd_slots(g);
  const long long nfilm = (long long)g.N * det.K * 2 * g.C, nwr = (long long)g.N * g.nwin();
  det.film = work; det.reg = work + nfilm;
  float* tmp = det.reg + nwr * g.R * g.C;
  cudaError_t e = cudaMemsetAsync(det.film, 0, (size_t)nfilm * sizeof(float), st);
  if (e != cudaSuccess) return set_error("attn_gather_bwd_det: %s", cudaGetErrorString(e));
  const long long rows = nwr * g.S();
  const unsigned grid = nblk(rows, 8 * 16);
  switch (g.C) {
    case 128: attn_gather_bwd_kernel<128, true><<<grid, 256, 0, st>>>(p, rows, det); break;
    case 256: attn_gather_bwd_kernel<256, true><<<grid, 256, 0, st>>>(p, rows, det); break;
    case 384: attn_gather_bwd_kernel<384, true><<<grid, 256, 0, st>>>(p, rows, det); break;
    default: attn_gather_bwd_kernel<512, true><<<grid, 256, 0, st>>>(p, rows, det); break;
  }
  int rc = check_launch("attn_gather_bwd_kernel (det)");
  if (!rc) rc = det_sum_run(det.film, g.N, det.K, 2 * g.C, 2LL * g.C, dfilm, 2LL * g.C, tmp, st);
  if (!rc && g.R > 0) {
    if (reg_per_field) rc = det_sum_run(det.reg, g.N, g.nwin(), g.R * g.C, (long long)g.R * g.C, dreg_in, (long long)g.R * g.C, tmp, st);
    else rc = det_sum_run(det.reg, 1, nwr, g.R * g.C, (long long)g.R * g.C, dreg_in, (long long)g.R * g.C, tmp, st);
  }
  return rc;
}

int attn_gather_bwd_run(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                        const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in, float* dfilm,
                        const AttnGeom& g, float eps, cudaStream_t st) {
  if (g.C != 128 && g.C != 256 && g.C != 384 && g.C != 512) return set_error("attn_gather_bwd: C=%d must be 128, 256, 384 or 512", g.C);
  AttnGatherBwdParams p;
  p.x = x; p.reg = reg; p.reg_per_field = reg_per_field; p.film = film; p.dtok = dtok; p.dx_out = dx_out; p.dreg_res = dreg_res;
  p.reg_scale = reg_scale; p.dx_in = dx_in; p.dreg_in = dreg_in; p.dfilm = dfilm; p.g = g; p.eps = eps;
  const long long rows = (long long)g.N * g.nwin() * g.S();
  const unsigned grid = nblk(rows, 8 * 16);
  switch (g.C) {
    case 128: attn_gather_bwd_kernel<128><<<grid, 256, 0, st>>>(p, rows, AttnDetSlots{}); break;
    case 256: attn_gather_bwd_kernel<256><<<grid, 256, 0, st>>>(p, rows, AttnDetSlots{}); break;
    case 384: attn_gather_bwd_kernel<384><<<grid, 256, 0, st>>>(p, rows, AttnDetSlots{}); break;
    default: attn_gather_bwd_kernel<512><<<grid, 256, 0, st>>>(p, rows, AttnDetSlots{}); break;
  }
  return check_launch("attn_gather_bwd_kernel");
}

}  // namespace vg
