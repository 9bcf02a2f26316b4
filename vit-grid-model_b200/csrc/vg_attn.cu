// Window / grid attention pieces (maxvit.py:170-219, 289-341).
//
//  attn_gather : window (block) or dilated (grid) partition folded into the load addressing + register-token
//                concat + LayerNorm (no affine) + FiLM  ->  token matrix (Nw*S, C)          [HBM-bound]
//  attn_core   : per (window, head): QK-RMSNorm, QK^T + relative-position bias (index computed arithmetically,
//                maxvit.py:160-167), softmax, PV                                               [v1: SIMT fp32 math]
// The QKV and output projections are shifted-row GEMMs (vg_gemm.cu); the output projection's epilogue adds the
// residual and scatters through the inverse partition map, so no partitioned tensor is ever materialised in
// NCHW/NHWC form.
#include "vg_common.cuh"
#include "vg_host.h"
#include "vg_rng.cuh"

namespace vg {

// token row r = wdx*S + tok,  wdx = n*nwin + x*Y + y  (windows field-major, x-major: maxvit.py:306-307); the pixel of a
// window token is attn_token_pixel (vg_host.h)

// test hook: the global pixel index every token row gathers from / scatters to (-1 for register-token rows)
__global__ void attn_partition_debug_kernel(const AttnGeom g, long long* __restrict__ out, long long rows) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int S = g.S(), nwin = g.nwin();
  const long long wdx = r / S;
  const int tok = (int)(r - wdx * S);
  const int n = (int)(wdx / nwin), wi = (int)(wdx - (long long)n * nwin);
  out[r] = tok < g.R ? -1 : (long long)n * g.Hl * g.Wl + attn_token_pixel(g, wi, tok - g.R);
}

template <typename T, typename TO>
__global__ void __launch_bounds__(256) attn_gather_kernel(const T* __restrict__ x, const float* __restrict__ reg, int reg_per_field,
                                                          const float* __restrict__ film, const AttnGeom g, float eps,
                                                          TO* __restrict__ tokens, long long rows) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const int S = g.S(), nwin = g.nwin(), C = g.C;
  const long long wdx = r / S;
  const int tok = (int)(r - wdx * S);
  const int n = (int)(wdx / nwin), wi = (int)(wdx - (long long)n * nwin);
  // C = 128*k: lane owns channels [lane*4 + 128*i, +4)
  float v[16];
  const int nv = C / 128;
  float s = 0.f;
  if (tok < g.R) {
    const float* src = reg + (reg_per_field ? (long long)n * g.R * C : 0) + (long long)tok * C;
    for (int i = 0; i < nv; ++i) {
      const float4 f = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
      v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
    }
  } else {
    const T* src = x + ((long long)n * g.Hl * g.Wl + attn_token_pixel(g, wi, tok - g.R)) * C;
    for (int i = 0; i < nv; ++i) {                                       // one 16- / 8-byte load per lane and 128 channels
      if constexpr (sizeof(T) == 4) {
        const float4 f = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
        v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
      } else {
        const uint2 u = *reinterpret_cast<const uint2*>(src + i * 128 + lane * 4);
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x)), b2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        v[4 * i] = a.x; v[4 * i + 1] = a.y; v[4 * i + 2] = b2.x; v[4 * i + 3] = b2.y;
      }
    }
  }
  for (int i = 0; i < 4 * nv; ++i) s += v[i];
  const float mean = warp_sum(s) / (float)C;
  float ss = 0.f;
  for (int i = 0; i < 4 * nv; ++i) { v[i] -= mean; ss += v[i] * v[i]; }
  const float rstd = rsqrtf(warp_sum(ss) / (float)C + eps);             // nn.LayerNorm, no affine (maxvit.py:137)
  const float* gam = film + (long long)n * 2 * C;                        // [gamma | beta], used raw (maxvit.py:187)
  TO* dst = tokens + r * C;
  for (int i = 0; i < nv; ++i) {
    const int c = i * 128 + lane * 4;
    const float4 ga = *reinterpret_cast<const float4*>(gam + c), be = *reinterpret_cast<const float4*>(gam + C + c);
    const float o0 = v[4 * i] * rstd * ga.x + be.x, o1 = v[4 * i + 1] * rstd * ga.y + be.y;
    const float o2 = v[4 * i + 2] * rstd * ga.z + be.z, o3 = v[4 * i + 3] * rstd * ga.w + be.w;
    if constexpr (sizeof(TO) == 4) {
      *reinterpret_cast<float4*>(dst + c) = make_float4(o0, o1, o2, o3);
    } else {
      uint2 u;
      *reinterpret_cast<__nv_bfloat162*>(&u.x) = __floats2bfloat162_rn(o0, o1);
      *reinterpret_cast<__nv_bfloat162*>(&u.y) = __floats2bfloat162_rn(o2, o3);
      *reinterpret_cast<uint2*>(dst + c) = u;
    }
  }
}

__device__ __forceinline__ float4 ld4f(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4f(const bf16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x)), b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// One block per (window, head), one query row per thread (ceil(S / 32) warps).  K-hat and V are staged in shared memory as fp32
// rows of DH floats (pad rows up to a multiple of 4 are zeros): DH/4 lanes stage one row with 16-byte loads and stores, the
// row norm by shuffles.  Every lane of a warp then reads the same key, so the reads are 16-byte broadcasts.  Keys go four at a
// time through the online softmax: four scores (each four partial sums -- a single 64-long FMA chain was the latency bound of
// the first version of this kernel, which also kept one (K, V) copy per warp: 113 KB per block, 8 warps per SM), one rescale
// of the output row per four keys.  BASELINE configs[4] (32 heads x 64, 360 windows): 0.93 -> see profiles/r02_summary.md.
template <typename T, int DH>
__global__ void __launch_bounds__(128, DH == 64 ? 3 : 5) attn_core_kernel(const T* __restrict__ qkv, const float* __restrict__ qgamma,
                                                        const float* __restrict__ kgamma, const float* __restrict__ bias_table,
                                                        const AttnGeom g, int heads, T* __restrict__ out, const DropCfg drop) {
  extern __shared__ __align__(16) float sm[];
  const int S = g.S(), Sp = (S + 3) & ~3, nb = (2 * g.win - 1) * (2 * g.win - 1) + 1;
  const int lane = threadIdx.x & 31;
  float* sk = sm;
  float* sv = sk + Sp * DH;
  float* sbias = sv + Sp * DH;
  const long long pair = blockIdx.x;
  const long long wdx = pair / heads;
  const int hd = (int)(pair - wdx * heads);
  const int inner = heads * DH;
  const T* base = qkv + wdx * S * 3 * inner + hd * DH;
  const float rs = sqrtf((float)DH);

  for (int i = threadIdx.x; i < nb; i += blockDim.x) sbias[i] = bias_table[i * heads + hd];
  {
    constexpr int LPR = DH / 4, RPP = 32 / LPR;              // lanes per row, rows per warp pass
    const int sub = lane / LPR, ch = lane - sub * LPR;
    const float4 kg = *reinterpret_cast<const float4*>(kgamma + hd * DH + ch * 4);
    // all the loads of a batch of UNR passes are issued before the first norm: one global round trip per batch, not per pass
    constexpr int UNR = 7;
    const int step = (blockDim.x >> 5) * RPP;
    for (int jb = (threadIdx.x >> 5) * RPP; jb < Sp; jb += step * UNR) {
      float4 k[UNR], v[UNR];
#pragma unroll
      for (int t = 0; t < UNR; ++t) {
        const int j = jb + t * step + sub;
        k[t] = make_float4(0.f, 0.f, 0.f, 0.f); v[t] = k[t];
        if (j < S) { const T* kp = base + (long long)j * 3 * inner + inner + ch * 4; k[t] = ld4f(kp); v[t] = ld4f(kp + inner); }
      }
#pragma unroll
      for (int t = 0; t < UNR; ++t) {
        if (jb + t * step < Sp) {                                // warp-uniform; then j < Sp too (Sp is a multiple of 4, RPP divides 4)
          const int j = jb + t * step + sub;
          float nrm = k[t].x * k[t].x + k[t].y * k[t].y + k[t].z * k[t].z + k[t].w * k[t].w;
#pragma unroll
          for (int o = LPR / 2; o; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
          const float inv = rs / fmaxf(sqrtf(nrm), 1e-12f);      // F.normalize eps (maxvit.py:30)
          *reinterpret_cast<float4*>(sk + j * DH + ch * 4) = make_float4(k[t].x * inv * kg.x, k[t].y * inv * kg.y, k[t].z * inv * kg.z, k[t].w * inv * kg.w);
          *reinterpret_cast<float4*>(sv + j * DH + ch * 4) = v[t];
        }
      }
    }
  }
  __syncthreads();

  const int i = threadIdx.x;
  if (i >= S) return;
  const int W2 = 2 * g.win - 1;
  float q[DH], o[DH], nrm = 0.f;
  const T* qp = base + (long long)i * 3 * inner;
#pragma unroll
  for (int d = 0; d < DH; d += 8) ld8(qp + d, q + d);
#pragma unroll
  for (int d = 0; d < DH; ++d) nrm += q[d] * q[d];
  const float inv = rs / fmaxf(sqrtf(nrm), 1e-12f);
#pragma unroll
  for (int d = 0; d < DH; ++d) { q[d] *= inv * qgamma[hd * DH + d]; o[d] = 0.f; }
  const int ti = i - g.R, ai = ti / g.win, bi = ti - ai * g.win;
  float m = -INFINITY, l = 0.f;
  const int slots = drop_slots(S);
  for (int j0 = 0; j0 < Sp; j0 += 4) {
    // nn.Dropout on the probabilities (maxvit.py:146): the same counter-based mask as the fused kernels (vg_rng.cuh; 128 slots
    // per window when S > 64)
    const uint32_t hsh = drop.thresh ? drop_hash(drop.seed, drop_row(wdx, i, slots), drop_group_prob(drop.salt, hd, j0 >> 2, slots)) : 0u;
    float sc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      const float4* kr = reinterpret_cast<const float4*>(sk + j * DH);
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        const float4 k = kr[c];
        s0 = fmaf(q[4 * c], k.x, s0); s1 = fmaf(q[4 * c + 1], k.y, s1); s2 = fmaf(q[4 * c + 2], k.z, s2); s3 = fmaf(q[4 * c + 3], k.w, s3);
      }
      int bidx = nb - 1;                                                 // register row/col -> shared last entry
      if (i >= g.R && j >= g.R && j < S) {
        const int tj = j - g.R, aj = tj / g.win, bj = tj - aj * g.win;
        bidx = (ai - aj + g.win - 1) * W2 + (bi - bj + g.win - 1);
      }
      sc[u] = j < S ? (s0 + s1) + (s2 + s3) + sbias[bidx] : -INFINITY;
    }
    const float mn = fmaxf(fmaxf(m, fmaxf(sc[0], sc[1])), fmaxf(sc[2], sc[3]));    // the first key of a group is always valid: finite
    const float corr = __expf(m - mn);
    float pm[4], ps = 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float p = __expf(sc[u] - mn);
      ps += p;                                                             // the normaliser l stays un-dropped
      pm[u] = !drop.thresh ? p : ((int)((hsh >> (8 * u)) & 255u) >= drop.thresh ? p * drop.scale : 0.f);
    }
    l = l * corr + ps;
    m = mn;
    const float4* v0 = reinterpret_cast<const float4*>(sv + j0 * DH);
#pragma unroll
    for (int c = 0; c < DH / 4; ++c) {
      const float4 a = v0[c], b = v0[c + DH / 4], cc = v0[c + 2 * (DH / 4)], dd = v0[c + 3 * (DH / 4)];
      o[4 * c]     = fmaf(pm[0], a.x, fmaf(pm[1], b.x, fmaf(pm[2], cc.x, fmaf(pm[3], dd.x, o[4 * c] * corr))));
      o[4 * c + 1] = fmaf(pm[0], a.y, fmaf(pm[1], b.y, fmaf(pm[2], cc.y, fmaf(pm[3], dd.y, o[4 * c + 1] * corr))));
      o[4 * c + 2] = fmaf(pm[0], a.z, fmaf(pm[1], b.z, fmaf(pm[2], cc.z, fmaf(pm[3], dd.z, o[4 * c + 2] * corr))));
      o[4 * c + 3] = fmaf(pm[0], a.w, fmaf(pm[1], b.w, fmaf(pm[2], cc.w, fmaf(pm[3], dd.w, o[4 * c + 3] * corr))));
    }
  }
  const float il = 1.0f / l;
#pragma unroll
  for (int d = 0; d < DH; ++d) o[d] *= il;
  T* op = out + (wdx * S + i) * inner + hd * DH;
#pragma unroll
  for (int d = 0; d < DH; d += 8) st8(op + d, o + d);
}

// ------------------------------------------------------------------------------------------------
// The same core on the tensor cores for the shapes of the un-fused path (S <= 64, no dropout): mma.sync m16n8k8 tf32, one block
// of four warps per (window, head), 16 query rows per warp.  SPLIT: every product as three tf32 products of the operands' hi / lo
// halves (hi*hi + hi*lo + lo*hi: fp32-grade, 24 accumulation steps per score) -- the 'tf32_conv' precision of wide networks; without
// SPLIT one tf32 product (10-bit operands, for bf16 storage).  K-hat and V sit in shared memory as fp32 rows of DH + 4 floats:
// the B-fragment reads (key g, dim t) and (key 2t, dim g) both touch 32 different banks.  The accumulator fragment of S holds keys
// (2t, 2t+1) of every 8-key tile where the A fragment of the next product wants (t, t+4): instead of moving P between lanes the
// contraction index of P.V is permuted -- the V fragment is read at keys (8k + 2t, 8k + 2t + 1).
__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t tf32_hi(float x) { return __float_as_uint(x) & 0xffffe000u; }
__device__ __forceinline__ uint32_t tf32_lo(float x, uint32_t hi) { return __float_as_uint(x - __uint_as_float(hi)) & 0xffffe000u; }

template <typename T, int DH, bool SPLIT>
__global__ void __launch_bounds__(128) attn_core_mma_kernel(const T* __restrict__ qkv, const float* __restrict__ qgamma,
                                                            const float* __restrict__ kgamma, const float* __restrict__ bias_table,
                                                            const AttnGeom g, int heads, T* __restrict__ out, int out_split) {
  constexpr int LD = DH + 4, KT = DH / 8;
  extern __shared__ __align__(16) float sm[];
  float* sk = sm;
  float* sv = sk + 64 * LD;
  float* sbias = sv + 64 * LD;
  int* skey = reinterpret_cast<int*>(sbias + (((2 * g.win - 1) * (2 * g.win - 1) + 1 + 3) & ~3));     // [64]: key -> (aj << 8 | bj), -1 = register token
  const int S = g.S(), nb = (2 * g.win - 1) * (2 * g.win - 1) + 1, W2 = 2 * g.win - 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long pair = blockIdx.x;
  const long long wdx = pair / heads;
  const int hd = (int)(pair - wdx * heads);
  const int inner = heads * DH;
  const T* base = qkv + wdx * S * 3 * inner + hd * DH;
  const float rs = sqrtf((float)DH);

  for (int i = threadIdx.x; i < nb; i += 128) sbias[i] = bias_table[i * heads + hd];
  if (threadIdx.x < 64) {
    const int tj = (int)threadIdx.x - g.R, aj = tj / g.win;
    skey[threadIdx.x] = tj < 0 ? -1 : ((aj << 8) | (tj - aj * g.win));
  }
  {
    constexpr int LPR = DH / 4, RPP = 32 / LPR, UNR = 64 / (4 * RPP);      // the block stages 64 rows in UNR passes of 4 * RPP rows
    const int sub = lane / LPR, ch = lane - sub * LPR;
    const float4 kg = *reinterpret_cast<const float4*>(kgamma + hd * DH + ch * 4);
    float4 k[UNR], v[UNR];
#pragma unroll
    for (int t = 0; t < UNR; ++t) {
      const int j = (t * 4 + warp) * RPP + sub;
      k[t] = make_float4(0.f, 0.f, 0.f, 0.f); v[t] = k[t];
      if (j < S) { const T* kp = base + (long long)j * 3 * inner + inner + ch * 4; k[t] = ld4f(kp); v[t] = ld4f(kp + inner); }
    }
#pragma unroll
    for (int t = 0; t < UNR; ++t) {
      const int j = (t * 4 + warp) * RPP + sub;
      float nrm = k[t].x * k[t].x + k[t].y * k[t].y + k[t].z * k[t].z + k[t].w * k[t].w;
#pragma unroll
      for (int o = LPR / 2; o; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
      const float inv = rs / fmaxf(sqrtf(nrm), 1e-12f);        // F.normalize eps (maxvit.py:30); pad rows stay zero
      *reinterpret_cast<float4*>(sk + j * LD + ch * 4) = make_float4(k[t].x * inv * kg.x, k[t].y * inv * kg.y, k[t].z * inv * kg.z, k[t].w * inv * kg.w);
      *reinterpret_cast<float4*>(sv + j * LD + ch * 4) = v[t];
    }
  }
  __syncthreads();
  const int r0 = warp * 16;
  if (r0 >= S) return;
  const int gq = lane >> 2, t4 = lane & 3;
  const int i0 = r0 + gq, i1 = i0 + 8;

  // Q-hat fragments: this thread holds dims t4 + 4m of rows i0 and i1 (the four lanes of a quad cover a row)
  uint32_t qh[2][2 * KT], ql[SPLIT ? 2 : 1][SPLIT ? 2 * KT : 1];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int i = r ? i1 : i0;
    float q[2 * KT], nrm = 0.f;
    const T* qp = base + (long long)i * 3 * inner;
#pragma unroll
    for (int m = 0; m < 2 * KT; ++m) { q[m] = i < S ? (float)qp[t4 + 4 * m] : 0.f; nrm = fmaf(q[m], q[m], nrm); }
    nrm += __shfl_xor_sync(0xffffffffu, nrm, 1);
    nrm += __shfl_xor_sync(0xffffffffu, nrm, 2);
    const float inv = rs / fmaxf(sqrtf(nrm), 1e-12f);
#pragma unroll
    for (int m = 0; m < 2 * KT; ++m) {
      const float x = q[m] * inv * qgamma[hd * DH + t4 + 4 * m];
      qh[r][m] = tf32_hi(x);
      if (SPLIT) ql[r][m] = tf32_lo(x, qh[r][m]);
    }
  }

  // consecutive MMAs go to different accumulators (the asm statements keep their order: a key-tile-outer loop would issue 3 * KT
  // dependent MMAs back to back)
  float sacc[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) sacc[nt][0] = sacc[nt][1] = sacc[nt][2] = sacc[nt][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < KT; ++kt) {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float* kr = sk + (8 * nt + gq) * LD + t4 + 8 * kt;
      const float k0 = kr[0], k1 = kr[4];
      const uint32_t b0 = tf32_hi(k0), b1 = tf32_hi(k1);
      if (SPLIT) {
        const uint32_t c0 = tf32_lo(k0, b0), c1 = tf32_lo(k1, b1);
        mma_tf32(sacc[nt], ql[0][2 * kt], ql[1][2 * kt], ql[0][2 * kt + 1], ql[1][2 * kt + 1], b0, b1);
        mma_tf32(sacc[nt], qh[0][2 * kt], qh[1][2 * kt], qh[0][2 * kt + 1], qh[1][2 * kt + 1], c0, c1);
      }
      mma_tf32(sacc[nt], qh[0][2 * kt], qh[1][2 * kt], qh[0][2 * kt + 1], qh[1][2 * kt + 1], b0, b1);
    }
  }

  // bias, mask of the pad keys, softmax over the row (16 keys per thread and row, the quad holds the row)
  const int ti0 = i0 - g.R, ai0 = ti0 / g.win, bi0 = ti0 - ai0 * g.win;
  const int ti1 = i1 - g.R, ai1 = ti1 / g.win, bi1 = ti1 - ai1 * g.win;
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int j = 8 * nt + 2 * t4 + e;
      const int kj = skey[j];
      const int aj = kj >> 8, bj = kj & 255;
      const int x0 = (ti0 < 0 || kj < 0 || i0 >= S) ? nb - 1 : (ai0 - aj + g.win - 1) * W2 + (bi0 - bj + g.win - 1);
      const int x1 = (ti1 < 0 || kj < 0 || i1 >= S) ? nb - 1 : (ai1 - aj + g.win - 1) * W2 + (bi1 - bj + g.win - 1);
      sacc[nt][e] = j < S ? sacc[nt][e] + sbias[x0] : -INFINITY;
      sacc[nt][2 + e] = j < S ? sacc[nt][2 + e] + sbias[x1] : -INFINITY;
      m0 = fmaxf(m0, sacc[nt][e]); m1 = fmaxf(m1, sacc[nt][2 + e]);
    }
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      sacc[nt][e] = __expf(sacc[nt][e] - m0); l0 += sacc[nt][e];
      sacc[nt][2 + e] = __expf(sacc[nt][2 + e] - m1); l1 += sacc[nt][2 + e];
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float il0 = 1.0f / l0, il1 = 1.0f / l1;

  // P (normalised) as the A operand: key tile ks, fragment columns (t, t+4) = keys (8ks + 2t, 8ks + 2t + 1)
  uint32_t ph[8][4], pl[SPLIT ? 8 : 1][4];
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const float p0 = sacc[ks][0] * il0, p1 = sacc[ks][2] * il1, p2 = sacc[ks][1] * il0, p3 = sacc[ks][3] * il1;
    ph[ks][0] = tf32_hi(p0); ph[ks][1] = tf32_hi(p1); ph[ks][2] = tf32_hi(p2); ph[ks][3] = tf32_hi(p3);
    if (SPLIT) { pl[ks][0] = tf32_lo(p0, ph[ks][0]); pl[ks][1] = tf32_lo(p1, ph[ks][1]); pl[ks][2] = tf32_lo(p2, ph[ks][2]); pl[ks][3] = tf32_lo(p3, ph[ks][3]); }
  }
  // out_split (fp32): the row is written as the left operand of a 3xTF32 GEMM, [hi | hi | lo] (vg_split3_tf32 pattern 0), 3 * inner long
  const int ldo = out_split ? 3 * inner : inner;
  T* op0 = out + (wdx * S + i0) * ldo + hd * DH + 2 * t4;
  T* op1 = out + (wdx * S + i1) * ldo + hd * DH + 2 * t4;
  float oacc[KT][4];
#pragma unroll
  for (int nd = 0; nd < KT; ++nd) oacc[nd][0] = oacc[nd][1] = oacc[nd][2] = oacc[nd][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
#pragma unroll
    for (int nd = 0; nd < KT; ++nd) {
      const float* vr = sv + (8 * ks + 2 * t4) * LD + 8 * nd + gq;
      const float v0 = vr[0], v1 = vr[LD];
      const uint32_t b0 = tf32_hi(v0), b1 = tf32_hi(v1);
      if (SPLIT) {
        const uint32_t c0 = tf32_lo(v0, b0), c1 = tf32_lo(v1, b1);
        mma_tf32(oacc[nd], pl[ks][0], pl[ks][1], pl[ks][2], pl[ks][3], b0, b1);
        mma_tf32(oacc[nd], ph[ks][0], ph[ks][1], ph[ks][2], ph[ks][3], c0, c1);
      }
      mma_tf32(oacc[nd], ph[ks][0], ph[ks][1], ph[ks][2], ph[ks][3], b0, b1);
    }
  }
#pragma unroll
  for (int nd = 0; nd < KT; ++nd) {
    const float* o = oacc[nd];
    if constexpr (sizeof(T) == 4) {
      if (out_split) {
        float h[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) h[e] = __uint_as_float(__float_as_uint(o[e]) & 0xffffe000u);
        if (i0 < S) {
          *reinterpret_cast<float2*>(op0 + 8 * nd) = make_float2(h[0], h[1]);
          *reinterpret_cast<float2*>(op0 + inner + 8 * nd) = make_float2(h[0], h[1]);
          *reinterpret_cast<float2*>(op0 + 2 * inner + 8 * nd) = make_float2(o[0] - h[0], o[1] - h[1]);
        }
        if (i1 < S) {
          *reinterpret_cast<float2*>(op1 + 8 * nd) = make_float2(h[2], h[3]);
          *reinterpret_cast<float2*>(op1 + inner + 8 * nd) = make_float2(h[2], h[3]);
          *reinterpret_cast<float2*>(op1 + 2 * inner + 8 * nd) = make_float2(o[2] - h[2], o[3] - h[3]);
        }
      } else {
        if (i0 < S) *reinterpret_cast<float2*>(op0 + 8 * nd) = make_float2(o[0], o[1]);
        if (i1 < S) *reinterpret_cast<float2*>(op1 + 8 * nd) = make_float2(o[2], o[3]);
      }
    } else {
      if (i0 < S) *reinterpret_cast<__nv_bfloat162*>(op0 + 8 * nd) = __floats2bfloat162_rn(o[0], o[1]);
      if (i1 < S) *reinterpret_cast<__nv_bfloat162*>(op1 + 8 * nd) = __floats2bfloat162_rn(o[2], o[3]);
    }
  }
}

// out_bf16: fp32 residual stream in, bf16 tokens out (the mixed-precision training backward re-materialises tokens in 16 bits)
int attn_gather_run(int dtype, const void* x, const float* reg, int reg_per_field, const float* film, const AttnGeom& g,
                    float eps, void* tokens, int out_bf16, cudaStream_t st) {
  if (g.C % 128 || g.C > 512) return set_error("attn_gather: C=%d must be a multiple of 128 (<=512)", g.C);
  const long long rows = (long long)g.N * g.nwin() * g.S();
  const unsigned grid = (unsigned)((rows + 7) / 8);
  if (dtype == 0) attn_gather_kernel<bf16, bf16><<<grid, 256, 0, st>>>(reinterpret_cast<const bf16*>(x), reg, reg_per_field, film, g, eps, reinterpret_cast<bf16*>(tokens), rows);
  else if (out_bf16) attn_gather_kernel<float, bf16><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), reg, reg_per_field, film, g, eps, reinterpret_cast<bf16*>(tokens), rows);
  else attn_gather_kernel<float, float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), reg, reg_per_field, film, g, eps, reinterpret_cast<float*>(tokens), rows);
  return check_launch("attn_gather_kernel");
}

int attn_partition_debug_run(const AttnGeom& g, long long* out, cudaStream_t st) {
  const long long rows = (long long)g.N * g.nwin() * g.S();
  attn_partition_debug_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(g, out, rows);
  return check_launch("attn_partition_debug_kernel");
}

template <typename T, int DH>
static int core_launch(const void* qkv, const float* qg, const float* kg, const float* bt, const AttnGeom& g, int heads, void* out, const DropCfg& drop, cudaStream_t st) {
  const int S = g.S(), Sp = (S + 3) & ~3, nb = (2 * g.win - 1) * (2 * g.win - 1) + 1;
  const size_t smem = (size_t)(2 * Sp * DH + nb) * sizeof(float);
  static PerDeviceSize attr_pd;                             // the size depends on the window geometry: raise the limit when it grows
  size_t& attr_bytes = attr_pd.cur();
  if (smem > attr_bytes) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_core_kernel<T, DH>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return set_error("attn_core smem attr: %s", cudaGetErrorString(e));
    attr_bytes = smem;
  }
  const long long pairs = (long long)g.N * g.nwin() * heads;
  attn_core_kernel<T, DH><<<(unsigned)pairs, 32 * ((S + 31) / 32), smem, st>>>(reinterpret_cast<const T*>(qkv), qg, kg, bt, g, heads, reinterpret_cast<T*>(out), drop);
  return check_launch("attn_core_kernel");
}

template <typename T, int DH, bool SPLIT>
static int core_mma_launch(const void* qkv, const float* qg, const float* kg, const float* bt, const AttnGeom& g, int heads, void* out, int out_split, cudaStream_t st) {
  const int nb = (2 * g.win - 1) * (2 * g.win - 1) + 1;
  const size_t smem = (size_t)(2 * 64 * (DH + 4) + ((nb + 3) & ~3) + 64) * sizeof(float);
  static PerDeviceSize attr_pd;
  size_t& attr_bytes = attr_pd.cur();
  if (smem > attr_bytes) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_mma_kernel<T, DH, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_core_mma_kernel<T, DH, SPLIT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return set_error("attn_core (mma) smem attr: %s", cudaGetErrorString(e));
    attr_bytes = smem;
  }
  const long long pairs = (long long)g.N * g.nwin() * heads;
  attn_core_mma_kernel<T, DH, SPLIT><<<(unsigned)pairs, 128, smem, st>>>(reinterpret_cast<const T*>(qkv), qg, kg, bt, g, heads, reinterpret_cast<T*>(out), out_split);
  return check_launch("attn_core_mma_kernel");
}

int attn_core_run(int dtype, const void* qkv, const float* qgamma, const float* kgamma, const float* bias_table,
                  const AttnGeom& g, int heads, int dh, void* out, unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st) {
  if (g.S() > 128) return set_error("attn_core: sequence %d too long", g.S());
  if (dtype != 0 && dtype != 1 && dtype != 2 && dtype != 4 && dtype != 6) return set_error("attn_core: dtype code %d (0 bf16, 1 fp32, 2 / 6 fp32 3xTF32, 4 fp32 tf32)", dtype);
  if (drop_thresh < 0 || drop_thresh > 255) return set_error("attn_core: dropout threshold %d outside [0, 255]", drop_thresh);
  if (drop_thresh && g.S() > 64 && heads > DROP_MAX_HEADS_LONG)
    return set_error("attn_core: dropout with %d heads at sequence %d > 64 (at most %d heads)", heads, g.S(), DROP_MAX_HEADS_LONG);
  DropCfg drop;
  drop.seed = seed; drop.salt = salt; drop.thresh = drop_thresh; drop.scale = 256.0f / (256.0f - (float)drop_thresh);
  // dtype 2 = fp32 storage with 3xTF32 tensor-core products (the 'tf32_conv' precision of wide networks); dtype 4 = fp32 storage and
  // bf16 storage (0) take single tf32 products (the mixed-precision modes).  Shapes outside the mma kernel (S > 64, attention dropout) and exact fp32 (dtype 1) run the SIMT kernel.
  const int out_split = dtype == 6;                        // dtype 6 = 2 with the output rows as the split operand [hi | hi | lo]
  if (out_split) dtype = 2;
  if (out_split && (drop_thresh || g.S() > 64 || (dh != 32 && dh != 64))) return set_error("attn_core: the split output (dtype 6) needs the tensor-core kernel (S <= 64, dim_head 32 / 64, no dropout)");
  if (dtype != 1 && drop_thresh == 0 && g.S() <= 64 && g.win <= 64) {
    if (dh == 64) return dtype == 0 ? core_mma_launch<bf16, 64, false>(qkv, qgamma, kgamma, bias_table, g, heads, out, 0, st)
                       : dtype == 4 ? core_mma_launch<float, 64, false>(qkv, qgamma, kgamma, bias_table, g, heads, out, out_split, st)
                                    : core_mma_launch<float, 64, true>(qkv, qgamma, kgamma, bias_table, g, heads, out, out_split, st);
    if (dh == 32) return dtype == 0 ? core_mma_launch<bf16, 32, false>(qkv, qgamma, kgamma, bias_table, g, heads, out, 0, st)
                       : dtype == 4 ? core_mma_launch<float, 32, false>(qkv, qgamma, kgamma, bias_table, g, heads, out, out_split, st)
                                    : core_mma_launch<float, 32, true>(qkv, qgamma, kgamma, bias_table, g, heads, out, out_split, st);
  }
  if (dtype == 2 || dtype == 4) dtype = 1;
  if (dh == 32) return dtype == 0 ? core_launch<bf16, 32>(qkv, qgamma, kgamma, bias_table, g, heads, out, drop, st)
                                  : core_launch<float, 32>(qkv, qgamma, kgamma, bias_table, g, heads, out, drop, st);
  if (dh == 64) return dtype == 0 ? core_launch<bf16, 64>(qkv, qgamma, kgamma, bias_table, g, heads, out, drop, st)
                                  : core_launch<float, 64>(qkv, qgamma, kgamma, bias_table, g, heads, out, drop, st);
  return set_error("attn_core: dim_head %d not supported (32 or 64)", dh);
}

}  // namespace vg
