// Backward kernels of the MetNet3 encoder / decoder (training step): everything around the dgrad / wgrad GEMMs is
// bandwidth-bound row-wise work on the padded-grid (PG) layout -- ChanLayerNorm + FiLM + ReLU backward with the
// parameter-gradient reductions fused in, head / max-pool / ConvTranspose gathers, the lead-time reduction of the
// de-duplicated stem, the analytic time-channel gradients, the conditioning MLPs and the embeddings.
//
// The reference has no hand-written backward (autograd of metnet3.py:86-430); each kernel names the forward lines it
// differentiates.  Gradients travel as fp32 [q][128] tensors; GEMM operands are written in the GEMM dtype.
#include "vg_common.cuh"
#include "vg_host.h"

namespace vg {

static inline unsigned nblk(long long total, int per) { return (unsigned)((total + per - 1) / per); }

// ================================================================================================
// Block backward (metnet3.py:110-126, 94-104):  y = ReLU((xhat*g + b) * (s+1) + sh),  xhat = (conv - mean) * rstd
//   dZ = dY * mask;  dxhat = dZ * g * (s+1);  dconv = rstd * (dxhat - mean_c(dxhat) - xhat * mean_c(dxhat*xhat))
//   per field n: sumA[n][c] += dZ*xhat, sumB[n][c] += dZ, sumD[n][c] += dconv  (parameter / FiLM / bias gradients)
// One warp per pixel (lane = 4 channels), 64 consecutive pixels per warp, 512 per block.
// ================================================================================================
struct ConvLnBwdParams {
  const float* dY;
  const void* xhat;
  const float* rstd;
  const unsigned* mask;
  const float* ln_g;
  const float* film;        // (N, 256) or null
  void* dconv;
  float* sumA; float* sumB; float* sumD;   // (N, 128) each, accumulated with atomics (zeroed by the caller)
  float* border;            // optional (N, 8, 128): sums of dconv over row 0, last row, col 0, last col, 4 corners
  float rstd_clamp;         // rsqrt(eps): rows whose variance was clamped have no variance gradient
  PGeom pg;
  float* slots;             // DET: (3, N, K, C) per-(field, warp) partials of sumA / sumB / sumD (zeroed by the launcher)
  int K;                    // DET: slots per field
};

// Fixed-order slot indices of the deterministic (DET) instantiations: the warps w that touch field n (whose PG rows are the
// pixels [n*R*P, (n+1)*R*P)) are numbered j = w - first warp of n, so a field has at most ceil(R*P / PPW) + 1 of them.
__host__ __device__ inline int det_field_slots(const PGeom& pg, int ppw) { return (int)(((long long)pg.R * pg.P + ppw - 1) / ppw) + 1; }
__device__ __forceinline__ int det_field_slot(const PGeom& pg, int ppw, long long warp_global, int n) {
  return (int)(warp_global - ((long long)n * pg.R * pg.P) / ppw);
}

// Half a warp per pixel (lane = 8 channels).  The kernel is a stream of ~1 KB rows with two 16-lane reductions each; what bounds it
// is how many bytes a warp keeps in flight.  Every warp owns a three-stage ring in shared memory; one lane fills a stage with
// the rows of four consecutive pixels (dY 2 KB + xhat 1 KB + mask + rstd: four bulk copies, cp.async.bulk -> mbarrier) two
// iterations ahead of the arithmetic, so ~6 KB per warp are always on their way from HBM without costing registers
// (loads issued from registers one iteration at a time reached 3.4 TB/s).
namespace lnb {
constexpr int C = 128, PPW = 64, G = 4, NST = 3;
template <typename T> __host__ __device__ constexpr int stage_bytes() { return ((G * C * 4 + G * C * (int)sizeof(T) + G * 16 + G * 4) + 127) / 128 * 128; }
}  // namespace lnb

__device__ __forceinline__ void bulk_g2s_b(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// DET: no atomics -- each half-warp stores its partial sums of a field into slot (n, 2 * warp-of-field + half) and the launcher
// reduces the slots in a fixed order; the border sums are left to border_sum_kernel (fp32 dconv).
template <typename T, typename TO, bool DET = false>
__global__ void __launch_bounds__(256) conv_ln_bwd_kernel(const ConvLnBwdParams p) {
  using namespace lnb;
  constexpr int XB = C * (int)sizeof(T), SB = stage_bytes<T>();
  extern __shared__ __align__(128) uint8_t ring_raw[];
  __shared__ float sacc[3][C];
  __shared__ uint64_t bars[8][NST];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, hl = lane & 15, sub = lane >> 4, c0 = hl * 8;
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ring_raw) + 127) & ~uintptr_t(127)) + (size_t)warp * NST * SB;
  const long long q_block = (long long)blockIdx.x * (8 * PPW);
  for (int i = threadIdx.x; i < 3 * C; i += 256) (&sacc[0][0])[i] = 0.f;
  if (lane == 0) { for (int s = 0; s < NST; ++s) mbar_init(&bars[warp][s], 1); fence_mbar_init(); }
  int nf0, hh, ww;
  p.pg.decode(q_block, nf0, hh, ww);
  if (nf0 >= p.pg.N) nf0 = p.pg.N - 1;
  __syncthreads();
  const T* xh = reinterpret_cast<const T*>(p.xhat);
  TO* dc = reinterpret_cast<TO*>(p.dconv);
  float A[8], B[8], D[8], gs[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) A[i] = B[i] = D[i] = gs[i] = 0.f;
  int n_cur = -1;
  auto flush = [&]() {
    if (n_cur < 0) return;
    if constexpr (DET) {
      const int j = det_field_slot(p.pg, PPW, q_block / PPW + warp, n_cur);
      const long long plane = (long long)p.pg.N * p.K * C;
      float* s = p.slots + ((long long)n_cur * p.K + 2 * j + sub) * C + c0;
      st8(s, A); st8(s + plane, B); st8(s + 2 * plane, D);
#pragma unroll
      for (int i = 0; i < 8; ++i) A[i] = B[i] = D[i] = 0.f;
      return;
    }
    float* dA = n_cur == nf0 ? &sacc[0][c0] : p.sumA + (long long)n_cur * C + c0;
    float* dB = n_cur == nf0 ? &sacc[1][c0] : p.sumB + (long long)n_cur * C + c0;
    float* dD = n_cur == nf0 ? &sacc[2][c0] : p.sumD + (long long)n_cur * C + c0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { atomicAdd(dA + i, A[i]); atomicAdd(dB + i, B[i]); atomicAdd(dD + i, D[i]); A[i] = B[i] = D[i] = 0.f; }
  };
  const long long q0 = q_block + warp * PPW;
  const long long npix = p.pg.pixels();
  auto issue = [&](int it) {                               // lane 0: the rows of pixels q0 + it*G .. +G-1 -> stage it % NST
    const long long q = q0 + (long long)it * G;
    if (it >= PPW / G || npix - q < G) return;             // (the last, partial group of the tensor is read straight from global memory:
    const uint32_t rows = G;                               //  bulk copies move multiples of 16 bytes, 4 bytes of rstd per pixel)
    uint8_t* st = ring + (it % NST) * SB;
    uint64_t* bar = &bars[warp][it % NST];
    mbar_arrive_expect_tx(bar, rows * (C * 4 + XB + 16 + 4));
    bulk_g2s_b(st, p.dY + q * C, rows * C * 4, bar);
    bulk_g2s_b(st + G * C * 4, xh + q * C, rows * XB, bar);
    bulk_g2s_b(st + G * C * 4 + G * XB, p.mask + q * 4, rows * 16, bar);
    bulk_g2s_b(st + G * C * 4 + G * XB + G * 16, p.rstd + q, rows * 4, bar);
  };
  if (lane == 0) { issue(0); issue(1); }
  // This half-warp visits pixels q0 + sub, +2, +4, ...: its PG coordinates advance incrementally (the two 32-bit divisions of a
  // decode per pixel were a third of the kernel's instructions, which ncu showed to be what bounds it: 61 % issue utilisation)
  long long q = q0 + sub;
  int col, rr_, n;
  {
    const long long row = q / p.pg.P;
    col = (int)(q - row * p.pg.P);
    n = (int)(row / p.pg.R);
    rr_ = (int)(row - (long long)n * p.pg.R);
  }
  TO* dcp = dc + q * C + c0;
  const int Pp = p.pg.P, Rr = p.pg.R, Nn = p.pg.N, HPm = p.pg.HP - 1, WPm = p.pg.WP - 1;
  for (int it = 0; it < PPW / G; ++it) {
    const long long qb = q0 + (long long)it * G;
    if (qb >= npix) break;
    __syncwarp();                                          // every lane is done with the stage that iteration it+2 refills
    if (lane == 0) issue(it + 2);
    const bool full = npix - qb >= G;
    uint8_t* st = ring + (it % NST) * SB;
    if (full) mbar_wait(&bars[warp][it % NST], (uint32_t)((it / NST) & 1));
#pragma unroll
    for (int u = 0; u < G / 2; ++u) {
      const int pi = 2 * u + sub;                          // pixel of this half-warp inside the group of four
      const bool inr = q < npix;
      const bool valid = inr && col >= 1 && rr_ >= 1 && n < Nn;
      const int h = rr_ - 1, w = col - 1;
      float dy[8], x[8], rstd = 0.f; unsigned bits = 0u;
#pragma unroll
      for (int i = 0; i < 8; ++i) dy[i] = x[i] = 0.f;
      if (valid) {
        if (full) {
          ld8(reinterpret_cast<const float*>(st) + pi * C + c0, dy);
          ld8(reinterpret_cast<const T*>(st + G * C * 4) + pi * C + c0, x);
          bits = reinterpret_cast<const unsigned*>(st + G * C * 4 + G * XB)[pi * 4 + (hl >> 2)] >> ((hl & 3) * 8);
          rstd = reinterpret_cast<const float*>(st + G * C * 4 + G * XB + G * 16)[pi];
        } else {                                           // the last, partial group of the tensor: straight from global memory
          ld8(p.dY + q * C + c0, dy);
          ld8(xh + q * C + c0, x);
          bits = p.mask[q * 4 + (hl >> 2)] >> ((hl & 3) * 8);
          rstd = p.rstd[q];
        }
      }
      if (valid && n != n_cur) {
        flush();
        n_cur = n;
#pragma unroll
        for (int i = 0; i < 8; ++i) gs[i] = p.ln_g[c0 + i] * (p.film ? p.film[(long long)n_cur * 2 * C + c0 + i] + 1.0f : 1.0f);
      }
      float dx[8], o[8], s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float dz = (bits & (1u << i)) ? dy[i] : 0.f;
        dx[i] = dz * gs[i]; s1 += dx[i]; s2 = fmaf(dx[i], x[i], s2);
        A[i] = fmaf(dz, x[i], A[i]); B[i] += dz;
      }
#pragma unroll
      for (int o2 = 8; o2 >= 1; o2 >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o2); s2 += __shfl_xor_sync(0xffffffffu, s2, o2); }
      s1 *= (1.0f / C);
      s2 = rstd >= p.rstd_clamp ? 0.f : s2 * (1.0f / C);           // var.clamp(min=eps): no gradient through a clamped variance
      const float rv = valid ? rstd : 0.f;                         // pad positions: zeros
#pragma unroll
      for (int i = 0; i < 8; ++i) { o[i] = rv * (dx[i] - s1 - x[i] * s2); D[i] += o[i]; }
      if (!DET && p.border && valid) {
        const bool r0 = h == 0, rl = h == HPm, k0 = w == 0, kl = w == WPm;
        if (r0 | rl | k0 | kl) {
          float* bb = p.border + (long long)n * 8 * C + c0;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (r0) atomicAdd(bb + 0 * C + i, o[i]);
            if (rl) atomicAdd(bb + 1 * C + i, o[i]);
            if (k0) atomicAdd(bb + 2 * C + i, o[i]);
            if (kl) atomicAdd(bb + 3 * C + i, o[i]);
            if (r0 && k0) atomicAdd(bb + 4 * C + i, o[i]);
            if (r0 && kl) atomicAdd(bb + 5 * C + i, o[i]);
            if (rl && k0) atomicAdd(bb + 6 * C + i, o[i]);
            if (rl && kl) atomicAdd(bb + 7 * C + i, o[i]);
          }
        }
      }
      if (inr) st8(dcp, o);
      // next pixel of this half-warp: q + 2
      q += 2; dcp += 2 * C; col += 2;
      if (col >= Pp) { col -= Pp; if (++rr_ == Rr) { rr_ = 0; ++n; } }
    }
  }
  flush();
  if constexpr (DET) return;
  __syncthreads();
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    if (sacc[0][c] != 0.f) atomicAdd(p.sumA + (long long)nf0 * C + c, sacc[0][c]);
    if (sacc[1][c] != 0.f) atomicAdd(p.sumB + (long long)nf0 * C + c, sacc[1][c]);
    if (sacc[2][c] != 0.f) atomicAdd(p.sumD + (long long)nf0 * C + c, sacc[2][c]);
  }
}

// Block backward at C = 128 * NV (n_start_channels 256 / 384 / 512; tf32_conv training): the math of conv_ln_bwd_kernel on fp32
// xhat / dconv.  One warp per pixel (lane owns channels v*128 + lane*4 .. +3, v < NV; ReLU mask word v*4 + lane/8 of the C/32
// words of a pixel), 32 consecutive pixels per warp, 256 per block.  The per-field sums of the block's first field collect in
// shared memory (most pixels of a block), the sums of any other field go to global atomics when the warp leaves the field.
// DET: as conv_ln_bwd_kernel, one slot per (field, warp-of-field)
template <int NV, bool DET = false>
__global__ void __launch_bounds__(256) conv_ln_bwd_wide_kernel(const ConvLnBwdParams p) {
  constexpr int C = 128 * NV, PPW = 32, MW = C / 32;
  __shared__ float sacc[3][C];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  const long long q_block = (long long)blockIdx.x * (8 * PPW);
  for (int i = threadIdx.x; i < 3 * C; i += 256) (&sacc[0][0])[i] = 0.f;
  int nf0, hh, ww;
  p.pg.decode(q_block, nf0, hh, ww);
  if (nf0 >= p.pg.N) nf0 = p.pg.N - 1;
  __syncthreads();
  const float* xh = reinterpret_cast<const float*>(p.xhat);
  float* dc = reinterpret_cast<float*>(p.dconv);
  float A[NV][4], B[NV][4], D[NV][4], gs[NV][4];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int i = 0; i < 4; ++i) A[v][i] = B[v][i] = D[v][i] = gs[v][i] = 0.f;
  int n_cur = -1;
  auto flush = [&]() {
    if (n_cur < 0) return;
    if constexpr (DET) {
      const int j = det_field_slot(p.pg, PPW, q_block / PPW + warp, n_cur);
      const long long plane = (long long)p.pg.N * p.K * C;
      float* s = p.slots + ((long long)n_cur * p.K + j) * C + c0;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        *reinterpret_cast<float4*>(s + v * 128) = make_float4(A[v][0], A[v][1], A[v][2], A[v][3]);
        *reinterpret_cast<float4*>(s + plane + v * 128) = make_float4(B[v][0], B[v][1], B[v][2], B[v][3]);
        *reinterpret_cast<float4*>(s + 2 * plane + v * 128) = make_float4(D[v][0], D[v][1], D[v][2], D[v][3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) A[v][i] = B[v][i] = D[v][i] = 0.f;
      }
      return;
    }
    const bool loc = n_cur == nf0;
#pragma unroll
    for (int v = 0; v < NV; ++v)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = v * 128 + c0 + i;
        const long long g = (long long)n_cur * C + c;
        atomicAdd(loc ? &sacc[0][c] : p.sumA + g, A[v][i]);
        atomicAdd(loc ? &sacc[1][c] : p.sumB + g, B[v][i]);
        atomicAdd(loc ? &sacc[2][c] : p.sumD + g, D[v][i]);
        A[v][i] = B[v][i] = D[v][i] = 0.f;
      }
  };
  const long long npix = p.pg.pixels();
  long long q = q_block + warp * PPW;
  const int Pp = p.pg.P, Rr = p.pg.R, Nn = p.pg.N, HPm = p.pg.HP - 1, WPm = p.pg.WP - 1;
  int col, rr_, n;
  {
    const long long row = q / Pp;
    col = (int)(q - row * Pp);
    n = (int)(row / Rr);
    rr_ = (int)(row - (long long)n * Rr);
  }
  for (int k = 0; k < PPW && q < npix; ++k) {
    const bool valid = col >= 1 && rr_ >= 1 && n < Nn;          // warp-uniform: the whole warp works on pixel q
    float o[NV][4];
#pragma unroll
    for (int v = 0; v < NV; ++v) o[v][0] = o[v][1] = o[v][2] = o[v][3] = 0.f;
    if (valid) {
      float dy[NV][4], x[NV][4];
      unsigned bits[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const float4 a = *reinterpret_cast<const float4*>(p.dY + q * C + v * 128 + c0);
        const float4 b = *reinterpret_cast<const float4*>(xh + q * C + v * 128 + c0);
        dy[v][0] = a.x; dy[v][1] = a.y; dy[v][2] = a.z; dy[v][3] = a.w;
        x[v][0] = b.x; x[v][1] = b.y; x[v][2] = b.z; x[v][3] = b.w;
        bits[v] = p.mask[q * MW + v * 4 + (lane >> 3)] >> ((lane & 7) * 4);
      }
      const float rstd = p.rstd[q];
      if (n != n_cur) {
        flush();
        n_cur = n;
#pragma unroll
        for (int v = 0; v < NV; ++v)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int c = v * 128 + c0 + i;
            gs[v][i] = p.ln_g[c] * (p.film ? p.film[(long long)n * 2 * C + c] + 1.0f : 1.0f);
          }
      }
      float dx[NV][4], s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int v = 0; v < NV; ++v)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float dz = (bits[v] & (1u << i)) ? dy[v][i] : 0.f;
          dx[v][i] = dz * gs[v][i]; s1 += dx[v][i]; s2 = fmaf(dx[v][i], x[v][i], s2);
          A[v][i] = fmaf(dz, x[v][i], A[v][i]); B[v][i] += dz;
        }
      s1 = warp_sum(s1) * (1.0f / C);
      s2 = warp_sum(s2);
      s2 = rstd >= p.rstd_clamp ? 0.f : s2 * (1.0f / C);          // var.clamp(min=eps): no gradient through a clamped variance
#pragma unroll
      for (int v = 0; v < NV; ++v)
#pragma unroll
        for (int i = 0; i < 4; ++i) { o[v][i] = rstd * (dx[v][i] - s1 - x[v][i] * s2); D[v][i] += o[v][i]; }
      if (!DET && p.border) {
        const int h = rr_ - 1, w = col - 1;
        const bool r0 = h == 0, rl = h == HPm, k0 = w == 0, kl = w == WPm;
        if (r0 | rl | k0 | kl) {
          float* bb = p.border + (long long)n * 8 * C + c0;
#pragma unroll
          for (int v = 0; v < NV; ++v)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float* b1 = bb + v * 128 + i;
              if (r0) atomicAdd(b1 + 0 * C, o[v][i]);
              if (rl) atomicAdd(b1 + 1 * C, o[v][i]);
              if (k0) atomicAdd(b1 + 2 * C, o[v][i]);
              if (kl) atomicAdd(b1 + 3 * C, o[v][i]);
              if (r0 && k0) atomicAdd(b1 + 4 * C, o[v][i]);
              if (r0 && kl) atomicAdd(b1 + 5 * C, o[v][i]);
              if (rl && k0) atomicAdd(b1 + 6 * C, o[v][i]);
              if (rl && kl) atomicAdd(b1 + 7 * C, o[v][i]);
            }
        }
      }
    }
#pragma unroll
    for (int v = 0; v < NV; ++v)
      *reinterpret_cast<float4*>(dc + q * C + v * 128 + c0) = make_float4(o[v][0], o[v][1], o[v][2], o[v][3]);
    ++q;
    if (++col == Pp) { col = 0; if (++rr_ == Rr) { rr_ = 0; ++n; } }
  }
  flush();
  if constexpr (DET) return;
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {
    if (sacc[0][c] != 0.f) atomicAdd(p.sumA + (long long)nf0 * C + c, sacc[0][c]);
    if (sacc[1][c] != 0.f) atomicAdd(p.sumB + (long long)nf0 * C + c, sacc[1][c]);
    if (sacc[2][c] != 0.f) atomicAdd(p.sumD + (long long)nf0 * C + c, sacc[2][c]);
  }
}

// parameter gradients of one Block from the per-field sums (one thread per channel; C / 32 blocks):
//   dg += sum_n A (s+1);  db += sum_n B (s+1);  dbias += sum_n D;  dfilm[n] = (A g + B b | B)
template <int C>
__global__ void __launch_bounds__(256) conv_ln_param_grads_kernel(const float* __restrict__ sumA, const float* __restrict__ sumB, const float* __restrict__ sumD,
                                           int N, const float* __restrict__ g, const float* __restrict__ b, const float* __restrict__ film,
                                           float* __restrict__ dg, float* __restrict__ db, float* __restrict__ dbias, float* __restrict__ dfilm) {
  __shared__ float red[3][8][32];
  const int l = threadIdx.x & 31, slice = threadIdx.x >> 5, c = blockIdx.x * 32 + l;     // 32 channels x 8 slices of the fields
  float ag = 0.f, ab = 0.f, ad = 0.f;
  for (int n = slice; n < N; n += 8) {
    const float A = sumA[n * C + c], B = sumB[n * C + c];
    const float s1 = film ? film[(long long)n * 2 * C + c] + 1.0f : 1.0f;
    ag += A * s1; ab += B * s1; ad += sumD[n * C + c];
    if (dfilm) { dfilm[(long long)n * 2 * C + c] = A * g[c] + B * b[c]; dfilm[(long long)n * 2 * C + C + c] = B; }
  }
  red[0][slice][l] = ag; red[1][slice][l] = ab; red[2][slice][l] = ad;
  __syncthreads();
  if (slice == 0) {
    ag = ab = ad = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) { ag += red[0][k][l]; ab += red[1][k][l]; ad += red[2][k][l]; }
    dg[c] += ag; db[c] += ab; dbias[c] += ad;
  }
}

// ================================================================================================
// head backward (metnet3.py:424-430): pred = (sum_c h*w + b)*std + mean on the un-padded window
//   dH[q][c] = dpred*std*w[c] inside the window, 0 elsewhere (incl. pads);  dw[c] += dpred*std*h;  db += dpred*std
// C = 128 * NV: lane owns channels v*128 + lane*4 .. +3 (v < NV)
// ================================================================================================
// DET: each warp stores (dw, db) partials into slot (block * 8 + warp) of dw ([slots][C + 1]); db is unused
template <int C, typename T, bool DET = false>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ dpred, const T* __restrict__ h, const float* __restrict__ w,
                                                       float stdv, PGeom pg, int H, int W, int pt, int pl, float* __restrict__ dH,
                                                       float* __restrict__ dw, float* __restrict__ db) {
  constexpr int PPW = 32, NV = C / 128;
  __shared__ float sw_[C + 1];
  for (int i = threadIdx.x; i < C + 1; i += 256) sw_[i] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  float4 w4[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) w4[v] = *reinterpret_cast<const float4*>(w + v * 128 + c0);
  float aw[NV][4] = {}, ab = 0.f;
  const long long q0 = ((long long)blockIdx.x * 8 + warp) * PPW;
#pragma unroll 1
  for (int k = 0; k < PPW; ++k) {
    const long long q = q0 + k;
    if (q >= pg.pixels()) break;
    int n, y, x;
    float4 o[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) o[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (pg.decode(q, n, y, x)) {
      const int hh = y - pt, ww = x - pl;
      if (hh >= 0 && hh < H && ww >= 0 && ww < W) {
        const float d = dpred[((long long)n * H + hh) * W + ww] * stdv;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          o[v] = make_float4(d * w4[v].x, d * w4[v].y, d * w4[v].z, d * w4[v].w);
#pragma unroll
          for (int i = 0; i < 4; ++i) aw[v][i] += d * Act<T>::ld(h + q * C + v * 128 + c0 + i);
        }
        ab += d;
      }
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) *reinterpret_cast<float4*>(dH + q * C + v * 128 + c0) = o[v];
  }
  if constexpr (DET) {
    float* s = dw + ((long long)blockIdx.x * 8 + warp) * (C + 1);
#pragma unroll
    for (int v = 0; v < NV; ++v)
#pragma unroll
      for (int i = 0; i < 4; ++i) s[v * 128 + c0 + i] = aw[v][i];
    if (lane == 0) s[C] = ab;
  } else {
#pragma unroll
    for (int v = 0; v < NV; ++v)
#pragma unroll
      for (int i = 0; i < 4; ++i) atomicAdd(&sw_[v * 128 + c0 + i], aw[v][i]);
    if (lane == 0) atomicAdd(&sw_[C], ab);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < (C + 255) / 256; ++k)
      if (k * 256 + threadIdx.x < C) atomicAdd(dw + k * 256 + threadIdx.x, sw_[k * 256 + threadIdx.x]);
    if (threadIdx.x == C % 256) atomicAdd(db, sw_[C]);
  }
}

// ================================================================================================
// max-pool 2x2 backward (metnet3.py:86): the gradient goes to the FIRST maximum of each window in row-major order
// (PyTorch's rule).  x: PG (N,HP,WP,C); dlow: CL (N,HP/2,WP/2,C) fp32; dx: PG fp32, every position written.
// ================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) maxpool2_bwd_kernel(const T* __restrict__ x, const float* __restrict__ dlow, float* __restrict__ dx,
                                                           PGeom pg, int C) {
  const int cv = C / 8;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pg.pixels() * cv) return;
  const long long q = i / cv;
  const int c8 = (int)(i - q * cv) * 8;
  int n, h, w;
  float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (pg.decode(q, n, h, w)) {
    const int ho = h >> 1, wo = w >> 1, me = (h & 1) * 2 + (w & 1);
    float v[4][8];
#pragma unroll
    for (int k = 0; k < 4; ++k) ld8(x + pg.q(n, 2 * ho + (k >> 1), 2 * wo + (k & 1)) * C + c8, v[k]);
    float g[8];
    ld8(dlow + (((long long)n * (pg.HP / 2) + ho) * (pg.WP / 2) + wo) * C + c8, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int best = 0; float m = v[0][j];
#pragma unroll
      for (int k = 1; k < 4; ++k) if (v[k][j] > m) { m = v[k][j]; best = k; }
      o[j] = best == me ? g[j] : 0.f;
    }
  }
  st8(dx + q * C + c8, o);
}

// ================================================================================================
// ConvTranspose2d(k2,s2) backward gather (metnet3.py:88-89): dUp PG (N,2Hl,2Wl,C) fp32 -> G [N*Hl*Wl][4C] in the GEMM
// dtype, column (di*2+dj)*C + co (the forward GEMM's column order), plus dbias[co] += sum.  C = 128 * NV.
// ================================================================================================
// DET: each warp stores its dbias partial into slot (block * 8 + warp) of dbias ([slots][C])
template <int C, typename TO, bool DET = false>
__global__ void __launch_bounds__(256) convT_bwd_gather_kernel(const float* __restrict__ dUp, TO* __restrict__ G, float* __restrict__ dbias,
                                                               PGeom pg, int Hl, int Wl, long long M) {
  constexpr int PPW = 16, NV = C / 128;
  __shared__ float sb[C];
#pragma unroll
  for (int k = 0; k < (C + 255) / 256; ++k)
    if (k * 256 + threadIdx.x < C) sb[k * 256 + threadIdx.x] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  float acc[NV][4];
#pragma unroll
  for (int u = 0; u < NV; ++u) acc[u][0] = acc[u][1] = acc[u][2] = acc[u][3] = 0.f;
  const long long r0 = ((long long)blockIdx.x * 8 + warp) * PPW;
  for (int k = 0; k < PPW; ++k) {
    const long long r = r0 + k;
    if (r >= M) break;
    const int n = (int)(r / (Hl * Wl));
    const int pp = (int)(r - (long long)n * Hl * Wl);
    const int i = pp / Wl, j = pp - i * Wl;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
#pragma unroll
      for (int u = 0; u < NV; ++u) {
        const float4 v = *reinterpret_cast<const float4*>(dUp + pg.q(n, 2 * i + (t >> 1), 2 * j + (t & 1)) * C + u * 128 + c0);
        acc[u][0] += v.x; acc[u][1] += v.y; acc[u][2] += v.z; acc[u][3] += v.w;
        TO* d = G + r * 4 * C + t * C + u * 128 + c0;
        Act<TO>::st(d, v.x); Act<TO>::st(d + 1, v.y); Act<TO>::st(d + 2, v.z); Act<TO>::st(d + 3, v.w);
      }
    }
  }
  if constexpr (DET) {
#pragma unroll
    for (int u = 0; u < NV; ++u)
      *reinterpret_cast<float4*>(dbias + ((long long)blockIdx.x * 8 + warp) * C + u * 128 + c0) = make_float4(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
  } else {
#pragma unroll
    for (int u = 0; u < NV; ++u)
#pragma unroll
      for (int i = 0; i < 4; ++i) atomicAdd(&sb[u * 128 + c0 + i], acc[u][i]);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < (C + 255) / 256; ++k)
      if (k * 256 + threadIdx.x < C) atomicAdd(dbias + k * 256 + threadIdx.x, sb[k * 256 + threadIdx.x]);
  }
}

// ================================================================================================
// stem: sum over the L lead times of a per-field tensor -> per-sample tensor (GEMM dtype), pads written as zeros:
//   out[b][h][w][c] = sum_l in[b*L + l][h][w][c]        (the transpose of the lead-time replication, metnet3.py:383)
// ================================================================================================
template <int C, typename TI, typename TO>
__global__ void __launch_bounds__(256) lead_sum_kernel(const TI* __restrict__ in, TO* __restrict__ out, PGeom pgN, PGeom pgB, int L) {
  constexpr int NV = C / 128;
  const long long qb = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (qb >= pgB.pixels()) return;
  const int lane = threadIdx.x & 31, c0 = lane * 4;
  int b, h, w;
  float a[NV][4];
#pragma unroll
  for (int v = 0; v < NV; ++v) a[v][0] = a[v][1] = a[v][2] = a[v][3] = 0.f;
  if (pgB.decode(qb, b, h, w)) {
    for (int l = 0; l < L; ++l) {
      const TI* s = in + pgN.q(b * L + l, h, w) * C + c0;
#pragma unroll
      for (int v = 0; v < NV; ++v)
#pragma unroll
        for (int i = 0; i < 4; ++i) a[v][i] += Act<TI>::ld(s + v * 128 + i);
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int i = 0; i < 4; ++i) Act<TO>::st(out + qb * C + v * 128 + c0 + i, a[v][i]);
}

// per-field sums over the frame pixels of an fp32 PG tensor: out[n][c] = sum_{h,w} in[n][h][w][c].  grid (chunks, N); C = 128 * NV
// DET: each warp stores its partial into slot ((n * chunks + chunk) * 8 + warp) of out ([N][chunks * 8][C])
template <int C, bool DET = false>
__global__ void __launch_bounds__(256) pg_field_sum_kernel(const float* __restrict__ in, float* __restrict__ out, PGeom pg) {
  constexpr int NV = C / 128;
  __shared__ float sb[C];
#pragma unroll
  for (int k = 0; k < (C + 255) / 256; ++k)
    if (k * 256 + threadIdx.x < C) sb[k * 256 + threadIdx.x] = 0.f;
  __syncthreads();
  const int n = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  const int npix = pg.HP * pg.WP;
  float a[NV][4];
#pragma unroll
  for (int u = 0; u < NV; ++u) a[u][0] = a[u][1] = a[u][2] = a[u][3] = 0.f;
  for (int i = blockIdx.x * 8 + warp; i < npix; i += gridDim.x * 8) {
    const int h = i / pg.WP, w = i - h * pg.WP;
#pragma unroll
    for (int u = 0; u < NV; ++u) {
      const float4 v = *reinterpret_cast<const float4*>(in + pg.q(n, h, w) * C + u * 128 + c0);
      a[u][0] += v.x; a[u][1] += v.y; a[u][2] += v.z; a[u][3] += v.w;
    }
  }
  if constexpr (DET) {
#pragma unroll
    for (int u = 0; u < NV; ++u)
      *reinterpret_cast<float4*>(out + (((long long)n * gridDim.x + blockIdx.x) * 8 + warp) * C + u * 128 + c0) = make_float4(a[u][0], a[u][1], a[u][2], a[u][3]);
  } else {
#pragma unroll
    for (int u = 0; u < NV; ++u)
#pragma unroll
      for (int i = 0; i < 4; ++i) atomicAdd(&sb[u * 128 + c0 + i], a[u][i]);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < (C + 255) / 256; ++k)
      if (k * 256 + threadIdx.x < C) atomicAdd(out + (long long)n * C + k * 256 + threadIdx.x, sb[k * 256 + threadIdx.x]);
  }
}

// ================================================================================================
// time-channel gradients of the stem (transpose of time_terms_kernel): from the border-class sums of dconv
// (border (N,8,C) + total sumD (N,C)) and the per-field sums of the residual gradient (tres_sum (N,C)):
//   V[n][tap][co] = sum of dconv over output pixels whose tap (ky,kx) falls inside the frame
//   dW3[co][c_data+ct][ky][kx] += sum_n temb[n][ct] V[n][tap][co];  dW1[co][c_data+ct] += sum_n temb[n][ct] tres_sum[n][co]
//   dtemb[n][ct] = sum_co sum_tap W3[co][c_data+ct][tap] V[n][tap][co] + sum_co W1[co][c_data+ct] tres_sum[n][co]
// ================================================================================================
struct TimeBwdParams {
  const float* border; const float* sumD; const float* tres_sum; const float* temb;
  const float* w3; const float* w1;
  float* dw3; float* dw1; float* dtemb; float* db1;
  int N, ntc, c_in, c_data, Cout;
};

__device__ __forceinline__ float valid_sum(const float* border, const float* sumD, int n, int co, int Cout, int ky, int kx) {
  const float* b = border + (long long)n * 8 * Cout + co;
  float v = sumD[(long long)n * Cout + co];
  if (ky == 0) v -= b[0 * Cout];
  if (ky == 2) v -= b[1 * Cout];
  if (kx == 0) v -= b[2 * Cout];
  if (kx == 2) v -= b[3 * Cout];
  if (ky == 0 && kx == 0) v += b[4 * Cout];
  if (ky == 0 && kx == 2) v += b[5 * Cout];
  if (ky == 2 && kx == 0) v += b[6 * Cout];
  if (ky == 2 && kx == 2) v += b[7 * Cout];
  return v;
}

// grid: one block per (co, tap10) -- tap 9 = the 1x1 res_conv; the per-field factor is computed once into shared memory, then a
// thread per time channel sums over the fields (a thread per (co, ct, tap) looping over N was 480 us of dependent L2 round trips)
__global__ void __launch_bounds__(128) time_w_bwd_kernel(const TimeBwdParams p) {
  extern __shared__ float sv[];                            // [N]
  const int tap = blockIdx.x % 10, co = blockIdx.x / 10;
  for (int n = threadIdx.x; n < p.N; n += 128)
    sv[n] = tap == 9 ? p.tres_sum[(long long)n * p.Cout + co] : valid_sum(p.border, p.sumD, n, co, p.Cout, tap / 3, tap % 3);
  __syncthreads();
  for (int ct = threadIdx.x; ct < p.ntc; ct += 128) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int n = 0;
    for (; n + 3 < p.N; n += 4) {
      a0 = fmaf(p.temb[n * p.ntc + ct], sv[n], a0); a1 = fmaf(p.temb[(n + 1) * p.ntc + ct], sv[n + 1], a1);
      a2 = fmaf(p.temb[(n + 2) * p.ntc + ct], sv[n + 2], a2); a3 = fmaf(p.temb[(n + 3) * p.ntc + ct], sv[n + 3], a3);
    }
    for (; n < p.N; ++n) a0 = fmaf(p.temb[n * p.ntc + ct], sv[n], a0);
    const float acc = (a0 + a1) + (a2 + a3);
    if (tap == 9) p.dw1[(long long)co * p.c_in + p.c_data + ct] += acc;
    else p.dw3[((long long)co * p.c_in + p.c_data + ct) * 9 + tap] += acc;
  }
}
// one block per field n: dtemb[n][ct]; thread 0.. also adds db1 (res_conv bias) = sum_n tres_sum (DET: left to a fixed-order
// reduction of tres_sum over the fields)
template <bool DET = false>
__global__ void __launch_bounds__(128) time_emb_bwd_kernel(const TimeBwdParams p) {
  const int n = blockIdx.x;
  __shared__ float red[128];
  for (int ct = 0; ct < p.ntc; ++ct) {
    float acc = 0.f;
    for (int co = threadIdx.x; co < p.Cout; co += 128) {
      for (int tap = 0; tap < 9; ++tap)
        acc += p.w3[((long long)co * p.c_in + p.c_data + ct) * 9 + tap] * valid_sum(p.border, p.sumD, n, co, p.Cout, tap / 3, tap % 3);
      acc += p.w1[(long long)co * p.c_in + p.c_data + ct] * p.tres_sum[(long long)n * p.Cout + co];
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s > 0; s >>= 1) { if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s]; __syncthreads(); }
    if (threadIdx.x == 0) p.dtemb[n * p.ntc + ct] = red[0];
    __syncthreads();
  }
  if constexpr (!DET)
    for (int co = threadIdx.x; co < p.Cout; co += 128) atomicAdd(p.db1 + co, p.tres_sum[(long long)n * p.Cout + co]);
}

// embedding gradients (transpose of time_embed_kernel, metnet3.py:389-416): dtemb (N, le+3te) and dcond (N, le)
__global__ void time_embed_bwd_kernel(const float* __restrict__ dtemb, const float* __restrict__ dcond, const float* __restrict__ ts,
                                      long long ts_sB, long long ts_sT, long long ts_sF, int B, int L, int le, int te,
                                      float* __restrict__ d_lead, float* __restrict__ d_m, float* __restrict__ d_d, float* __restrict__ d_h, int* err) {
  const int N = B * L, ntc = le + 3 * te;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * ntc) return;
  const int n = i / ntc, c = i - n * ntc;
  const float g = dtemb[i];
  if (c < le) {
    atomicAdd(d_lead + ((n % L) + 1) * le + c, g + (dcond ? dcond[n * le + c] : 0.f));
  } else {
    const int f = n * 3 * te + (c - le);
    const int r = f / te, col = f - r * te;
    const int which = r / N, idx = r - which * N;
    const int b = idx / L;
    const int k = (int)ts[(long long)b * ts_sB + 6 * ts_sT + (long long)(1 + which) * ts_sF];
    float* e = which == 0 ? d_m : (which == 1 ? d_d : d_h);
    const int rows = which == 0 ? 13 : (which == 1 ? 32 : 25);
    if (k < 0 || k >= rows) { if (err) atomicOr(err, VG_DEVERR_TIMESTAMP); return; }   // forward already poisoned this field
    atomicAdd(e + k * te + col, g);
  }
}

// deterministic time_embed_bwd_kernel: one thread per output element sums its contributions in field order.
//   lead rows l+1 (l < L): d_lead[l+1][c] += sum_b (dtemb[b*L+l][c] + dcond[b*L+l][c])
//   table `which` (month / day / hour), row k, column col: every r = which*N + idx whose timestamp index is k contributes
//   dtemb at flat offset f = r*te + col of the (N, 3te) model-time block (the dim-0 concat quirk of metnet3.py:395-401)
__global__ void time_embed_bwd_det_kernel(const float* __restrict__ dtemb, const float* __restrict__ dcond, const float* __restrict__ ts,
                                          long long ts_sB, long long ts_sT, long long ts_sF, int B, int L, int le, int te,
                                          float* __restrict__ d_lead, float* __restrict__ d_m, float* __restrict__ d_d, float* __restrict__ d_h,
                                          int* err) {
  const int N = B * L, ntc = le + 3 * te, nlead = L * le;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  auto tindex = [&](int which, int idx) { return (int)ts[(long long)(idx / L) * ts_sB + 6 * ts_sT + (long long)(1 + which) * ts_sF]; };
  if (i < nlead) {
    const int l = i / le, c = i - l * le;
    float acc = 0.f;
    for (int b = 0; b < B; ++b) {
      const int n = b * L + l;
      acc += dtemb[n * ntc + c] + (dcond ? dcond[n * le + c] : 0.f);
    }
    d_lead[(l + 1) * le + c] += acc;
    return;
  }
  int j = i - nlead;
  const int nrows[3] = {13, 32, 25};
  for (int which = 0; which < 3; ++which) {
    if (j < nrows[which] * te) {
      const int k = j / te, col = j - k * te;
      float acc = 0.f;
      for (int idx = 0; idx < N; ++idx) {
        const int kk = tindex(which, idx);
        if (kk < 0 || kk >= nrows[which]) { if (err && k == 0 && col == 0) atomicOr(err, VG_DEVERR_TIMESTAMP); continue; }
        if (kk != k) continue;
        const long long f = ((long long)which * N + idx) * te + col;
        const int n = (int)(f / (3 * te)), c = le + (int)(f - (long long)n * 3 * te);
        acc += dtemb[(long long)n * ntc + c];
      }
      float* e = which == 0 ? d_m : (which == 1 ? d_d : d_h);
      e[k * te + col] += acc;
      return;
    }
    j -= nrows[which] * te;
  }
}

// ================================================================================================
// Fixed-order reductions of the deterministic (_det) entry points: out[g][w] += sum_{s < S} in[g*S + s][w] (rows of ld floats).
// A block sums the slots [z*ch, z*ch + ch) of 32 columns (eight slot lanes, then the eight lane sums in order); with more than
// one chunk the chunk sums go to tmp and a second pass reduces them.  The order depends on S alone.
// ================================================================================================
__global__ void __launch_bounds__(256) slot_sum_kernel(const float* __restrict__ in, int S, int W, long long ld, int ch,
                                                       float* __restrict__ out, long long out_ld, int accumulate) {
  __shared__ float red[8][33];
  const int l = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int w = blockIdx.x * 32 + l, g = blockIdx.y, z = blockIdx.z;
  const int s0 = z * ch, s1 = min(S, s0 + ch);
  float a = 0.f;
  if (w < W)
    for (int s = s0 + sl; s < s1; s += 8) a += in[((long long)g * S + s) * ld + w];
  red[sl][l] = a;
  __syncthreads();
  if (sl == 0 && w < W) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][l];
    float* o = out + ((long long)g * gridDim.z + z) * out_ld + w;
    *o = accumulate ? *o + t : t;
  }
}

static int det_chunk(long long S) { int c = 64; while ((long long)c * c < S) c *= 2; return c; }

long long det_sum_tmp_elems(int G, long long S, int W) {
  const int ch = det_chunk(S);
  return S <= ch ? 0 : (long long)G * ((S + ch - 1) / ch) * W;
}

int det_sum_run(const float* in, int G, long long S, int W, long long ld, float* out, long long out_ld, float* tmp, cudaStream_t st) {
  if (G <= 0 || W <= 0) return 0;
  const int ch = det_chunk(S);
  const unsigned gx = (unsigned)((W + 31) / 32);
  if (S <= ch) {
    slot_sum_kernel<<<dim3(gx, G, 1), 256, 0, st>>>(in, (int)S, W, ld, ch, out, out_ld, 1);
    return check_launch("slot_sum_kernel");
  }
  const int nz = (int)((S + ch - 1) / ch);
  slot_sum_kernel<<<dim3(gx, G, nz), 256, 0, st>>>(in, (int)S, W, ld, ch, tmp, W, 0);
  int rc = check_launch("slot_sum_kernel");
  if (rc) return rc;
  slot_sum_kernel<<<dim3(gx, G, 1), 256, 0, st>>>(tmp, nz, W, W, ch, out, out_ld, 1);
  return check_launch("slot_sum_kernel");
}

// border (N, 8, C) += the sums of an fp32 dconv PG tensor over row 0, the last row, column 0, the last column and the four corners
// (what conv_ln_bwd_kernel accumulates with atomics), each a loop in pixel order; grid (N, 8)
__global__ void __launch_bounds__(128) border_sum_kernel(const float* __restrict__ dconv, float* __restrict__ border, PGeom pg, int C) {
  const int n = blockIdx.x, k = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += 128) {
    float s = 0.f;
    if (k < 2) {
      const int h = k == 0 ? 0 : pg.HP - 1;
      for (int w = 0; w < pg.WP; ++w) s += dconv[pg.q(n, h, w) * C + c];
    } else if (k < 4) {
      const int w = k == 2 ? 0 : pg.WP - 1;
      for (int h = 0; h < pg.HP; ++h) s += dconv[pg.q(n, h, w) * C + c];
    } else {
      s = dconv[pg.q(n, (k - 4) & 2 ? pg.HP - 1 : 0, (k - 4) & 1 ? pg.WP - 1 : 0) * C + c];
    }
    border[((long long)n * 8 + k) * C + c] += s;
  }
}

// ================================================================================================
// conditioning MLP backward (metnet3.py:140-143 ReLU->Linear; maxvit.py:130-135 Linear->SiLU->Linear)
// One block per field: recomputes the hidden layer, writes the per-field quantities the weight-gradient reductions
// need (xin (N,cd) = pre(cond), dpre (N,hid), hact (N,hid)) and accumulates dcond (N,cd).
// ================================================================================================
__global__ void __launch_bounds__(256) cond_mlp_bwd_kernel(const float* __restrict__ cond, int cd, int pre_relu, const float* __restrict__ W0,
                                                           const float* __restrict__ b0, int hid, const float* __restrict__ W1, int od,
                                                           const float* __restrict__ dout, float* __restrict__ xin, float* __restrict__ dpre,
                                                           float* __restrict__ hact, float* __restrict__ dcond) {
  extern __shared__ float sh[];          // cd + hid (dpre) + od (dout)
  float* sc = sh; float* sd = sh + cd; float* so = sd + hid;
  const int n = blockIdx.x;
  for (int i = threadIdx.x; i < cd; i += blockDim.x) {
    const float v = cond[n * cd + i];
    sc[i] = pre_relu ? fmaxf(v, 0.f) : v;
    xin[n * cd + i] = sc[i];
  }
  if (W1) for (int o = threadIdx.x; o < od; o += blockDim.x) so[o] = dout[(long long)n * od + o];
  __syncthreads();
  for (int j = threadIdx.x; j < hid; j += blockDim.x) {
    float g;
    if (W1) {
      float a = b0 ? b0[j] : 0.f;
      for (int i = 0; i < cd; ++i) a += W0[j * cd + i] * sc[i];
      const float sg = 1.0f / (1.0f + expf(-a));
      hact[(long long)n * hid + j] = a * sg;
      // (eight loads in flight: a rolled loop waits out one L2 round trip per iteration -- 42 us per launch for 0.3 MB of weights)
      float d8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      int o = 0;
      for (; o + 7 < od; o += 8) {
        float w8[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) w8[u] = W1[(long long)(o + u) * hid + j];
#pragma unroll
        for (int u = 0; u < 8; ++u) d8[u] = fmaf(w8[u], so[o + u], d8[u]);
      }
      for (; o < od; ++o) d8[0] = fmaf(W1[(long long)o * hid + j], so[o], d8[0]);
      const float dh = ((d8[0] + d8[1]) + (d8[2] + d8[3])) + ((d8[4] + d8[5]) + (d8[6] + d8[7]));
      g = dh * (sg * (1.0f + a * (1.0f - sg)));                 // d silu
    } else {
      g = dout[(long long)n * hid + j];
    }
    dpre[(long long)n * hid + j] = g;
    sd[j] = g;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < cd; i += blockDim.x) {
    float a8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    int j = 0;
    for (; j + 7 < hid; j += 8) {
      float w8[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w8[u] = W0[(j + u) * cd + i];
#pragma unroll
      for (int u = 0; u < 8; ++u) a8[u] = fmaf(w8[u], sd[j + u], a8[u]);
    }
    for (; j < hid; ++j) a8[0] = fmaf(W0[j * cd + i], sd[j], a8[0]);
    float a = ((a8[0] + a8[1]) + (a8[2] + a8[3])) + ((a8[4] + a8[5]) + (a8[6] + a8[7]));
    if (pre_relu && cond[n * cd + i] <= 0.f) a = 0.f;
    dcond[n * cd + i] += a;
  }
}

// dW[o][i] += sum_n G[n][o] * X[n][i];  db[o] += sum_n G[n][o]   (tiny reductions over the fields)
// A 32 x 32 output tile per block (256 threads, four outputs each); the fields are walked in chunks of 32 through shared memory,
// so every G / X element is read once per tile row / column instead of once per output (a thread -- later a warp -- per output:
// 68 / 48 us per launch for a 12 MFLOP product).
__global__ void __launch_bounds__(256) outer_sum_kernel(const float* __restrict__ G, const float* __restrict__ X, int N, int O, int I,
                                                        float* __restrict__ dW, float* __restrict__ db) {
  __shared__ float sg[32][33], sx[32][33];
  const int o0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;        // ty 0..7
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, bsum[4] = {0.f, 0.f, 0.f, 0.f};
  for (int n0 = 0; n0 < N; n0 += 32) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int n = n0 + ty + 8 * k;
      sg[ty + 8 * k][tx] = (n < N && o0 + tx < O) ? G[(long long)n * O + o0 + tx] : 0.f;
      sx[ty + 8 * k][tx] = (n < N && i0 + tx < I) ? X[(long long)n * I + i0 + tx] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int n = 0; n < 32; ++n) {
      const float xv = sx[n][tx];
#pragma unroll
      for (int k = 0; k < 4; ++k) { const float gv = sg[n][ty + 8 * k]; acc[k] = fmaf(gv, xv, acc[k]); bsum[k] += gv; }
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int o = o0 + ty + 8 * k, i = i0 + tx;
    if (o < O && i < I) dW[(long long)o * I + i] += acc[k];
    if (db && blockIdx.x == 0 && tx == 0 && o < O) db[o] += bsum[k];
  }
}

// ================================================================================================
// fused AdamW step over a flat parameter / gradient / moment buffer
// ================================================================================================
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, long long n, float lr, float b1, float b2, float eps,
                                                    float wd, float c1, float c2, float gscale) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * gscale;
  const float mi = b1 * m[i] + (1.0f - b1) * gi;
  const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
  m[i] = mi; v[i] = vi;
  float pi = p[i];
  pi -= lr * wd * pi;
  pi -= lr * (mi / c1) / (sqrtf(vi / c2) + eps);
  p[i] = pi;
}

// ================================================================================================
// host launchers
// ================================================================================================
int conv_ln_bwd_run(int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const unsigned* mask,
                    const float* ln_g, const float* film, float eps, void* dconv, float* sumA, float* sumB, float* sumD,
                    float* border, int N, int HP, int WP, cudaStream_t st) {
  ConvLnBwdParams p;
  p.dY = dY; p.xhat = xhat; p.rstd = rstd; p.mask = mask; p.ln_g = ln_g; p.film = film; p.dconv = dconv;
  p.sumA = sumA; p.sumB = sumB; p.sumD = sumD; p.border = border; p.rstd_clamp = 1.0f / sqrtf(eps) * (1.0f - 1e-6f);
  p.pg = make_pgeom(N, HP, WP);
  const unsigned g = nblk(p.pg.pixels(), 512);
  // the bulk copies need 16-byte aligned rows (torch allocations are; views at odd offsets are not)
  if ((reinterpret_cast<uintptr_t>(dY) | reinterpret_cast<uintptr_t>(xhat) | reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(rstd)) & 15)
    return set_error("conv_ln_bwd: dY / xhat / mask / rstd must be 16-byte aligned");
  const size_t sm16 = 8 * lnb::NST * lnb::stage_bytes<bf16>() + 128, sm32 = 8 * lnb::NST * lnb::stage_bytes<float>() + 128;
  static PerDeviceFlag attr_pd;
  bool& attr = attr_pd.cur();
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_ln_bwd_kernel<bf16, bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm16);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_ln_bwd_kernel<bf16, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm16);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_ln_bwd_kernel<float, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm32);
    if (e != cudaSuccess) return set_error("conv_ln_bwd smem attr: %s", cudaGetErrorString(e));
    attr = true;
  }
  if (xdtype == 0 && odtype == 0) conv_ln_bwd_kernel<bf16, bf16><<<g, 256, sm16, st>>>(p);
  else if (xdtype == 0 && odtype == 1) conv_ln_bwd_kernel<bf16, float><<<g, 256, sm16, st>>>(p);
  else if (xdtype == 1 && odtype == 1) conv_ln_bwd_kernel<float, float><<<g, 256, sm32, st>>>(p);
  else return set_error("conv_ln_bwd: unsupported dtype combination (%d, %d)", xdtype, odtype);
  return check_launch("conv_ln_bwd_kernel");
}

static int wide_c_check(const char* what, int C) {
  if (C != 128 && C != 256 && C != 384 && C != 512) return set_error("%s: C=%d must be 128, 256, 384 or 512", what, C);
  return 0;
}

// expands BODY with the compile-time width CW = C (128, 256, 384 or 512; checked by the caller)
#define VG_WIDTH_SWITCH(C, BODY)                           \
  switch (C) {                                             \
    case 128: { constexpr int CW = 128; BODY; } break;     \
    case 256: { constexpr int CW = 256; BODY; } break;     \
    case 384: { constexpr int CW = 384; BODY; } break;     \
    default:  { constexpr int CW = 512; BODY; } break;     \
  }

int conv_ln_bwd_wide_run(int C, const float* dY, const float* xhat, const float* rstd, const unsigned* mask, const float* ln_g,
                         const float* film, float eps, float* dconv, float* sumA, float* sumB, float* sumD, float* border, int N,
                         int HP, int WP, cudaStream_t st) {
  if (wide_c_check("conv_ln_bwd_wide", C)) return 1;
  ConvLnBwdParams p;
  p.dY = dY; p.xhat = xhat; p.rstd = rstd; p.mask = mask; p.ln_g = ln_g; p.film = film; p.dconv = dconv;
  p.sumA = sumA; p.sumB = sumB; p.sumD = sumD; p.border = border; p.rstd_clamp = 1.0f / sqrtf(eps) * (1.0f - 1e-6f);
  p.pg = make_pgeom(N, HP, WP);
  const unsigned g = nblk(p.pg.pixels(), 256);
  VG_WIDTH_SWITCH(C, (conv_ln_bwd_wide_kernel<CW / 128><<<g, 256, 0, st>>>(p)));
  return check_launch("conv_ln_bwd_wide_kernel");
}

int conv_ln_param_grads_run(const float* sumA, const float* sumB, const float* sumD, int N, const float* g, const float* b,
                            const float* film, float* dg, float* db, float* dbias, float* dfilm, int C, cudaStream_t st) {
  if (wide_c_check("conv_ln_param_grads", C)) return 1;
  VG_WIDTH_SWITCH(C, (conv_ln_param_grads_kernel<CW><<<CW / 32, 256, 0, st>>>(sumA, sumB, sumD, N, g, b, film, dg, db, dbias, dfilm)));
  return check_launch("conv_ln_param_grads_kernel");
}

int head_bwd_run(int dtype, const float* dpred, const void* h, const float* w, float stdv, int N, int HP, int WP, int H, int W,
                 int pt, int pl, float* dH, float* dw, float* db, int C, cudaStream_t st) {
  if (wide_c_check("head_bwd", C)) return 1;
  PGeom pg = make_pgeom(N, HP, WP);
  const unsigned g = nblk(pg.pixels(), 256);
  if (dtype == 0) VG_WIDTH_SWITCH(C, (head_bwd_kernel<CW, bf16><<<g, 256, 0, st>>>(dpred, reinterpret_cast<const bf16*>(h), w, stdv, pg, H, W, pt, pl, dH, dw, db)))
  else VG_WIDTH_SWITCH(C, (head_bwd_kernel<CW, float><<<g, 256, 0, st>>>(dpred, reinterpret_cast<const float*>(h), w, stdv, pg, H, W, pt, pl, dH, dw, db)))
  return check_launch("head_bwd_kernel");
}

int maxpool2_bwd_run(int dtype, const void* x, const float* dlow, float* dx, int N, int HP, int WP, int C, cudaStream_t st) {
  if (C % 8 || HP % 2 || WP % 2) return set_error("maxpool2_bwd: bad shape");
  PGeom pg = make_pgeom(N, HP, WP);
  const long long total = pg.pixels() * (C / 8);
  if (dtype == 0) maxpool2_bwd_kernel<bf16><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<const bf16*>(x), dlow, dx, pg, C);
  else maxpool2_bwd_kernel<float><<<nblk(total, 256), 256, 0, st>>>(reinterpret_cast<const float*>(x), dlow, dx, pg, C);
  return check_launch("maxpool2_bwd_kernel");
}

int convT_bwd_gather_run(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, cudaStream_t st) {
  if (wide_c_check("convT_bwd_gather", C)) return 1;
  PGeom pg = make_pgeom(N, 2 * Hl, 2 * Wl);
  const long long M = (long long)N * Hl * Wl;
  const unsigned g = nblk(M, 8 * 16);
  if (odtype == 0) VG_WIDTH_SWITCH(C, (convT_bwd_gather_kernel<CW, bf16><<<g, 256, 0, st>>>(dUp, reinterpret_cast<bf16*>(G), dbias, pg, Hl, Wl, M)))
  else VG_WIDTH_SWITCH(C, (convT_bwd_gather_kernel<CW, float><<<g, 256, 0, st>>>(dUp, reinterpret_cast<float*>(G), dbias, pg, Hl, Wl, M)))
  return check_launch("convT_bwd_gather_kernel");
}

int lead_sum_run(int idtype, int odtype, const void* in, void* out, int B, int L, int HP, int WP, int C, cudaStream_t st) {
  if (wide_c_check("lead_sum", C)) return 1;
  PGeom pgN = make_pgeom(B * L, HP, WP), pgB = make_pgeom(B, HP, WP);
  const unsigned g = nblk(pgB.pixels(), 8);
  if (idtype == 0 && odtype == 0) VG_WIDTH_SWITCH(C, (lead_sum_kernel<CW, bf16, bf16><<<g, 256, 0, st>>>(reinterpret_cast<const bf16*>(in), reinterpret_cast<bf16*>(out), pgN, pgB, L)))
  else if (idtype == 1 && odtype == 0) VG_WIDTH_SWITCH(C, (lead_sum_kernel<CW, float, bf16><<<g, 256, 0, st>>>(reinterpret_cast<const float*>(in), reinterpret_cast<bf16*>(out), pgN, pgB, L)))
  else if (idtype == 1 && odtype == 1) VG_WIDTH_SWITCH(C, (lead_sum_kernel<CW, float, float><<<g, 256, 0, st>>>(reinterpret_cast<const float*>(in), reinterpret_cast<float*>(out), pgN, pgB, L)))
  else return set_error("lead_sum: unsupported dtype combination (%d, %d)", idtype, odtype);
  return check_launch("lead_sum_kernel");
}

int pg_field_sum_run(const float* in, float* out, int N, int HP, int WP, int C, cudaStream_t st) {
  if (wide_c_check("pg_field_sum", C)) return 1;
  PGeom pg = make_pgeom(N, HP, WP);
  int chunks = (HP * WP + 255) / 256;
  if (chunks > 32) chunks = 32;
  VG_WIDTH_SWITCH(C, (pg_field_sum_kernel<CW><<<dim3(chunks, N), 256, 0, st>>>(in, out, pg)));
  return check_launch("pg_field_sum_kernel");
}

int time_terms_bwd_run(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                       const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                       float* dtemb, cudaStream_t st) {
  TimeBwdParams p;
  p.border = border; p.sumD = sumD; p.tres_sum = tres_sum; p.temb = temb; p.w3 = w3; p.w1 = w1;
  p.dw3 = dw3; p.dw1 = dw1; p.dtemb = dtemb; p.db1 = db1; p.N = N; p.ntc = ntc; p.c_in = c_in; p.c_data = c_data; p.Cout = Cout;
  time_w_bwd_kernel<<<Cout * 10, 128, (size_t)N * sizeof(float), st>>>(p);
  int rc = check_launch("time_w_bwd_kernel");
  if (rc) return rc;
  time_emb_bwd_kernel<<<N, 128, 0, st>>>(p);
  return check_launch("time_emb_bwd_kernel");
}

int time_embed_bwd_run(const float* dtemb, const float* dcond, const float* ts, long long sB, long long sT, long long sF, int B,
                       int L, int le, int te, float* d_lead, float* d_m, float* d_d, float* d_h, cudaStream_t st) {
  const int N = B * L, ntc = le + 3 * te;
  time_embed_bwd_kernel<<<nblk((long long)N * ntc, 128), 128, 0, st>>>(dtemb, dcond, ts, sB, sT, sF, B, L, le, te, d_lead, d_m, d_d, d_h, device_error_ptr());
  return check_launch("time_embed_bwd_kernel");
}

int cond_mlp_bwd_run(const float* cond, int N, int cd, int pre_relu, const float* W0, const float* b0, int hid, const float* W1,
                     int od, const float* dout, float* dW0, float* db0, float* dW1, float* db1, float* dcond, float* work,
                     long long work_elems, cudaStream_t st) {
  const long long need = (long long)N * (cd + 2 * hid);
  if (work_elems < need) return set_error("cond_mlp_bwd: workspace too small (%lld < %lld)", work_elems, need);
  float* xin = work; float* dpre = xin + (long long)N * cd; float* hact = dpre + (long long)N * hid;
  cond_mlp_bwd_kernel<<<N, 256, (cd + hid + od) * sizeof(float), st>>>(cond, cd, pre_relu, W0, b0, hid, W1, od, dout, xin, dpre, hact, dcond);
  int rc = check_launch("cond_mlp_bwd_kernel");
  if (rc) return rc;
  outer_sum_kernel<<<dim3((cd + 31) / 32, (hid + 31) / 32), 256, 0, st>>>(dpre, xin, N, hid, cd, dW0, db0);
  rc = check_launch("outer_sum_kernel");
  if (rc || !W1) return rc;
  outer_sum_kernel<<<dim3((hid + 31) / 32, (od + 31) / 32), 256, 0, st>>>(dout, hact, N, od, hid, dW1, db1);
  return check_launch("outer_sum_kernel");
}

int outer_sum_run(const float* G, const float* X, int N, int O, int I, float* dW, float* db, cudaStream_t st) {
  outer_sum_kernel<<<dim3((I + 31) / 32, (O + 31) / 32), 256, 0, st>>>(G, X, N, O, I, dW, db);
  return check_launch("outer_sum_kernel");
}

// ------------------------------------------------------------------------------------------------
// deterministic variants: per-warp partials in fixed slots of the caller's workspace, then det_sum_run
// ------------------------------------------------------------------------------------------------
static int det_work_check(const char* what, long long need, float* work, long long work_elems) {
  if (need > 0 && (!work || work_elems < need)) return set_error("%s: workspace too small (%lld < %lld floats)", what, work_elems, need);
  return 0;
}

static int conv_ln_slots(int C, const PGeom& pg) { return C == 128 ? 2 * det_field_slots(pg, lnb::PPW) : det_field_slots(pg, 32); }

long long conv_ln_bwd_det_workspace_elems(int C, int N, int HP, int WP) {
  const PGeom pg = make_pgeom(N, HP, WP);
  const int K = conv_ln_slots(C, pg);
  return 3LL * N * K * C + det_sum_tmp_elems(N, K, C);
}

int conv_ln_bwd_det_run(int C, int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const unsigned* mask,
                        const float* ln_g, const float* film, float eps, void* dconv, float* sumA, float* sumB, float* sumD,
                        float* border, int N, int HP, int WP, float* work, long long work_elems, cudaStream_t st) {
  if (wide_c_check("conv_ln_bwd_det", C)) return 1;
  if (border && odtype != 1) return set_error("conv_ln_bwd_det: the border sums need an fp32 dconv (odtype 1)");
  ConvLnBwdParams p;
  p.dY = dY; p.xhat = xhat; p.rstd = rstd; p.mask = mask; p.ln_g = ln_g; p.film = film; p.dconv = dconv;
  p.sumA = sumA; p.sumB = sumB; p.sumD = sumD; p.border = nullptr; p.rstd_clamp = 1.0f / sqrtf(eps) * (1.0f - 1e-6f);
  p.pg = make_pgeom(N, HP, WP);
  p.K = conv_ln_slots(C, p.pg);
  const long long nslots = 3LL * N * p.K * C;
  if (det_work_check("conv_ln_bwd_det", conv_ln_bwd_det_workspace_elems(C, N, HP, WP), work, work_elems)) return 1;
  p.slots = work;
  float* tmp = work + nslots;
  cudaError_t e = cudaMemsetAsync(p.slots, 0, (size_t)nslots * sizeof(float), st);
  if (e != cudaSuccess) return set_error("conv_ln_bwd_det: %s", cudaGetErrorString(e));
  if (C == 128) {
    const unsigned g = nblk(p.pg.pixels(), 512);
    if ((reinterpret_cast<uintptr_t>(dY) | reinterpret_cast<uintptr_t>(xhat) | reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(rstd)) & 15)
      return set_error("conv_ln_bwd_det: dY / xhat / mask / rstd must be 16-byte aligned");
    const size_t sm16 = 8 * lnb::NST * lnb::stage_bytes<bf16>() + 128, sm32 = 8 * lnb::NST * lnb::stage_bytes<float>() + 128;
    static PerDeviceFlag attr_pd;
    bool& attr = attr_pd.cur();
    if (!attr) {
      cudaError_t e2 = cudaFuncSetAttribute(conv_ln_bwd_kernel<bf16, bf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm16);
      if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(conv_ln_bwd_kernel<bf16, float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm16);
      if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(conv_ln_bwd_kernel<float, float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm32);
      if (e2 != cudaSuccess) return set_error("conv_ln_bwd_det smem attr: %s", cudaGetErrorString(e2));
      attr = true;
    }
    if (xdtype == 0 && odtype == 0) conv_ln_bwd_kernel<bf16, bf16, true><<<g, 256, sm16, st>>>(p);
    else if (xdtype == 0 && odtype == 1) conv_ln_bwd_kernel<bf16, float, true><<<g, 256, sm16, st>>>(p);
    else if (xdtype == 1 && odtype == 1) conv_ln_bwd_kernel<float, float, true><<<g, 256, sm32, st>>>(p);
    else return set_error("conv_ln_bwd_det: unsupported dtype combination (%d, %d)", xdtype, odtype);
  } else {
    const unsigned g = nblk(p.pg.pixels(), 256);
    VG_WIDTH_SWITCH(C, (conv_ln_bwd_wide_kernel<CW / 128, true><<<g, 256, 0, st>>>(p)));
  }
  int rc = check_launch("conv_ln_bwd_kernel (det)");
  float* outs[3] = {sumA, sumB, sumD};
  for (int k = 0; k < 3 && !rc; ++k) rc = det_sum_run(p.slots + k * (nslots / 3), N, p.K, C, C, outs[k], C, tmp, st);
  if (rc || !border) return rc;
  border_sum_kernel<<<dim3(N, 8), 128, 0, st>>>(reinterpret_cast<const float*>(dconv), border, p.pg, C);
  return check_launch("border_sum_kernel");
}

static long long head_warps(const PGeom& pg) { return (long long)nblk(pg.pixels(), 256) * 8; }

long long head_bwd_det_workspace_elems(int N, int HP, int WP, int C) {
  const long long S = head_warps(make_pgeom(N, HP, WP));
  return S * (C + 1) + det_sum_tmp_elems(1, S, C);
}

int head_bwd_det_run(int dtype, const float* dpred, const void* h, const float* w, float stdv, int N, int HP, int WP, int H, int W,
                     int pt, int pl, float* dH, float* dw, float* db, int C, float* work, long long work_elems, cudaStream_t st) {
  if (wide_c_check("head_bwd_det", C)) return 1;
  if (det_work_check("head_bwd_det", head_bwd_det_workspace_elems(N, HP, WP, C), work, work_elems)) return 1;
  PGeom pg = make_pgeom(N, HP, WP);
  const unsigned g = nblk(pg.pixels(), 256);
  const long long S = head_warps(pg);
  float* tmp = work + S * (C + 1);
  if (dtype == 0) VG_WIDTH_SWITCH(C, (head_bwd_kernel<CW, bf16, true><<<g, 256, 0, st>>>(dpred, reinterpret_cast<const bf16*>(h), w, stdv, pg, H, W, pt, pl, dH, work, nullptr)))
  else VG_WIDTH_SWITCH(C, (head_bwd_kernel<CW, float, true><<<g, 256, 0, st>>>(dpred, reinterpret_cast<const float*>(h), w, stdv, pg, H, W, pt, pl, dH, work, nullptr)))
  int rc = check_launch("head_bwd_kernel (det)");
  if (!rc) rc = det_sum_run(work, 1, S, C, C + 1, dw, C, tmp, st);
  if (!rc) rc = det_sum_run(work + C, 1, S, 1, C + 1, db, 1, tmp, st);
  return rc;
}

long long convT_bwd_gather_det_workspace_elems(int N, int Hl, int Wl, int C) {
  const long long S = (long long)nblk((long long)N * Hl * Wl, 8 * 16) * 8;
  return S * C + det_sum_tmp_elems(1, S, C);
}

int convT_bwd_gather_det_run(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, float* work,
                             long long work_elems, cudaStream_t st) {
  if (wide_c_check("convT_bwd_gather_det", C)) return 1;
  if (det_work_check("convT_bwd_gather_det", convT_bwd_gather_det_workspace_elems(N, Hl, Wl, C), work, work_elems)) return 1;
  PGeom pg = make_pgeom(N, 2 * Hl, 2 * Wl);
  const long long M = (long long)N * Hl * Wl;
  const unsigned g = nblk(M, 8 * 16);
  const long long S = (long long)g * 8;
  if (odtype == 0) VG_WIDTH_SWITCH(C, (convT_bwd_gather_kernel<CW, bf16, true><<<g, 256, 0, st>>>(dUp, reinterpret_cast<bf16*>(G), work, pg, Hl, Wl, M)))
  else VG_WIDTH_SWITCH(C, (convT_bwd_gather_kernel<CW, float, true><<<g, 256, 0, st>>>(dUp, reinterpret_cast<float*>(G), work, pg, Hl, Wl, M)))
  int rc = check_launch("convT_bwd_gather_kernel (det)");
  return rc ? rc : det_sum_run(work, 1, S, C, C, dbias, C, work + S * C, st);
}

static int field_sum_chunks(int HP, int WP) { int c = (HP * WP + 255) / 256; return c > 32 ? 32 : c; }

long long pg_field_sum_det_workspace_elems(int N, int HP, int WP, int C) {
  const long long S = (long long)field_sum_chunks(HP, WP) * 8;
  return (long long)N * S * C + det_sum_tmp_elems(N, S, C);
}

int pg_field_sum_det_run(const float* in, float* out, int N, int HP, int WP, int C, float* work, long long work_elems, cudaStream_t st) {
  if (wide_c_check("pg_field_sum_det", C)) return 1;
  if (det_work_check("pg_field_sum_det", pg_field_sum_det_workspace_elems(N, HP, WP, C), work, work_elems)) return 1;
  PGeom pg = make_pgeom(N, HP, WP);
  const int chunks = field_sum_chunks(HP, WP);
  VG_WIDTH_SWITCH(C, (pg_field_sum_kernel<CW, true><<<dim3(chunks, N), 256, 0, st>>>(in, work, pg)));
  int rc = check_launch("pg_field_sum_kernel (det)");
  return rc ? rc : det_sum_run(work, N, chunks * 8, C, C, out, C, work + (long long)N * chunks * 8 * C, st);
}

long long time_terms_bwd_det_workspace_elems(int N, int Cout) { return det_sum_tmp_elems(1, N, Cout); }

int time_terms_bwd_det_run(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                           const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                           float* dtemb, float* work, long long work_elems, cudaStream_t st) {
  if (det_work_check("time_terms_bwd_det", time_terms_bwd_det_workspace_elems(N, Cout), work, work_elems)) return 1;
  TimeBwdParams p;
  p.border = border; p.sumD = sumD; p.tres_sum = tres_sum; p.temb = temb; p.w3 = w3; p.w1 = w1;
  p.dw3 = dw3; p.dw1 = dw1; p.dtemb = dtemb; p.db1 = db1; p.N = N; p.ntc = ntc; p.c_in = c_in; p.c_data = c_data; p.Cout = Cout;
  time_w_bwd_kernel<<<Cout * 10, 128, (size_t)N * sizeof(float), st>>>(p);
  int rc = check_launch("time_w_bwd_kernel");
  if (rc) return rc;
  time_emb_bwd_kernel<true><<<N, 128, 0, st>>>(p);
  rc = check_launch("time_emb_bwd_kernel (det)");
  return rc ? rc : det_sum_run(tres_sum, 1, N, Cout, Cout, db1, Cout, work, st);
}

int time_embed_bwd_det_run(const float* dtemb, const float* dcond, const float* ts, long long sB, long long sT, long long sF, int B,
                           int L, int le, int te, float* d_lead, float* d_m, float* d_d, float* d_h, cudaStream_t st) {
  const long long total = (long long)L * le + 70LL * te;
  time_embed_bwd_det_kernel<<<nblk(total, 128), 128, 0, st>>>(dtemb, dcond, ts, sB, sT, sF, B, L, le, te, d_lead, d_m, d_d, d_h, device_error_ptr());
  return check_launch("time_embed_bwd_det_kernel");
}

int adamw_run(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps, float wd,
              int step, float gscale, cudaStream_t st) {
  const float c1 = 1.0f - powf(b1, (float)step), c2 = 1.0f - powf(b2, (float)step);
  adamw_kernel<<<nblk(n, 256), 256, 0, st>>>(p, g, m, v, n, lr, b1, b2, eps, wd, c1, c2, gscale);
  return check_launch("adamw_kernel");
}

}  // namespace vg
