// Row-wise GEMM epilogues shared by the tcgen05 kernel (accumulator row read from TMEM, one thread per
// row) and the fp32-mode SIMT path (accumulator row read from a global scratch).  A "Loader" exposes
//     void load(int chunk, float v[32])   // columns [n0 + 32*chunk, +32) of this thread's accumulator row
// and MUST be called uniformly by all threads of a warp (the TMEM load is warp-collective); only the global
// stores are predicated on row validity.
#pragma once
#include "vg_common.cuh"
#include "vg_rng.cuh"

namespace vg {

enum EpiKind : int {
  EPI_STORE = 0,      // y = act(acc*scale + shift | acc + bias) (+ res)                 -> [row][ldo]
  EPI_CONV_LN = 1,    // conv3x3 block: +bias, channel LayerNorm, FiLM, ReLU, (+res), zero pads (PG layout)
  EPI_ATTN_OUT = 2,   // attention out-projection: + residual, scatter through the inverse window/grid map
  EPI_CONVT = 3,      // ConvTranspose2d k2 s2 as GEMM: + bias, depth-to-space into the PG layout
  EPI_CONV_LN_TRAIN = 4,  // EPI_CONV_LN that also saves what the backward pass needs (normalised activations, rstd, ReLU mask)
};

struct EpiParams {
  void* out;
  long long ldo;
  int out_f32;               // output element type: 0 = activation dtype T, 1 = fp32, 2 = bf16, 3 = fp16 (coalesced store epilogue)
  int n_total;               // total number of GEMM columns
  const float* bias;         // [n_total] (EPI_CONVT: [C])
  const float* col_scale;    // folded BatchNorm: y = acc*scale + shift (bias already folded into shift)
  const float* col_shift;
  int act;                   // 0 none, 1 GELU(erf), 2 ReLU
  const void* res;           // residual, same row indexing as out
  long long ldres;
  // EPI_CONV_LN
  const float* ln_g;
  const float* ln_b;
  float ln_eps;
  const float* film;         // [fields][2C]  (scale | shift), applied as v*(scale+1)+shift; null = none
  PGeom pg;                  // output geometry (EPI_CONV_LN, EPI_CONVT)
  int res_f32;               // EPI_CONV_LN: the residual is fp32 (skip connections keep full precision)
  float* out2;               // optional fp32 copy of the output (EPI_CONV_LN, EPI_CONVT), same indexing as out
  // EPI_CONV_LN_TRAIN: saved for backward -- xhat (activation dtype, [q][C], zeros at pads), rstd (fp32 [q]),
  // relu_mask (4 x 32 bits per pixel: bit c%32 of word c/32 = ReLU input > 0)
  void* xhat;
  float* rstd_out;
  unsigned* relu_mask;
  // optional fused 1x1 head + unpad + de-normalisation (metnet3.py:424-430): head_out[n][h-pt][w-pl]
  const float* head_w;       // [C]; null = no head
  float* head_out;           // (N, H, W) fp32
  float head_b, head_std, head_mean;
  int head_H, head_W, head_pt, head_pl;
  // EPI_ATTN_OUT
  int S, R, nwin, grid_mode, win, X, Y, Hl, Wl;
  const void* x_in;          // (N, Hl*Wl, C) residual stream the window tokens came from
  const float* reg_in;       // register-token residual: [R][C] (shared) or [N][R][C] (per field)
  int reg_in_per_field;
  float* reg_out;            // [Nw][R][C] register-token outputs (block attention) or null
  unsigned drop_seed, drop_salt; int drop_thresh; float drop_scale;   // nn.Dropout after to_out (maxvit.py:151); thresh 0 = off
};

// store 8 consecutive outputs at element offset `off` of ep.out in the selected output type
template <typename T>
__device__ __forceinline__ void st8_out(const EpiParams& ep, long long off, const float* v) {
  if (ep.out_f32 == 1) st8(reinterpret_cast<float*>(ep.out) + off, v);
  else if (ep.out_f32 == 2) st8(reinterpret_cast<bf16*>(ep.out) + off, v);
  else st8(reinterpret_cast<T*>(ep.out) + off, v);
}

template <typename T, class Loader>
__device__ __forceinline__ void epi_store(const EpiParams& ep, long long row, bool ok, int n0, Loader& ld) {
  float v[32];
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    ld.load(ch, v);
    const int c0 = n0 + ch * 32;
    if (!ok || c0 >= ep.n_total) continue;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float x = v[j];
      if (ep.col_scale) x = x * __ldg(ep.col_scale + c0 + j) + __ldg(ep.col_shift + c0 + j);
      else if (ep.bias) x += __ldg(ep.bias + c0 + j);
      if (ep.act == 1) x = gelu_erf(x);
      else if (ep.act == 2) x = fmaxf(x, 0.f);
      v[j] = x;
    }
    if (ep.res && ep.res_f32) {
      const float* r = reinterpret_cast<const float*>(ep.res) + row * ep.ldres + c0;
#pragma unroll
      for (int j = 0; j < 32; j += 8) { float t[8]; ld8(r + j, t);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[j + i] += t[i]; }
    } else if (ep.res) {
      const T* r = reinterpret_cast<const T*>(ep.res) + row * ep.ldres + c0;
#pragma unroll
      for (int j = 0; j < 32; j += 8) { float t[8]; ld8(r + j, t);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[j + i] += t[i]; }
    }
#pragma unroll
    for (int j = 0; j < 32; j += 8) st8_out<T>(ep, row * ep.ldo + c0 + j, v + j);
  }
}

// plain fp32 row store (+ optional fp32 residual) of a 128-column accumulator row, 256-bit global accesses: the epilogue of the
// convolution's data gradient in the halo kernel
__device__ __forceinline__ void ld8_256(const float* p, float* v) {
  asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]),
               "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}
template <class Loader>
__device__ __forceinline__ void epi_store_f32_rows(const EpiParams& ep, long long row, bool ok, Loader& ld) {
  float v[32];
  float* o = reinterpret_cast<float*>(ep.out) + row * ep.ldo;
  const float* r = ep.res ? reinterpret_cast<const float*>(ep.res) + row * ep.ldres : nullptr;
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    float rr[32];
    if (ok && r) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) ld8_256(r + ch * 32 + j, rr + j);
    }
    ld.load(ch, v);
    if (!ok) continue;
    if (r) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += rr[j];
    }
#pragma unroll
    for (int j = 0; j < 32; j += 8) st8_256(o + ch * 32 + j, v + j);
  }
}

// EPI_STORE with a 16-bit output and nothing else to do (no scale / bias / activation / residual): every thread converts its row's 32
// accumulator columns and writes them as two 256-bit stores (64 contiguous bytes).  The transposing epilogue below needs 8 + 8
// shared-memory instructions and 8 stores per 32 columns for the same 64 sectors; with one epilogue warp pair per scheduler that
// instruction count, not HBM, bounded the QKV re-materialisation GEMM of the training step (0.88 ms for 1.9 GB of output)
template <typename T>
__device__ __forceinline__ bool epi_store_rows16_ok(const EpiParams& ep) {
  const bool out16 = ep.out_f32 == 2 || ep.out_f32 == 3 || (ep.out_f32 == 0 && sizeof(T) == 2);
  return out16 && !ep.res && !ep.col_scale && !ep.bias && ep.act == 0 && (ep.n_total & 31) == 0 && (ep.ldo & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(ep.out) & 31) == 0;
}
template <class Loader>
__device__ __forceinline__ void epi_store_rows16(const EpiParams& ep, long long row, bool ok, int n0, Loader& ld, int ch_begin = 0, int ch_end = 4) {
  float v[32];
#pragma unroll 1
  for (int ch = ch_begin; ch < ch_end; ++ch) {
    const int c0 = n0 + ch * 32;
    ld.load(ch, v);
    if (c0 >= ep.n_total || !ok) continue;
    const long long off = row * ep.ldo + c0;
    if (ep.out_f32 == 3) { __half* o = reinterpret_cast<__half*>(ep.out) + off; st16_256(o, v); st16_256(o + 16, v + 16); }
    else { bf16* o = reinterpret_cast<bf16*>(ep.out) + off; st16_256(o, v); st16_256(o + 16, v + 16); }
  }
}

// EPI_STORE for the tcgen05 kernel: same math as epi_store, but the 32x32 block a warp reads from TMEM (one row per
// thread) is transposed through a padded shared-memory tile so that every global access is a run of four full
// 128-byte row segments per warp instruction instead of 32 scattered 16-byte pieces (the row-per-thread stores made
// the wide 1x1 / projection GEMMs LSU-transaction-bound).  `row0` = global row of lane 0, `nvalid` = valid rows of
// this warp's 32 (rows are consecutive), stg = this warp's [32][36] float tile.
template <typename T, class Loader>
__device__ __forceinline__ void epi_store_coalesced(const EpiParams& ep, long long row0, int nvalid, int n0, Loader& ld,
                                                    float* stg, int lane, int ch_begin = 0, int ch_end = 4) {
  constexpr int LDS_ = 36;                                 // row stride of the tile: 16-byte aligned, conflict-free for 128-bit access
  float v[32];
  const int rr = lane >> 3, cq = (lane & 7) * 4;
#pragma unroll 1
  for (int ch = ch_begin; ch < ch_end; ++ch) {
    const int c0 = n0 + ch * 32;
    // this lane's four output columns are the same for every row of the transposed phase: fetch their parameters once
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c0 < ep.n_total) {
      if (ep.col_scale) { sc = __ldg(reinterpret_cast<const float4*>(ep.col_scale + c0 + cq)); sh = __ldg(reinterpret_cast<const float4*>(ep.col_shift + c0 + cq)); }
      else if (ep.bias) sh = __ldg(reinterpret_cast<const float4*>(ep.bias + c0 + cq));
    }
    ld.load(ch, v);
    if (c0 >= ep.n_total) continue;                       // warp-uniform
#pragma unroll
    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(stg + lane * LDS_ + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    __syncwarp();
    // activation first, for all eight row groups at once and without branches: the GELU is a chain of ~20 dependent operations
    // and two MUFU round trips per element, and only two epilogue warps share a scheduler -- eight independent chains per
    // thread hide it (with the row-validity branch around each group the compiler kept the groups serial)
    float o8[8][4];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const float4 a4 = *reinterpret_cast<const float4*>(stg + (it * 4 + rr) * LDS_ + cq);
      o8[it][0] = fmaf(a4.x, sc.x, sh.x); o8[it][1] = fmaf(a4.y, sc.y, sh.y); o8[it][2] = fmaf(a4.z, sc.z, sh.z); o8[it][3] = fmaf(a4.w, sc.w, sh.w);
    }
    if (ep.act == 1) {
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const float2 g0 = gelu_erf2(make_float2(o8[it][0], o8[it][1])), g1 = gelu_erf2(make_float2(o8[it][2], o8[it][3]));
        o8[it][0] = g0.x; o8[it][1] = g0.y; o8[it][2] = g1.x; o8[it][3] = g1.y;
      }
    } else if (ep.act == 2) {
#pragma unroll
      for (int it = 0; it < 8; ++it) { o8[it][0] = fmaxf(o8[it][0], 0.f); o8[it][1] = fmaxf(o8[it][1], 0.f); o8[it][2] = fmaxf(o8[it][2], 0.f); o8[it][3] = fmaxf(o8[it][3], 0.f); }
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int r = it * 4 + rr;
      if (r < nvalid) {
        const long long row = row0 + r;
        float* o = o8[it];
        if (ep.res) {
          if (ep.res_f32 || sizeof(T) == 4) {
            const float4 q = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ep.res) + row * ep.ldres + c0 + cq);
            o[0] += q.x; o[1] += q.y; o[2] += q.z; o[3] += q.w;
          } else {
            const bf16* q = reinterpret_cast<const bf16*>(ep.res) + row * ep.ldres + c0 + cq;
            const uint2 u = *reinterpret_cast<const uint2*>(q);
            const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
            const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
            o[0] += a.x; o[1] += a.y; o[2] += b.x; o[3] += b.y;
          }
        }
        const long long off = row * ep.ldo + c0 + cq;
        const bool f32out = ep.out_f32 == 1 || (ep.out_f32 == 0 && sizeof(T) == 4);
        if (f32out) *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out) + off) = make_float4(o[0], o[1], o[2], o[3]);
        else if (ep.out_f32 == 3) {
          uint2 u;
          *reinterpret_cast<__half2*>(&u.x) = __floats2half2_rn(o[0], o[1]);
          *reinterpret_cast<__half2*>(&u.y) = __floats2half2_rn(o[2], o[3]);
          *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(ep.out) + off) = u;
        } else {
          uint2 u;
          *reinterpret_cast<__nv_bfloat162*>(&u.x) = __floats2bfloat162_rn(o[0], o[1]);
          *reinterpret_cast<__nv_bfloat162*>(&u.y) = __floats2bfloat162_rn(o[2], o[3]);
          *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(ep.out) + off) = u;
        }
      }
    }
    __syncwarp();
  }
}

// Per-channel parameters of the conv epilogue; the tcgen05 kernel stages them in shared memory once per CTA,
// the fp32-mode row kernel points them at global memory.
struct EpiCtx {
  const float* bias;
  const float* ln_g;
  const float* ln_b;
  // the tcgen05 kernels stage bias / ln_g / ln_b (and gb) in shared memory: read them with ld.shared.  Through a generic
  // pointer every one of these warp-uniform 16-byte reads (128 per row) is an LD.E.128 that costs 2.4 LSU wavefronts instead
  // of one broadcast -- 55 M of the kernel's wavefronts with the LSU data pipe at 80 % (ncu, round 2)
  bool params_smem = false;
  // FiLM folded into the LayerNorm affine, staged per tile by the epilogue warpgroup (tcgen05 kernel only):
  // gb[f][0..127] = g*(scale+1), gb[f][128..255] = b*(scale+1)+shift for the fields n_first+f, f in {0,1}
  const float* gb;
  int n_first;
  // fp32 residual rows delivered by TMA (conv_halo_kernel): the warp owns two [32 rows][128 B] SWIZZLE_128B buffers and
  // a pair of mbarriers; chunk g of the warp's running sequence (4 per tile) lands in buffer g & 1, parity (g >> 1) & 1.
  // A row-per-thread LDG.128 of a 512-byte-stride residual costs ~36 L1 wavefronts per warp instruction (ncu), which made
  // the residual variants LSU-bound; the TMA path leaves only conflict-free 128-bit shared loads on the LSU.
  const CUtensorMap* res_map = nullptr;
  uint8_t* res_buf = nullptr;
  uint64_t* res_bar = nullptr;
  uint32_t res_g0 = 0;             // running chunk index of this tile's chunk 0
  long long res_row0 = 0;          // row of lane 0 in this tile
  long long res_next_row0 = -1;    // row of lane 0 in the CTA's next tile, -1 = none
  // fp32 copy of the output (out2) through the SAME buffers: after the residual is added, the finished [32 rows][32 columns]
  // block goes back into the chunk's buffer and leaves as one TMA tensor store; the refill of the buffer waits for the store
  // to have read it.  16 of a row's 24 epilogue store instructions disappear from the LSU, which bounded these launches.
  const CUtensorMap* out2_map = nullptr;
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(m), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ float4 ldp4(const EpiCtx& cx, const float* p) {
  if (cx.params_smem) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)));
    return v;
  }
  return *reinterpret_cast<const float4*>(p);
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// residual row: issued before the accumulator is ready so the DRAM latency hides behind the MMAs
template <typename T>
__device__ __forceinline__ void epi_conv_ln_prefetch(const EpiParams& ep, long long row, bool ok) {
  if (!ep.res || !ok || row >= ep.pg.pixels()) return;
  const char* r = reinterpret_cast<const char*>(ep.res) + row * ep.ldres * (ep.res_f32 ? 4 : (long long)sizeof(T));
  const int bytes = 128 * (ep.res_f32 ? 4 : (int)sizeof(T));
  for (int o = 0; o < bytes; o += 128) prefetch_l2(r + o);
}

// Requires the whole channel row in one tile: n0 == 0, C == 128.
template <typename T, bool TRAIN, class Loader>
__device__ __forceinline__ void epi_conv_ln(const EpiParams& ep, const EpiCtx& cx, long long row, bool ok, int n0, Loader& ld) {
  (void)n0;
  constexpr int C = 128;
  float v[32];
  int n, h, w;
  const bool in_buf = ok && row < ep.pg.pixels();
  const bool valid = ep.pg.decode(row, n, h, w) && in_buf;
  // pass 1: shifted one-pass statistics of x = acc + bias (shift = first element, so E[d^2]-E[d]^2 does not cancel)
  float s1 = 0.f, s2 = 0.f, x0 = 0.f;
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    ld.load(ch, v);
    if (ch == 0) x0 = v[0] + ldp4(cx, cx.bias).x;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b4 = ldp4(cx, cx.bias + ch * 32 + j);
      const float d0 = v[j] + b4.x - x0, d1 = v[j + 1] + b4.y - x0, d2 = v[j + 2] + b4.z - x0, d3 = v[j + 3] + b4.w - x0;
      s1 += (d0 + d1) + (d2 + d3);
      s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
    }
  }
  const float md = s1 * (1.0f / C);
  const float mean = x0 + md;
  const float var = fmaxf(s2 * (1.0f / C) - md * md, 0.f);             // biased variance
  const float rstd = rsqrtf(fmaxf(var, ep.ln_eps));                    // var.clamp(min=eps).rsqrt()  (metnet3.py:104)
  // affine = LayerNorm (g, b) with the per-field FiLM (scale+1, shift) folded in when staged; else applied explicitly
  const float* film = (ep.film && valid && !cx.gb) ? ep.film + (long long)n * 2 * C : nullptr;
  const float* pg_ = cx.ln_g;
  const float* pb_ = cx.ln_b;
  if (cx.gb) { const int f = (valid && n > cx.n_first) ? 1 : 0; pg_ = cx.gb + f * 256; pb_ = pg_ + 128; }
  T* o = ep.out ? reinterpret_cast<T*>(ep.out) + row * ep.ldo : nullptr;
  float* o2 = ep.out2 ? ep.out2 + row * ep.ldo : nullptr;
  const T* r = (ep.res && !ep.res_f32 && valid) ? reinterpret_cast<const T*>(ep.res) + row * ep.ldres : nullptr;
  const bool rtma = cx.res_map != nullptr;
  const bool o2tma = rtma && cx.out2_map != nullptr && ep.out2 != nullptr;      // warp-uniform
  const int lane_ = threadIdx.x & 31;
  const float* rf = (ep.res && ep.res_f32 && valid && !rtma) ? reinterpret_cast<const float*>(ep.res) + row * ep.ldres : nullptr;
  float head = 0.f;
  T* xo = (TRAIN && ep.xhat) ? reinterpret_cast<T*>(ep.xhat) + row * ep.ldo : nullptr;
  if (TRAIN && in_buf) {
    if (ep.rstd_out) ep.rstd_out[row] = valid ? rstd : 0.f;
  }
  // pass 2: normalise, FiLM, ReLU, residual, store (zeros at pad positions); the residual of chunk ch+1 is in
  // flight while chunk ch is processed
  float rr[32];
  if (rf) {
#pragma unroll
    for (int j = 0; j < 32; j += 8) ld8(rf + j, rr + j);
  } else if (r) {
#pragma unroll
    for (int j = 0; j < 32; j += 8) ld8(r + j, rr + j);
  }
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    ld.load(ch, v);
    if (rtma) {                                              // warp-uniform
      const uint32_t g = cx.res_g0 + ch;
      uint8_t* buf = cx.res_buf + (g & 1) * 4096;
      uint64_t* bar = cx.res_bar + (g & 1);
      mbar_wait(bar, (g >> 1) & 1);
      const uint8_t* p = buf + lane_ * 128;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 q4 = *reinterpret_cast<const float4*>(p + ((j ^ (lane_ & 7)) << 4));
        rr[4 * j] = q4.x; rr[4 * j + 1] = q4.y; rr[4 * j + 2] = q4.z; rr[4 * j + 3] = q4.w;
      }
      __syncwarp();
      if (lane_ == 0 && !o2tma) {                            // refill the buffer with chunk g + 2
        const long long r0 = ch < 2 ? cx.res_row0 : cx.res_next_row0;
        if (r0 >= 0) {
          fence_proxy_async_smem();
          mbar_arrive_expect_tx(bar, 4096);
          tma_load_2d(buf, cx.res_map, bar, ((ch + 2) & 3) * 32, (int)r0);
        }
      }
    }
    if (in_buf) {
    unsigned mbits = 0u;
    float xh[TRAIN ? 32 : 1];
    if (valid) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const int c = ch * 32 + j;
        const float4 b4 = ldp4(cx, cx.bias + c), g4 = ldp4(cx, pg_ + c), e4 = ldp4(cx, pb_ + c);
        float y0 = fmaf((v[j] + b4.x - mean) * rstd, g4.x, e4.x), y1 = fmaf((v[j + 1] + b4.y - mean) * rstd, g4.y, e4.y);
        float y2 = fmaf((v[j + 2] + b4.z - mean) * rstd, g4.z, e4.z), y3 = fmaf((v[j + 3] + b4.w - mean) * rstd, g4.w, e4.w);
        if (film) {
          const float4 sc = __ldg(reinterpret_cast<const float4*>(film + c)), sh = __ldg(reinterpret_cast<const float4*>(film + C + c));
          y0 = fmaf(y0, sc.x + 1.0f, sh.x); y1 = fmaf(y1, sc.y + 1.0f, sh.y);
          y2 = fmaf(y2, sc.z + 1.0f, sh.z); y3 = fmaf(y3, sc.w + 1.0f, sh.w);
        }
        if (TRAIN) {
          mbits |= (y0 > 0.f ? 1u : 0u) << j; mbits |= (y1 > 0.f ? 1u : 0u) << (j + 1);
          mbits |= (y2 > 0.f ? 1u : 0u) << (j + 2); mbits |= (y3 > 0.f ? 1u : 0u) << (j + 3);
          xh[j] = (v[j] + b4.x - mean) * rstd; xh[j + 1] = (v[j + 1] + b4.y - mean) * rstd;
          xh[j + 2] = (v[j + 2] + b4.z - mean) * rstd; xh[j + 3] = (v[j + 3] + b4.w - mean) * rstd;
        }
        v[j] = fmaxf(y0, 0.f); v[j + 1] = fmaxf(y1, 0.f); v[j + 2] = fmaxf(y2, 0.f); v[j + 3] = fmaxf(y3, 0.f);
      }
      if (TRAIN && xo) {
#pragma unroll
        for (int j = 0; j < 32; j += 16) st16_256(xo + ch * 32 + j, xh + j);
      }
      if (rf || r || rtma) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += rr[j];
        if (ch < 3) {
          if (rf) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) ld8(rf + (ch + 1) * 32 + j, rr + j);
          } else if (r) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) ld8(r + (ch + 1) * 32 + j, rr + j);
          }
        }
      }
      if (ep.head_w) {
#pragma unroll
        for (int j = 0; j < 32; ++j) head = fmaf(v[j], __ldg(ep.head_w + ch * 32 + j), head);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = 0.f;
      if (TRAIN && xo) {
#pragma unroll
        for (int j = 0; j < 32; j += 16) st16_256(xo + ch * 32 + j, v + j);
      }
    }
    if (TRAIN && ep.relu_mask) ep.relu_mask[row * 4 + ch] = mbits;
    if (o) {
#pragma unroll
      for (int j = 0; j < 32; j += 16) st16_256(o + ch * 32 + j, v + j);
    }
    if (o2 && !o2tma) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) st8_256(o2 + ch * 32 + j, v + j);
    }
    }                                                        // in_buf
    if (o2tma) {
      const uint32_t g = cx.res_g0 + ch;
      uint8_t* buf = cx.res_buf + (g & 1) * 4096;
      if (in_buf) {
        uint8_t* p = buf + lane_ * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<float4*>(p + ((j ^ (lane_ & 7)) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane_ == 0) {
        tma_store_2d(cx.out2_map, buf, ch * 32, (int)cx.res_row0);      // rows beyond the tensor are clipped by the map
        bulk_commit_group();
        const long long r0 = ch < 2 ? cx.res_row0 : cx.res_next_row0;
        bulk_wait_read_all();                                           // the store has read the buffer: it may be refilled
        if (r0 >= 0) {
          uint64_t* bar = cx.res_bar + (g & 1);
          mbar_arrive_expect_tx(bar, 4096);
          tma_load_2d(buf, cx.res_map, bar, ((ch + 2) & 3) * 32, (int)r0);
        }
      }
      __syncwarp();
    }
  }
  if (ep.head_w && valid) {
    const int hh = h - ep.head_pt, ww = w - ep.head_pl;
    if (hh >= 0 && hh < ep.head_H && ww >= 0 && ww < ep.head_W)
      ep.head_out[((long long)n * ep.head_H + hh) * ep.head_W + ww] = (head + ep.head_b) * ep.head_std + ep.head_mean;
  }
}

template <typename T, class Loader>
__device__ __forceinline__ void epi_attn_out(const EpiParams& ep, long long row, bool ok, int n0, Loader& ld) {
  const int C = ep.n_total;
  const long long wdx = row / ep.S;
  const int tok = (int)(row - wdx * ep.S);
  const int n = (int)(wdx / ep.nwin);
  const int wi = (int)(wdx - (long long)n * ep.nwin);
  const T* rsrc = nullptr; T* dst = nullptr; const float* rreg = nullptr; float* dreg = nullptr;
  if (ok) {
    if (tok < ep.R) {
      if (ep.reg_out) {
        rreg = ep.reg_in + (ep.reg_in_per_field ? (long long)n * ep.R * C : 0) + (long long)tok * C;
        dreg = ep.reg_out + (wdx * ep.R + tok) * C;
      }
    } else {
      AttnGeom g;
      g.Hl = ep.Hl; g.Wl = ep.Wl; g.win = ep.win; g.X = ep.X; g.Y = ep.Y; g.grid_mode = ep.grid_mode;
      const long long pix = (long long)n * ep.Hl * ep.Wl + attn_token_pixel(g, wi, tok - ep.R);     // maxvit.py:298 / :322
      rsrc = reinterpret_cast<const T*>(ep.x_in) + pix * C;
      dst = reinterpret_cast<T*>(ep.out) + pix * C;
    }
  }
  float v[32];
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    ld.load(ch, v);
    const int c0 = n0 + ch * 32;
    if (c0 >= C) continue;
    if (ep.drop_thresh && ok) {                              // nn.Dropout after to_out, before the residual (maxvit.py:151, 310)
      const uint32_t rid = drop_row(wdx, tok, drop_slots(ep.S));       // 128 slots per window when S > 64 (vg_rng.cuh)
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const uint32_t hsh = drop_hash(ep.drop_seed, rid, drop_group_out(ep.drop_salt, (c0 + j) >> 2));
#pragma unroll
        for (int k = 0; k < 4; ++k) v[j + k] *= (int)((hsh >> (8 * k)) & 255u) >= ep.drop_thresh ? ep.drop_scale : 0.f;
      }
    }
    if (dst) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) { float t[8]; ld8(rsrc + c0 + j, t);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[j + i] += t[i];
        st8(dst + c0 + j, v + j); }
    } else if (dreg) {
#pragma unroll
      for (int j = 0; j < 32; ++j) dreg[c0 + j] = v[j] + __ldg(rreg + c0 + j);
    }
  }
}

template <typename T, class Loader>
__device__ __forceinline__ void epi_convt(const EpiParams& ep, long long row, bool ok, int n0, Loader& ld) {
  const int C = ep.n_total / 4;
  const int tap = n0 / C, cbase = n0 - tap * C;
  const int lo = ep.Hl * ep.Wl;
  const int n = (int)(row / lo);
  const int p = (int)(row - (long long)n * lo);
  const int i = p / ep.Wl, j0 = p - i * ep.Wl;
  const long long o = ep.pg.q(n, 2 * i + (tap >> 1), 2 * j0 + (tap & 1)) * ep.ldo + cbase;
  float v[32];
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    ld.load(ch, v);
    if (!ok || cbase + ch * 32 >= C) continue;
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] += __ldg(ep.bias + cbase + ch * 32 + j);
#pragma unroll
    for (int j = 0; j < 32; j += 8) st8_out<T>(ep, o + ch * 32 + j, v + j);
    if (ep.out2) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) st8(ep.out2 + o + ch * 32 + j, v + j);
    }
  }
}

// EPI_CONVT for the tcgen05 kernel with the same shared-memory transposition as epi_store_coalesced: every output pixel's
// 128 channels of one tap are contiguous in the PG buffer, so a warp instruction writes four full row segments.
template <typename T, class Loader>
__device__ __forceinline__ void epi_convt_coalesced(const EpiParams& ep, long long row, bool ok, int n0, Loader& ld, float* stg, int lane) {
  constexpr int LDS_ = 36;
  const int C = ep.n_total / 4;
  const int tap = n0 / C, cbase = n0 - tap * C;
  const int lo = ep.Hl * ep.Wl;
  long long o = -1;                                        // element offset of this lane's row in the output (or -1)
  if (ok) {
    const int n = (int)(row / lo);
    const int p = (int)(row - (long long)n * lo);
    const int i = p / ep.Wl, j0 = p - i * ep.Wl;
    o = ep.pg.q(n, 2 * i + (tap >> 1), 2 * j0 + (tap & 1)) * ep.ldo + cbase;
  }
  const int rr = lane >> 3, cq = (lane & 7) * 4;
  float v[32];
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    const bool live = cbase + ch * 32 < C;                 // warp-uniform
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) b4 = __ldg(reinterpret_cast<const float4*>(ep.bias + cbase + ch * 32 + cq));
    ld.load(ch, v);
    if (!live) continue;
#pragma unroll
    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(stg + lane * LDS_ + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int r = it * 4 + rr;
      const long long orow = __shfl_sync(0xffffffffu, o, r);
      if (orow >= 0) {
        const float4 a4 = *reinterpret_cast<const float4*>(stg + r * LDS_ + cq);
        const float4 y = make_float4(a4.x + b4.x, a4.y + b4.y, a4.z + b4.z, a4.w + b4.w);
        const long long off = orow + ch * 32 + cq;
        const bool f32out = ep.out_f32 == 1 || (ep.out_f32 == 0 && sizeof(T) == 4);
        if (f32out) *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out) + off) = y;
        else {
          uint2 u;
          *reinterpret_cast<__nv_bfloat162*>(&u.x) = __floats2bfloat162_rn(y.x, y.y);
          *reinterpret_cast<__nv_bfloat162*>(&u.y) = __floats2bfloat162_rn(y.z, y.w);
          *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(ep.out) + off) = u;
        }
        if (ep.out2) *reinterpret_cast<float4*>(ep.out2 + off) = y;
      }
    }
    __syncwarp();
  }
}

template <int KIND, typename T, class Loader>
__device__ __forceinline__ void run_epilogue(const EpiParams& ep, const EpiCtx& cx, long long row, bool ok, int n0, Loader& ld) {
  if constexpr (KIND == EPI_STORE) epi_store<T>(ep, row, ok, n0, ld);
  else if constexpr (KIND == EPI_CONV_LN) epi_conv_ln<T, false>(ep, cx, row, ok, n0, ld);
  else if constexpr (KIND == EPI_CONV_LN_TRAIN) epi_conv_ln<T, true>(ep, cx, row, ok, n0, ld);
  else if constexpr (KIND == EPI_ATTN_OUT) epi_attn_out<T>(ep, row, ok, n0, ld);
  else epi_convt<T>(ep, row, ok, n0, ld);
}

}  // namespace vg
