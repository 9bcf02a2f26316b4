// Shifted-row GEMM for sm_100a: D[m][n] = sum_tap sum_c A[m + shift(tap)][c] * B[n][tap*Ca + c]
//
// One kernel serves every tensor-core contraction on the path: 3x3 convolutions over the padded-grid layout
// (9 taps = 9 row shifts of the same 2-D A tensor, see vg_common.cuh), 1x1 convolutions / linear layers
// (1 tap) and ConvTranspose2d-as-GEMM.  bf16 mode: persistent warp-specialised tcgen05 kernel, operands
// streamed by TMA into a 128B-swizzled multi-stage ring, fp32 accumulators double-buffered in TMEM, row-wise
// fused epilogues (vg_epilogue.cuh).  fp32 mode: SIMT FFMA kernel + the same epilogues run row-wise.
#include <stdio.h>
#include <stdlib.h>

#include "vg_epilogue.cuh"
#include "vg_host.h"

namespace vg {

struct GemmShape {
  long long M;              // valid output rows (all batches)
  int num_m_tiles, num_n_tiles;
  int k_blocks, cblocks;    // 128-byte-wide K blocks (64 bf16 / 32 tf32 elements): total and per tap
  int tap_shift[9];
  int tiles_per_batch;      // m-tiles per batch (== num_m_tiles when not batched)
  long long rows_per_batch; // A / output rows per batch (== M when not batched)
  int b_rows_per_batch;     // B row offset per batch (per-field weights)
  int f16;                  // 16-bit operands are fp16, not bf16 (kind::f16 with the fp16 operand format)
};

constexpr int BM = 256, BN = 128, BK = 64, STAGES = 4;        // tile = 256 rows (two M=128 MMAs sharing one B stage) x 128 cols
constexpr int A_BYTES = BM * BK * 2;                          // 32 KiB: rows 0..127 then rows 128..255, 128 B per row
constexpr int B_BYTES = BN * BK * 2;                          // 16 KiB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;                // 48 KiB
constexpr int PARAM_FLOATS = 3 * 128 + 2 * 2 * 256;           // conv epilogue: bias | ln_g | ln_b | per-WG folded FiLM affine [2 fields][256]
constexpr int TC_SMEM_BYTES = STAGES * STAGE_BYTES + PARAM_FLOATS * 4 + 1024 /*align slack*/ + 256 /*barriers*/;
// EPI_STORE kernels are epilogue / HBM-bound: 3 stages, and the freed space holds the 8 per-warp [32][33] fp32 tiles the
// coalesced store epilogue transposes through ([32][36] each)
constexpr int STORE_STAGES = 3;
constexpr int STORE_STG_FLOATS = 8 * 32 * 36;
constexpr int TC_SMEM_BYTES_STORE = STORE_STAGES * STAGE_BYTES + STORE_STG_FLOATS * 4 + 1024 + 256;
// EPI_STORE runs SIXTEEN epilogue warps (640 threads): four per TMEM lane quadrant, two column chunks of the tile each.  With eight,
// two warps per scheduler ran the whole epilogue (fixed-latency dependency stalls, 45 % issue utilisation in ncu) while the
// tensor pipe idled: the 1x1 expand + BN + GELU GEMM took 0.97 ms against 0.32 ms of GELU issue time and 0.27 ms of HBM time.
constexpr int STORE_EPI_WARPS = 16;
constexpr int TC_THREADS_STORE = 128 + 32 * STORE_EPI_WARPS;
constexpr int TC_SMEM_BYTES_STORE16 = STORE_STAGES * STAGE_BYTES + 2 * STORE_STG_FLOATS * 4 + 1024 + 256;
constexpr int TMEM_COLS = 512;                                // 2 tiles in flight x 2 row halves x 128 fp32 columns
constexpr int TC_THREADS = 384;                               // warp 0 TMA, 1 MMA, 2 TMEM alloc, 3 idle, 4-7 / 8-11 epilogue WGs

struct TmemLoader {
  uint32_t taddr;
  __device__ __forceinline__ void load(int chunk, float* v) {
    tmem_ld32(taddr + chunk * 32, v);
    tmem_wait_ld();
  }
};

// TF32 = 0: bf16 operands (64 per 128-byte K block, UMMA K = 16); TF32 = 1: fp32 operands read as tf32 (32 per K
// block, UMMA K = 8).  The smem tiles are [rows][128 bytes] either way, so the pipeline is identical.
// Epilogue warpgroup e (warps 4+4e .. 7+4e) owns rows [128e, 128e+128) of every tile.
template <int KIND, int TF32>
__global__ void __launch_bounds__(KIND == EPI_STORE ? TC_THREADS_STORE : TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
               const GemmShape gs, const EpiParams ep) {
  constexpr bool STAGED = KIND == EPI_STORE || KIND == EPI_CONVT;      // epilogues that transpose through shared memory
  constexpr int STAGES = STAGED ? STORE_STAGES : vg::STAGES;
  constexpr int EPI_WARPS = KIND == EPI_STORE ? STORE_EPI_WARPS : 8;
  constexpr int PARAM_BYTES = STAGED ? (EPI_WARPS / 8) * STORE_STG_FLOATS * 4 : PARAM_FLOATS * 4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* sparam = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + PARAM_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapB); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull + s, 1); mbar_init(tempty + s, EPI_WARPS); }
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  if (KIND == EPI_CONV_LN || KIND == EPI_CONV_LN_TRAIN) {
    for (int i = threadIdx.x; i < 128; i += TC_THREADS) {
      sparam[i] = ep.bias[i]; sparam[128 + i] = ep.ln_g[i]; sparam[256 + i] = ep.ln_b[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform: lets the MMA issue use uniform registers (no per-MMA elect/broadcast loop)

  const int total_tiles = gs.num_m_tiles * gs.num_n_tiles;
  constexpr int BKE = TF32 ? 32 : 64;                        // elements per K block

  if (warp == 0) {
    if (lane == 0) {                                         // ===== TMA producer =====
      int stage = 0; uint32_t phase = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int m_tile = t / gs.num_n_tiles, n_tile = t - m_tile * gs.num_n_tiles;
        const int batch = m_tile / gs.tiles_per_batch, mt = m_tile - batch * gs.tiles_per_batch;
        const long long row0 = (long long)batch * gs.rows_per_batch + (long long)mt * BM;
        const int brow0 = batch * gs.b_rows_per_batch + n_tile * BN;
        for (int kb = 0; kb < gs.k_blocks; ++kb) {
          const int tap = kb / gs.cblocks, cb = kb - tap * gs.cblocks;
          mbar_wait(empty + stage, phase ^ 1);
          mbar_arrive_expect_tx(full + stage, STAGE_BYTES);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          tma_load_2d(sa, &mapA, full + stage, cb * BKE, (int)(row0 + gs.tap_shift[tap]));      // 256-row box
          tma_load_2d(sa + A_BYTES, &mapB, full + stage, kb * BKE, brow0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {                                                        // ===== MMA issuer: the warp runs converged, an elected lane issues (see elect_one) =====
      const uint32_t idesc = TF32 ? umma_idesc_tf32(128, BN) : (gs.f16 ? umma_idesc_f16(128, BN) : umma_idesc_bf16(128, BN));
      int stage = 0; uint32_t phase = 0; int it = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
        const int as = it & 1; const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(tempty + as, aphase ^ 1);                  // both epilogue warpgroups have drained this buffer
        tc_fence_after();
        const uint32_t d0 = tmem_base + as * 256, d1 = d0 + 128;
        for (int kb = 0; kb < gs.k_blocks; ++kb) {
          mbar_wait(full + stage, phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          if (elect_one()) {
            const uint64_t da0 = umma_desc_k128(sa), da1 = umma_desc_k128(sa + A_BYTES / 2), db = umma_desc_k128(sa + A_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k) {                    // 4 x 32 B per K block, +32 B inside the swizzle atom
              const uint32_t acc = (kb | k) ? 1u : 0u;
              if (TF32) { tc_mma_tf32(d0, da0 + 2 * k, db + 2 * k, idesc, acc); tc_mma_tf32(d1, da1 + 2 * k, db + 2 * k, idesc, acc); }
              else { tc_mma_bf16(d0, da0 + 2 * k, db + 2 * k, idesc, acc); tc_mma_bf16(d1, da1 + 2 * k, db + 2 * k, idesc, acc); }
            }
            tc_commit(empty + stage);                        // frees the smem slot when these MMAs retire
            if (kb == gs.k_blocks - 1) tc_commit(tfull + as);   // accumulators complete -> epilogue
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {                                    // ===== epilogue: 2 x 128 threads, one row each =====
    const int lg = warp & 3;                                 // TMEM lane group this warp may access
    const int e = ((warp - 4) >> 2) & 1;                     // row half of the tile
    const int ch0 = EPI_WARPS == 16 ? ((warp - 4) >> 3) * 2 : 0, ch1 = EPI_WARPS == 16 ? ch0 + 2 : 4;      // column chunks (32 each) of this warp
    EpiCtx cx;
    cx.bias = sparam; cx.ln_g = sparam + 128; cx.ln_b = sparam + 256; cx.gb = nullptr; cx.n_first = 0; cx.params_smem = true;
    float* sgb = sparam + 384 + e * 512;                     // this warpgroup's staging buffer
    const int wt = (warp & 3) * 32 + lane;                   // thread index inside the warpgroup
    int it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
      const int m_tile = t / gs.num_n_tiles, n_tile = t - m_tile * gs.num_n_tiles;
      const int batch = m_tile / gs.tiles_per_batch, mt = m_tile - batch * gs.tiles_per_batch;
      const long long lrow = (long long)mt * BM + e * 128 + lg * 32 + lane;
      const long long row = (long long)batch * gs.rows_per_batch + lrow;
      const bool ok = lrow < gs.rows_per_batch && row < gs.M;
      const int as = it & 1; const uint32_t aphase = (it >> 1) & 1;
      if (KIND == EPI_CONV_LN || KIND == EPI_CONV_LN_TRAIN) {
        if (TF32) epi_conv_ln_prefetch<float>(ep, row, ok); else epi_conv_ln_prefetch<bf16>(ep, row, ok);
        if (ep.film) {
          // fold FiLM of the (at most two) fields this warpgroup's 128 rows touch into the LayerNorm affine
          const long long r0 = (long long)batch * gs.rows_per_batch + (long long)mt * BM + e * 128;
          int nf = (int)((r0 / ep.pg.P) / ep.pg.R);
          if (nf > ep.pg.N - 1) nf = ep.pg.N - 1;
          asm volatile("bar.sync %0, 128;" ::"r"(2 + e) : "memory");          // previous tile's readers are done
          for (int i = wt; i < 256; i += 128) {
            const int f = i >> 7, c = i & 127;
            const int n2 = (nf + f < ep.pg.N) ? nf + f : nf;
            const float sc = ep.film[(long long)n2 * 256 + c] + 1.0f, sh = ep.film[(long long)n2 * 256 + 128 + c];
            sgb[f * 256 + c] = sparam[128 + c] * sc;
            sgb[f * 256 + 128 + c] = fmaf(sparam[256 + c], sc, sh);
          }
          asm volatile("bar.sync %0, 128;" ::"r"(2 + e) : "memory");
          cx.gb = sgb; cx.n_first = nf;
        }
      }
      mbar_wait(tfull + as, aphase);
      tc_fence_after();
      TmemLoader ld{tmem_base + as * 256 + e * 128 + ((uint32_t)(lg * 32) << 16)};
      if constexpr (KIND == EPI_STORE) {
        // rows of this warp are consecutive: lane 0 holds lrow - lane
        const long long lrow0 = lrow - lane;
        long long nv = gs.rows_per_batch - lrow0;
        const long long nv2 = gs.M - ((long long)batch * gs.rows_per_batch + lrow0);
        if (nv2 < nv) nv = nv2;
        const int nvalid = nv < 0 ? 0 : (nv > 32 ? 32 : (int)nv);
        float* stg = sparam + (warp - 4) * (32 * 36);
        // the plain 16-bit store has no arithmetic to overlap: eight warps saturate the store path, the upper eight only keep the
        // accumulator hand-shake (measured: 0.87 ms with eight, 0.95 ms with sixteen for the QKV re-materialisation)
        if (TF32) {
          if (epi_store_rows16_ok<float>(ep)) { if (warp < 12) epi_store_rows16(ep, row, ok, n_tile * BN, ld, 0, 4); }
          else epi_store_coalesced<float>(ep, row - lane, nvalid, n_tile * BN, ld, stg, lane, ch0, ch1);
        } else {
          if (epi_store_rows16_ok<bf16>(ep)) { if (warp < 12) epi_store_rows16(ep, row, ok, n_tile * BN, ld, 0, 4); }
          else epi_store_coalesced<bf16>(ep, row - lane, nvalid, n_tile * BN, ld, stg, lane, ch0, ch1);
        }
      } else if constexpr (KIND == EPI_CONVT) {
        float* stg = sparam + (warp - 4) * (32 * 36);
        if (TF32) epi_convt_coalesced<float>(ep, row, ok, n_tile * BN, ld, stg, lane);
        else epi_convt_coalesced<bf16>(ep, row, ok, n_tile * BN, ld, stg, lane);
      } else {
        if (TF32) run_epilogue<KIND, float>(ep, cx, row, ok, n_tile * BN, ld);
        else run_epilogue<KIND, bf16>(ep, cx, row, ok, n_tile * BN, ld);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty + as);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// 3x3 convolution with halo reuse (bf16, Cin = Cout = 128, PG layout).
//
// The generic kernel above re-reads the A operand from L2 once per tap (9x).  Here a tile of 256 output pixels loads
// its input rows ONCE, with the halo of P+1 rows on each side, as two [HR rows x 128 B] channel-block tiles
// (SWIZZLE_128B, written by TMA); tap (dy,dx) is then the same smem tile addressed through a UMMA descriptor whose
// start address is shifted by (P+1 + dy*P + dx) rows (128 B each; the descriptor's base-offset field stays 0: the 128B
// swizzle is applied to absolute shared-memory address bits, so a row-shifted start into a 1024-B-aligned tile needs no
// phase correction -- measured on B200).  Only the weights (16 KiB per tap and channel block) stream through a ring.
// K order: channel block 0 taps 0..8, then channel block 1 taps 0..8, so each A half-buffer is reloaded for the next
// tile while the other half is being consumed.  L2->SM traffic per 256-pixel tile: 100 KiB (A) + 288 KiB (B)
// instead of 576 + 288 KiB.
// ------------------------------------------------------------------------------------------------
constexpr int HALO_MAX_ROWS = 416;                            // HR <= 416 (two TMA boxes of <= 208 rows)
constexpr int HB_STAGES = 3;                                  // weight ring
constexpr int HALO_RES_BYTES = 8 * 2 * 4096;                  // per epilogue warp: two [32 rows][128 B] fp32 residual chunks (TMA)
constexpr int HALO_A_BYTES = HALO_MAX_ROWS * 128;             // per channel block
constexpr int HALO_SMEM_BYTES = 2 * HALO_A_BYTES + HB_STAGES * B_BYTES + HALO_RES_BYTES + PARAM_FLOATS * 4 + 1024 + 256;

struct HaloShape {
  long long M;          // flat pixels (rows of the [q][128] matrices)
  int num_tiles;        // 256-pixel tiles
  int P;                // row pitch (pixels)
  int HR;               // halo rows loaded per tile (multiple of 16)
  int res_tma;          // the fp32 residual arrives through mapR (else: per-thread global loads)
  int flip;             // data gradient: tap t of the weights is applied with the input shift of tap 8 - t (the negated shift)
  int out2_tma;         // the fp32 copy of the output leaves through mapO (TMA tensor stores from the residual buffers)
};

__device__ __forceinline__ uint64_t umma_desc_k128_shift(uint32_t tile_addr, int row) {
  const uint32_t a = tile_addr + (uint32_t)row * 128u;
  return (uint64_t)((a & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

// MODE 0: conv + ChanLN / FiLM / ReLU / residual epilogue; 1: the same, saving xhat / rstd / mask for backward; 2: plain fp32 store
// (+ fp32 residual) -- the DATA GRADIENT of the convolution runs through the same halo pipeline with the tap order flipped
template <int MODE>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                 const __grid_constant__ CUtensorMap mapR, const __grid_constant__ CUtensorMap mapO, const HaloShape hs, const EpiParams ep) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem + 2 * HALO_A_BYTES;
  uint8_t* sres = sB + HB_STAGES * B_BYTES;
  float* sparam = reinterpret_cast<float*>(sres + HALO_RES_BYTES);
  uint64_t* full = reinterpret_cast<uint64_t*>(sres + HALO_RES_BYTES + PARAM_FLOATS * 4);
  uint64_t* empty = full + HB_STAGES;
  uint64_t* a_full = empty + HB_STAGES;    // [2]
  uint64_t* a_free = a_full + 2;           // [2]
  uint64_t* tfull = a_free + 2;            // [2]
  uint64_t* tempty = tfull + 2;            // [2]
  uint64_t* res_full = tempty + 2;         // [8 epilogue warps][2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 16);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapB); if (hs.res_tma) tma_prefetch_desc(&mapR); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < HB_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(a_full + s, 1); mbar_init(a_free + s, 1); mbar_init(tfull + s, 1); mbar_init(tempty + s, 8); }
    for (int s = 0; s < 16; ++s) mbar_init(res_full + s, 1);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  if (MODE != 2) {
    for (int i = threadIdx.x; i < 128; i += TC_THREADS) {
      sparam[i] = ep.bias[i]; sparam[128 + i] = ep.ln_g[i]; sparam[256 + i] = ep.ln_b[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform: lets the MMA issue use uniform registers (no per-MMA elect/broadcast loop)
  const int halo = hs.P + 1;                                 // rows in front of the tile's first output pixel
  if (warp == 0) {
    if (lane == 0) {                                         // ===== TMA producer =====
      int stage = 0; uint32_t phase = 0; uint32_t it = 0;
      const int half_rows = hs.HR / 2;
      for (int t = blockIdx.x; t < hs.num_tiles; t += gridDim.x, ++it) {
        const long long q0 = (long long)t * BM;
        for (int cb = 0; cb < 2; ++cb) {
          mbar_wait(a_free + cb, (it & 1) ^ 1);              // previous tile's taps on this half have retired
          mbar_arrive_expect_tx(a_full + cb, hs.HR * 128);
          uint8_t* sa = smem + cb * HALO_A_BYTES;
          tma_load_2d(sa, &mapA, a_full + cb, cb * 64, (int)(q0 - halo));
          tma_load_2d(sa + half_rows * 128, &mapA, a_full + cb, cb * 64, (int)(q0 - halo + half_rows));
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(empty + stage, phase ^ 1);
            mbar_arrive_expect_tx(full + stage, B_BYTES);
            tma_load_2d(sB + stage * B_BYTES, &mapB, full + stage, (hs.flip ? 8 - tap : tap) * 128 + cb * 64, 0);
            if (++stage == HB_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    {                                                        // ===== MMA issuer: the warp runs converged, an elected lane issues (see elect_one) =====
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
      int stage = 0; uint32_t phase = 0; uint32_t it = 0;
      for (int t = blockIdx.x; t < hs.num_tiles; t += gridDim.x, ++it) {
        const int as = it & 1; const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(tempty + as, aphase ^ 1);
        tc_fence_after();
        const uint32_t d0 = tmem_base + as * 256, d1 = d0 + 128;
        for (int cb = 0; cb < 2; ++cb) {
          mbar_wait(a_full + cb, it & 1);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + cb * HALO_A_BYTES);
          for (int tap = 0; tap < 9; ++tap) {
            const int r0 = halo + (tap / 3 - 1) * hs.P + (tap % 3 - 1);       // first input row of this tap
            mbar_wait(full + stage, phase);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t da0 = umma_desc_k128_shift(sa, r0), da1 = umma_desc_k128_shift(sa, r0 + 128);
              const uint64_t db = umma_desc_k128(smem_u32(sB + stage * B_BYTES));
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t acc = (cb | tap | k) ? 1u : 0u;
                tc_mma_bf16(d0, da0 + 2 * k, db + 2 * k, idesc, acc);
                tc_mma_bf16(d1, da1 + 2 * k, db + 2 * k, idesc, acc);
              }
              tc_commit(empty + stage);
              if (tap == 8) {
                tc_commit(a_free + cb);
                if (cb == 1) tc_commit(tfull + as);
              }
            }
            __syncwarp();
            if (++stage == HB_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp >= 4) {                                    // ===== epilogue: 2 x 128 threads, one pixel row each =====
    const int lg = warp & 3;
    const int e = (warp - 4) >> 2;
    EpiCtx cx;
    cx.bias = sparam; cx.ln_g = sparam + 128; cx.ln_b = sparam + 256; cx.gb = nullptr; cx.n_first = 0; cx.params_smem = true;
    if (hs.res_tma) {
      cx.res_map = &mapR; cx.res_buf = sres + (warp - 4) * 8192; cx.res_bar = res_full + (warp - 4) * 2;
      if (hs.out2_tma) cx.out2_map = &mapO;
      if (lane == 0 && (int)blockIdx.x < hs.num_tiles) {     // chunks 0 and 1 of the first tile
        const int r0 = (int)((long long)blockIdx.x * BM + e * 128 + lg * 32);
        for (int c = 0; c < 2; ++c) {
          mbar_arrive_expect_tx(cx.res_bar + c, 4096);
          tma_load_2d(cx.res_buf + c * 4096, &mapR, cx.res_bar + c, c * 32, r0);
        }
      }
    }
    uint32_t it = 0;
    for (int t = blockIdx.x; t < hs.num_tiles; t += gridDim.x, ++it) {
      const long long row = (long long)t * BM + e * 128 + lg * 32 + lane;
      const bool ok = row < hs.M;
      const int as = it & 1; const uint32_t aphase = (it >> 1) & 1;
      if (hs.res_tma) {
        cx.res_g0 = it * 4; cx.res_row0 = row - lane;
        cx.res_next_row0 = (t + (int)gridDim.x < hs.num_tiles) ? cx.res_row0 + (long long)gridDim.x * BM : -1;
      } else if (MODE != 2) {
        epi_conv_ln_prefetch<bf16>(ep, row, ok);
      }
      mbar_wait(tfull + as, aphase);
      tc_fence_after();
      TmemLoader ld{tmem_base + as * 256 + e * 128 + ((uint32_t)(lg * 32) << 16)};
      if constexpr (MODE == 2) epi_store_f32_rows(ep, row, ok && row < hs.M, ld);
      else run_epilogue<MODE == 1 ? EPI_CONV_LN_TRAIN : EPI_CONV_LN, bf16>(ep, cx, row, ok, 0, ld);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty + as);
    }
    if (hs.out2_tma && lane == 0) bulk_wait_all();           // outstanding tensor stores have been performed before the CTA exits
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// fp32 mode: SIMT GEMM into a scratch accumulator + row-wise epilogue kernel
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gemm_simt_kernel(const float* __restrict__ A, long long rowsA, int Ca, const float* __restrict__ B, int Ktot,
                 const GemmShape gs, float* __restrict__ scratch, int Ntot) {
  __shared__ float sA[16][65], sB[16][65];
  const int batch = blockIdx.z;
  const long long lrow0 = (long long)blockIdx.x * 64;
  const int n0 = blockIdx.y * 64;
  const long long grow0 = (long long)batch * gs.rows_per_batch + lrow0;
  const float* Bb = B + (long long)batch * gs.b_rows_per_batch * Ktot;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  const int ntaps = gs.k_blocks / gs.cblocks;
  for (int tap = 0; tap < ntaps; ++tap) {
    for (int c0 = 0; c0 < Ca; c0 += 16) {
      for (int i = threadIdx.x; i < 64 * 16; i += 256) {
        const int r = i >> 4, c = i & 15;
        const long long ar = grow0 + r + gs.tap_shift[tap];
        sA[c][r] = (ar >= 0 && ar < rowsA && c0 + c < Ca) ? A[ar * Ca + c0 + c] : 0.f;
        const int bn = n0 + r;
        sB[c][r] = (bn < Ntot && c0 + c < Ca) ? Bb[(long long)bn * Ktot + tap * Ca + c0 + c] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a[i] = sA[k][ty * 4 + i]; b[i] = sB[k][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long lr = lrow0 + ty * 4 + i;
    const long long gr = grow0 + ty * 4 + i;
    if (lr >= gs.rows_per_batch || gr >= gs.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < Ntot) scratch[gr * Ntot + n] = acc[i][j];
    }
  }
}

struct ScratchLoader {
  const float* p;   // scratch + row*Ntot + n0 (null when the row is out of range)
  int ncols;        // valid columns from n0
  __device__ __forceinline__ void load(int chunk, float* v) {
#pragma unroll
    for (int j = 0; j < 32; ++j) { const int c = chunk * 32 + j; v[j] = (p && c < ncols) ? p[c] : 0.f; }
  }
};

template <int KIND>
__global__ void __launch_bounds__(128)
epilogue_rows_kernel(const float* __restrict__ scratch, int Ntot, const GemmShape gs, const EpiParams ep) {
  const long long row = (long long)blockIdx.x * 128 + threadIdx.x;
  const int n0 = blockIdx.y * BN;
  const bool ok = row < gs.M;
  ScratchLoader ld{ok ? scratch + row * Ntot + n0 : nullptr, Ntot - n0};
  EpiCtx cx;
  cx.bias = ep.bias; cx.ln_g = ep.ln_g; cx.ln_b = ep.ln_b; cx.gb = nullptr; cx.n_first = 0;
  run_epilogue<KIND, float>(ep, cx, row, ok, n0, ld);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess || !p)
      return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D tensor [outer][inner] (inner contiguous, bf16 or fp32), box (128 bytes) x box_outer, 128B swizzle, zero OOB fill
static int make_map_2d(CUtensorMap* m, bool f32, const void* ptr, long long inner, long long outer, int box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)inner * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {f32 ? 32u : 64u, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error("cuTensorMapEncodeTiled failed (%d) ptr=%p inner=%lld outer=%lld", (int)r, ptr, inner, outer);
  return 0;
}

static int num_sms() {
  static int n_sms[64] = {};
  int dev = 0; cudaGetDevice(&dev);
  int& n = n_sms[dev & 63];
  if (!n) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int KIND, int TF32>
static int launch_tc(const CUtensorMap& ma, const CUtensorMap& mb, const GemmShape& gs, const EpiParams& ep, cudaStream_t st) {
  static PerDeviceFlag attr_pd;
  bool& attr_set = attr_pd.cur();
  constexpr int SMEM = KIND == EPI_STORE ? TC_SMEM_BYTES_STORE16 : (KIND == EPI_CONVT ? TC_SMEM_BYTES_STORE : TC_SMEM_BYTES);
  constexpr int THREADS = KIND == EPI_STORE ? TC_THREADS_STORE : TC_THREADS;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<KIND, TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  const int total = gs.num_m_tiles * gs.num_n_tiles;
  const int grid = total < num_sms() ? total : num_sms();
  gemm_tc_kernel<KIND, TF32><<<grid, THREADS, SMEM, st>>>(ma, mb, gs, ep);
  return check_launch("gemm_tc_kernel");
}

template <int KIND>
static int launch_simt_epi(const float* scratch, int Ntot, const GemmShape& gs, const EpiParams& ep, cudaStream_t st) {
  dim3 grid((unsigned)((gs.M + 127) / 128), (unsigned)((Ntot + BN - 1) / BN));
  epilogue_rows_kernel<KIND><<<grid, 128, 0, st>>>(scratch, Ntot, gs, ep);
  return check_launch("epilogue_rows_kernel");
}

// bf16 3x3 conv (Cin = Cout = 128) over a PG buffer with halo reuse; returns -1 when the shape does not fit
int conv_halo_run_mp(const void* x, const void* Wt, long long M, int P, const EpiParams& ep, int mode_k, int flip, cudaStream_t st);

int conv_halo_run(const void* x, const void* Wt, const PGeom& pg, const EpiParams& ep, int train, cudaStream_t st) {
  return conv_halo_run_mp(x, Wt, pg.pixels(), pg.P, ep, train ? 1 : 0, 0, st);
}

// mode 0 / 1: forward (+ training outputs); 2: plain fp32 store (+ fp32 residual); flip: data gradient (negated tap shifts)
int conv_halo_run_mp(const void* x, const void* Wt, long long M, int P, const EpiParams& ep, int mode_k, int flip, cudaStream_t st) {
  const int train = mode_k == 1;
  const int HR = ((BM + 2 * (P + 1)) + 15) / 16 * 16;
  if (HR > HALO_MAX_ROWS) return -1;
  CUtensorMap ma, mb, mr;
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable");
  const bool res_tma = mode_k != 2 && ep.res && ep.res_f32 && ep.ldres == 128 && (reinterpret_cast<uintptr_t>(ep.res) & 15) == 0;
  if (res_tma) {
    int rc = make_map_2d(&mr, true, ep.res, 128, M, 32);
    if (rc) return rc;
  }
  {
    cuuint64_t dims[2] = {128, (cuuint64_t)M};
    cuuint64_t strides[1] = {256};
    cuuint32_t box[2] = {64u, (cuuint32_t)(HR / 2)};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = fn(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(x), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error("conv_halo: A tensor map failed (%d)", (int)r);
  }
  int rc = make_map_2d(&mb, false, Wt, 9 * 128, 128, BN);
  if (rc) return rc;
  HaloShape hs;
  hs.M = M; hs.num_tiles = (int)((hs.M + BM - 1) / BM); hs.P = P; hs.HR = HR; hs.res_tma = res_tma ? 1 : 0;
  hs.flip = flip;
  // fp32 copy through TMA stores (needs the residual buffers: fp32-residual launches only; the others store it per thread)
  CUtensorMap mo = ma;
  hs.out2_tma = 0;
  if (res_tma && ep.out2 && ep.ldo == 128 && (reinterpret_cast<uintptr_t>(ep.out2) & 15) == 0) {
    int rc2 = make_map_2d(&mo, true, ep.out2, 128, M, 32);
    if (rc2) return rc2;
    hs.out2_tma = 1;
  }
  static PerDeviceFlag attr_pd;
  bool& attr_set = attr_pd.cur();
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_halo_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, HALO_SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_halo_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, HALO_SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_halo_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, HALO_SMEM_BYTES);
    if (e != cudaSuccess) return set_error("cudaFuncSetAttribute(conv_halo): %s", cudaGetErrorString(e));
    attr_set = true;
  }
  const int grid = hs.num_tiles < num_sms() ? hs.num_tiles : num_sms();
  if (!res_tma) mr = ma;                                     // unused by the kernel
  if (mode_k == 2) conv_halo_kernel<2><<<grid, TC_THREADS, HALO_SMEM_BYTES, st>>>(ma, mb, mr, mo, hs, ep);
  else if (train) conv_halo_kernel<1><<<grid, TC_THREADS, HALO_SMEM_BYTES, st>>>(ma, mb, mr, mo, hs, ep);
  else conv_halo_kernel<0><<<grid, TC_THREADS, HALO_SMEM_BYTES, st>>>(ma, mb, mr, mo, hs, ep);
  return check_launch("conv_halo_kernel");
}

// The one host entry used by the C ABI (vg_api.cu).  dtype: 0 = bf16 (tcgen05), 1 = fp32 (SIMT FFMA),
// 2 = fp32 storage with TF32 tcgen05 MMA.
int gemm_run(int dtype, int kind, const void* A, long long rowsA, int Ca, const void* B, int Ntot, int ntaps,
             const int* tap_shift, long long M, long long rows_per_batch, int b_rows_per_batch,
             const EpiParams& ep, float* scratch, long long scratch_elems, cudaStream_t st) {
  // dtype 3: fp16 operands -- the bf16 pipeline (2-byte elements, same tensor maps) with the fp16 instruction descriptor
  const bool f16 = dtype == 3;
  if (f16) { dtype = 0; if (kind != EPI_STORE) return set_error("gemm: fp16 operands are built for the plain store epilogue"); }
  const int bke = dtype == 2 ? 32 : 64;
  if (dtype != 1 && Ca % bke) return set_error("gemm: channels (%d) must be a multiple of %d", Ca, bke);   // SIMT path: any Ca
  if (ntaps < 1 || ntaps > 9) return set_error("gemm: bad tap count %d", ntaps);
  if (M <= 0) return 0;
  GemmShape gs;
  gs.M = M; gs.f16 = f16 ? 1 : 0;
  gs.cblocks = dtype == 1 ? 1 : Ca / bke;                    // the SIMT kernel only uses k_blocks / cblocks = ntaps
  gs.k_blocks = gs.cblocks * ntaps;
  for (int i = 0; i < 9; ++i) gs.tap_shift[i] = i < ntaps ? tap_shift[i] : 0;
  const bool batched = rows_per_batch > 0 && rows_per_batch < M;
  gs.rows_per_batch = batched ? rows_per_batch : M;
  gs.b_rows_per_batch = batched ? b_rows_per_batch : 0;
  const long long nbatch = (M + gs.rows_per_batch - 1) / gs.rows_per_batch;
  gs.tiles_per_batch = (int)((gs.rows_per_batch + BM - 1) / BM);
  gs.num_m_tiles = (int)(gs.tiles_per_batch * nbatch);
  gs.num_n_tiles = (Ntot + BN - 1) / BN;
  const int Ktot = Ca * ntaps;
  if ((kind == EPI_CONV_LN || kind == EPI_CONV_LN_TRAIN) && Ntot != BN) return set_error("gemm: conv+LN epilogue needs exactly %d output channels (got %d)", BN, Ntot);

  // The data gradient of a 128 -> 128 3x3 convolution (bf16 operands, fp32 output, optional fp32 residual, tap shifts = the
  // negated -- or plain -- shifts of a row pitch P) runs through the halo-reuse kernel: 1.7x the generic shifted-row GEMM
  if (dtype == 0 && !f16 && kind == EPI_STORE && ntaps == 9 && Ca == 128 && Ntot == 128 && !batched && rowsA == M && ep.out_f32 == 1 &&
      !ep.col_scale && !ep.bias && ep.act == 0 && (!ep.res || (ep.res_f32 && ep.ldres == 128)) && ep.ldo == 128) {
    const int P = tap_shift[3] - tap_shift[0];                 // (ky) step of the shift pattern, signed
    const int sgn = P < 0 ? -1 : 1, aP = P < 0 ? -P : P;
    bool pattern = aP > 2;
    for (int t = 0; t < 9 && pattern; ++t) pattern = tap_shift[t] == sgn * ((t / 3 - 1) * aP + (t % 3 - 1));
    if (pattern) {
      const int rc = conv_halo_run_mp(A, B, M, aP, ep, 2, sgn < 0 ? 1 : 0, st);
      if (rc >= 0) return rc;
    }
  }
  if (dtype == 0 || dtype == 2) {
    CUtensorMap ma, mb;
    int rc = make_map_2d(&ma, dtype == 2, A, Ca, rowsA, BM);       // one 256-row box per K block
    if (rc) return rc;
    rc = make_map_2d(&mb, dtype == 2, B, Ktot, (long long)Ntot * (batched ? nbatch : 1), BN);
    if (rc) return rc;
    if (dtype == 0) {
      switch (kind) {
        case EPI_STORE: return launch_tc<EPI_STORE, 0>(ma, mb, gs, ep, st);
        case EPI_CONV_LN: return launch_tc<EPI_CONV_LN, 0>(ma, mb, gs, ep, st);
        case EPI_ATTN_OUT: return launch_tc<EPI_ATTN_OUT, 0>(ma, mb, gs, ep, st);
        case EPI_CONVT: return launch_tc<EPI_CONVT, 0>(ma, mb, gs, ep, st);
        case EPI_CONV_LN_TRAIN: return launch_tc<EPI_CONV_LN_TRAIN, 0>(ma, mb, gs, ep, st);
      }
    } else {
      switch (kind) {
        case EPI_STORE: return launch_tc<EPI_STORE, 1>(ma, mb, gs, ep, st);
        case EPI_CONV_LN: return launch_tc<EPI_CONV_LN, 1>(ma, mb, gs, ep, st);
        case EPI_ATTN_OUT: return launch_tc<EPI_ATTN_OUT, 1>(ma, mb, gs, ep, st);
        case EPI_CONVT: return launch_tc<EPI_CONVT, 1>(ma, mb, gs, ep, st);
        case EPI_CONV_LN_TRAIN: return launch_tc<EPI_CONV_LN_TRAIN, 1>(ma, mb, gs, ep, st);
      }
    }
    return set_error("gemm: bad epilogue kind %d", kind);
  }
  if (dtype != 1) return set_error("gemm: bad dtype %d", dtype);
  if (scratch_elems < M * (long long)Ntot) return set_error("gemm(fp32): scratch too small (%lld < %lld)", scratch_elems, M * (long long)Ntot);
  dim3 grid((unsigned)((gs.rows_per_batch + 63) / 64), (unsigned)((Ntot + 63) / 64), (unsigned)nbatch);
  gemm_simt_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(A), rowsA, Ca, reinterpret_cast<const float*>(B),
                                         Ktot, gs, scratch, Ntot);
  int rc = check_launch("gemm_simt_kernel");
  if (rc) return rc;
  switch (kind) {
    case EPI_STORE: return launch_simt_epi<EPI_STORE>(scratch, Ntot, gs, ep, st);
    case EPI_CONV_LN: return launch_simt_epi<EPI_CONV_LN>(scratch, Ntot, gs, ep, st);
    case EPI_ATTN_OUT: return launch_simt_epi<EPI_ATTN_OUT>(scratch, Ntot, gs, ep, st);
    case EPI_CONVT: return launch_simt_epi<EPI_CONVT>(scratch, Ntot, gs, ep, st);
    case EPI_CONV_LN_TRAIN: return launch_simt_epi<EPI_CONV_LN_TRAIN>(scratch, Ntot, gs, ep, st);
  }
  return set_error("gemm: bad epilogue kind %d", kind);
}

}  // namespace vg
