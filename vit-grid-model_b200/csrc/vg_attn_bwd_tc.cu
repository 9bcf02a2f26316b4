// Attention core backward on the 5th-generation tensor cores (maxvit.py:189-213 differentiated: QK-RMSNorm, sim + relative
// position bias, softmax, dropout, attn @ v).  Replaces the mma.sync kernel (vg_bwd_vit.cu attn_core_bwd_bf16_kernel) for the
// mixed-precision training step; same inputs, outputs and numerics contract (bf16 operands, fp32 accumulation, bf16 tensors).
//
// One persistent CTA works on items (field n, head h); an item is the field's windows taken two at a time: a tile of
// 2 x 64 token slots = the 128 rows (TMEM lanes) of an M=128 tcgen05.mma.  Per tile
//
//   TMA          raw q | k | v | dO rows of both windows (boxes [S rows x 32 dims] of the bf16 qkv / datt tensors)  -> smem
//   staging      q^ = q / |q|, k^ = log2e rs^2 gq gk k / |k| (bf16) -> QK tile [128 rows][q^ 64 B | k^ 64 B]; v | dO -> VD tile   (SWIZZLE_128B rows)
//   S  = q^ k^T   M128 N128 K32   both operands K-major from the QK tile
//   dP = dO v^T   M128 N128 K32   both K-major from the VD tile                (only the diagonal 64 x 64 blocks are read)
//   softmax      P = softmax(S + bias), P' = P mask, dS = P (dP mask - sum_j P' dP)    -> two bf16 smem tiles
//   dV  = P'^T dO   M128 N32 K128   A MN-major (the P' tile read transposed), B = dO MN-major
//   dK^ = dS^T q^   M128 N32 K128   A MN-major, B = q^ MN-major
//   dQ^ = dS k^     M128 N32 K128   A K-major,  B = k^ MN-major
//   att = P' v      M128 N32 K128   A K-major,  B = v  MN-major              (re-materialised forward output for the to_out weight gradient)
//   epilogue     RMSNorm backward of dQ^ / dK^, gamma gradients, bf16 stores of dq | dk | dv | att
//
// The SAME bytes serve as K-major and as MN-major operands: a SWIZZLE_128B tile is rows of 128 bytes either way, only the
// descriptor says whether a row is an M/N index (K-major) or a K index (MN-major).  P' and dS are block diagonal (a window's
// queries only see its own keys); each is stored as [window-A block 8 KB][zeros 8 KB][window-B block 8 KB], so that the
// K atom "keys of window A" is (A block, zeros), the K atom "keys of window B" is (zeros, B block) -- the zero block is shared.
//
// Warp roles (576 threads): warps 0..15 compute (row = TMEM lane, four threads per row: 16 of the 64 score columns, 8 of the
// 32 head dims, one of the four raw matrices each), warp 16 TMA, warp 17 MMA issuer.  Compute order per tile:
// softmax(t) -> staging(t+1) -> epilogue(t), so the four output products of tile t run under staging(t+1) and S / dP of
// tile t+1 under epilogue(t).
#include "vg_common.cuh"
#include "vg_host.h"
#include "vg_rng.cuh"

namespace vg {

namespace ab {
constexpr int DH = 32;
constexpr int QK_OFF = 0;                        // 2 buffers x [128 rows x 128 B]
constexpr int VD_OFF = QK_OFF + 2 * 16384;       // 2 buffers x [128 rows x 128 B]
constexpr int P_OFF = VD_OFF + 2 * 16384;        // [A block 8 KB][zeros 8 KB][B block 8 KB]
constexpr int DS_OFF = P_OFF + 24576;
constexpr int RAW_OFF = DS_OFF + 24576;          // 2 stages x [2 windows][q, k, v, dO][64 rows x 64 B]
constexpr int RAW_STAGE = 2 * 4 * 4096;
constexpr int MAX_OFF = RAW_OFF + 2 * RAW_STAGE; // float[128][4]      row maxima of the four column quarters
constexpr int SUM_OFF = MAX_OFF + 2048;          // float2[128][4]     (sum e, sum e dP)
constexpr int DOT_OFF = SUM_OFF + 4096;          // float2[128][4]     (g.u of q, of k) partial dots of the RMSNorm backward
constexpr int INV_OFF = DOT_OFF + 4096;          // float[2 buffers][2][128]   1 / |q|, 1 / |k|
constexpr int GAM_OFF = INV_OFF + 2048;          // float[4][32]: rs gq, 1 / (rs gq), rs gk, 1 / (rs gk)
constexpr int BIAS_OFF = GAM_OFF + 512;          // float[256] bias column of this head, float[256] its gradient
constexpr int GRED_OFF = BIAS_OFF + 2048;        // float[16 warps][32]: per-warp gamma-gradient column sums, + float[16] register-token bias partials
constexpr int BX_LD = 68;                        // floats per row of the expanded bias table (272 B: conflict-free 16-byte row reads)
constexpr int BX_OFF = GRED_OFF + 2048 + 64;     // float[64][BX_LD]: bias of (query slot, key slot) for this head
constexpr int BAR_OFF = BX_OFF + 64 * BX_LD * 4;
constexpr int SMEM_BYTES = BAR_OFF + 256 + 1024;
constexpr int THREADS = 576;
constexpr int T_S = 0, T_DP = 128, T_OUT = 256;  // TMEM columns: S, dP, then dV | dQ^ | dK^ | att (32 each)
constexpr int T_DG = 448;                        // 32 columns (k rows): per-row gamma-gradient terms dK"_d u_d, reduced over rows once per item
constexpr int T_DB = 384;                        // 64 columns: the bias-gradient accumulators of the item (sum of dS over its tiles), thread-private
}  // namespace ab

struct AttnBwdTcParams {
  const float* qgamma; const float* kgamma;      // [heads*DH]
  const float* bias_table;                       // [nb][heads]
  bf16* dqkv;                                    // [rows][3*inner]
  bf16* att_out;                                 // [rows][inner] or null
  float* dqgamma; float* dkgamma; float* dbias_table;
  AttnGeom g;
  int heads;
  DropCfg drop;
};

namespace {

__device__ __forceinline__ uint32_t sw128(int r, int c16) { return (uint32_t)(r * 128 + ((c16 ^ (r & 7)) << 4)); }
__device__ __forceinline__ uint4 lds128u(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds128f(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float2 lds64f(uint32_t a) { float2 v; asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ float lds32f(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts32f(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts64f(uint32_t a, float x, float y) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ float ex2a(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ void sts128u(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t pkbf(float a, float b) { __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ float2 unbf(uint32_t w) { return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w)); }
__device__ __forceinline__ void tmld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmst16(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// K-major SWIZZLE_128B descriptor: umma_desc_k128.  MN-major SWIZZLE_128B: a 128-byte row is one K index and 64 M/N elements;
// 8-row groups SBO = 1024 B apart, the next 64 M/N elements LBO bytes away (cute: ((T,8,m),(8,k)):((1,T,LBO),(8T,SBO)))
__device__ __forceinline__ uint64_t desc_mn128(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

}  // namespace

__global__ void __launch_bounds__(ab::THREADS, 1)
attn_core_bwd_tc_kernel(const __grid_constant__ CUtensorMap mapQKV, const __grid_constant__ CUtensorMap mapD, const AttnBwdTcParams p) {
  using namespace ab;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BAR_OFF);
  uint64_t* raw_full = bars;            // [2]  TMA -> compute
  uint64_t* raw_free = bars + 2;        // [2]  16 compute warps -> TMA
  uint64_t* staged = bars + 4;          // [2]  16 compute warps -> MMA: operand tiles of buffer b written, S / dP accumulators drained
  uint64_t* sdp_done = bars + 6;        //      MMA -> compute
  uint64_t* pds_ready = bars + 7;       //      16 compute warps -> MMA: P' and dS tiles written, output accumulators drained
  uint64_t* out_done = bars + 8;        // [4]  MMA -> compute, one per output product (dV, dQ^, dK^, att): a warp waits for its own only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const AttnGeom g_ = p.g;
  const int S = g_.S(), nwin = g_.nwin(), R = g_.R, win = g_.win, W2 = 2 * win - 1, nb = W2 * W2 + 1;
  const int heads = p.heads, inner = heads * DH;
  const int ntile = (nwin + 1) >> 1;
  const int items = g_.N * heads;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(raw_full + s, 1); mbar_init(raw_free + s, 16); mbar_init(staged + s, 16); }
    mbar_init(sdp_done, 1); mbar_init(pds_ready, 16);
    for (int s = 0; s < 4; ++s) mbar_init(out_done + s, 1);
    fence_mbar_init();
    tma_prefetch_desc(&mapQKV); tma_prefetch_desc(&mapD);
  }
  if (warp == 17) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  // the P' / dS tiles start as zeros (the shared zero blocks stay zero for the whole kernel); so do the raw stages (rows >= S
  // of a stage are never written by TMA and are never read as data, but keep them finite)
  for (int i = threadIdx.x; i < (2 * 24576 + 2 * RAW_STAGE) / 16; i += THREADS)
    reinterpret_cast<uint4*>(smem + P_OFF)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const uint32_t sb = smem_u32(smem);

  if (warp == 16) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      uint32_t T = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int n = item / heads, hd = item - n * heads;
        for (int tt = 0; tt < ntile; ++tt, ++T) {
          const uint32_t st = T & 1;
          if (T >= 2) mbar_wait_tag(raw_free + st, ((T >> 1) - 1) & 1, 401);
          const int nw = (nwin - 2 * tt) < 2 ? 1 : 2;
          mbar_arrive_expect_tx(raw_full + st, (uint32_t)(nw * 4 * S * 64));
          for (int half = 0; half < nw; ++half) {
            const int row = (n * nwin + 2 * tt + half) * S;
            uint8_t* dst = smem + RAW_OFF + st * RAW_STAGE + half * 16384;
            for (int m = 0; m < 3; ++m) tma_load_2d(dst + m * 4096, &mapQKV, raw_full + st, m * inner + hd * DH, row);
            tma_load_2d(dst + 3 * 4096, &mapD, raw_full + st, hd * DH, row);
          }
        }
      }
    }
  } else if (warp == 17) {
    // ============================== MMA issuer ==============================
    constexpr uint32_t id_sdp = umma_idesc_bf16(128, 128);
    constexpr uint32_t id_kmn = umma_idesc_bf16(128, 32) | (1u << 16);                 // A K-major, B MN-major
    constexpr uint32_t id_mnmn = umma_idesc_bf16(128, 32) | (1u << 15) | (1u << 16);   // A and B MN-major
    uint32_t T = 0;
    auto issue_sdp = [&](uint32_t Tn) {
      const uint32_t b = Tn & 1;
      mbar_wait_tag(staged + b, (Tn >> 1) & 1, 402);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dqk = umma_desc_k128(sb + QK_OFF + b * 16384), dvd = umma_desc_k128(sb + VD_OFF + b * 16384);
#pragma unroll
        for (int k = 0; k < 2; ++k) tc_mma_bf16(tmem + T_S, dqk + 2 * k, dqk + 4 + 2 * k, id_sdp, k ? 1u : 0u);      // q^ . k^
#pragma unroll
        for (int k = 0; k < 2; ++k) tc_mma_bf16(tmem + T_DP, dvd + 4 + 2 * k, dvd + 2 * k, id_sdp, k ? 1u : 0u);     // dO . v
        tc_commit(sdp_done);
      }
      __syncwarp();
    };
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      for (int tt = 0; tt < ntile; ++tt, ++T) {
        if (tt == 0) issue_sdp(T);
        const uint32_t b = T & 1;
        mbar_wait_tag(pds_ready, T & 1, 403);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t qk = sb + QK_OFF + b * 16384, vd = sb + VD_OFF + b * 16384;
          // the longest epilogues first (dK^: RMSNorm backward + gamma terms, then dQ^), each product with its own barrier
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)      // dK^[key][d] += dS[q][key] q^[q][d]: K = 16 query rows per step
            tc_mma_bf16(tmem + T_OUT + 64, desc_mn128(sb + DS_OFF + ks * 2048, 8192), desc_mn128(qk + ks * 2048, 16), id_mnmn, ks ? 1u : 0u);
          tc_commit(out_done + 2);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)      // dQ^[q][d] += dS[q][key] k^[key][d]: K = 16 keys per step
            tc_mma_bf16(tmem + T_OUT + 32, umma_desc_k128(sb + DS_OFF + (ks >> 2) * 8192 + (ks & 3) * 32), desc_mn128(qk + 64 + ks * 2048, 16),
                        id_kmn, ks ? 1u : 0u);
          tc_commit(out_done + 1);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)      // dV[key][d] += P'[q][key] dO[q][d]
            tc_mma_bf16(tmem + T_OUT, desc_mn128(sb + P_OFF + ks * 2048, 8192), desc_mn128(vd + 64 + ks * 2048, 16), id_mnmn, ks ? 1u : 0u);
          tc_commit(out_done + 0);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)      // att[q][d] += P'[q][key] v[key][d]
            tc_mma_bf16(tmem + T_OUT + 96, umma_desc_k128(sb + P_OFF + (ks >> 2) * 8192 + (ks & 3) * 32), desc_mn128(vd + ks * 2048, 16),
                        id_kmn, ks ? 1u : 0u);
          tc_commit(out_done + 3);
        }
        __syncwarp();
        if (tt + 1 < ntile) issue_sdp(T + 1);
      }
    }
  } else {
    // ============================== compute warps ==============================
    const int lg = warp & 3;                                 // TMEM lane quadrant
    const int cq = warp >> 2;                                // column quarter / raw matrix / head-dim octet of this thread
    const int t = lg * 32 + lane;                            // tile row == TMEM lane
    const int half = t >> 6, i = t & 63;                     // window within the tile, token slot
    const uint32_t lane_addr = tmem + ((uint32_t)(lg * 32) << 16);
    float* sgam = reinterpret_cast<float*>(smem + GAM_OFF);
    float* sbias = reinterpret_cast<float*>(smem + BIAS_OFF);
    float* gred = reinterpret_cast<float*>(smem + GRED_OFF);
    const int ct = warp * 32 + lane;                         // 0..511
    const float rs = sqrtf((float)DH);
    float* sbx = reinterpret_cast<float*>(smem + BX_OFF);
    const uint32_t a_gam = sb + GAM_OFF, a_inv = sb + INV_OFF, a_bx = sb + BX_OFF + (uint32_t)(i * BX_LD + cq * 16) * 4u;
    // exchange arrays are [column quarter][row]: a warp's stores and loads touch consecutive words (the [row][quarter] layout cost 8-way conflicts)
    const uint32_t a_max = sb + MAX_OFF + (uint32_t)t * 4u, a_sum = sb + SUM_OFF + (uint32_t)t * 8u;
    constexpr float LOG2E = 1.4426950408889634f;
    float* gpart = gred;                                     // [16][32]
    float* wpart = gred + 512;                               // [16]
    // relative-position-bias index of (query slot qi, key slot kj) (maxvit.py:158-168): nb-1 when either is a register token
    auto pair_index = [&](int qi, int kj) {
      if (qi < R || kj < R) return nb - 1;
      const int ti = qi - R, a = ti / win, b = ti - a * win, tj = kj - R, c = tj / win, d = tj - c * win;
      return (a - c + win - 1) * W2 + (b - d + win - 1);
    };
    // the four 8-KB data blocks of the P' / dS tiles double as the fp32 staging [128 rows][64 keys] of the item flush
    auto flush_addr = [&](int row, int c16) {
      const int blk = row >> 5;
      return sb + (uint32_t)((blk & 2 ? DS_OFF : P_OFF) + (blk & 1) * 16384 + (row & 31) * 256 + ((c16 ^ (row & 7)) << 4));
    };
    // The scale of the scores sits on the K side only: u = x / |x| for q, K" = log2e rs^2 gq gk k / |k| -- S comes out in the exp2
    // domain, the q rows need one multiply per element, and ONE gamma-gradient reduction (on dK") serves both gammas:
    //   G = rs^2 gq gk,  dG_d = sum_rows dK"_d u_k,d,  dgq_d = dG_d rs^2 gk_d,  dgk_d = dG_d rs^2 gq_d
    auto stage = [&](uint32_t Tn, int tt_n) {
      const uint32_t st = Tn & 1, buf = Tn & 1;
      mbar_wait_tag(raw_full + st, (Tn >> 1) & 1, 404);
      const bool valid = i < S && (2 * tt_n + half) < nwin;
      const int sx = (i >> 1) & 3;                           // TMA SWIZZLE_64B rows: 16-byte chunk c of row i sits at chunk c ^ ((i >> 1) & 3)
      auto stage_matrix = [&](int mi) {                      // mi: 0 q, 1 k, 2 v, 3 dO
        const uint32_t src = sb + RAW_OFF + st * RAW_STAGE + half * 16384 + mi * 4096 + i * 64;
        uint4 w[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) w[c] = valid ? lds128u(src + ((c ^ sx) << 4)) : make_uint4(0u, 0u, 0u, 0u);
        if (mi < 2) {                                        // q or k: unit vector (maxvit.py:30); k also takes the whole scale (maxvit.py:197)
          float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;      // (the row stays packed: 16 registers instead of 32 floats)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float2 a = unbf(w[c].x), b = unbf(w[c].y), cc = unbf(w[c].z), d = unbf(w[c].w);
            s0 = fmaf(a.x, a.x, s0); s1 = fmaf(a.y, a.y, s1); s2 = fmaf(b.x, b.x, s2); s3 = fmaf(b.y, b.y, s3);
            s0 = fmaf(cc.x, cc.x, s0); s1 = fmaf(cc.y, cc.y, s1); s2 = fmaf(d.x, d.x, s2); s3 = fmaf(d.y, d.y, s3);
          }
          const float inv = rsqrtf(fmaxf((s0 + s1) + (s2 + s3), 1e-24f));     // 1 / max(|x|, 1e-12)  (F.normalize eps, maxvit.py:30)
          if (mi == 0) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float2 a = unbf(w[c].x), b = unbf(w[c].y), cc = unbf(w[c].z), d = unbf(w[c].w);
              w[c].x = pkbf(a.x * inv, a.y * inv); w[c].y = pkbf(b.x * inv, b.y * inv);
              w[c].z = pkbf(cc.x * inv, cc.y * inv); w[c].w = pkbf(d.x * inv, d.y * inv);
            }
          } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float4 g0 = lds128f(a_gam + 32 * c), g1 = lds128f(a_gam + 32 * c + 16);
              const float2 a = unbf(w[c].x), b = unbf(w[c].y), cc = unbf(w[c].z), d = unbf(w[c].w);
              w[c].x = pkbf(a.x * inv * g0.x, a.y * inv * g0.y); w[c].y = pkbf(b.x * inv * g0.z, b.y * inv * g0.w);
              w[c].z = pkbf(cc.x * inv * g1.x, cc.y * inv * g1.y); w[c].w = pkbf(d.x * inv * g1.z, d.y * inv * g1.w);
            }
          }
          sts32f(a_inv + (buf * 256 + mi * 128 + t) * 4, inv);
        }
        const uint32_t dst = sb + ((mi < 2) ? QK_OFF : VD_OFF) + buf * 16384;
#pragma unroll
        for (int c = 0; c < 4; ++c) sts128u(dst + sw128(t, (mi & 1) * 4 + c), w[c]);
      };
      // roles by epilogue weight: the dK^ warps (cq 2, the longest epilogue) stage nothing, the att warps (cq 3, the shortest) stage k and dO
      if (cq == 0) stage_matrix(0);
      else if (cq == 1) stage_matrix(2);
      else if (cq == 3) { stage_matrix(1); stage_matrix(3); }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(raw_free + st); mbar_arrive(staged + buf); }
    };

    uint32_t T = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int n = item / heads, hd = item - n * heads;
      bar_sync(5, 512);                                      // the previous item's flush has read the tables
      for (int k = ct; k < nb; k += 512) sbias[k] = p.bias_table[k * heads + hd];
      if (ct >= 64 && ct < 64 + DH) {
        const int d = ct - 64;
        const float G = rs * rs * p.qgamma[hd * DH + d] * p.kgamma[hd * DH + d];
        sgam[d] = G * LOG2E; sgam[DH + d] = G != 0.f ? 1.0f / (G * LOG2E) : 0.f;       // K" scale, and back to the unit vector
        sgam[2 * DH + d] = G;
      }
      bar_sync(5, 512);
      for (int k = ct; k < 64 * 64; k += 512) {
        const int qi = k >> 6, kj = k & 63;
        // exp2 domain; -inf for the pad keys (they drop out of max, sum and P without a per-element test)
        sbx[qi * BX_LD + kj] = kj >= S ? -INFINITY : (qi < S ? sbias[pair_index(qi, kj)] * LOG2E : 0.f);
      }
      bar_sync(5, 512);
      {                                                      // bias-gradient accumulators live in TMEM (16 registers per thread less)
        float z[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) z[e] = 0.f;
        tmst16(lane_addr + T_DB + cq * 16, z);
        if (cq == 2) { tmst16(lane_addr + T_DG, z); tmst16(lane_addr + T_DG + 16, z); }
        tmem_wait_st();
      }

      stage(T, 0);
      for (int tt = 0; tt < ntile; ++tt, ++T) {
        const uint32_t buf = T & 1;
        const int wdx_i = n * nwin + 2 * tt + half;
        const bool row_ok = i < S && (2 * tt + half) < nwin;
        // ---------------- softmax + dS ----------------
        {
          mbar_wait_tag(sdp_done, T & 1, 405);
          tc_fence_after();
          float s[16], dp[16];
          tmld16(lane_addr + T_S + half * 64 + cq * 16, s);
          tmld16(lane_addr + T_DP + half * 64 + cq * 16, dp);
          tmem_wait_ld();
          float m = -INFINITY;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 bq = lds128f(a_bx + 16 * c);
            s[4 * c] += bq.x; s[4 * c + 1] += bq.y; s[4 * c + 2] += bq.z; s[4 * c + 3] += bq.w;
          }
#pragma unroll
          for (int e = 0; e < 16; ++e) m = fmaxf(m, s[e]);
          sts32f(a_max + cq * 512, m);
          bar_sync(1 + lg, 128);
          {
            m = fmaxf(fmaxf(lds32f(a_max), lds32f(a_max + 512)), fmaxf(lds32f(a_max + 1024), lds32f(a_max + 1536)));
          }
          float se = 0.f, sed = 0.f;
          // dropout on the probabilities (maxvit.py:146): one hash = the mask bytes of 4 keys; a per-byte compare turns them
          // into 0xFF / 0x00, PRMT (sign-replicate mode) widens a byte to a 32-bit AND mask for the scaled value
          uint32_t m4[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
          const float mscale = p.drop.thresh ? p.drop.scale : 1.0f;
          if (p.drop.thresh) {
            const uint32_t th4 = (uint32_t)p.drop.thresh * 0x01010101u;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4)
              m4[q4] = __vcmpgeu4(drop_hash(p.drop.seed, drop_row((long long)wdx_i, i), drop_group_prob(p.drop.salt, hd, cq * 4 + q4)), th4);
          }
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float ex = ex2a(s[e] - m);                 // scores and bias are in the exp2 domain
            dp[e] = __uint_as_float(__float_as_uint(dp[e] * mscale) & __byte_perm(m4[e >> 2], 0u, 0x8888u + 0x1111u * (e & 3)));   // dP through the mask
            s[e] = ex;
            se += ex; sed = fmaf(ex, dp[e], sed);
          }
          sts64f(a_sum + cq * 1024, se, sed);
          bar_sync(1 + lg, 128);
          {
            const float2 e0 = lds64f(a_sum), e1 = lds64f(a_sum + 1024), e2 = lds64f(a_sum + 2048), e3 = lds64f(a_sum + 3072);
            se = (e0.x + e1.x) + (e2.x + e3.x); sed = (e0.y + e1.y) + (e2.y + e3.y);
          }
          const float inv = row_ok ? __frcp_rn(se) : 0.f;
          const float delta = sed * inv;
          uint32_t pw[8], dw[8];
          float db[16];
          tmld16(lane_addr + T_DB + cq * 16, db);
          tmem_wait_ld();
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            float pm[4], ds[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int e = q4 * 4 + k;
              const float pr = s[e] * inv;
              pm[k] = __uint_as_float(__float_as_uint(pr * mscale) & __byte_perm(m4[q4], 0u, 0x8888u + 0x1111u * k));
              ds[k] = pr * (dp[e] - delta);
              db[e] += ds[k];
            }
            pw[2 * q4] = pkbf(pm[0], pm[1]); pw[2 * q4 + 1] = pkbf(pm[2], pm[3]);
            dw[2 * q4] = pkbf(ds[0], ds[1]); dw[2 * q4 + 1] = pkbf(ds[2], ds[3]);
          }
          tmst16(lane_addr + T_DB + cq * 16, db);
          const uint32_t blk = (uint32_t)half * 16384u;      // A block at +0, B block at +16384 (zeros in between)
          sts128u(sb + P_OFF + blk + sw128(i, 2 * cq), make_uint4(pw[0], pw[1], pw[2], pw[3]));
          sts128u(sb + P_OFF + blk + sw128(i, 2 * cq + 1), make_uint4(pw[4], pw[5], pw[6], pw[7]));
          sts128u(sb + DS_OFF + blk + sw128(i, 2 * cq), make_uint4(dw[0], dw[1], dw[2], dw[3]));
          sts128u(sb + DS_OFF + blk + sw128(i, 2 * cq + 1), make_uint4(dw[4], dw[5], dw[6], dw[7]));
          fence_proxy_async_smem();
          tmem_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(pds_ready);
        }
        // ---------------- operands of the next tile (the four output products of this one run meanwhile) ----------------
        if (tt + 1 < ntile) stage(T + 1, tt + 1);
        // ---------------- epilogue: thread (row, cq) owns the whole 32-dim row of output cq (dV, dQ^, dK^, att) ----------------
        {
          mbar_wait_tag(out_done + cq, T & 1, 406);
          tc_fence_after();
          const long long rg = (long long)wdx_i * S + i;
          const uint32_t tacc = lane_addr + T_OUT + cq * 32;
          if (cq == 1 || cq == 2) {
            // RMSNorm backward, in halves of 16 dims with the accumulator row read twice from TMEM (32 live registers less):
            //   q: dq = (du - u (du.u)) / |q|,  du = dS K" / log2e  (the score scale log2e sits in K"),  u = q^
            //   k: dk = (g - u (g.u)) / |k|,    g = G dK",  u = K" / (log2e G),  so g.u = dK".K" / log2e;   dG += dK" u: the per-row
            //      terms accumulate in TMEM, the sum over the rows is taken once per item (flush)
            const bool isk = cq == 2;
            const float invn = lds32f(a_inv + (buf * 256 + (isk ? 128 : 0) + t) * 4) * (isk ? 1.0f : 1.0f / LOG2E);
            const uint32_t xrow = sb + QK_OFF + buf * 16384;
            const int cb = isk ? 4 : 0;                      // k^ sits in chunks 4..7 of the row
            float d0 = 0.f, d1 = 0.f;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              float acc[16];
              tmld16(tacc + 16 * hh, acc);
              const uint4 x0 = lds128u(xrow + sw128(t, cb + 2 * hh)), x1 = lds128u(xrow + sw128(t, cb + 2 * hh + 1));
              const uint32_t xw[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
              tmem_wait_ld();
#pragma unroll
              for (int k = 0; k < 8; ++k) { const float2 xx = unbf(xw[k]); d0 = fmaf(acc[2 * k], xx.x, d0); d1 = fmaf(acc[2 * k + 1], xx.y, d1); }
            }
            const float dot = (d0 + d1) * (isk ? 1.0f / LOG2E : 1.0f);
            bf16* dst = p.dqkv + rg * 3 * inner + (isk ? inner : 0) + hd * DH;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              float acc[16];
              tmld16(tacc + 16 * hh, acc);
              const uint4 x0 = lds128u(xrow + sw128(t, cb + 2 * hh)), x1 = lds128u(xrow + sw128(t, cb + 2 * hh + 1));
              const uint32_t xw[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
              if (!isk) {
                tmem_wait_ld();
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                  const float2 xx = unbf(xw[k]);
                  acc[2 * k] = invn * fmaf(-xx.x, dot, acc[2 * k]); acc[2 * k + 1] = invn * fmaf(-xx.y, dot, acc[2 * k + 1]);
                }
              } else {
                float dg[16];
                tmld16(lane_addr + T_DG + 16 * hh, dg);
                tmem_wait_ld();
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4) {
                  const int kk = 4 * hh + k4;
                  const float4 ig = lds128f(a_gam + (DH + 4 * kk) * 4), gg = lds128f(a_gam + (2 * DH + 4 * kk) * 4);
                  const float2 xa = unbf(xw[2 * k4]), xb = unbf(xw[2 * k4 + 1]);
                  const float u0 = xa.x * ig.x, u1 = xa.y * ig.y, u2 = xb.x * ig.z, u3 = xb.y * ig.w;
                  dg[4 * k4] = fmaf(acc[4 * k4], u0, dg[4 * k4]); dg[4 * k4 + 1] = fmaf(acc[4 * k4 + 1], u1, dg[4 * k4 + 1]);
                  dg[4 * k4 + 2] = fmaf(acc[4 * k4 + 2], u2, dg[4 * k4 + 2]); dg[4 * k4 + 3] = fmaf(acc[4 * k4 + 3], u3, dg[4 * k4 + 3]);
                  acc[4 * k4] = invn * fmaf(-u0, dot, acc[4 * k4] * gg.x); acc[4 * k4 + 1] = invn * fmaf(-u1, dot, acc[4 * k4 + 1] * gg.y);
                  acc[4 * k4 + 2] = invn * fmaf(-u2, dot, acc[4 * k4 + 2] * gg.z); acc[4 * k4 + 3] = invn * fmaf(-u3, dot, acc[4 * k4 + 3] * gg.w);
                }
                tmst16(lane_addr + T_DG + 16 * hh, dg);
              }
              if (row_ok) st16_256(dst + 16 * hh, acc);
            }
            if (isk) tmem_wait_st();
          } else {
            float acc[32];
            tmem_ld32(tacc, acc);
            tmem_wait_ld();
            if (row_ok) {
              if (cq == 0) { bf16* dst = p.dqkv + rg * 3 * inner + 2 * inner + hd * DH; st16_256(dst, acc); st16_256(dst + 16, acc + 16); }
              else if (p.att_out) { bf16* dst = p.att_out + rg * inner + hd * DH; st16_256(dst, acc); st16_256(dst + 16, acc + 16); }
            }
          }
        }
      }
      // ---------------- item flush: bias and gamma gradients, no shared-memory atomics (fp32 ones are CAS loops) ----------------
      // The staging below overwrites the P' / dS blocks: EVERY output product of the last tile must have retired, not only the one
      // this warp's epilogue waited for (att is committed last; commits complete in issue order).
      mbar_wait_tag(out_done + 3, (T - 1) & 1, 407);
      {
        float db[16];
        tmld16(lane_addr + T_DB + cq * 16, db);
        tmem_wait_ld();
        float wsum = 0.f;                                    // pairs with a register token: one table entry for all of them
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const int kj = cq * 16 + e;
          if (i < S && kj < S && (i < R || kj < R)) wsum += db[e];
        }
        wsum = warp_sum(wsum);
        if (lane == 0) wpart[warp] = wsum;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(flush_addr(t, cq * 4 + c)), "f"(db[4 * c]), "f"(db[4 * c + 1]),
                       "f"(db[4 * c + 2]), "f"(db[4 * c + 3]) : "memory");
        if (cq == 2) {
          // dG: column sums over the warp's 32 rows by a transposing butterfly (lane d ends with column d), once per item
          float csum = 0.f;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            float acc[16];
            tmld16(lane_addr + T_DG + 16 * hh, acc);
            tmem_wait_ld();
#pragma unroll
            for (int sft = 8; sft >= 1; sft >>= 1) {
              const bool hi = (lane & sft) != 0;
#pragma unroll
              for (int k = 0; k < sft; ++k) {
                const float send = hi ? acc[k] : acc[k + sft];
                const float keepv = hi ? acc[k + sft] : acc[k];
                acc[k] = keepv + __shfl_xor_sync(0xffffffffu, send, sft);
              }
            }
            acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 16);
            if ((lane >> 4) == hh) csum = acc[0];
          }
          gpart[lg * 32 + lane] = csum;
        }
      }
      bar_sync(5, 512);
      if (ct < nb - 1) {                                     // entry (da, db): all window-token pairs with that relative offset, both windows
        const int da = ct / W2 - (win - 1), dbb = ct - (ct / W2) * W2 - (win - 1);
        float acc = 0.f;
        for (int a = (da > 0 ? da : 0); a < win + (da < 0 ? da : 0); ++a)
          for (int b = (dbb > 0 ? dbb : 0); b < win + (dbb < 0 ? dbb : 0); ++b) {
            const int qi = R + a * win + b, kj = R + (a - da) * win + (b - dbb);
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
              float v;
              asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(flush_addr(h2 * 64 + qi, kj >> 2) + (uint32_t)(kj & 3) * 4u));
              acc += v;
            }
          }
        atomicAdd(p.dbias_table + ct * heads + hd, acc);
      } else if (ct == nb - 1) {
        float acc = 0.f;
        for (int k = 0; k < 16; ++k) acc += wpart[k];
        atomicAdd(p.dbias_table + ct * heads + hd, acc);
      } else if (ct >= 256 && ct < 256 + DH) {
        const int d = ct - 256;
        const float dG = (gpart[d] + gpart[32 + d]) + (gpart[64 + d] + gpart[96 + d]);
        atomicAdd(p.dqgamma + hd * DH + d, dG * rs * rs * p.kgamma[hd * DH + d]);
        atomicAdd(p.dkgamma + hd * DH + d, dG * rs * rs * p.qgamma[hd * DH + d]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 17) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ------------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn3)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn3 encode_fn3() {
  static EncodeTiledFn3 fn = nullptr;
  if (!fn) {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn3>(q);
  }
  return fn;
}

static int rows_map(CUtensorMap* m, const void* base, long long cols, long long rows, int box_rows) {
  EncodeTiledFn3 fn = encode_fn3();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error("attn_core_bwd_tc: tensor map failed (%d)", (int)r);
  return 0;
}

int attn_core_bwd_tc_run(const void* qkv, const void* datt, const float* qgamma, const float* kgamma, const float* bias_table,
                         const AttnGeom& g, int heads, void* dqkv, float* dqgamma, float* dkgamma, float* dbias_table,
                         void* att_out, unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st) {
  const int S = g.S(), nb = (2 * g.win - 1) * (2 * g.win - 1) + 1;
  if (S < 1 || S > 64) return set_error("attn_core_bwd_tc: sequence %d outside [1, 64]", S);
  if (nb > 256) return set_error("attn_core_bwd_tc: %d bias-table rows > 256 (window %d)", nb, g.win);
  const long long rows = (long long)g.N * g.nwin() * S;
  if (rows >= (1ll << 31)) return set_error("attn_core_bwd_tc: %lld rows >= 2^31", rows);
  if (rows * 3 * heads * ab::DH >= (1ll << 40)) return set_error("attn_core_bwd_tc: qkv of %lld elements >= 2^40", rows * 3 * heads * ab::DH);
  if ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(datt) | reinterpret_cast<uintptr_t>(dqkv) |
       reinterpret_cast<uintptr_t>(att_out)) & 15) return set_error("attn_core_bwd_tc: qkv, datt, dqkv and att_out must be 16-byte aligned");
  CUtensorMap mq, md;
  int rc = rows_map(&mq, qkv, 3ll * heads * ab::DH, rows, S);
  if (rc) return rc;
  rc = rows_map(&md, datt, (long long)heads * ab::DH, rows, S);
  if (rc) return rc;
  static PerDeviceFlag attr_pd;
  bool& attr = attr_pd.cur();
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_core_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ab::SMEM_BYTES);
    if (e != cudaSuccess) return set_error("attn_core_bwd_tc smem attr: %s", cudaGetErrorString(e));
    attr = true;
  }
  static PerDeviceSize sms_pd;
  size_t& sms_c = sms_pd.cur();
  int sms = (int)sms_c;
  if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; sms_c = (size_t)sms; }
  AttnBwdTcParams p;
  p.qgamma = qgamma; p.kgamma = kgamma; p.bias_table = bias_table; p.dqkv = reinterpret_cast<bf16*>(dqkv);
  p.att_out = reinterpret_cast<bf16*>(att_out); p.dqgamma = dqgamma; p.dkgamma = dkgamma; p.dbias_table = dbias_table;
  p.g = g; p.heads = heads;
  p.drop.seed = seed; p.drop.salt = salt; p.drop.thresh = drop_thresh; p.drop.scale = 256.0f / (256.0f - (float)drop_thresh);
  const int items = g.N * heads;
  const int grid = items < sms ? items : sms;
  attn_core_bwd_tc_kernel<<<grid, ab::THREADS, ab::SMEM_BYTES, st>>>(mq, md, p);
  return check_launch("attn_core_bwd_tc_kernel");
}

}  // namespace vg
