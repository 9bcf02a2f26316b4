// Weight-gradient GEMM for sm_100a:   dW[n][tap*Ca + c] (+)= sum_m dY[m][n] * A[m + shift(tap)][c]
//
// The reduction runs over the ROW index m (pixels / tokens, millions of them) of two row-major activations, so both
// MMA operands are "MN-major" (the contiguous memory dimension is the MMA M / N dimension, not K).  tcgen05 reads such
// tiles directly from the 128B-swizzled [K rows][128 bytes] boxes TMA writes (transpose bits of the instruction
// descriptor; LBO = distance between 128-byte column groups, SBO = 1024 B between 8-row groups), so no transposed copy
// of an activation ever exists.  One CTA owns one 128-row n-tile x up to four 128-wide column tiles (e.g. three taps of
// a 3x3 convolution: the dY tile is loaded once per K step and reused for every column tile) over a slice of the
// reduction range; fp32 partial results go to a caller-provided workspace [ksplit][Ntot][Ktot] and a second kernel sums
// the slices into dW (deterministic, no atomics).  3x3 convolutions over the padded-grid layout need no im2col: tap
// (dy,dx) is the same A tensor loaded at a shifted row coordinate (zero padding = stored zeros / TMA OOB fill).
//
// fp32 mode: SIMT FFMA kernel with the same decomposition and workspace.
#include <stdlib.h>

#include "vg_common.cuh"
#include "vg_host.h"

namespace vg {

namespace wg {
constexpr int THREADS = 192;            // warp 0 TMA, warp 1 MMA issuer, warps 2..5 epilogue (TMEM lane group = warp & 3)
constexpr int TILE_BYTES = 16384;       // one operand tile: 128 elements x KT rows (KT = 64 bf16 / 32 tf32)
constexpr int MAX_ACC = 4;              // 4 x 128 fp32 columns = the whole TMEM
}  // namespace wg

struct WgradShape {
  long long M;                 // reduction rows
  int Ntot, Ca, ntaps, Ktot;   // dW is [Ntot][Ktot], Ktot = ntaps * Ca
  int tap_shift[9];
  int n_tiles;                 // ceil(Ntot / 128)
  int col_tiles;               // ntaps * (Ca / 128)
  int groups;                  // ceil(col_tiles / acc_per_cta)
  int acc_per_cta;
  int ksplit;
  long long rows_per_split;    // multiple of KT
  int stages;
};

// MN-major 128-byte-swizzled operand: 128-byte column groups `lbo` bytes apart, K row groups `sbo` bytes apart.
// 16-bit types: SWIZZLE_128B (layout type 2, 16-byte chunks XOR row%8, K groups of 8 rows).
// 32-bit types (tf32): the only MN-major layout is SWIZZLE_128B_BASE32B (layout type 1: 32-byte chunks XOR row%4,
// K groups of 4 rows), written by TMA with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
__device__ __forceinline__ uint64_t umma_desc_mn128(uint32_t smem_addr, uint32_t lbo, uint32_t sbo, uint32_t layout_type) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
         (1ull << 46) | ((uint64_t)layout_type << 61);
}

template <int TF32>
__global__ void __launch_bounds__(wg::THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap mapY, const __grid_constant__ CUtensorMap mapA, const WgradShape ws,
                float* __restrict__ part) {
  using namespace wg;
  constexpr int E = TF32 ? 32 : 64;          // elements per 128 bytes
  constexpr int KT = TF32 ? 32 : 64;         // reduction rows per stage
  constexpr int BOXES = 128 / E;             // 128-byte column groups per 128-element tile
  constexpr int BOX_BYTES = KT * 128;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = (1 + ws.acc_per_cta) * TILE_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + ws.stages * stage_bytes);
  uint64_t* empty = full + 8;
  uint64_t* done = empty + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  // unit -> (n tile, column group, k split)
  int u = blockIdx.x;
  const int ks = u % ws.ksplit; u /= ws.ksplit;
  const int grp = u % ws.groups;
  const int n_tile = u / ws.groups;
  const int ct0 = grp * ws.acc_per_cta;
  const int nacc = min(ws.acc_per_cta, ws.col_tiles - ct0);
  const long long m_begin = (long long)ks * ws.rows_per_split;
  long long m_end = m_begin + ws.rows_per_split;
  if (m_end > ws.M) m_end = ws.M;
  const int k_steps = m_end > m_begin ? (int)((m_end - m_begin + KT - 1) / KT) : 0;
  const int cblocks = ws.Ca / 128;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&mapY); tma_prefetch_desc(&mapA); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < ws.stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    mbar_init(done, 1);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot, 0);        // warp-uniform: lets the MMA issue use uniform registers (no per-MMA elect/broadcast loop)

  if (warp == 0) {
    if (lane == 0) {                                           // ===== TMA producer =====
      int stage = 0; uint32_t phase = 0;
      for (int kb = 0; kb < k_steps; ++kb) {
        const long long m0 = m_begin + (long long)kb * KT;
        mbar_wait(empty + stage, phase ^ 1);
        mbar_arrive_expect_tx(full + stage, (1 + nacc) * TILE_BYTES);
        uint8_t* sy = smem + stage * stage_bytes;
#pragma unroll
        for (int b = 0; b < BOXES; ++b) tma_load_2d(sy + b * BOX_BYTES, &mapY, full + stage, n_tile * 128 + b * E, (int)m0);
        for (int a = 0; a < nacc; ++a) {
          const int ct = ct0 + a, tap = ct / cblocks, cb = ct - tap * cblocks;
          uint8_t* sa = sy + (1 + a) * TILE_BYTES;
#pragma unroll
          for (int b = 0; b < BOXES; ++b)
            tma_load_2d(sa + b * BOX_BYTES, &mapA, full + stage, cb * 128 + b * E, (int)(m0 + ws.tap_shift[tap]));
        }
        if (++stage == ws.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    {                                                          // ===== MMA issuer: converged warp, an elected lane issues (see elect_one) =====
      // both operands MN-major (transpose bits 15 / 16)
      constexpr uint32_t idesc = (TF32 ? umma_idesc_tf32(128, 128) : umma_idesc_bf16(128, 128)) | (1u << 15) | (1u << 16);
      constexpr int KSTEP_ROWS = TF32 ? 8 : 16;                // rows consumed per MMA
      constexpr uint32_t KGROUP_BYTES = TF32 ? 512u : 1024u;   // 4 rows (tf32) / 8 rows (bf16) of 128 bytes
      constexpr uint32_t LAYOUT = TF32 ? 1u : 2u;
      constexpr uint32_t lbo = (uint32_t)BOX_BYTES, sbo = KGROUP_BYTES;
      int stage = 0; uint32_t phase = 0;
      for (int kb = 0; kb < k_steps; ++kb) {
        mbar_wait(full + stage, phase);
        tc_fence_after();
        const uint32_t sy = smem_u32(smem + stage * stage_bytes);
#pragma unroll 1
        for (int a = 0; a < nacc; ++a) {
          if (elect_one()) {
            const uint32_t sa = sy + (1 + a) * TILE_BYTES;
#pragma unroll
            for (int k = 0; k < KT / KSTEP_ROWS; ++k) {
              const uint64_t dy = umma_desc_mn128(sy + k * KSTEP_ROWS * 128, lbo, sbo, LAYOUT);
              const uint64_t da = umma_desc_mn128(sa + k * KSTEP_ROWS * 128, lbo, sbo, LAYOUT);
              if (TF32) tc_mma_tf32(tmem + a * 128, dy, da, idesc, (kb | k) ? 1u : 0u);
              else tc_mma_bf16(tmem + a * 128, dy, da, idesc, (kb | k) ? 1u : 0u);
            }
            if (a == nacc - 1) tc_commit(empty + stage);
          }
          __syncwarp();
        }
        if (++stage == ws.stages) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) tc_commit(done);
      __syncwarp();
    }
  } else {                                                     // ===== epilogue: lane = dW row n =====
    const int lg = warp & 3;
    const int n = n_tile * 128 + lg * 32 + lane;
    mbar_wait(done, 0);
    tc_fence_after();
    float* prow = part + ((long long)ks * ws.Ntot + n) * ws.Ktot;
    float v[32];
    for (int a = 0; a < nacc; ++a) {
      const int ct = ct0 + a;                                  // column tile = (tap, channel block): columns [ct*128, +128)
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        if (k_steps > 0) { tmem_ld32(tmem + ((uint32_t)(lg * 32) << 16) + a * 128 + ch * 32, v); tmem_wait_ld(); }
        else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        if (n < ws.Ntot) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(prow + ct * 128 + ch * 32 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// fp32 mode / generic shapes: one block = 64 (n) x 64 (columns of one tap) outputs over one reduction slice
__global__ void __launch_bounds__(256)
wgrad_simt_kernel(const float* __restrict__ dY, const float* __restrict__ A, long long rowsA, const WgradShape ws,
                  float* __restrict__ part) {
  __shared__ float sY[16][65], sA[16][65];
  const int cpt = (ws.Ca + 63) / 64;                       // column tiles per tap
  const int tap = blockIdx.x / cpt, c0 = (blockIdx.x - tap * cpt) * 64;
  const int n0 = blockIdx.y * 64;
  const int ks = blockIdx.z;
  const long long m_begin = (long long)ks * ws.rows_per_split;
  long long m_end = m_begin + ws.rows_per_split;
  if (m_end > ws.M) m_end = ws.M;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int shift = ws.tap_shift[tap];
  float acc[4][4] = {};
  for (long long m0 = m_begin; m0 < m_end; m0 += 16) {
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      const int r = i >> 6, c = i & 63;
      const long long m = m0 + r;
      const long long ar = m + shift;
      sY[r][c] = (m < m_end && n0 + c < ws.Ntot) ? dY[m * ws.Ntot + n0 + c] : 0.f;
      sA[r][c] = (m < m_end && ar >= 0 && ar < rowsA && c0 + c < ws.Ca) ? A[ar * ws.Ca + c0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float y[4], a[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { y[i] = sY[k][ty * 4 + i]; a[i] = sA[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(y[i], a[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= ws.Ntot) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + tx * 4 + j;
      if (c < ws.Ca) part[((long long)ks * ws.Ntot + n) * ws.Ktot + tap * ws.Ca + c] = acc[i][j];
    }
  }
}

// dW[i] = beta * dW[i] + sum_ks part[ks][i]
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, int ksplit, long long n, float beta,
                                                           float* __restrict__ dW) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  if (i + 4 <= n) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < ksplit; ++k) {
      const float4 v = *reinterpret_cast<const float4*>(part + (long long)k * n + i);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    float4* d = reinterpret_cast<float4*>(dW + i);
    if (beta != 0.f) { const float4 o = *d; s.x += beta * o.x; s.y += beta * o.y; s.z += beta * o.z; s.w += beta * o.w; }
    *d = s;
  } else {
    for (long long j = i; j < n; ++j) {
      float s = 0.f;
      for (int k = 0; k < ksplit; ++k) s += part[(long long)k * n + j];
      dW[j] = (beta != 0.f ? beta * dW[j] : 0.f) + s;
    }
  }
}

// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_rows_map(CUtensorMap* m, bool f32, const void* ptr, long long inner, long long outer, int box_rows) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qr) != cudaSuccess || !q)
      return set_error("cuTensorMapEncodeTiled entry point unavailable");
    fn = reinterpret_cast<EncodeTiledFn>(q);
  }
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)inner * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {f32 ? 32u : 64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, f32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error("wgrad: cuTensorMapEncodeTiled failed (%d) inner=%lld outer=%lld", (int)r, inner, outer);
  return 0;
}

static int wgrad_plan(WgradShape& ws, int dtype, long long M, int Ntot, int Ca, int ntaps, const int* tap_shift) {
  ws.M = M; ws.Ntot = Ntot; ws.Ca = Ca; ws.ntaps = ntaps; ws.Ktot = ntaps * Ca;
  for (int i = 0; i < 9; ++i) ws.tap_shift[i] = i < ntaps ? tap_shift[i] : 0;
  int sms = 148, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (sms <= 0) sms = 148;
  const int kt = dtype == 2 ? 32 : (dtype == 0 ? 64 : 16);
  if (dtype == 1) {
    ws.n_tiles = (Ntot + 63) / 64;
    ws.col_tiles = ntaps * ((Ca + 63) / 64);
    ws.groups = ws.col_tiles; ws.acc_per_cta = 1; ws.stages = 0;
  } else {
    ws.n_tiles = (Ntot + 127) / 128;
    ws.col_tiles = ntaps * (Ca / 128);
    // three taps of one kernel row per CTA for 3x3 convolutions, otherwise up to four column tiles
    ws.acc_per_cta = (ntaps == 9 && Ca == 128) ? 3 : (ws.col_tiles < wg::MAX_ACC ? ws.col_tiles : wg::MAX_ACC);
    ws.groups = (ws.col_tiles + ws.acc_per_cta - 1) / ws.acc_per_cta;
    const int stage_bytes = (1 + ws.acc_per_cta) * wg::TILE_BYTES;
    ws.stages = 200 * 1024 / stage_bytes;
    if (ws.stages > 6) ws.stages = 6;
  }
  const long long units = (long long)ws.n_tiles * ws.groups;
  long long want = (dtype == 1 ? 4LL * sms : (long long)sms) / units;          // reduction slices
  const long long max_split = (M + 8LL * kt - 1) / (8LL * kt);                 // at least 8 K steps per slice
  if (want > max_split) want = max_split;
  if (want > 64) want = 64;
  if (want < 1) want = 1;
  ws.ksplit = (int)want;
  long long rps = (M + ws.ksplit - 1) / ws.ksplit;
  rps = (rps + kt - 1) / kt * kt;
  ws.rows_per_split = rps;
  ws.ksplit = (int)((M + rps - 1) / rps);
  return 0;
}

long long wgrad_workspace_elems(int dtype, long long M, int Ntot, int Ca, int ntaps) {
  if (M <= 0) return 0;                                        // an empty reduction needs no slices (wgrad_plan divides by M)
  WgradShape ws;
  int shifts[9] = {0};
  wgrad_plan(ws, dtype, M, Ntot, Ca, ntaps, shifts);
  return (long long)ws.ksplit * Ntot * ws.Ktot;
}

// dtype 0: bf16 operands, 1: fp32 SIMT, 2: fp32 operands as tf32.  dW fp32 [Ntot][ntaps*Ca]; dW = beta*dW + result.
int wgrad_run(int dtype, const void* dY, const void* A, long long rowsA, long long M, int Ntot, int Ca, int ntaps,
              const int* tap_shift, float* dW, float beta, float* work, long long work_elems, cudaStream_t st) {
  if (ntaps < 1 || ntaps > 9) return set_error("wgrad: bad tap count %d", ntaps);
  if (M < 0) return set_error("wgrad: negative row count %lld", M);
  if (dtype != 1 && (Ca % 128 || Ntot % 64)) return set_error("wgrad: tensor-core path needs Ca %% 128 == 0 and Ntot %% 64 == 0 (got %d, %d)", Ca, Ntot);
  if (M == 0) {                                                // the sum over no rows is zero: dW = beta * dW, as for any M
    const long long n = (long long)Ntot * ntaps * Ca;
    wgrad_reduce_kernel<<<(unsigned)((n / 4 + 256) / 256), 256, 0, st>>>(work, 0, n, beta, dW);
    return check_launch("wgrad_reduce_kernel");
  }
  WgradShape ws;
  wgrad_plan(ws, dtype, M, Ntot, Ca, ntaps, tap_shift);
  const long long need = (long long)ws.ksplit * Ntot * ws.Ktot;
  if (work_elems < need) return set_error("wgrad: workspace too small (%lld < %lld floats)", work_elems, need);
  if (dtype == 1) {
    dim3 grid((unsigned)ws.col_tiles, (unsigned)ws.n_tiles, (unsigned)ws.ksplit);
    wgrad_simt_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(dY), reinterpret_cast<const float*>(A), rowsA, ws, work);
    int rc = check_launch("wgrad_simt_kernel");
    if (rc) return rc;
  } else {
    CUtensorMap my, ma;
    const int kt = dtype == 2 ? 32 : 64;
    int rc = make_rows_map(&my, dtype == 2, dY, Ntot, M, kt);
    if (rc) return rc;
    rc = make_rows_map(&ma, dtype == 2, A, Ca, rowsA, kt);
    if (rc) return rc;
    const int smem = ws.stages * (1 + ws.acc_per_cta) * wg::TILE_BYTES + 1024 + 256;
    static PerDeviceSize attr_pd[2];
    size_t& attr_cur = attr_pd[dtype == 2].cur();
    if (attr_cur < (size_t)smem) {
      cudaError_t e = dtype == 2 ? cudaFuncSetAttribute(wgrad_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)
                                 : cudaFuncSetAttribute(wgrad_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return set_error("wgrad smem attr: %s", cudaGetErrorString(e));
      attr_cur = 227 * 1024;
    }
    const int grid = ws.n_tiles * ws.groups * ws.ksplit;
    if (dtype == 2) wgrad_tc_kernel<1><<<grid, wg::THREADS, smem, st>>>(my, ma, ws, work);
    else wgrad_tc_kernel<0><<<grid, wg::THREADS, smem, st>>>(my, ma, ws, work);
    rc = check_launch("wgrad_tc_kernel");
    if (rc) return rc;
  }
  const long long n = (long long)Ntot * ws.Ktot;
  wgrad_reduce_kernel<<<(unsigned)((n / 4 + 256) / 256), 256, 0, st>>>(work, ws.ksplit, n, beta, dW);
  return check_launch("wgrad_reduce_kernel");
}

}  // namespace vg
