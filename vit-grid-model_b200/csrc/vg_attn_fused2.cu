// Fused window / grid attention for sm_100a, second generation (maxvit.py:170-219 + the partition / residual code around it,
// :298-340).  In place on the residual stream: xio += to_out(attention(LN/FiLM(gather(xio)))).
//
// One persistent CTA processes tiles of TWO windows (2 x 64 token slots = the 128 rows of a tcgen05 M=128 MMA).
//
//  * The window / grid partition IS the TMA tensor map (SURVEY App. C): block partition = boxes (32 ch, 7, 7) of the 3-D view
//    (C, Wl, N*Hl); grid partition = boxes (32 ch, 1, 7, 1, 7) of the 5-D view (C, Y, 7, X, 7N) -- Hl = 7X, Wl = 7Y, so the
//    dilated gather 'b d (w1 x) (w2 y)' is plain box addressing.  The TMA warp prefetches the 49 token rows of both windows of the NEXT
//    tile (four 32-channel SWIZZLE_128B planes) while this tile computes; the result goes back through the SAME maps with
//    cp.reduce.async.bulk.tensor (.add): the residual add happens in the TMA unit / L2, the SMs never re-read the input rows.
//  * Per tile: LN + FiLM of the prefetched rows -> X tile (fp16, 64 TMEM columns: the A operand of all 32 QKV projections).
//  * Per head h (weights and per-head tables streamed by TMA):
//      QKV_h = X Wqkv_h^T            kind::f16 (fp16 operands) M128 N96 K128, A from TMEM            -> TMEM (single buffer)
//      staging: q^ = q log2e/|q| (fp16), K" = k 32 gq gk/|k| (fp16) -> ONE 128-byte-row tile (q^ | K"), V^T (bf16)  -> smem
//      S = q^ K"^T                   kind::f16 M128 N128 K32                                           -> TMEM
//      softmax(S + bias) in registers (exp2 domain), P (bf16 pairs)                                    -> TMEM (tcgen05.st)
//      O_h = P V                     kind::f16 M128 N32 K128, A = P from TMEM                           -> TMEM
//      Out += O_h Wout_h^T           kind::tf32 M128 N128 K32, A = O_h read in place from TMEM          -> TMEM
//  * TWO compute groups of eight warps work on ALTERNATE heads: each group stages its head's operands and then runs its
//    softmax, so the dependent phases of one head (barrier polls, TMEM round trips, the exp2 chain) overlap the other group's.
//    The QKV accumulator is released as soon as the staging group holds q, k, v in registers, the S accumulator as soon as
//    the softmax group holds its half rows -- single buffers, all 512 TMEM columns in use.
//
// Warp roles (640 threads): warp 0 = TMA (weights, tables, token rows); THREE MMA issuers -- warp 1: QKV projections, warp 19:
// S products, warp 18: PV and out-projection -- because a tcgen05.mma issue blocks while the tensor pipe's queue is full
// (8 QKV instructions hold their issuer ~450 cycles) and a single issuer puts that, nine barrier polls per head and the
// PV -> out wait in front of the S product the softmax group is waiting for; every TMEM hand-over between the three streams
// goes through an mbarrier; each issuer runs converged with an elected lane issuing; warps 2..9 = compute group 0 (even
// heads; builds the X tile of the next tile), warps 10..17 = compute group 1 (odd heads; runs the tile epilogue).  Two threads
// per token row (= TMEM lane) in each group.
#include "vg_common.cuh"
#include "vg_host.h"
#include "vg_rng.cuh"

namespace vg {

namespace fb {
constexpr int C = 128, DH = 32;
constexpr int WIN = 7, REG = 4, SEQ = REG + WIN * WIN;
constexpr int WQ_BYTES = 2 * 12288;              // fp16: 2 k-blocks x [96 rows x 128 B]
constexpr int WQ_OFF = 0;                        // 2 buffers (heads alternate)
constexpr int WO_OFF = WQ_OFF + 2 * WQ_BYTES;    // tf32 [128 rows x 128 B], 2 buffers
constexpr int QK_OFF = WO_OFF + 2 * 16384;       // per group: [128 rows x 128 B]: q^ (fp16, bytes 0..63) | K" (fp16, bytes 64..127)
constexpr int VT_OFF = QK_OFF + 2 * 16384;       // V (bf16, MN-major B operand of PV): [128 key rows x 128 B], group g in bytes g*64 .. g*64+63
constexpr int RAW_OFF = VT_OFF + 2 * 8192;       // token rows of a tile: 4 channel planes x [128 rows x 128 B], SWIZZLE_128B
constexpr int RAW_BYTES = 4 * 16384;
constexpr int TAB_SR = 12, TAB_SB = 180, TAB_T169 = 7 * TAB_SB;
constexpr int TAB_FLOATS = TAB_T169 + 8 + 64;    // the per-head table of ops.pack_head_tables
constexpr int TAB_OFF = RAW_OFF + RAW_BYTES;     // 2 x TAB_FLOATS floats
constexpr int FILM_OFF = TAB_OFF + 2 * TAB_FLOATS * 4;   // 2 windows x (gamma[128] | beta[128])
constexpr int REGS_OFF = FILM_OFF + 2 * 1024;    // 2 windows x register-token rows [4][128]
constexpr int RED_OFF = REGS_OFF + 2 * 2048;     // softmax pair exchange: 2 groups x float[128][2][2]; then LN exchange float[128][2][2]
constexpr int BAR_OFF = RED_OFF + 2 * 2048 + 2048;
constexpr int SMEM_BYTES = BAR_OFF + 512 + 1024;
constexpr int THREADS = 640;
constexpr int BOX_BYTES = WIN * WIN * 128;       // one 32-channel plane of one window
// TMEM columns (all 512 in use)
constexpr int T_QKV = 0;       // 96   q | k | v accumulator (single buffer)
constexpr int T_P = 96;        // 64   P: 128 keys as bf16 pairs (A operand of PV)
constexpr int T_O = 160;       // 32   O_h (D of PV, A operand of the out-projection)
constexpr int T_X = 192;       // 64   X tile as fp16 pairs
constexpr int T_S = 256;       // 128
constexpr int T_OUT = 384;     // 128
constexpr float LOG2E = 1.4426950408889634f;
}  // namespace fb

struct Fused2Params {
  float* xio;                          // residual stream, updated in place (CL (N, Hl, Wl, 128))
  const float* reg_in; int reg_per_field; float* reg_out;
  const float* film;                   // (N, 2C) gamma | beta
  const float* head_tab;               // [heads][TAB_FLOATS]
  AttnGeom g;
  int heads;
  float ln_eps;
  long long n_windows;
  DropCfg drop;
};

namespace {

__device__ __forceinline__ uint32_t sw128b(int r, int c16) { return (uint32_t)(r * 128 + ((c16 ^ (r & 7)) << 4)); }
__device__ __forceinline__ void sts128f(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void sts128w(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void sts16b(uint32_t a, unsigned short v) { asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "h"(v) : "memory"); }
__device__ __forceinline__ float4 lds128f(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float2 fadd2b(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<uint64_t&>(d)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float2 fmul2b(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<uint64_t&>(d)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ uint32_t pk_f16(float a, float b) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ uint32_t pk_bf16(float a, float b) { __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ void tm_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tm_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void mma_ts_f16(uint32_t d, uint32_t a, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
               ::"r"(d), "r"(a), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_ts_tf32(uint32_t d, uint32_t a, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
               ::"r"(d), "r"(a), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
               ::"r"(smem_u32(dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// global[box] += smem[box] through the tensor map (fp32 add in the TMA unit / L2)
__device__ __forceinline__ void tma_red_add_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(m), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_red_add_5d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.reduce.async.bulk.tensor.5d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
               ::"l"(m), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// named barriers: 2 + 4*grp + lg = the two warps of a group that share a TMEM lane quadrant; 10 + grp = the whole group
__device__ __forceinline__ void pair_bar(int grp, int lg) { asm volatile("bar.sync %0, 64;" ::"r"(2 + 4 * grp + lg) : "memory"); }
__device__ __forceinline__ void group_bar(int grp) { asm volatile("bar.sync %0, 256;" ::"r"(10 + grp) : "memory"); }

// mbarrier operations on precomputed 32-bit shared addresses (the generic-pointer helpers of vg_common.cuh re-derive the
// aligned dynamic-shared-memory base -- eight uniform-datapath instructions -- at every call site of the hot loop)
__device__ __forceinline__ bool mbar_try_a(uint32_t a, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(a), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t a, uint32_t parity, int tag) {
  if (mbar_try_a(a, parity)) return;
  long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_a(a, parity)) {
    if (((++spins) & 0x3ff) == 0 && (clock64() - t0) > 1000000000LL) {
      printf("vitgrid: mbarrier wait timeout tag %d parity %u (block %d thread %d)\n", tag, parity, (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t a) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory"); }
__device__ __forceinline__ void sts64f(uint32_t a, float x, float y) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ float lds32f(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts32f(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ float2 lds64f(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ float rcpf(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// Up to three barriers polled by three different lanes at once, then the warp re-converges: a try_wait issued by all 32 lanes
// of a warp on one barrier was measured at ~190 cycles even when the phase is long complete, and a role that polls three
// barriers back to back pays it three times.  (__syncwarp orders the waiting lanes' acquire before the other lanes' accesses.)
#ifndef VG_LANE_POLL
#define VG_LANE_POLL 0
#endif
__device__ __forceinline__ void wait3(int lane, uint64_t* b0, uint32_t p0, uint64_t* b1, uint32_t p1, uint64_t* b2, uint32_t p2, int tag) {
#if VG_LANE_POLL
  uint64_t* b = lane == 0 ? b0 : (lane == 1 ? b1 : b2);
  const uint32_t par = lane == 0 ? p0 : (lane == 1 ? p1 : p2);
  if (lane < 3 && b != nullptr) mbar_wait_tag(b, par, tag + lane);
  __syncwarp();
#else
  if (b0) mbar_wait_tag(b0, p0, tag);
  if (b1) mbar_wait_tag(b1, p1, tag + 1);
  if (b2) mbar_wait_tag(b2, p2, tag + 2);
#endif
}

// window `half` (0 / 1) of a tile -> (valid, field n, window-in-field coordinates)
struct WinPos { bool valid; int n, xw, yw; long long wdx; };
__device__ __forceinline__ WinPos win_pos(const Fused2Params& p, long long tile, int half) {
  WinPos w;
  w.wdx = tile * 2 + half;
  w.valid = w.wdx < p.n_windows;
  const int nwin = p.g.nwin();
  w.n = w.valid ? (int)(w.wdx / nwin) : 0;
  const int wi = w.valid ? (int)(w.wdx - (long long)w.n * nwin) : 0;
  w.xw = wi / p.g.Y; w.yw = wi - w.xw * p.g.Y;
  return w;
}

}  // namespace

// DROP: training instantiation with the dropout code -- compiled out of the inference instantiations, whose cold paths share
// an instruction cache with five hot role loops
// NOMAX: the caller proved |logit + bias| <= 115 in the exp2 domain (unit q-hat / k-hat: |logit| <= log2e * dh * max|gamma_q gamma_k|), so
// neither exp2 (>= 2^-115, a normal number) nor the row sum of 53 of them (< 2^121) can leave the fp32 range and the softmax skips the
// running maximum: 32 FMNMX + 16 packed subtractions per thread and head, and two exp2 of the pair exchange
template <bool DROP, bool NOMAX>
__global__ void __launch_bounds__(fb::THREADS, 1)
attn_fused2_kernel(const __grid_constant__ CUtensorMap mapWq, const __grid_constant__ CUtensorMap mapWo,
                   const __grid_constant__ CUtensorMap mapX, const Fused2Params p) {
  using namespace fb;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BAR_OFF);
  uint64_t* wq_full = bars + 0;   uint64_t* wq_free = bars + 2;       // [2] each
  uint64_t* wo_full = bars + 4;   uint64_t* wo_free = bars + 6;       // [2] each
  uint64_t* tab_full = bars + 8;  uint64_t* tab_free = bars + 10;     // [2] each (per group)
  uint64_t* qkv_done = bars + 12;                                      // [2] per group: "stage ready" = 3 arrivals per head: the head's table has
                                                                       // landed (TMA), QKV(j) has retired, PV(j-2) has retired (this group's V bytes
                                                                       // are free) -- one poll at the start of staging instead of three
  uint64_t* qk_ready = bars + 14;                                      // [2] per group
  uint64_t* s_done = bars + 16;                                        // [2] per group
  uint64_t* p_ready = bars + 18;                                       // [2] per group
  uint64_t* pv_done = bars + 20;                                       // [2] per group
  uint64_t* qkv_free = bars + 22;                                      // staging group holds q, k, v in registers
  uint64_t* s_free = bars + 23;                                        // softmax group holds S in registers
  uint64_t* x_ready = bars + 24;  uint64_t* x_free = bars + 25;
  uint64_t* raw_full = bars + 26; uint64_t* raw_consumed = bars + 27; uint64_t* epi_done = bars + 28;
  uint64_t* tile_done = bars + 29; uint64_t* out_free = bars + 30;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int heads = p.heads;

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(wq_full + i, 1); mbar_init(wq_free + i, 1); mbar_init(wo_full + i, 1); mbar_init(wo_free + i, 1);
      mbar_init(tab_full + i, 1); mbar_init(tab_free + i, 8);
      mbar_init(qkv_done + i, 3); mbar_init(qk_ready + i, 8); mbar_init(s_done + i, 1); mbar_init(p_ready + i, 8);
      mbar_init(pv_done + i, 1);
    }
    mbar_init(qkv_free, 8); mbar_init(s_free, 8);
    mbar_init(x_ready, 8); mbar_init(x_free, 1);
    mbar_init(raw_full, 1); mbar_init(raw_consumed, 8); mbar_init(epi_done, 1);
    mbar_init(tile_done, 1); mbar_init(out_free, 8);
    fence_mbar_init();
  }
  if (warp == 0) {
    if (lane == 0) { tma_prefetch_desc(&mapWq); tma_prefetch_desc(&mapWo); tma_prefetch_desc(&mapX); }
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  // 32-bit counters in the role loops: a 64-bit division is a ~400-cycle software routine, and the MMA warp's issue loop is
  // the clock of the whole kernel
  const long long n_tiles = (p.n_windows + 1) / 2;
  const int my_tiles = (int)(((long long)blockIdx.x < n_tiles) ? (n_tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0);
  const int total = my_tiles * heads;                        // heads this CTA processes, numbered j = tl * heads + h

  if (warp == 0) {
    // ============================== TMA: token rows per tile, weights and tables per head ==============================
    if (lane == 0) {
      auto load_raw = [&](int tl) {                           // token rows, FiLM rows and register tokens of CTA-local tile tl
        const long long tile = blockIdx.x + (long long)tl * gridDim.x;
        if (tl >= 1) mbar_wait_tag(raw_consumed, (uint32_t)((tl - 1) & 1), 301);   // build_x(tl-1) has read the buffer
        if (tl >= 2) mbar_wait_tag(epi_done, (uint32_t)((tl - 2) & 1), 302);       // epilogue(tl-2)'s store has read it
        const WinPos w0 = win_pos(p, tile, 0), w1 = win_pos(p, tile, 1);
        const uint32_t per = 4 * BOX_BYTES + 2048 + 1024;
        mbar_arrive_expect_tx(raw_full, per * ((w0.valid ? 1u : 0u) + (w1.valid ? 1u : 0u)));
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const WinPos& w = half ? w1 : w0;
          if (!w.valid) continue;
#pragma unroll
          for (int pl = 0; pl < 4; ++pl) {
            uint8_t* dst = smem + RAW_OFF + pl * 16384 + (half * 64 + REG) * 128;
            if (p.g.grid_mode) tma_load_5d(dst, &mapX, raw_full, pl * 32, w.yw, 0, w.xw, w.n * WIN);
            else tma_load_3d(dst, &mapX, raw_full, pl * 32, w.yw * WIN, w.n * p.g.Hl + w.xw * WIN);
          }
          bulk_g2s(smem + REGS_OFF + half * 2048, p.reg_in + (p.reg_per_field ? (long long)w.n * REG * C : 0), 2048, raw_full);
          bulk_g2s(smem + FILM_OFF + half * 1024, p.film + (long long)w.n * 2 * C, 1024, raw_full);
        }
      };
      auto load_wq = [&](int j, int h) {
        const uint32_t b = (uint32_t)(j & 1);
        mbar_wait_tag(wq_free + b, (uint32_t)(((j >> 1) & 1) ^ 1), 303);
        mbar_arrive_expect_tx(wq_full + b, WQ_BYTES);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
          tma_load_2d(smem + WQ_OFF + b * WQ_BYTES + kb * 12288, &mapWq, wq_full + b, kb * 64, h * 96);
      };
      auto load_tab = [&](int j, int h) {
        const uint32_t b = (uint32_t)(j & 1);
        mbar_wait_tag(tab_free + b, (uint32_t)(((j >> 1) & 1) ^ 1), 304);
        mbar_arrive_expect_tx(qkv_done + b, TAB_FLOATS * 4);
        bulk_g2s(smem + TAB_OFF + b * TAB_FLOATS * 4, p.head_tab + (long long)h * TAB_FLOATS, TAB_FLOATS * 4, qkv_done + b);
      };
      if (total > 0) load_raw(0);
      for (int j = 0; j < 2 && j < total; ++j) { load_wq(j, j % heads); load_tab(j, j % heads); }
      const int raw_h = heads > 6 ? 6 : heads - 1;
      int h = 0, tl = 0, h2 = 2 % heads;                       // head of j, tile of j, head of j + 2
      for (int j = 0; j < total; ++j) {
        const uint32_t b = (uint32_t)(j & 1);
        mbar_wait_tag(wo_free + b, (uint32_t)(((j >> 1) & 1) ^ 1), 305);
        mbar_arrive_expect_tx(wo_full + b, 16384);
        tma_load_2d(smem + WO_OFF + b * 16384, &mapWo, wo_full + b, 0, h * 128);
        if (j + 2 < total) { load_wq(j + 2, h2); load_tab(j + 2, h2); }
        // the next tile's rows: once the previous tile's epilogue is certainly behind us (a few heads into this tile)
        if (h == raw_h && tl + 1 < my_tiles) load_raw(tl + 1);
        if (++h == heads) { h = 0; ++tl; }
        if (++h2 == heads) h2 = 0;
      }
    }
  } else if (warp == 1) {
    // ============================== QKV issuer: QKV(j+1) as soon as staging(j) holds the accumulator in registers ==============================
    constexpr uint32_t id_qkv = umma_idesc_f16(128, 96);
    const uint32_t sWQ = smem_u32(smem + WQ_OFF);
    auto issue_qkv = [&](int j, int h, int tl) {   // QKV(j): needs X of its tile, WQ(j), and the accumulator released by staging(j-1)
        const uint32_t b = (uint32_t)(j & 1);
        wait3(lane, h == 0 ? x_ready : nullptr, (uint32_t)(tl & 1), j > 0 ? qkv_free : nullptr, (uint32_t)((j - 1) & 1),
              wq_full + b, (uint32_t)((j >> 1) & 1), 311);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t db = umma_desc_k128(sWQ + b * WQ_BYTES);
#pragma unroll
          for (int st = 0; st < 8; ++st) {
            const int kb = st >> 2, k = st & 3;
            mma_ts_f16(tmem + T_QKV, tmem + T_X + 8 * st, db + kb * (12288 >> 4) + 2 * k, id_qkv, st ? 1u : 0u);
          }
          tc_commit(qkv_done + b);
          tc_commit(wq_free + b);
          if (h == heads - 1) tc_commit(x_free);
        }
        __syncwarp();
    };
    if (total > 0) issue_qkv(0, 0, 0);
    int hq = 1 % heads, tlq = heads == 1 ? 1 : 0;            // (head, tile) of j + 1
    for (int j = 0; j + 1 < total; ++j) {
      issue_qkv(j + 1, hq, tlq);
      if (++hq == heads) { hq = 0; ++tlq; }
    }
  } else if (warp == 19) {
    // ============================== S issuer: S(j) = q^ K"^T as soon as its operands are staged ==============================
    constexpr uint32_t id_s = umma_idesc_f16(128, 128);
    const uint32_t sQK = smem_u32(smem + QK_OFF);
    for (int j = 0; j < total; ++j) {
      const uint32_t b = (uint32_t)(j & 1);
      // s_free(j-1) first (the other group took S(j-1) long ago); the operands of head j arrive over a hardware named
      // barrier: an mbarrier poll by a whole warp costs ~190 cycles, and this hand-over is in front of every softmax
      if (j > 0) mbar_wait_tag(s_free, (uint32_t)((j - 1) & 1), 315);
      asm volatile("bar.sync %0, 288;" ::"r"(12 + (int)b) : "memory");
      tc_fence_after();
      if (elect_one()) {
        const uint64_t da = umma_desc_k128(sQK + b * 16384);
#pragma unroll
        for (int k = 0; k < 2; ++k) tc_mma_bf16(tmem + T_S, da + 2 * k, da + 4 + 2 * k, id_s, k ? 1u : 0u);
        tc_commit(s_done + b);
      }
      __syncwarp();
    }
  } else if (warp == 18) {
    // ============================== back-end MMA issuer: PV(k), out(k) ==============================
    constexpr uint32_t id_pv = umma_idesc_bf16(128, 32) | (1u << 16);       // B (= V) is MN-major: key rows x head dims
    constexpr uint32_t id_out = umma_idesc_tf32(128, 128);
    const uint32_t sWO = smem_u32(smem + WO_OFF), sVT = smem_u32(smem + VT_OFF);
    int h = 0, tl = 0;
    if (lane == 0) { mbar_arrive(qkv_done + 0); mbar_arrive(qkv_done + 1); }      // heads 0 and 1 have no PV(j-2) to wait for
    for (int k = 0; k < total; ++k) {
      const uint32_t b = (uint32_t)(k & 1);
      mbar_wait_tag(wo_full + b, (uint32_t)((k >> 1) & 1), 316);
      if (h == 0 && tl > 0) mbar_wait_tag(out_free, (uint32_t)((tl - 1) & 1), 317);
      asm volatile("bar.sync %0, 288;" ::"r"(14 + (int)b) : "memory");      // P(k) stored by the 8 warps of group b
      tc_fence_after();
      if (elect_one()) {
        // MN-major SWIZZLE_128B operand: 16 key rows (2048 B) per K step, 8-row groups 1024 B apart; this head's 64 bytes
        // start at byte b*64 of every row
        const uint64_t dv = (uint64_t)(((sVT + b * 64) & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
#pragma unroll
        for (int st = 0; st < 8; ++st) mma_ts_f16(tmem + T_O, tmem + T_P + 8 * st, dv + st * (2048 >> 4), id_pv, st ? 1u : 0u);
        tc_commit(pv_done + b);
        if (k + 2 < total) tc_commit(qkv_done + b);          // staging(k+2) may overwrite this group's V bytes
      }
      __syncwarp();
      // a TMEM A operand is not ordered behind the MMA that writes it: wait for PV(k) to retire before out(k)
      wait3(lane, pv_done + b, (uint32_t)((k >> 1) & 1), nullptr, 0, nullptr, 0, 319);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dwo = umma_desc_k128(sWO + b * 16384);
#pragma unroll
        for (int st = 0; st < 4; ++st) mma_ts_tf32(tmem + T_OUT, tmem + T_O + 8 * st, dwo + 2 * st, id_out, (h | st) ? 1u : 0u);
        tc_commit(wo_free + b);
        if (h == heads - 1) tc_commit(tile_done);
      }
      __syncwarp();
      if (++h == heads) { h = 0; ++tl; }
    }
  } else {
    // ============================== compute groups ==============================
    const int grp = (warp - 2) >> 3;                         // 0: even heads (+ builds X), 1: odd heads (+ tile epilogue)
    const int lg = warp & 3;                                 // TMEM lane quadrant this warp may access
    const int ch = ((warp - 2) >> 2) & 1;                    // column half handled by this thread
    const int t = lg * 32 + lane;                            // tile row == TMEM lane
    const int half = t >> 6, i = t & 63;                     // window within the tile, token slot
    const uint32_t lane_addr = tmem + ((uint32_t)(lg * 32) << 16);
    // the aligned base as a 32-bit shared address computed from the raw array's shared address (a compile-time constant): derived
    // from the generic pointer it made every barrier address below depend on the 64-bit shared-window chain (S2R SR_SWINHI, S2UR
    // SR_CgaCtaId, two 64-bit adds), which the compiler rebuilt in every head iteration rather than keep ten addresses in registers
    const uint32_t s_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t s_bar = s_base + BAR_OFF;
    const bool is_reg = i < REG;
    const int ti = (i >= REG && i < SEQ) ? i - REG : 0;
    const int ai = ti / WIN, bi = ti - ai * WIN;
    const uint32_t red = s_base + RED_OFF + grp * 2048 + t * 16;             // this row: [2 threads] x (max, sum)
    const uint32_t a_stage = s_bar + 8 * (12 + grp), a_qkv_free = s_bar + 8 * 22, a_s_done = s_bar + 8 * (16 + grp);
    const uint32_t a_s_free = s_bar + 8 * 23, a_tab_free = s_bar + 8 * (10 + grp), a_pv_other = s_bar + 8 * (20 + (grp ^ 1));
    const uint32_t lnred = s_base + RED_OFF + 4096;                          // float [128][2] sums | [128][2] square sums
    // barriers of the tile-boundary work by 32-bit shared address: generic pointers in this role made the compiler rebuild the 64-bit
    // shared-window address (S2R SR_SWINHI, S2UR SR_CgaCtaId, 64-bit adds) in every head iteration
    const uint32_t a_x_ready = s_bar + 8 * 24, a_x_free = s_bar + 8 * 25, a_raw_full = s_bar + 8 * 26, a_raw_consumed = s_bar + 8 * 27;
    const uint32_t a_epi_done = s_bar + 8 * 28, a_tile_done = s_bar + 8 * 29, a_out_free = s_bar + 8 * 30;
    const uint32_t b_off = is_reg ? (uint32_t)TAB_T169 * 4u : (uint32_t)(bi * TAB_SB + (ai + 6) * TAB_SR) * 4u;
    const uint32_t b_step = is_reg ? 0u : (uint32_t)TAB_SR * 4u;
    const uint32_t QK = s_base + QK_OFF + grp * 16384;
    const uint32_t VT = s_base + VT_OFF;
    const uint32_t tab = s_base + TAB_OFF + grp * TAB_FLOATS * 4;

    // ---------------- tile prologue (group 0): LN + FiLM of the prefetched rows -> X tile (fp16, TMEM) ----------------
    auto build_x = [&](int tl) {
      const long long tile = blockIdx.x + (long long)tl * gridDim.x;
      const WinPos w = win_pos(p, tile, half);
      if (tl > 0) mbar_wait_a(a_x_free, (uint32_t)((tl - 1) & 1), 321);      // every QKV projection of the previous tile has retired
      mbar_wait_a(a_raw_full, (uint32_t)(tl & 1), 322);
      tc_fence_after();
      const bool valid = w.valid && i < SEQ;
      float4 v[16];
      float sm = 0.f;
      if (valid) {
        if (is_reg) {
          const uint32_t src = s_base + REGS_OFF + half * 2048 + i * 512 + ch * 256;
#pragma unroll
          for (int c = 0; c < 16; ++c) v[c] = lds128f(src + c * 16);
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) v[c] = lds128f(s_base + RAW_OFF + (ch * 2 + (c >> 3)) * 16384 + sw128b(t, c & 7));
        }
      } else {
#pragma unroll
        for (int c = 0; c < 16; ++c) v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int c = 0; c < 16; ++c) sm += (v[c].x + v[c].y) + (v[c].z + v[c].w);
      sts32f(lnred + (t * 2 + ch) * 4, sm);
      pair_bar(grp, lg);
      const float2 sm2 = lds64f(lnred + t * 8);
      const float mean = (sm2.x + sm2.y) * (1.0f / C);
      float ss = 0.f;
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        v[c].x -= mean; v[c].y -= mean; v[c].z -= mean; v[c].w -= mean;
        ss += (v[c].x * v[c].x + v[c].y * v[c].y) + (v[c].z * v[c].z + v[c].w * v[c].w);
      }
      sts32f(lnred + (256 + t * 2 + ch) * 4, ss);
      pair_bar(grp, lg);
      const float2 ss2 = lds64f(lnred + (256 + t * 2) * 4);
      const float rstd = rsqrtf((ss2.x + ss2.y) * (1.0f / C) + p.ln_eps);
      const uint32_t film = s_base + FILM_OFF + half * 1024 + ch * 256;       // gamma at +0, beta at +512
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t pk[16];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          pk[2 * c] = 0u; pk[2 * c + 1] = 0u;
          if (valid) {
            const float4 xv = v[hf * 8 + c];
            const float4 ga = lds128f(film + (hf * 8 + c) * 16), be = lds128f(film + 512 + (hf * 8 + c) * 16);
            pk[2 * c] = pk_f16(xv.x * rstd * ga.x + be.x, xv.y * rstd * ga.y + be.y);
            pk[2 * c + 1] = pk_f16(xv.z * rstd * ga.z + be.z, xv.w * rstd * ga.w + be.w);
          }
        }
        tm_st16(lane_addr + T_X + ch * 32 + hf * 16, pk);
      }
      tm_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive_a(a_x_ready); mbar_arrive_a(a_raw_consumed); }
    };

    // ---------------- tile epilogue (group 1): Out -> the staging planes -> TMA reduce-add through the partition map ----------------
    auto epilogue = [&](int tl) {
      const long long tile = blockIdx.x + (long long)tl * gridDim.x;
      const WinPos w = win_pos(p, tile, half);
      mbar_wait_a(a_tile_done, (uint32_t)(tl & 1), 331);
      // the staging buffer holds the NEXT tile's prefetched rows until group 0 has built its X tile
      const int last_build = (tl + 1 < my_tiles) ? tl + 1 : tl;
      mbar_wait_a(a_raw_consumed, (uint32_t)(last_build & 1), 332);
      tc_fence_after();
      const bool valid = w.valid && i < SEQ;
#pragma unroll 1
      for (int q = 0; q < 2; ++q) {
        const int c0 = ch * 64 + q * 32;
        float v[32];
        tmem_ld32(lane_addr + T_OUT + c0, v); tmem_wait_ld();
        if (q == 1) {                                          // Out is in registers: the next tile's out-projections may start
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_a(a_out_free);
        }
        if (DROP && p.drop.thresh) {                           // nn.Dropout after to_out (maxvit.py:151)
          const uint32_t rid = drop_row(w.wdx, i);
#pragma unroll
          for (int c = 0; c < 32; c += 4) {
            const uint32_t hsh = drop_hash(p.drop.seed, rid, drop_group_out(p.drop.salt, (c0 + c) >> 2));
#pragma unroll
            for (int k = 0; k < 4; ++k) v[c + k] *= (int)((hsh >> (8 * k)) & 255u) >= p.drop.thresh ? p.drop.scale : 0.f;
          }
        }
        if (valid && !is_reg) {
          const uint32_t dst = s_base + RAW_OFF + (c0 >> 5) * 16384;
#pragma unroll
          for (int c = 0; c < 8; ++c) sts128f(dst + sw128b(t, c), v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        } else if (valid && p.reg_out) {                       // register-token rows: reg_out = reg_in + Out (plain stores, 8 rows per tile)
          const float* rin = p.reg_in + (p.reg_per_field ? (long long)w.n * REG * C : 0) + (long long)i * C + c0;
          float* rout = p.reg_out + (w.wdx * REG + i) * C + c0;
#pragma unroll
          for (int c = 0; c < 32; c += 4) {
            const float4 rr = __ldg(reinterpret_cast<const float4*>(rin + c));
            *reinterpret_cast<float4*>(rout + c) = make_float4(v[c] + rr.x, v[c + 1] + rr.y, v[c + 2] + rr.z, v[c + 3] + rr.w);
          }
        }
      }
      fence_proxy_async_smem();
      group_bar(grp);
      if (warp == 10 && lane == 0) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const WinPos wh = win_pos(p, tile, hf);
          if (!wh.valid) continue;
#pragma unroll
          for (int pl = 0; pl < 4; ++pl) {
            const uint8_t* src = smem + RAW_OFF + pl * 16384 + (hf * 64 + REG) * 128;
            if (p.g.grid_mode) tma_red_add_5d(&mapX, src, pl * 32, wh.yw, 0, wh.xw, wh.n * WIN);
            else tma_red_add_3d(&mapX, src, pl * 32, wh.yw * WIN, wh.n * p.g.Hl + wh.xw * WIN);
          }
        }
        bulk_commit();
        bulk_wait_read0();                                     // the staging planes may be overwritten (next prefetch)
        mbar_arrive_a(a_epi_done);
      }
    };

    if (grp == 0) {
      // P rows are block diagonal: the key columns of the OTHER window of a row are zero and no head ever writes them --
      // cleared once here (both groups write the same columns of the same rows)
      uint32_t z[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) z[c] = 0u;
      tm_st16(lane_addr + T_P + (half ^ 1) * 32 + ch * 16, z);
      tm_wait_st();
      if (my_tiles > 0) build_x(0);
    }

    int h = grp, tl = 0;                                     // (head, tile) of j; heads is even
    long long wdx = (long long)blockIdx.x * 2 + half;        // window of this row (dropout row id)
    for (int j = grp; j < total; j += 2) {
      const uint32_t u = (uint32_t)(j >> 1);                  // sequence number inside this group

      // ---------------- staging: q^ | K" (fp16) and V^T (bf16) of head j ----------------
      // one barrier: the table of this head has landed, PV(j-2) has read this group's V bytes, QKV(j) has retired
      mbar_wait_a(a_stage, u & 1, 341);
      tc_fence_after();
      {
        float a[32], vv[16];
        tmem_ld32(lane_addr + T_QKV + ch * 32, a);                       // ch 0: q, ch 1: k
        tm_ld16(lane_addr + T_QKV + 64 + ch * 16, vv);                   // v[ch*16, +16)
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_a(a_qkv_free);                        // QKV(j+1) may overwrite the accumulator
        // V (bf16), MN-major: key row t holds its 32 head dims contiguously (64 bytes, chunks grp*4 .. grp*4+3 of the 128-byte
        // row): two 16-byte stores per thread instead of 16 transposing 2-byte stores
#pragma unroll
        for (int c = 0; c < 2; ++c)
          sts128w(VT + sw128b(t, grp * 4 + ch * 2 + c), pk_bf16(vv[8 * c], vv[8 * c + 1]), pk_bf16(vv[8 * c + 2], vv[8 * c + 3]),
                  pk_bf16(vv[8 * c + 4], vv[8 * c + 5]), pk_bf16(vv[8 * c + 6], vv[8 * c + 7]));
        float2* a2 = reinterpret_cast<float2*>(a);
        float2 n2a = make_float2(0.f, 0.f), n2b = make_float2(0.f, 0.f);
#pragma unroll
        for (int d = 0; d < 16; d += 2) { n2a = f2_fma(a2[d], a2[d], n2a); n2b = f2_fma(a2[d + 1], a2[d + 1], n2b); }
        const float nn = (n2a.x + n2a.y) + (n2b.x + n2b.y);
        // F.normalize(eps=1e-12) (maxvit.py:30): x / max(|x|, 1e-12) = x * rsqrt(max(|x|^2, 1e-24))
        const float inv = rsqrtf(fmaxf(nn, 1e-24f));
        if (ch == 0) {
          const float sc = inv * LOG2E;                                  // the softmax works in the exp2 domain
          const float2 s2 = make_float2(sc, sc);
#pragma unroll
          for (int d = 0; d < 16; ++d) a2[d] = f2_mul(a2[d], s2);
#pragma unroll
          for (int c = 0; c < 4; ++c)
            sts128w(QK + sw128b(t, c), pk_f16(a[8 * c], a[8 * c + 1]), pk_f16(a[8 * c + 2], a[8 * c + 3]),
                    pk_f16(a[8 * c + 4], a[8 * c + 5]), pk_f16(a[8 * c + 6], a[8 * c + 7]));
        } else {
          const uint32_t gm = tab + (TAB_T169 + 8) * 4;                  // 32 * gamma_q * gamma_k of this head
          const float2 i2 = make_float2(inv, inv);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 g0 = lds128f(gm + c * 32), g1 = lds128f(gm + c * 32 + 16);
            a2[4 * c] = f2_mul(f2_mul(a2[4 * c], i2), make_float2(g0.x, g0.y));
            a2[4 * c + 1] = f2_mul(f2_mul(a2[4 * c + 1], i2), make_float2(g0.z, g0.w));
            a2[4 * c + 2] = f2_mul(f2_mul(a2[4 * c + 2], i2), make_float2(g1.x, g1.y));
            a2[4 * c + 3] = f2_mul(f2_mul(a2[4 * c + 3], i2), make_float2(g1.z, g1.w));
            sts128w(QK + sw128b(t, 4 + c), pk_f16(a[8 * c], a[8 * c + 1]), pk_f16(a[8 * c + 2], a[8 * c + 3]),
                    pk_f16(a[8 * c + 4], a[8 * c + 5]), pk_f16(a[8 * c + 6], a[8 * c + 7]));
          }
        }
      }
      fence_proxy_async_smem();
      asm volatile("bar.arrive %0, 288;" ::"r"(12 + grp) : "memory");      // q^ | K" staged: the S issuer (warp 19) syncs on this barrier

      // ---------------- softmax of head j ----------------
      mbar_wait_a(a_s_done, u & 1, 344);
      tc_fence_after();
      {
        float2 sc2[16];
        float* sc = reinterpret_cast<float*>(sc2);
        tmem_ld32(lane_addr + T_S + half * 64 + ch * 32, sc);
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_a(a_s_free);                          // S(j+1) may overwrite the accumulator
        const uint32_t brow = tab + b_off;
        float m = NOMAX ? 0.f : -INFINITY;
        if (ch == 0) {
          // keys 0..3 are register tokens, keys 4..31 are window rows aj = 0..3
          const float t169 = lds32f(tab + TAB_T169 * 4);                  // (a generic load here made the compiler rebuild the 64-bit smem pointer per head)
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) sc[jj] += t169;
#pragma unroll
          for (int aj = 0; aj < 4; ++aj) {
            const uint32_t a = brow - aj * b_step;
            const float4 b0 = lds128f(a), b1 = lds128f(a + 16);
            float* q = sc + 4 + aj * 7;
            q[0] += b0.x; q[1] += b0.y; q[2] += b0.z; q[3] += b0.w; q[4] += b1.x; q[5] += b1.y; q[6] += b1.z;
          }
          if (!NOMAX) {
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) m = fmaxf(m, sc[jj]);
          }
        } else {
          // keys 32..52 are window rows aj = 4..6; keys 53..63 are padding
#pragma unroll
          for (int aj = 4; aj < 7; ++aj) {
            const uint32_t a = brow - aj * b_step;
            const float4 b0 = lds128f(a), b1 = lds128f(a + 16);
            float* q = sc + (aj - 4) * 7;
            q[0] += b0.x; q[1] += b0.y; q[2] += b0.z; q[3] += b0.w; q[4] += b1.x; q[5] += b1.y; q[6] += b1.z;
          }
          if (!NOMAX) {
#pragma unroll
            for (int jj = 0; jj < 21; ++jj) m = fmaxf(m, sc[jj]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_a(a_tab_free);                        // last read of this head's tables
        // the P buffer is single: PV(j-1) (the other group's head) must have retired before this head's P is stored.  Polled
        // here, where the thread has independent work in flight; a completed poll costs ~190 cycles at the hand-over otherwise
        const bool p_free = j > 0 ? mbar_try_a(a_pv_other, (uint32_t)(((j - 1) >> 1) & 1)) : true;
        const float2 nm = make_float2(-m, -m);
        float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
        if (ch == 0) {
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            if (!NOMAX) sc2[k] = fadd2b(sc2[k], nm);
            sc2[k].x = ex2f(sc2[k].x); sc2[k].y = ex2f(sc2[k].y);
            if (k & 1) acc1 = fadd2b(acc1, sc2[k]); else acc0 = fadd2b(acc0, sc2[k]);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 10; ++k) {
            if (!NOMAX) sc2[k] = fadd2b(sc2[k], nm);
            sc2[k].x = ex2f(sc2[k].x); sc2[k].y = ex2f(sc2[k].y);
            if (k & 1) acc1 = fadd2b(acc1, sc2[k]); else acc0 = fadd2b(acc0, sc2[k]);
          }
          sc[20] = ex2f(NOMAX ? sc[20] : sc[20] - m); sc[21] = 0.f;
          acc0 = fadd2b(acc0, sc2[10]);
#pragma unroll
          for (int k = 11; k < 16; ++k) sc2[k] = make_float2(0.f, 0.f);
        }
        acc0 = fadd2b(acc0, acc1);
        const float s_own = acc0.x + acc0.y;
        sts64f(red + ch * 8, m, s_own);
        pair_bar(grp, lg);                                               // partner's (max, sum) is visible
        const float2 oth = lds64f(red + (ch ^ 1) * 8);
        float inv_sum;
        if (NOMAX) {
          inv_sum = rcpf(s_own + oth.y);
        } else {
          const float mrow = fmaxf(m, oth.x);
          const float f_own = ex2f(m - mrow), f_oth = ex2f(oth.x - mrow);
          inv_sum = f_own * rcpf(fmaf(s_own, f_own, oth.y * f_oth));
        }
        if (DROP && p.drop.thresh) {                                     // nn.Dropout on the probabilities (maxvit.py:146, 209)
          // one hash -> four mask bytes -> per-byte compare (0xFF where kept) -> PRMT sign-replicate -> AND: the backward kernel's form
          const float ks = inv_sum * p.drop.scale;
          const float2 ks2 = make_float2(ks, ks);
          const uint32_t rid = drop_row(wdx, i), th4 = (uint32_t)p.drop.thresh * 0x01010101u;
#pragma unroll
          for (int k = 0; k < 16; ++k) sc2[k] = fmul2b(sc2[k], ks2);
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const uint32_t keep = __vcmpgeu4(drop_hash(p.drop.seed, rid, drop_group_prob(p.drop.salt, h, ch * 8 + c)), th4);
#pragma unroll
            for (int k = 0; k < 4; ++k) sc[4 * c + k] = __uint_as_float(__float_as_uint(sc[4 * c + k]) & __byte_perm(keep, 0u, 0x8888u + 0x1111u * k));
          }
        } else {
          const float2 is2 = make_float2(inv_sum, inv_sum);
#pragma unroll
          for (int k = 0; k < 16; ++k) sc2[k] = fmul2b(sc2[k], is2);
        }
        // P (bf16 pairs, one 32-bit TMEM column per two keys): own 32 keys -> columns [half*32 + ch*16, +16); the same keys of
        // the other window are zero.  The P buffer is single: PV(j-1) (the other group's head) must have retired.
        if (!p_free) mbar_wait_a(a_pv_other, (uint32_t)(((j - 1) >> 1) & 1), 345);
        tc_fence_after();
        uint32_t pk[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) pk[c] = pk_bf16(sc[2 * c], sc[2 * c + 1]);
        tm_st16(lane_addr + T_P + half * 32 + ch * 16, pk);          // (the other window's key columns of this row stay zero)
        tm_wait_st();
      }
      tc_fence_before();
      asm volatile("bar.arrive %0, 288;" ::"r"(14 + grp) : "memory");      // P(j) is in TMEM: the back-end issuer (warp 18) syncs on this barrier

      // ---------------- tile boundary work after this group's last head of the tile ----------------
      if (h == heads - 2 + grp) {
        if (grp == 0) { if (tl + 1 < my_tiles) build_x(tl + 1); }
        else epilogue(tl);
      }
      h += 2;
      if (h >= heads) { h -= heads; ++tl; wdx += 2LL * gridDim.x; }
    }
  }
  // outstanding TMA reduce-adds must have been performed before the CTA exits
  if (warp == 10 && lane == 0) bulk_wait_all0();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn2 encode_fn() {
  static EncodeTiledFn2 fn = nullptr;
  if (!fn) {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qr) != cudaSuccess || !q) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn2>(q);
  }
  return fn;
}

static int make_w_map2(CUtensorMap* m, const void* ptr, long long inner, long long outer, int box_outer, bool f16) {
  EncodeTiledFn2 fn = encode_fn();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable");
  const int esz = f16 ? 2 : 4;
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)inner * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error("attn_fused2: cuTensorMapEncodeTiled (weights) failed (%d)", (int)r);
  return 0;
}

// The partition as a tensor map over the fp32 residual stream (N, Hl, Wl, 128) (SURVEY App. C):
//   block (maxvit.py:298)  3-D (C, Wl, N*Hl), box (32, 7, 7)            at (c0, yw*7, n*Hl + xw*7)
//   grid  (maxvit.py:322)  5-D (C, Y, 7, X, 7N), box (32, 1, 7, 1, 7)   at (c0, yw, 0, xw, 7n):  pixel (w1*X + x, w2*Y + y)
// Box rows arrive token-major (w1*7 + w2), 128 bytes (32 channels) each, SWIZZLE_128B.
int attn_partition_map(CUtensorMap* m, const float* x, const AttnGeom& g) {
  EncodeTiledFn2 fn = encode_fn();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable");
  const cuuint64_t C = (cuuint64_t)g.C, W = (cuuint64_t)g.Wl, H = (cuuint64_t)g.Hl, X = (cuuint64_t)g.X, Y = (cuuint64_t)g.Y;
  const cuuint32_t win = (cuuint32_t)g.win;
  CUresult r;
  if (!g.grid_mode) {
    cuuint64_t dims[3] = {C, W, (cuuint64_t)g.N * H};
    cuuint64_t strides[2] = {C * 4, W * C * 4};
    cuuint32_t box[3] = {32u, win, win};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    cuuint64_t dims[5] = {C, Y, (cuuint64_t)win, X, (cuuint64_t)win * g.N};
    cuuint64_t strides[4] = {C * 4, Y * C * 4, W * C * 4, X * W * C * 4};
    cuuint32_t box[5] = {32u, 1u, win, 1u, win};
    cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
    r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) return set_error("attn_fused2: cuTensorMapEncodeTiled (partition map, %s) failed (%d)", g.grid_mode ? "grid" : "block", (int)r);
  return 0;
}

// wqkv_h: fp16 [heads*96][128]; wout_h: fp32 [heads*128][32]; xio: residual stream, updated in place
int attn_fused2_run(float* xio, const float* reg_in, int reg_per_field, float* reg_out, const float* film, const void* wqkv_h,
                    const float* wout_h, const float* head_tab, const AttnGeom& g, int heads, int dh, float ln_eps, unsigned seed,
                    unsigned salt, int drop_thresh, float logit_bound, cudaStream_t st) {
  if (drop_thresh < 0 || drop_thresh > 255) return set_error("attn_fused2: dropout threshold %d outside [0, 255]", drop_thresh);
  if (g.C != fb::C || dh != fb::DH) return set_error("attn_fused2: needs C=128, dim_head=32 (got C=%d, dh=%d)", g.C, dh);
  if (heads < 2 || (heads & 1)) return set_error("attn_fused2: the two compute groups alternate heads: heads must be even (got %d)", heads);
  if (g.win != fb::WIN || g.R != fb::REG) return set_error("attn_fused2: specialised for 7x7 windows + 4 register tokens (got %d, %d)", g.win, g.R);
  CUtensorMap mq, mo, mx;
  int rc = make_w_map2(&mq, wqkv_h, 128, (long long)heads * 96, 96, true);
  if (rc) return rc;
  rc = make_w_map2(&mo, wout_h, 32, (long long)heads * 128, 128, false);
  if (rc) return rc;
  rc = attn_partition_map(&mx, xio, g);
  if (rc) return rc;
  Fused2Params p;
  p.xio = xio; p.reg_in = reg_in; p.reg_per_field = reg_per_field; p.reg_out = reg_out; p.film = film;
  p.head_tab = head_tab; p.g = g; p.heads = heads; p.ln_eps = ln_eps; p.n_windows = (long long)g.N * g.nwin();
  p.drop.seed = seed; p.drop.salt = salt; p.drop.thresh = drop_thresh; p.drop.scale = 256.0f / (256.0f - (float)drop_thresh);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static bool attr[64] = {};
  if (dev < 0 || dev >= 64) return set_error("attn_fused2: device ordinal %d out of range", dev);
  if (!attr[dev]) {
    cudaError_t e = cudaFuncSetAttribute(attn_fused2_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fb::SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_fused2_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fb::SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_fused2_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fb::SMEM_BYTES);
    if (e != cudaSuccess) return set_error("attn_fused2 smem attr: %s", cudaGetErrorString(e));
    attr[dev] = true;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long n_tiles = (p.n_windows + 1) / 2;
  const int grid = (int)(n_tiles < sms ? n_tiles : sms);
  // logit_bound: the caller's bound of |logit + bias| in the exp2 domain (0 = none given: keep the running maximum)
  const bool nomax = logit_bound > 0.f && logit_bound <= 115.f;
  if (drop_thresh) attn_fused2_kernel<true, false><<<grid, fb::THREADS, fb::SMEM_BYTES, st>>>(mq, mo, mx, p);
  else if (nomax) attn_fused2_kernel<false, true><<<grid, fb::THREADS, fb::SMEM_BYTES, st>>>(mq, mo, mx, p);
  else attn_fused2_kernel<false, false><<<grid, fb::THREADS, fb::SMEM_BYTES, st>>>(mq, mo, mx, p);
  return check_launch("attn_fused2_kernel");
}

}  // namespace vg
