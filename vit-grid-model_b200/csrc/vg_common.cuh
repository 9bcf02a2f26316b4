// Common device helpers for the sm_100a kernels: mbarrier, TMA, tcgen05/TMEM wrappers (inline PTX),
// activation-dtype traits and the padded-grid geometry shared by every kernel.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace vg {

typedef __nv_bfloat16 bf16;

// ----------------------------------------------------------------------------------------------
// Padded-grid geometry ("PG" layout) used by every full-resolution (HP x WP) feature map.
//
// A field's HP x WP frame (already padded to a multiple of 14 by MetNet3, metnet3.py:324-333) is stored
// channels-last with ONE shared zero column between image rows and ONE shared zero row between images:
//     flat pixel  q = (n*(HP+1) + h + 1) * (WP+1) + (w + 1),   row pitch P = WP+1
// so tap (dy,dx) of a 3x3/pad-1 convolution is the plain row offset dy*P + dx and a conv becomes a GEMM
// whose A operand is the same 2-D [q][C] tensor loaded at 9 shifted row coordinates (zero padding comes
// from the stored zero pads, or from TMA out-of-bounds fill at the two ends of the buffer).
// Every writer stores zeros at pad positions, so pads stay zero.
// ----------------------------------------------------------------------------------------------
struct PGeom {
  int HP, WP;     // frame height / width
  int P;          // row pitch in pixels = WP + 1
  int R;          // rows per image    = HP + 1
  int N;          // number of images
  __host__ __device__ long long rows() const { return (long long)N * R + 1; }
  __host__ __device__ long long pixels() const { return rows() * P; }         // flat q range
  __host__ __device__ long long q(int n, int h, int w) const { return ((long long)n * R + h + 1) * P + (w + 1); }
  // decode q -> (n,h,w); returns false for pad / out-of-range positions
  __host__ __device__ bool decode(long long qq, int& n, int& h, int& w) const {
    long long row = qq / P;
    int col = (int)(qq - row * P);
    n = (int)(row / R);
    int r = (int)(row - (long long)n * R);
    h = r - 1; w = col - 1;
    return (col >= 1) && (r >= 1) && (n < N) && (qq >= 0);
  }
  // the same for 0 <= qq < 2^31 (32-bit divisions: the 64-bit ones are ~400-cycle software routines)
  __host__ __device__ bool decode32(unsigned qq, int& n, int& h, int& w) const {
    const unsigned row = qq / (unsigned)P;
    const int col = (int)(qq - row * (unsigned)P);
    n = (int)(row / (unsigned)R);
    const int r = (int)(row - (unsigned)n * (unsigned)R);
    h = r - 1; w = col - 1;
    return (col >= 1) && (r >= 1) && (n < N);
  }
};
inline PGeom make_pgeom(int N, int HP, int WP) { PGeom g; g.HP = HP; g.WP = WP; g.P = WP + 1; g.R = HP + 1; g.N = N; return g; }

// ----------------------------------------------------------------------------------------------
// attention geometry and the window / grid partition map
// ----------------------------------------------------------------------------------------------
struct AttnGeom {
  int N, Hl, Wl, C;        // fields, low-res map, channels
  int win, R, X, Y;        // window size, register tokens, windows per column / row
  int grid_mode;           // 0 block partition (maxvit.py:298), 1 grid partition (maxvit.py:322)
  __host__ __device__ int S() const { return R + win * win; }
  __host__ __device__ int nwin() const { return X * Y; }
};
// THE partition map of the package (every kernel that gathers or scatters tokens calls this one function; the device
// test vg_attn_partition_debug dumps it against the einops-generated golden tables): pixel offset, inside its field, of
// window token t (0 .. win*win-1, row-major inside the window) of window wi = x*Y + y.
//   block partition  'b d (x w1) (y w2) -> b x y w1 w2 d'  (maxvit.py:298):  pixel (x*win + w1, y*win + w2)
//   grid partition   'b d (w1 x) (w2 y) -> b x y w1 w2 d'  (maxvit.py:322):  pixel (w1*X + x,  w2*Y + y)
__host__ __device__ __forceinline__ long long attn_token_pixel(const AttnGeom& g, int wi, int t) {
  const int a = t / g.win, b = t - a * g.win;
  const int x = wi / g.Y, y = wi - x * g.Y;
  const int ph = g.grid_mode ? a * g.X + x : x * g.win + a;
  const int pw = g.grid_mode ? b * g.Y + y : y * g.win + b;
  return (long long)ph * g.Wl + pw;
}

// slots of the deterministic (DET) instantiations of the attention core and gather backward
// kernels (vg_bwd_vit.cu, vg_attn_bwd_tc.cu): a kernel parameter of its own after
// the others, so that the parameters of the atomic instantiations keep their offsets
struct AttnDetSlots {
  float* gamma;            // core: [N][2][heads*DH] per-field q / k gamma gradients
  float* bias;             // core: [N][nb][heads] per-field bias-table gradients
  float* film; int K;      // gather: [N][K][2C] per-(field, warp-of-field) dfilm partials (zeroed by the launcher)
  float* reg;              // gather: [N*nwin][R][C] register-row gradients of every window
};

// ----------------------------------------------------------------------------------------------
// dtype traits: activations are bf16 ("bf16 mode") or float ("fp32 mode")
// ----------------------------------------------------------------------------------------------
template <typename T> struct Act;
template <> struct Act<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct Act<bf16> {
  static __device__ __forceinline__ float ld(const bf16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(bf16* p, float v) { *p = __float2bfloat16(v); }
};

// 8 consecutive activations <-> 8 floats (16-byte vector for bf16, 2 x 16 bytes for float)
__device__ __forceinline__ void ld8(const bf16* p, float* v) {
  uint4 u = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void ld8(const float* p, float* v) {
  float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void st8(bf16* p, const float* v) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = u;
}
__device__ __forceinline__ void st8(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// 256-bit global stores (sm_100: STG.E.ENL2.256).  A row-per-thread epilogue store touches 32 different 128-byte lines per warp
// instruction whatever its width; 32 bytes per thread halve the number of store instructions (and LSU wavefronts) per row.
// p must be 32-byte aligned.
__device__ __forceinline__ void st8_256(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void st16_256(bf16* p, const float* v) {
  uint32_t u[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]); u[i] = *reinterpret_cast<uint32_t*>(&h); }
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]),
               "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]) : "memory");
}
__device__ __forceinline__ void st16_256(float* p, const float* v) { st8_256(p, v); st8_256(p + 8, v + 8); }
__device__ __forceinline__ void st16_256(__half* p, const float* v) {
  uint32_t u[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]); u[i] = *reinterpret_cast<uint32_t*>(&h); }
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]),
               "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]) : "memory");
}

// erf by Abramowitz & Stegun 7.1.26 (|error| < 6.1e-7 in fp32 arithmetic, checked against double over [-6, 6]): five FMAs and
// two MUFU ops instead of libdevice erff's two polynomial branches -- the exact-erf GELU (nn.GELU(), maxvit.py:45,48) of
// the 1x1 expand epilogue and the depthwise kernel costs as many issue slots as the convolution arithmetic around it
__device__ __forceinline__ float erf_as(float x) {
  const float ax = fabsf(x);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.0f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  return copysignf(fmaf(-p, __expf(-ax * ax), 1.0f), x);
}
// Two GELUs at once with packed fp32 pairs (FMUL2 / FFMA2 / FADD2 on sm_100: half the issue slots of the polynomial; the two MUFU
// ops per element stay).  Same A&S 7.1.26 arithmetic as erf_as, evaluated as 0.5 x (1 + sign(x) (1 - p(t) e^{-x^2/2})).
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<uint64_t&>(d)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(reinterpret_cast<uint64_t&>(d)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)), "l"(reinterpret_cast<uint64_t&>(c)));
  return d;
}
__device__ __forceinline__ float2 gelu_erf2(float2 x) {
#ifdef VG_EXACT_ERFF
  return make_float2(0.5f * x.x * (1.0f + erff(x.x * 0.70710678118654752440f)), 0.5f * x.y * (1.0f + erff(x.y * 0.70710678118654752440f)));
#else
  const float2 z = f2_mul(x, make_float2(0.70710678118654752440f, 0.70710678118654752440f));
  const float2 az = make_float2(fabsf(z.x), fabsf(z.y));
  const float2 den = f2_fma(make_float2(0.3275911f, 0.3275911f), az, make_float2(1.0f, 1.0f));
  float2 t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(den.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(den.y));
  float2 pp = f2_fma(make_float2(1.061405429f, 1.061405429f), t, make_float2(-1.453152027f, -1.453152027f));
  pp = f2_fma(pp, t, make_float2(1.421413741f, 1.421413741f));
  pp = f2_fma(pp, t, make_float2(-0.284496736f, -0.284496736f));
  pp = f2_fma(pp, t, make_float2(0.254829592f, 0.254829592f));
  pp = f2_mul(pp, t);
  // e^{-z^2} = 2^{x^2 (-log2(e) / 2)}: the exp2 argument straight from x on the packed pipe (no scalar scaling multiply per element)
  const float2 ea = f2_mul(f2_mul(x, x), make_float2(-0.72134752044448170368f, -0.72134752044448170368f));
  float2 e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(ea.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(ea.y));
  const float2 one_m = f2_fma(make_float2(-pp.x, -pp.y), e, make_float2(1.0f, 1.0f));     // erf(|z|)
  const float2 er = make_float2(copysignf(one_m.x, z.x), copysignf(one_m.y, z.y));
  const float2 hx = f2_mul(x, make_float2(0.5f, 0.5f));
  return f2_fma(hx, er, hx);                                                // 0.5 x (1 + erf)
#endif
}
#ifdef VG_EXACT_ERFF
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
#else
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752440f)); }
#endif
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ----------------------------------------------------------------------------------------------
// mbarrier / TMA / tcgen05 (sm_100a)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (-> CUDA error in the host call), never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (((++spins) & 0x3ff) == 0 && (clock64() - t0) > 4000000000LL) {   // ~2 s at 2 GHz
      printf("vitgrid: mbarrier wait timeout (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

// same, with a tag that names the barrier in the timeout message (protocol debugging)
__device__ __forceinline__ void mbar_wait_tag(uint64_t* bar, uint32_t parity, int tag) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (((++spins) & 0x3ff) == 0 && (clock64() - t0) > 1000000000LL) {
      printf("vitgrid: mbarrier wait timeout tag %d parity %u (block %d thread %d)\n", tag, parity, (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// One lane of a CONVERGED warp.  Issue tcgen05.mma / tcgen05.commit inside `if (elect_one()) { ... }` with the whole warp
// running the role code: nvcc then emits back-to-back UTCHMMA.  Under `if (lane == 0)` it wraps EVERY instruction in an
// ELECT / BRA.U.ANY waterfall loop (~60 cycles of issue latency per MMA, whatever its size).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> f32, issued by ONE thread
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// same, operands are fp32 in shared memory read as TF32 (K = 8 per instruction)
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i of the warp = lane base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major operand, SWIZZLE_128B, rows of 64 bf16 (128 B), 8-row atoms 1024 B apart.
// (bits: [0,14) addr>>4, [16,30) LBO>>4 (=1, unused for swizzled K-major), [32,46) SBO>>4 (=64), [46,48) version=1,
//  [61,64) layout=2 (SWIZZLE_128B); base_offset 0 because every stage buffer is 1024-B aligned.)
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// UMMA instruction descriptor: D=f32, A=B=bf16, both K-major, M x N tile
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D=f32, A=B=fp16 (kind::f16 with the fp16 operand format), both K-major
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D=f32, A=B=tf32 (fp32 storage), both K-major
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace vg
