// extern "C" entry points of libvitgrid.so (declared in include/vitgrid.h).
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "../../include/vitgrid.h"
#include "vg_epilogue.cuh"
#include "vg_host.h"

namespace vg {

static thread_local char g_err[512] = "";

int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

static unsigned long long g_launches = 0;

int check_launch(const char* what) {
  ++g_launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error("%s: %s", what, cudaGetErrorString(e));
  return 0;
}

static int* g_deverr_host = nullptr;
static int* g_deverr_dev = nullptr;

int* device_error_ptr() {
  if (!g_deverr_host) {
    int* h = nullptr;
    if (cudaHostAlloc(&h, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    *h = 0;
    int* d = nullptr;
    if (cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) { cudaGetLastError(); cudaFreeHost(h); return nullptr; }
    g_deverr_host = h; g_deverr_dev = d;
  }
  return g_deverr_dev;
}

static EpiParams epi_zero() {
  EpiParams ep;
  memset(&ep, 0, sizeof(ep));
  return ep;
}

}  // namespace vg

using namespace vg;

extern "C" {

int vg_version(void) { return 100; }

long long vg_launch_count(void) { return (long long)g_launches; }

const char* vg_last_error(void) { return g_err; }

int vg_device_error(int clear) {
  if (!g_deverr_host) return 0;
  const int v = *reinterpret_cast<volatile int*>(g_deverr_host);
  if (clear) *reinterpret_cast<volatile int*>(g_deverr_host) = 0;
  return v;
}

int vg_device_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error("no CUDA device: %s", cudaGetErrorString(e));
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) return set_error("libvitgrid is built for sm_100a only; device is sm_%d%d", major, minor);
  return 0;
}

long long vg_pg_pixels(int N, int HP, int WP) { return make_pgeom(N, HP, WP).pixels(); }

int vg_prepare_fwd(int dtype, const float* x, const long long* xstride, int B, int T, int C, int H, int W, int pad_top,
                   int pad_left, int HP, int WP, int Cpad, float pm_mean, float pm_std, void* out, void* stream) {
  return prepare_run(dtype, x, 0, 0, xstride, B, T, C, H, W, pad_top, pad_left, HP, WP, Cpad, pm_mean, pm_std, out,
                     (cudaStream_t)stream);
}

int vg_prepare_packed_fwd(int dtype, const void* x_bf16, const long long* xstride, int B, int T, int C, int H, int W, int pad_top,
                          int pad_left, int HP, int WP, int Cpad, void* out, void* stream) {
  return prepare_run(dtype, x_bf16, 1, 1, xstride, B, T, C, H, W, pad_top, pad_left, HP, WP, Cpad, 0.f, 1.f, out,
                     (cudaStream_t)stream);
}

int vg_prepare_bwd(const float* g, int B, int T, int C, int H, int W, int pad_top, int pad_left, int HP, int WP, int Cpad,
                   float pm_std, int extra_channel, float* dx, void* stream) {
  return prepare_bwd_run(g, B, T, C, H, W, pad_top, pad_left, HP, WP, Cpad, pm_std, extra_channel, dx, (cudaStream_t)stream);
}

int vg_standardise_channel(float* x, const long long* xstride, int B, int T, int C, int H, int W, int channel, float pm_mean,
                           float pm_std, void* stream) {
  return standardise_channel_run(x, xstride, B, T, C, H, W, channel, pm_mean, pm_std, (cudaStream_t)stream);
}

int vg_split3_tf32(const float* in, long long rows, int K, float* out, int pattern, void* stream) {
  return split3_tf32_run(in, rows, K, out, pattern, (cudaStream_t)stream);
}

int vg_time_terms_fwd(const float* ts, long long ts_sB, long long ts_sT, long long ts_sF, int B, int L, int le, int te,
                      const float* emb_lead, const float* emb_month, const float* emb_day, const float* emb_hour,
                      const float* w3, const float* w1, int c_in, int c_data, int Cout, float* temb, float* cond,
                      float* tt, float* tres, void* stream) {
  TimeParams p;
  p.ts = ts; p.ts_sB = ts_sB; p.ts_sT = ts_sT; p.ts_sF = ts_sF;
  p.B = B; p.L = L; p.le = le; p.te = te;
  p.emb_lead = emb_lead; p.emb_m = emb_month; p.emb_d = emb_day; p.emb_h = emb_hour;
  p.w3 = w3; p.w1 = w1; p.c_in = c_in; p.c_data = c_data; p.Cout = Cout;
  p.temb = temb; p.cond = cond; p.tt = tt; p.tres = tres;
  p.err = device_error_ptr();
  return time_terms_run(p, (cudaStream_t)stream);
}

int vg_dense_rows_fwd(const float* in, int N, int in_dim, int pre_relu, const float* W, const float* b, int od, int act,
                      float* out, void* stream) {
  return dense_rows_run(in, N, in_dim, pre_relu, W, b, od, act, out, (cudaStream_t)stream);
}

int vg_cond_mlp_fwd(const float* cond, int N, int cond_dim, int pre_relu, const float* W0, const float* b0, int hid,
                    const float* W1, const float* b1, int od, float* out, void* stream) {
  return cond_mlp_run(cond, N, cond_dim, pre_relu, W0, b0, hid, W1, b1, od, out, (cudaStream_t)stream);
}

int vg_gemm_fwd(int dtype, const void* A, long long rowsA, int Ca, const void* Wt, int Ntot, int ntaps,
                const int* tap_shift, long long M, long long rows_per_batch, int b_rows_per_batch, const float* bias,
                const float* scale, const float* shift, int act, const void* res, long long ldres, int res_f32,
                void* out, long long ldo, int out_f32, float* scratch, long long scratch_elems, void* stream) {
  EpiParams ep = epi_zero();
  ep.out = out; ep.ldo = ldo; ep.out_f32 = out_f32; ep.n_total = Ntot;
  ep.bias = bias; ep.col_scale = scale; ep.col_shift = shift; ep.act = act; ep.res = res; ep.ldres = ldres;
  ep.res_f32 = res_f32;
  if ((scale == nullptr) != (shift == nullptr)) return set_error("gemm: scale and shift must be given together");
  return gemm_run(dtype, EPI_STORE, A, rowsA, Ca, Wt, Ntot, ntaps, tap_shift, M, rows_per_batch, b_rows_per_batch, ep,
                  scratch, scratch_elems, (cudaStream_t)stream);
}

int vg_conv3x3_ln_fwd(int dtype, const void* x, int Ca, const void* Wt, const float* bias, const float* ln_g,
                      const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, void* out,
                      float* out_f32_copy, int N, int HP, int WP, const float* head_w, float head_b, float head_std,
                      float head_mean, int H, int W, int pad_top, int pad_left, float* head_out, float* scratch,
                      long long scratch_elems, void* stream) {
  PGeom pg = make_pgeom(N, HP, WP);
  EpiParams ep = epi_zero();
  ep.out = out; ep.ldo = 128; ep.n_total = 128; ep.bias = bias; ep.ln_g = ln_g; ep.ln_b = ln_b; ep.ln_eps = ln_eps;
  ep.film = film; ep.res = res; ep.ldres = 128; ep.pg = pg; ep.res_f32 = res_f32; ep.out2 = out_f32_copy;
  ep.head_w = head_w; ep.head_out = head_out; ep.head_b = head_b; ep.head_std = head_std; ep.head_mean = head_mean;
  ep.head_H = H; ep.head_W = W; ep.head_pt = pad_top; ep.head_pl = pad_left;
  if (!out && !head_w) return set_error("conv3x3_ln: no output requested");
  if (head_w && !head_out) return set_error("conv3x3_ln: head_w without head_out");
  if (dtype == 0 && Ca == 128) {                     // halo-reuse kernel (falls through when the row pitch is too large)
    const int rc = conv_halo_run(x, Wt, pg, ep, 0, (cudaStream_t)stream);
    if (rc >= 0) return rc;
  }
  int shifts[9];
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) shifts[ky * 3 + kx] = (ky - 1) * pg.P + (kx - 1);
  return gemm_run(dtype, EPI_CONV_LN, x, pg.pixels(), Ca, Wt, 128, 9, shifts, pg.pixels(), 0, 0, ep, scratch,
                  scratch_elems, (cudaStream_t)stream);
}

int vg_conv3x3_ln_train_fwd(int dtype, const void* x, int Ca, const void* Wt, const float* bias, const float* ln_g,
                            const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, void* out,
                            float* out_f32_copy, void* xhat, float* rstd, void* relu_mask, int N, int HP, int WP,
                            float* scratch, long long scratch_elems, void* stream) {
  PGeom pg = make_pgeom(N, HP, WP);
  EpiParams ep = epi_zero();
  ep.out = out; ep.ldo = 128; ep.n_total = 128; ep.bias = bias; ep.ln_g = ln_g; ep.ln_b = ln_b; ep.ln_eps = ln_eps;
  ep.film = film; ep.res = res; ep.ldres = 128; ep.pg = pg; ep.res_f32 = res_f32; ep.out2 = out_f32_copy;
  ep.xhat = xhat; ep.rstd_out = rstd; ep.relu_mask = reinterpret_cast<unsigned*>(relu_mask);
  if (!out || !xhat || !rstd || !relu_mask) return set_error("conv3x3_ln_train: out, xhat, rstd and relu_mask are required");
  if (dtype == 0 && Ca == 128) {
    const int rc = conv_halo_run(x, Wt, pg, ep, 1, (cudaStream_t)stream);
    if (rc >= 0) return rc;
  }
  int shifts[9];
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) shifts[ky * 3 + kx] = (ky - 1) * pg.P + (kx - 1);
  return gemm_run(dtype, EPI_CONV_LN_TRAIN, x, pg.pixels(), Ca, Wt, 128, 9, shifts, pg.pixels(), 0, 0, ep, scratch,
                  scratch_elems, (cudaStream_t)stream);
}

int vg_stem_finish_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                       const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                       const float* film, int B, int L, int HP, int WP, void* h1, float* res, void* stream) {
  StemParams p;
  p.raw3 = raw3; p.rawres = rawres; p.bias3 = bias3; p.bias1 = bias1; p.tt = tt; p.tres = tres;
  p.ln_g = ln_g; p.ln_b = ln_b; p.eps = ln_eps; p.film = film; p.L = L;
  p.xhat = nullptr; p.rstd = nullptr; p.mask = nullptr;
  p.pgB = make_pgeom(B, HP, WP); p.pgN = make_pgeom(B * L, HP, WP);
  return stem_finish_run(dtype, p, h1, res, (cudaStream_t)stream);
}

int vg_stem_finish_train_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                             const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                             const float* film, int B, int L, int HP, int WP, void* h1, float* res, void* xhat, float* rstd,
                             void* relu_mask, void* stream) {
  StemParams p;
  p.raw3 = raw3; p.rawres = rawres; p.bias3 = bias3; p.bias1 = bias1; p.tt = tt; p.tres = tres;
  p.ln_g = ln_g; p.ln_b = ln_b; p.eps = ln_eps; p.film = film; p.L = L;
  p.xhat = xhat; p.rstd = rstd; p.mask = reinterpret_cast<unsigned*>(relu_mask);
  if (!xhat || !rstd || !relu_mask) return set_error("stem_finish_train: xhat, rstd and relu_mask are required");
  p.pgB = make_pgeom(B, HP, WP); p.pgN = make_pgeom(B * L, HP, WP);
  return stem_finish_run(dtype, p, h1, res, (cudaStream_t)stream);
}

int vg_conv3x3_ln_wide_fwd(int dtype, const void* x, int C, const void* Wt, const float* bias, const float* ln_g,
                           const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, void* out,
                           float* out_f32_copy, int N, int HP, int WP, const float* head_w, float head_b, float head_std,
                           float head_mean, int H, int W, int pad_top, int pad_left, float* head_out, float* scratch,
                           long long scratch_elems, void* stream) {
  PGeom pg = make_pgeom(N, HP, WP);
  if (!out && !head_w) return set_error("conv3x3_ln_wide: no output requested");
  if (head_w && !head_out) return set_error("conv3x3_ln_wide: head_w without head_out");
  if (C % 128 || C < 128 || C > 512) return set_error("conv3x3_ln_wide: C=%d must be 128, 256, 384 or 512", C);
  const long long need = pg.pixels() * (long long)C * (dtype == 1 ? 2 : 1);
  if (scratch_elems < need) return set_error("conv3x3_ln_wide: scratch too small (%lld < %lld floats)", scratch_elems, need);
  int shifts[9];
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) shifts[ky * 3 + kx] = (ky - 1) * pg.P + (kx - 1);
  // 1. shifted-row GEMM, fp32 result [q][C]   (fp32 mode: the SIMT kernel accumulates in the second half of the scratch)
  EpiParams ep = epi_zero();
  ep.out = scratch; ep.ldo = C; ep.out_f32 = 1; ep.n_total = C;
  int rc = gemm_run(dtype, EPI_STORE, x, pg.pixels(), C, Wt, C, 9, shifts, pg.pixels(), 0, 0, ep, scratch + pg.pixels() * (long long)C,
                    scratch_elems - pg.pixels() * (long long)C, (cudaStream_t)stream);
  if (rc) return rc;
  // 2. bias, channel LayerNorm, FiLM, ReLU, residual, pads, optional head
  return conv_ln_rows_run(dtype, scratch, C, bias, ln_g, ln_b, ln_eps, film, res, res_f32, out, out_f32_copy, pg, head_w, head_b,
                          head_std, head_mean, H, W, pad_top, pad_left, head_out, (cudaStream_t)stream);
}

int vg_stem_finish_wide_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                            const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                            const float* film, int B, int L, int HP, int WP, int C, void* h1, float* res, void* stream) {
  StemParams p;
  p.raw3 = raw3; p.rawres = rawres; p.bias3 = bias3; p.bias1 = bias1; p.tt = tt; p.tres = tres;
  p.ln_g = ln_g; p.ln_b = ln_b; p.eps = ln_eps; p.film = film; p.L = L;
  p.xhat = nullptr; p.rstd = nullptr; p.mask = nullptr;
  p.pgB = make_pgeom(B, HP, WP); p.pgN = make_pgeom(B * L, HP, WP);
  return stem_finish_wide_run(dtype, p, C, h1, res, (cudaStream_t)stream);
}

int vg_conv3x3_ln_wide_train_fwd(int dtype, const void* x, int C, const void* Wt, const float* bias, const float* ln_g,
                                 const float* ln_b, float ln_eps, const float* film, const void* res, int res_f32, float* out,
                                 float* out_f32_copy, float* xhat, float* rstd, void* relu_mask, int N, int HP, int WP, float* scratch,
                                 long long scratch_elems, void* stream) {
  PGeom pg = make_pgeom(N, HP, WP);
  if (dtype != 1 && dtype != 2) return set_error("conv3x3_ln_wide_train: dtype %d (1 = fp32 SIMT, 2 = tf32 tensor cores)", dtype);
  if (!out || !xhat || !rstd || !relu_mask) return set_error("conv3x3_ln_wide_train: out, xhat, rstd and relu_mask are required");
  if (C % 128 || C < 128 || C > 512) return set_error("conv3x3_ln_wide_train: C=%d must be 128, 256, 384 or 512", C);
  const long long need = pg.pixels() * (long long)C * (dtype == 1 ? 2 : 1);
  if (scratch_elems < need) return set_error("conv3x3_ln_wide_train: scratch too small (%lld < %lld floats)", scratch_elems, need);
  int shifts[9];
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) shifts[ky * 3 + kx] = (ky - 1) * pg.P + (kx - 1);
  EpiParams ep = epi_zero();
  ep.out = scratch; ep.ldo = C; ep.out_f32 = 1; ep.n_total = C;
  int rc = gemm_run(dtype, EPI_STORE, x, pg.pixels(), C, Wt, C, 9, shifts, pg.pixels(), 0, 0, ep, scratch + pg.pixels() * (long long)C,
                    scratch_elems - pg.pixels() * (long long)C, (cudaStream_t)stream);
  if (rc) return rc;
  return conv_ln_rows_train_run(scratch, C, bias, ln_g, ln_b, ln_eps, film, res, res_f32, out, out_f32_copy, xhat, rstd,
                                reinterpret_cast<unsigned*>(relu_mask), pg, (cudaStream_t)stream);
}

int vg_stem_finish_wide_train_fwd(int dtype, const float* raw3, const float* rawres, const float* bias3, const float* bias1,
                                  const float* tt, const float* tres, const float* ln_g, const float* ln_b, float ln_eps,
                                  const float* film, int B, int L, int HP, int WP, int C, float* h1, float* res, float* xhat,
                                  float* rstd, void* relu_mask, void* stream) {
  if (!xhat || !rstd || !relu_mask) return set_error("stem_finish_wide_train: xhat, rstd and relu_mask are required");
  StemParams p;
  p.raw3 = raw3; p.rawres = rawres; p.bias3 = bias3; p.bias1 = bias1; p.tt = tt; p.tres = tres;
  p.ln_g = ln_g; p.ln_b = ln_b; p.eps = ln_eps; p.film = film; p.L = L;
  p.xhat = xhat; p.rstd = rstd; p.mask = reinterpret_cast<unsigned*>(relu_mask);
  p.pgB = make_pgeom(B, HP, WP); p.pgN = make_pgeom(B * L, HP, WP);
  return stem_finish_wide_run(dtype, p, C, h1, res, (cudaStream_t)stream);
}

int vg_pool2_fwd(int dtype, int out_f32, const void* in, void* out, int N, int HP, int WP, int C, void* stream) {
  return maxpool2_run(dtype, out_f32, in, out, N, HP, WP, C, (cudaStream_t)stream);
}

int vg_dw3x3_bnact_fwd(int dtype, const void* in, const float* w9, const float* scale, const float* shift, void* out,
                       float* psum, int N, int H, int W, int C, void* stream) {
  return dwconv_run(dtype, in, w9, scale, shift, out, psum, N, H, W, C, (cudaStream_t)stream);
}

int vg_se_scale_fwd(int dtype, void* x, const float* gate, int N, long long HW, int C, void* stream) {
  return se_scale_run(dtype, x, gate, N, HW, C, (cudaStream_t)stream);
}

static int make_attn_geom(AttnGeom& g, int N, int Hl, int Wl, int C, int win, int R, int grid_mode) {
  if (win <= 0 || Hl % win || Wl % win) return set_error("attention: map %dx%d not divisible by window %d", Hl, Wl, win);
  g.N = N; g.Hl = Hl; g.Wl = Wl; g.C = C; g.win = win; g.R = R; g.X = Hl / win; g.Y = Wl / win; g.grid_mode = grid_mode;
  return 0;
}

int vg_attn_partition_debug(int N, int Hl, int Wl, int win, int R, int grid_mode, long long* pixel_index, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, 128, win, R, grid_mode)) return 1;
  return attn_partition_debug_run(g, pixel_index, (cudaStream_t)stream);
}

int vg_attn_gather_fwd(int dtype, const void* x, const float* reg, int reg_per_field, const float* film, int N, int Hl,
                       int Wl, int C, int win, int R, int grid_mode, float ln_eps, void* tokens, int tokens_bf16, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, grid_mode)) return 1;
  return attn_gather_run(dtype, x, reg, reg_per_field, film, g, ln_eps, tokens, tokens_bf16, (cudaStream_t)stream);
}

int vg_attn_core_fwd(int dtype, const void* qkv, const float* q_gamma, const float* k_gamma, const float* bias_table,
                     int N, int Hl, int Wl, int win, int R, int heads, int dh, void* out, long long drop_seed, int drop_salt,
                     int drop_thresh, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, 0, win, R, 0)) return 1;
  return attn_core_run(dtype, qkv, q_gamma, k_gamma, bias_table, g, heads, dh, out, (unsigned)drop_seed, (unsigned)drop_salt,
                       drop_thresh, (cudaStream_t)stream);
}

int vg_attn_out_fwd(int dtype, const void* attn, int inner, const void* Wt, const void* x_in, const float* reg_in,
                    int reg_per_field, float* reg_out, void* x_out, int N, int Hl, int Wl, int C, int win, int R,
                    int grid_mode, long long drop_seed, int drop_salt, int drop_thresh, float* scratch, long long scratch_elems,
                    void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, grid_mode)) return 1;
  EpiParams ep = epi_zero();
  ep.out = x_out; ep.n_total = C; ep.S = g.S(); ep.R = R; ep.nwin = g.nwin(); ep.grid_mode = grid_mode; ep.win = win;
  ep.X = g.X; ep.Y = g.Y; ep.Hl = Hl; ep.Wl = Wl; ep.x_in = x_in; ep.reg_in = reg_in;
  ep.reg_in_per_field = reg_per_field; ep.reg_out = reg_out;
  if (drop_thresh < 0 || drop_thresh > 255) return set_error("attn_out: dropout threshold %d outside [0, 255]", drop_thresh);
  ep.drop_seed = (unsigned)drop_seed; ep.drop_salt = (unsigned)drop_salt; ep.drop_thresh = drop_thresh;
  ep.drop_scale = 256.0f / (256.0f - (float)drop_thresh);
  const long long M = (long long)N * g.nwin() * g.S();
  const int shift0 = 0;
  return gemm_run(dtype, EPI_ATTN_OUT, attn, M, inner, Wt, C, 1, &shift0, M, 0, 0, ep, scratch, scratch_elems,
                  (cudaStream_t)stream);
}

int vg_attn_fused2_fwd(float* xio, const float* reg_in, int reg_per_field, float* reg_out, const float* film, const void* wqkv_h,
                       const float* wout_h, const float* head_tab, int N, int Hl, int Wl, int C, int win, int R, int grid_mode, int heads,
                       int dh, float ln_eps, long long drop_seed, int drop_salt, int drop_thresh, float logit_bound, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, grid_mode)) return 1;
  return attn_fused2_run(xio, reg_in, reg_per_field, reg_out, film, wqkv_h, wout_h, head_tab, g, heads, dh, ln_eps,
                         (unsigned)drop_seed, (unsigned)drop_salt, drop_thresh, logit_bound, (cudaStream_t)stream);
}

int vg_reg_mean_fwd(const float* in, float* out, int N, int nwin, int RC, void* stream) {
  return reg_mean_run(in, out, N, nwin, RC, (cudaStream_t)stream);
}

int vg_convT2_fwd(int dtype, int out_bf16, const void* x, const void* Wt, const float* bias, void* out, float* out_f32_copy,
                  int N, int Hl, int Wl, int C, float* scratch, long long scratch_elems, void* stream) {
  EpiParams ep = epi_zero();
  ep.out = out; ep.ldo = C; ep.out_f32 = out_bf16 ? 2 : 0; ep.out2 = out_f32_copy; ep.n_total = 4 * C; ep.bias = bias; ep.Hl = Hl; ep.Wl = Wl;
  ep.pg = make_pgeom(N, 2 * Hl, 2 * Wl);
  if (C % 128) return set_error("convT2: C=%d must be a multiple of 128", C);
  const long long M = (long long)N * Hl * Wl;
  const int shift0 = 0;
  return gemm_run(dtype, EPI_CONVT, x, M, C, Wt, 4 * C, 1, &shift0, M, 0, 0, ep, scratch, scratch_elems,
                  (cudaStream_t)stream);
}

int vg_head_fwd(int dtype, const void* h, const float* w, float bias, float pm_std, float pm_mean, int N, int HP, int WP,
                int C, int H, int W, int pad_top, int pad_left, float* out, void* stream) {
  return head_run(dtype, h, w, bias, pm_std, pm_mean, N, HP, WP, C, H, W, pad_top, pad_left, out, (cudaStream_t)stream);
}

long long vg_eval_metrics_workspace(int B, int L, int P) { return eval_metrics_workspace_run(B, L, P); }

int vg_eval_metrics(float* preds, const float* truth, const void* truth_class, int class_is_i64, const float* persist,
                    const float* sim_21h, const float* sim_avg, int B, int L, int P, float b1, float b2, float b3,
                    int clamp_preds, void* counts, double* sums, double* glob, void* nonzero, double* loss_sum, double* work,
                    long long work_elems, void* stream) {
  if (!preds || !truth || !truth_class || !persist || !sim_21h || !sim_avg) return set_error("eval_metrics: null input");
  if (!counts || !sums || !glob || !nonzero || !loss_sum || !work) return set_error("eval_metrics: null accumulator");
  return eval_metrics_run(preds, truth, truth_class, class_is_i64, persist, sim_21h, sim_avg, B, L, P, b1, b2, b3, clamp_preds,
                          reinterpret_cast<unsigned long long*>(counts), sums, glob, reinterpret_cast<unsigned long long*>(nonzero),
                          loss_sum, work, work_elems, (cudaStream_t)stream);
}

int vg_focal_r_fwd(const float* pred, const float* target, long long n, float beta, float gamma, int mse, float* partial,
                   int nblocks, float* loss, void* stream) {
  return focal_r_fwd_run(pred, target, n, beta, gamma, mse, partial, nblocks, loss, (cudaStream_t)stream);
}

int vg_focal_r_bwd(const float* pred, const float* target, long long n, float beta, float gamma, int mse, float gscale,
                   float* grad, void* stream) {
  return focal_r_bwd_run(pred, target, n, beta, gamma, mse, gscale, grad, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ training
int vg_conv_ln_bwd(int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const void* relu_mask,
                   const float* ln_g, const float* film, float ln_eps, void* dconv, float* sumA, float* sumB, float* sumD,
                   float* border, int N, int HP, int WP, void* stream) {
  return conv_ln_bwd_run(xdtype, odtype, dY, xhat, rstd, reinterpret_cast<const unsigned*>(relu_mask), ln_g, film, ln_eps,
                         dconv, sumA, sumB, sumD, border, N, HP, WP, (cudaStream_t)stream);
}

int vg_conv_ln_param_grads(const float* sumA, const float* sumB, const float* sumD, int N, const float* ln_g,
                           const float* ln_b, const float* film, float* dg, float* db, float* dbias, float* dfilm,
                           void* stream) {
  return conv_ln_param_grads_run(sumA, sumB, sumD, N, ln_g, ln_b, film, dg, db, dbias, dfilm, 128, (cudaStream_t)stream);
}

int vg_conv_ln_bwd_wide(int C, const float* dY, const float* xhat, const float* rstd, const void* relu_mask, const float* ln_g,
                        const float* film, float ln_eps, float* dconv, float* sumA, float* sumB, float* sumD, float* border, int N,
                        int HP, int WP, void* stream) {
  return conv_ln_bwd_wide_run(C, dY, xhat, rstd, reinterpret_cast<const unsigned*>(relu_mask), ln_g, film, ln_eps, dconv, sumA, sumB,
                              sumD, border, N, HP, WP, (cudaStream_t)stream);
}

int vg_conv_ln_param_grads_wide(const float* sumA, const float* sumB, const float* sumD, int N, int C, const float* ln_g,
                                const float* ln_b, const float* film, float* dg, float* db, float* dbias, float* dfilm, void* stream) {
  return conv_ln_param_grads_run(sumA, sumB, sumD, N, ln_g, ln_b, film, dg, db, dbias, dfilm, C, (cudaStream_t)stream);
}

long long vg_wgrad_workspace(int dtype, long long M, int Ntot, int Ca, int ntaps) {
  return wgrad_workspace_elems(dtype, M, Ntot, Ca, ntaps);
}

int vg_wgrad(int dtype, const void* dY, const void* A, long long rowsA, long long M, int Ntot, int Ca, int ntaps,
             const int* tap_shift, float* dW, float beta, float* work, long long work_elems, void* stream) {
  return wgrad_run(dtype, dY, A, rowsA, M, Ntot, Ca, ntaps, tap_shift, dW, beta, work, work_elems, (cudaStream_t)stream);
}

int vg_head_bwd(int dtype, const float* dpred, const void* h, const float* w, float pm_std, int N, int HP, int WP, int H,
                int W, int pad_top, int pad_left, float* dH, float* dw, float* db, void* stream) {
  return head_bwd_run(dtype, dpred, h, w, pm_std, N, HP, WP, H, W, pad_top, pad_left, dH, dw, db, 128, (cudaStream_t)stream);
}

int vg_head_bwd_wide(int dtype, const float* dpred, const void* h, const float* w, float pm_std, int N, int HP, int WP, int C, int H,
                     int W, int pad_top, int pad_left, float* dH, float* dw, float* db, void* stream) {
  return head_bwd_run(dtype, dpred, h, w, pm_std, N, HP, WP, H, W, pad_top, pad_left, dH, dw, db, C, (cudaStream_t)stream);
}

int vg_pool2_bwd(int dtype, const void* x, const float* dlow, float* dx, int N, int HP, int WP, int C, void* stream) {
  return maxpool2_bwd_run(dtype, x, dlow, dx, N, HP, WP, C, (cudaStream_t)stream);
}

int vg_convT2_bwd_gather(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, void* stream) {
  return convT_bwd_gather_run(odtype, dUp, G, dbias, N, Hl, Wl, C, (cudaStream_t)stream);
}

int vg_lead_sum(int idtype, int odtype, const void* in, void* out, int B, int L, int HP, int WP, void* stream) {
  return lead_sum_run(idtype, odtype, in, out, B, L, HP, WP, 128, (cudaStream_t)stream);
}

int vg_lead_sum_wide(int idtype, int odtype, const void* in, void* out, int B, int L, int HP, int WP, int C, void* stream) {
  return lead_sum_run(idtype, odtype, in, out, B, L, HP, WP, C, (cudaStream_t)stream);
}

int vg_pg_field_sum(const float* in, float* out, int N, int HP, int WP, void* stream) {
  return pg_field_sum_run(in, out, N, HP, WP, 128, (cudaStream_t)stream);
}

int vg_pg_field_sum_wide(const float* in, float* out, int N, int HP, int WP, int C, void* stream) {
  return pg_field_sum_run(in, out, N, HP, WP, C, (cudaStream_t)stream);
}

int vg_time_terms_bwd(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                      const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                      float* dtemb, void* stream) {
  return time_terms_bwd_run(border, sumD, tres_sum, temb, w3, w1, N, ntc, c_in, c_data, Cout, dw3, dw1, db1, dtemb,
                            (cudaStream_t)stream);
}

int vg_time_embed_bwd(const float* dtemb, const float* dcond, const float* ts, long long ts_sB, long long ts_sT,
                      long long ts_sF, int B, int L, int le, int te, float* d_lead, float* d_month, float* d_day,
                      float* d_hour, void* stream) {
  return time_embed_bwd_run(dtemb, dcond, ts, ts_sB, ts_sT, ts_sF, B, L, le, te, d_lead, d_month, d_day, d_hour,
                            (cudaStream_t)stream);
}

int vg_cond_mlp_bwd(const float* cond, int N, int cond_dim, int pre_relu, const float* W0, const float* b0, int hid,
                    const float* W1, int od, const float* dout, float* dW0, float* db0, float* dW1, float* db1,
                    float* dcond, float* work, long long work_elems, void* stream) {
  return cond_mlp_bwd_run(cond, N, cond_dim, pre_relu, W0, b0, hid, W1, od, dout, dW0, db0, dW1, db1, dcond, work,
                          work_elems, (cudaStream_t)stream);
}

int vg_adamw_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, float gscale, void* stream) {
  return adamw_run(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step, gscale, (cudaStream_t)stream);
}

long long vg_bn_workspace(long long M, int C) { return bn_workspace_elems(M, C); }

int vg_bn_stats(const float* x, long long M, int C, const float* gamma, const float* beta, float eps, float momentum,
                float* running_mean, float* running_var, float* mean, float* rstd, float* scale, float* shift,
                float* work, long long work_elems, void* stream) {
  return bn_stats_run(x, M, C, gamma, beta, eps, momentum, running_mean, running_var, mean, rstd, scale, shift, work,
                      work_elems, (cudaStream_t)stream);
}

int vg_bn_act(const float* raw, const float* scale, const float* shift, int act, const float* res, float* out,
              long long M, int C, void* stream) {
  return bn_act_run(raw, scale, shift, act, res, out, M, C, (cudaStream_t)stream);
}

int vg_bn_bwd(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean,
              const float* rstd, const float* gamma, int act, const float* fgate, const float* fadd,
              long long rows_per_field, long long M, int C, float* dgamma, float* dbeta, float* draw, float* work,
              long long work_elems, void* stream) {
  return bn_bwd_run(dOut, raw, scale, shift, mean, rstd, gamma, act, fgate, fadd, rows_per_field, M, C, dgamma, dbeta, draw,
                    work, work_elems, (cudaStream_t)stream);
}

int vg_bn_bwd_frozen(const float* dOut, const float* raw, const float* scale, const float* shift, const float* running_mean,
                     const float* running_rstd, int act, const float* fgate, const float* fadd, long long rows_per_field, long long M,
                     int C, float* dgamma, float* dbeta, float* draw, float* work, long long work_elems, void* stream) {
  return bn_bwd_frozen_run(dOut, raw, scale, shift, running_mean, running_rstd, act, fgate, fadd, rows_per_field, M, C, dgamma, dbeta,
                           draw, work, work_elems, (cudaStream_t)stream);
}

int vg_colsum(const float* x, long long M, int C, float* out, void* stream) { return colsum_run(x, M, C, out, (cudaStream_t)stream); }

int vg_dw_strips(int W) { return dwconv_strips(W); }

int vg_dw3x3_fwd(int dtype, const void* in, const float* w9, const float* scale, const float* shift, int act, void* out,
                 float* psum, int N, int H, int W, int C, void* stream) {
  return dwconv_march_run(dtype, in, w9, scale, shift, act, out, psum, N, H, W, C, (cudaStream_t)stream);
}

int vg_dw3x3_wgrad(const float* x, const float* dY, int N, int H, int W, int C, float* dw9, float* dbias, float* work,
                   long long work_elems, void* stream) {
  return dw_wgrad_run(x, dY, N, H, W, C, dw9, dbias, work, work_elems, (cudaStream_t)stream);
}

int vg_se_gate_train_fwd(const float* psum, int N, int nparts, long long HW, const float* W1, const float* W2, int C,
                         int se, float* gate, float* mean, float* hid, void* stream) {
  return se_gate_train_run(psum, N, nparts, HW, W1, W2, C, se, gate, mean, hid, (cudaStream_t)stream);
}

int vg_field_parts(long long HW) { return field_parts(HW); }

int vg_field_dot(const float* a, const float* b, float* out, int N, long long HW, int C, void* stream) {
  return field_dot_run(a, b, out, N, HW, C, (cudaStream_t)stream);
}

int vg_se_fold_weights(const float* W, const float* gate, void* out, int out_f16, int N, int Cout, int C, void* stream) {
  return se_fold_run(W, gate, out, out_f16, N, Cout, C, (cudaStream_t)stream);
}

int vg_se_scale_oop(const float* x, const float* gate, float* out, int N, long long HW, int C, void* stream) {
  return se_scale_oop_run(x, gate, out, N, HW, C, (cudaStream_t)stream);
}

int vg_se_bwd(const float* dh4, const float* h3, const float* gate, const float* mean, const float* hid, const float* W1,
              const float* W2, int N, long long HW, int C, int se, float* dW1, float* dW2, float* dmean, float* work,
              long long work_elems, void* stream) {
  return se_bwd_run(dh4, h3, gate, mean, hid, W1, W2, N, HW, C, se, dW1, dW2, dmean, work, work_elems, (cudaStream_t)stream);
}

int vg_attn_out_bwd_gather(const float* dx_out, const float* dreg, float reg_scale, int N, int Hl, int Wl, int C, int win,
                           int R, int grid_mode, void* dproj, int dproj_bf16, long long drop_seed, int drop_salt, int drop_thresh,
                           void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, grid_mode)) return 1;
  return attn_out_bwd_gather_run(dx_out, dreg, reg_scale, g, dproj, dproj_bf16, (unsigned)drop_seed, (unsigned)drop_salt, drop_thresh,
                                 (cudaStream_t)stream);
}

int vg_dropout_mask_debug(long long drop_seed, int drop_salt, int drop_thresh, long long n_windows, int heads, int C,
                          int slots, void* prob_mask, void* out_mask, void* stream) {
  return dropout_mask_debug_run((unsigned)drop_seed, (unsigned)drop_salt, drop_thresh, n_windows, heads, C, slots,
                                reinterpret_cast<unsigned char*>(prob_mask), reinterpret_cast<unsigned char*>(out_mask),
                                (cudaStream_t)stream);
}

int vg_attn_core_bwd(const void* qkv, const void* datt, const float* q_gamma, const float* k_gamma,
                     const float* bias_table, int N, int Hl, int Wl, int win, int R, int heads, int dh, void* dqkv,
                     float* dq_gamma, float* dk_gamma, float* dbias_table, int use_tf32, void* att_out, long long drop_seed,
                     int drop_salt, int drop_thresh, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, 0, win, R, 0)) return 1;
  return attn_core_bwd_run(reinterpret_cast<const float*>(qkv), reinterpret_cast<const float*>(datt), q_gamma, k_gamma, bias_table, g, heads, dh, reinterpret_cast<float*>(dqkv), dq_gamma, dk_gamma, dbias_table,
                           use_tf32, reinterpret_cast<float*>(att_out), (unsigned)drop_seed, (unsigned)drop_salt, drop_thresh, (cudaStream_t)stream);
}

int vg_attn_gather_bwd(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                       const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in,
                       float* dfilm, int N, int Hl, int Wl, int C, int win, int R, int grid_mode, float ln_eps,
                       void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, grid_mode)) return 1;
  return attn_gather_bwd_run(x, reg, reg_per_field, film, dtok, dx_out, dreg_res, reg_scale, dx_in, dreg_in, dfilm, g, ln_eps,
                             (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ deterministic backward
long long vg_conv_ln_bwd_det_workspace(int C, int N, int HP, int WP) { return conv_ln_bwd_det_workspace_elems(C, N, HP, WP); }

int vg_conv_ln_bwd_det(int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const void* relu_mask,
                       const float* ln_g, const float* film, float ln_eps, void* dconv, float* sumA, float* sumB, float* sumD,
                       float* border, int N, int HP, int WP, float* work, long long work_elems, void* stream) {
  return conv_ln_bwd_det_run(128, xdtype, odtype, dY, xhat, rstd, reinterpret_cast<const unsigned*>(relu_mask), ln_g, film, ln_eps,
                             dconv, sumA, sumB, sumD, border, N, HP, WP, work, work_elems, (cudaStream_t)stream);
}

int vg_conv_ln_bwd_wide_det(int C, const float* dY, const float* xhat, const float* rstd, const void* relu_mask,
                            const float* ln_g, const float* film, float ln_eps, float* dconv, float* sumA, float* sumB,
                            float* sumD, float* border, int N, int HP, int WP, float* work, long long work_elems, void* stream) {
  if (C == 128) return set_error("conv_ln_bwd_wide_det: C=128 is vg_conv_ln_bwd_det");
  return conv_ln_bwd_det_run(C, 1, 1, dY, xhat, rstd, reinterpret_cast<const unsigned*>(relu_mask), ln_g, film, ln_eps, dconv,
                             sumA, sumB, sumD, border, N, HP, WP, work, work_elems, (cudaStream_t)stream);
}

long long vg_head_bwd_det_workspace(int N, int HP, int WP, int C) { return head_bwd_det_workspace_elems(N, HP, WP, C); }

int vg_head_bwd_det(int dtype, const float* dpred, const void* h, const float* w, float pm_std, int N, int HP, int WP, int C,
                    int H, int W, int pad_top, int pad_left, float* dH, float* dw, float* db, float* work, long long work_elems,
                    void* stream) {
  return head_bwd_det_run(dtype, dpred, h, w, pm_std, N, HP, WP, H, W, pad_top, pad_left, dH, dw, db, C, work, work_elems,
                          (cudaStream_t)stream);
}

long long vg_convT2_bwd_gather_det_workspace(int N, int Hl, int Wl, int C) { return convT_bwd_gather_det_workspace_elems(N, Hl, Wl, C); }

int vg_convT2_bwd_gather_det(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, float* work,
                             long long work_elems, void* stream) {
  return convT_bwd_gather_det_run(odtype, dUp, G, dbias, N, Hl, Wl, C, work, work_elems, (cudaStream_t)stream);
}

long long vg_pg_field_sum_det_workspace(int N, int HP, int WP, int C) { return pg_field_sum_det_workspace_elems(N, HP, WP, C); }

int vg_pg_field_sum_det(const float* in, float* out, int N, int HP, int WP, int C, float* work, long long work_elems,
                        void* stream) {
  return pg_field_sum_det_run(in, out, N, HP, WP, C, work, work_elems, (cudaStream_t)stream);
}

long long vg_time_terms_bwd_det_workspace(int N, int Cout) { return time_terms_bwd_det_workspace_elems(N, Cout); }

int vg_time_terms_bwd_det(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                          const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                          float* dtemb, float* work, long long work_elems, void* stream) {
  return time_terms_bwd_det_run(border, sumD, tres_sum, temb, w3, w1, N, ntc, c_in, c_data, Cout, dw3, dw1, db1, dtemb, work,
                                work_elems, (cudaStream_t)stream);
}

long long vg_time_embed_bwd_det_workspace(int, int, int, int) { return 0; }

int vg_time_embed_bwd_det(const float* dtemb, const float* dcond, const float* ts, long long ts_sB, long long ts_sT,
                          long long ts_sF, int B, int L, int le, int te, float* d_lead, float* d_month, float* d_day,
                          float* d_hour, float*, long long, void* stream) {
  return time_embed_bwd_det_run(dtemb, dcond, ts, ts_sB, ts_sT, ts_sF, B, L, le, te, d_lead, d_month, d_day, d_hour,
                                (cudaStream_t)stream);
}

long long vg_colsum_det_workspace(long long M, int C) { return colsum_det_workspace_elems(M, C); }

int vg_colsum_det(const float* x, long long M, int C, float* out, float* work, long long work_elems, void* stream) {
  return colsum_det_run(x, M, C, out, work, work_elems, (cudaStream_t)stream);
}

long long vg_attn_core_bwd_det_workspace(int N, int Hl, int Wl, int win, int R, int heads, int dh) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, 0, win, R, 0)) return -1;
  return attn_core_bwd_det_workspace_elems(g, heads, dh);
}

int vg_attn_core_bwd_det(const void* qkv, const void* datt, const float* q_gamma, const float* k_gamma,
                         const float* bias_table, int N, int Hl, int Wl, int win, int R, int heads, int dh, void* dqkv,
                         float* dq_gamma, float* dk_gamma, float* dbias_table, int use_tf32, void* att_out, long long drop_seed,
                         int drop_salt, int drop_thresh, float* work, long long work_elems, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, 0, win, R, 0)) return 1;
  return attn_core_bwd_det_run(reinterpret_cast<const float*>(qkv), reinterpret_cast<const float*>(datt), q_gamma, k_gamma,
                               bias_table, g, heads, dh, reinterpret_cast<float*>(dqkv), dq_gamma, dk_gamma, dbias_table, use_tf32,
                               reinterpret_cast<float*>(att_out), (unsigned)drop_seed, (unsigned)drop_salt, drop_thresh, work,
                               work_elems, (cudaStream_t)stream);
}

long long vg_attn_gather_bwd_det_workspace(int N, int Hl, int Wl, int C, int win, int R, int reg_per_field) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, 0)) return -1;
  return attn_gather_bwd_det_workspace_elems(g, reg_per_field);
}

int vg_attn_gather_bwd_det(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                           const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in,
                           float* dfilm, int N, int Hl, int Wl, int C, int win, int R, int grid_mode, float ln_eps,
                           float* work, long long work_elems, void* stream) {
  AttnGeom g;
  if (make_attn_geom(g, N, Hl, Wl, C, win, R, grid_mode)) return 1;
  return attn_gather_bwd_det_run(x, reg, reg_per_field, film, dtok, dx_out, dreg_res, reg_scale, dx_in, dreg_in, dfilm, g, ln_eps,
                                 work, work_elems, (cudaStream_t)stream);
}

}  // extern "C"
