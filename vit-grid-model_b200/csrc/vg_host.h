// Host-side helpers shared by the translation units of libvitgrid (error reporting, launch checks,
// internal entry points).  Not part of the public C ABI (that is include/vitgrid.h).
#pragma once
#include <cuda_runtime.h>

#include "vg_common.cuh"

namespace vg {

struct EpiParams;

// cudaFuncSetAttribute and the SM count belong to a DEVICE: "already done" caches are kept per device ordinal, so a process that
// drives several GPUs (the reference wraps its model in nn.DataParallel) configures every one of them.
struct PerDeviceFlag { bool done[64] = {}; bool& cur() { int d = 0; cudaGetDevice(&d); return done[d & 63]; } };
struct PerDeviceSize { size_t v[64] = {}; size_t& cur() { int d = 0; cudaGetDevice(&d); return v[d & 63]; } };

// printf-style: records the message for vg_last_error() and returns a non-zero error code
int set_error(const char* fmt, ...);
// cudaGetLastError() after a launch; 0 when clean
int check_launch(const char* what);
// Sticky device-side error word (one mapped, pinned int shared by every device of the process): kernels that meet input a
// PyTorch op would have raised on (e.g. an embedding row out of range) OR a bit into it instead of touching memory; the host reads
// it with vg_device_error() after a synchronisation.  Returns the device-visible pointer (nullptr if the allocation failed).
int* device_error_ptr();
enum { VG_DEVERR_TIMESTAMP = 1 };

int conv_halo_run(const void* x, const void* Wt, const PGeom& pg, const EpiParams& ep, int train, cudaStream_t st);
int split3_tf32_run(const float* in, long long rows, int K, float* out, int pattern, cudaStream_t st);
int gemm_run(int dtype, int kind, const void* A, long long rowsA, int Ca, const void* B, int Ntot, int ntaps,
             const int* tap_shift, long long M, long long rows_per_batch, int b_rows_per_batch,
             const EpiParams& ep, float* scratch, long long scratch_elems, cudaStream_t st);

struct PrepParams {
  const void* x;                  // fp32, or bf16 (packed host batches)
  long long sB, sT, sC, sH, sW;   // element strides of x
  int B, T, C, H, W;
  int pad_top, pad_left;
  int Cpad;
  float mean, stdv;
  int prestd;                     // 1: the PM2.5 channels of x are already standardised
  PGeom pg;
  int w_fast;                     // 1: x contiguous along W (tile transposed through smem along w)
};

struct TimeParams {
  const float* ts; long long ts_sB, ts_sT, ts_sF;  // timestamps (B, n_ts, 4) strides
  int B, L, le, te;
  const float* emb_lead;   // (L+1, le)
  const float* emb_m; const float* emb_d; const float* emb_h;  // (13|32|25, te)
  const float* w3;         // (Cout, c_in, 3, 3) original layout
  const float* w1;         // (Cout, c_in, 1, 1)
  int c_in, c_data, Cout;
  float* temb;             // (N, le+3te)
  float* cond;             // (N, le)
  float* tt;               // (N, 9, Cout)
  float* tres;             // (N, Cout)
  int* err;                // device error word (device_error_ptr())
};

struct StemParams {
  // training only (null in inference): saved for backward, same meaning as the EPI_CONV_LN_TRAIN outputs
  void* xhat; float* rstd; unsigned* mask;
  const float* raw3; const float* rawres;   // [q_b][C] fp32 over the B-image PG geometry
  const float* bias3; const float* bias1;
  const float* tt; const float* tres;       // (N,9,C), (N,C)
  const float* ln_g; const float* ln_b; float eps;
  const float* film;                        // (N, 2C)
  int L;
  PGeom pgB, pgN;
};

int prepare_run(int dtype, const void* x, int x_bf16, int prestd, const long long* xs, int B, int T, int C, int H, int W, int pad_top,
                int pad_left, int HP, int WP, int Cpad, float mean, float stdv, void* out, cudaStream_t st);
int prepare_bwd_run(const float* g, int B, int T, int C, int H, int W, int pad_top, int pad_left, int HP, int WP, int Cpad,
                    float stdv, int extra, float* dx, cudaStream_t st);
int time_terms_run(const TimeParams& p, cudaStream_t st);
int standardise_channel_run(float* x, const long long* xs, int B, int T, int C, int H, int W, int ch, float mean, float stdv, cudaStream_t st);
int dense_rows_run(const float* in, int N, int cd, int pre_relu, const float* W, const float* b, int od, int act, float* out,
                   cudaStream_t st);
int cond_mlp_run(const float* cond, int N, int cd, int pre_relu, const float* W0, const float* b0, int hid,
                 const float* W1, const float* b1, int od, float* out, cudaStream_t st);
int stem_finish_run(int dtype, const StemParams& p, void* h1, float* res, cudaStream_t st);
int stem_finish_wide_run(int dtype, const StemParams& p, int C, void* h1, float* res, cudaStream_t st);
int conv_ln_rows_run(int dtype, const float* acc, int C, const float* bias, const float* ln_g, const float* ln_b, float eps,
                     const float* film, const void* res, int res_f32, void* out, float* out2, const PGeom& pg,
                     const float* head_w, float head_b, float head_std, float head_mean, int H, int W, int pad_top,
                     int pad_left, float* head_out, cudaStream_t st);
// training instantiation of conv_ln_rows_kernel: also writes xhat (fp32 [q][C]), rstd ([q]) and the ReLU mask ([q][C/32])
int conv_ln_rows_train_run(const float* acc, int C, const float* bias, const float* ln_g, const float* ln_b, float eps,
                           const float* film, const void* res, int res_f32, float* out, float* out2, float* xhat, float* rstd,
                           unsigned* mask, const PGeom& pg, cudaStream_t st);
int maxpool2_run(int dtype, int out_f32, const void* in, void* out, int N, int HP, int WP, int C, cudaStream_t st);
int dwconv_run(int dtype, const void* in, const float* w9, const float* scale, const float* shift, void* out, float* psum,
               int N, int H, int W, int C, cudaStream_t st);
int se_scale_run(int dtype, void* x, const float* gate, int N, long long HW, int C, cudaStream_t st);
int reg_mean_run(const float* in, float* out, int N, int nwin, int RC, cudaStream_t st);
int head_run(int dtype, const void* h, const float* w, float bias, float stdv, float mean, int N, int HP, int WP, int C,
             int H, int W, int pad_top, int pad_left, float* out, cudaStream_t st);
long long eval_metrics_workspace_run(int B, int L, int P);
int eval_metrics_run(float* preds, const float* truth, const void* tcls, int cls_i64, const float* persist, const float* sim21,
                     const float* simavg, int B, int L, int P, float b1, float b2, float b3, int clamp_preds,
                     unsigned long long* counts, double* sums, double* glob, unsigned long long* nonzero, double* loss_sum,
                     double* work, long long work_elems, cudaStream_t st);
int focal_r_fwd_run(const float* pred, const float* tgt, long long n, float beta, float gamma, int mse, float* partial,
                    int nb, float* loss, cudaStream_t st);
int focal_r_bwd_run(const float* pred, const float* tgt, long long n, float beta, float gamma, int mse, float gscale,
                    float* grad, cudaStream_t st);

// attention (vg_attn.cu); AttnGeom / attn_token_pixel live in vg_common.cuh
int attn_partition_debug_run(const AttnGeom& g, long long* out, cudaStream_t st);
int attn_gather_run(int dtype, const void* x, const float* reg, int reg_per_field, const float* film, const AttnGeom& g,
                    float eps, void* tokens, int out_bf16, cudaStream_t st);
int attn_core_run(int dtype, const void* qkv, const float* qgamma, const float* kgamma, const float* bias_table,
                  const AttnGeom& g, int heads, int dh, void* out, unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st);

// fused attention (vg_attn_fused2.cu): in place on the residual stream, partition through TMA tensor maps
int attn_fused2_run(float* xio, const float* reg_in, int reg_per_field, float* reg_out, const float* film, const void* wqkv_h,
                    const float* wout_h, const float* head_tab, const AttnGeom& g, int heads, int dh, float ln_eps, unsigned seed,
                    unsigned salt, int drop_thresh, float logit_bound, cudaStream_t st);
int attn_partition_map(CUtensorMap* m, const float* x, const AttnGeom& g);

// ---- training (vg_wgrad.cu, vg_bwd.cu, vg_bwd_vit.cu)
long long wgrad_workspace_elems(int dtype, long long M, int Ntot, int Ca, int ntaps);
int wgrad_run(int dtype, const void* dY, const void* A, long long rowsA, long long M, int Ntot, int Ca, int ntaps,
              const int* tap_shift, float* dW, float beta, float* work, long long work_elems, cudaStream_t st);
int conv_ln_bwd_run(int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const unsigned* mask,
                    const float* ln_g, const float* film, float eps, void* dconv, float* sumA, float* sumB, float* sumD,
                    float* border, int N, int HP, int WP, cudaStream_t st);
int conv_ln_bwd_wide_run(int C, const float* dY, const float* xhat, const float* rstd, const unsigned* mask, const float* ln_g,
                         const float* film, float eps, float* dconv, float* sumA, float* sumB, float* sumD, float* border, int N,
                         int HP, int WP, cudaStream_t st);
int conv_ln_param_grads_run(const float* sumA, const float* sumB, const float* sumD, int N, const float* g, const float* b,
                            const float* film, float* dg, float* db, float* dbias, float* dfilm, int C, cudaStream_t st);
int head_bwd_run(int dtype, const float* dpred, const void* h, const float* w, float stdv, int N, int HP, int WP, int H, int W,
                 int pt, int pl, float* dH, float* dw, float* db, int C, cudaStream_t st);
int maxpool2_bwd_run(int dtype, const void* x, const float* dlow, float* dx, int N, int HP, int WP, int C, cudaStream_t st);
int convT_bwd_gather_run(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, cudaStream_t st);
int lead_sum_run(int idtype, int odtype, const void* in, void* out, int B, int L, int HP, int WP, int C, cudaStream_t st);
int pg_field_sum_run(const float* in, float* out, int N, int HP, int WP, int C, cudaStream_t st);
int time_terms_bwd_run(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                       const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                       float* dtemb, cudaStream_t st);
int time_embed_bwd_run(const float* dtemb, const float* dcond, const float* ts, long long sB, long long sT, long long sF, int B,
                       int L, int le, int te, float* d_lead, float* d_m, float* d_d, float* d_h, cudaStream_t st);
int cond_mlp_bwd_run(const float* cond, int N, int cd, int pre_relu, const float* W0, const float* b0, int hid, const float* W1,
                     int od, const float* dout, float* dW0, float* db0, float* dW1, float* db1, float* dcond, float* work,
                     long long work_elems, cudaStream_t st);
int outer_sum_run(const float* G, const float* X, int N, int O, int I, float* dW, float* db, cudaStream_t st);
int adamw_run(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps, float wd,
              int step, float gscale, cudaStream_t st);

long long bn_workspace_elems(long long M, int C);
int bn_stats_run(const float* X, long long M, int C, const float* gamma, const float* beta, float eps, float momentum,
                 float* run_mean, float* run_var, float* mean, float* rstd, float* scale, float* shift, float* work,
                 long long work_elems, cudaStream_t st);
int bn_act_run(const float* raw, const float* scale, const float* shift, int act, const float* res, float* out, long long M, int C,
               cudaStream_t st);
int bn_bwd_run(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean, const float* rstd,
               const float* gamma, int act, const float* fgate, const float* fadd, long long rows_per_field, long long M, int C,
               float* dgamma, float* dbeta, float* draw, float* work, long long work_elems, cudaStream_t st);
int bn_bwd_frozen_run(const float* dOut, const float* raw, const float* scale, const float* shift, const float* mean, const float* rstd,
                      int act, const float* fgate, const float* fadd, long long rows_per_field, long long M, int C, float* dgamma,
                      float* dbeta, float* draw, float* work, long long work_elems, cudaStream_t st);
int colsum_run(const float* X, long long M, int C, float* out, cudaStream_t st);
int dwconv_march_run(int dtype, const void* in, const float* w9, const float* scale, const float* shift, int act, void* out,
                     float* psum, int N, int H, int W, int C, cudaStream_t st);
int dwconv_strips(int W);
int dw_wgrad_run(const float* X, const float* dY, int N, int H, int W, int C, float* dw9, float* dbias, float* work,
                 long long work_elems, cudaStream_t st);
int se_gate_train_run(const float* psum, int N, int nparts, long long HW, const float* W1, const float* W2, int C, int se,
                      float* gate, float* mean, float* hid, cudaStream_t st);
int field_parts(long long HW);
int field_dot_run(const float* a, const float* b, float* out, int N, long long HW, int C, cudaStream_t st);
int se_fold_run(const float* W, const float* gate, void* out, int out_f16, int N, int Cout, int C, cudaStream_t st);
int se_scale_oop_run(const float* x, const float* gate, float* out, int N, long long HW, int C, cudaStream_t st);
int se_bwd_run(const float* dh4, const float* h3, const float* gate, const float* mean, const float* hid, const float* W1,
               const float* W2, int N, long long HW, int C, int se, float* dW1, float* dW2, float* dmean, float* work,
               long long work_elems, cudaStream_t st);
int attn_out_bwd_gather_run(const float* dx_out, const float* dreg, float reg_scale, const AttnGeom& g, void* dproj, int out_bf16,
                            unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st);
int dropout_mask_debug_run(unsigned seed, unsigned salt, int drop_thresh, long long n_windows, int heads, int C, int slots, unsigned char* prob_mask,
                           unsigned char* out_mask, cudaStream_t st);
int attn_core_bwd_run(const float* qkv, const float* datt, const float* qgamma, const float* kgamma, const float* bias_table,
                      const AttnGeom& g, int heads, int dh, float* dqkv, float* dqgamma, float* dkgamma, float* dbias_table,
                      int use_tf32, float* att_out, unsigned seed, unsigned salt, int drop_thresh, cudaStream_t st);
int attn_gather_bwd_run(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                        const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in, float* dfilm,
                        const AttnGeom& g, float eps, cudaStream_t st);

// ---- deterministic training-backward variants (fixed-order reductions over per-warp / per-block slots; vg_bwd.cu, vg_bwd_vit.cu)
long long det_sum_tmp_elems(int G, long long S, int W);
int det_sum_run(const float* in, int G, long long S, int W, long long ld, float* out, long long out_ld, float* tmp, cudaStream_t st);
long long conv_ln_bwd_det_workspace_elems(int C, int N, int HP, int WP);
int conv_ln_bwd_det_run(int C, int xdtype, int odtype, const float* dY, const void* xhat, const float* rstd, const unsigned* mask,
                        const float* ln_g, const float* film, float eps, void* dconv, float* sumA, float* sumB, float* sumD,
                        float* border, int N, int HP, int WP, float* work, long long work_elems, cudaStream_t st);
long long head_bwd_det_workspace_elems(int N, int HP, int WP, int C);
int head_bwd_det_run(int dtype, const float* dpred, const void* h, const float* w, float stdv, int N, int HP, int WP, int H, int W,
                     int pt, int pl, float* dH, float* dw, float* db, int C, float* work, long long work_elems, cudaStream_t st);
long long convT_bwd_gather_det_workspace_elems(int N, int Hl, int Wl, int C);
int convT_bwd_gather_det_run(int odtype, const float* dUp, void* G, float* dbias, int N, int Hl, int Wl, int C, float* work,
                             long long work_elems, cudaStream_t st);
long long pg_field_sum_det_workspace_elems(int N, int HP, int WP, int C);
int pg_field_sum_det_run(const float* in, float* out, int N, int HP, int WP, int C, float* work, long long work_elems, cudaStream_t st);
long long time_terms_bwd_det_workspace_elems(int N, int Cout);
int time_terms_bwd_det_run(const float* border, const float* sumD, const float* tres_sum, const float* temb, const float* w3,
                           const float* w1, int N, int ntc, int c_in, int c_data, int Cout, float* dw3, float* dw1, float* db1,
                           float* dtemb, float* work, long long work_elems, cudaStream_t st);
int time_embed_bwd_det_run(const float* dtemb, const float* dcond, const float* ts, long long sB, long long sT, long long sF, int B,
                           int L, int le, int te, float* d_lead, float* d_m, float* d_d, float* d_h, cudaStream_t st);
long long colsum_det_workspace_elems(long long M, int C);
int colsum_det_run(const float* X, long long M, int C, float* out, float* work, long long work_elems, cudaStream_t st);
long long attn_core_bwd_det_workspace_elems(const AttnGeom& g, int heads, int dh);
int attn_core_bwd_det_run(const float* qkv, const float* datt, const float* qgamma, const float* kgamma, const float* bias_table,
                          const AttnGeom& g, int heads, int dh, float* dqkv, float* dqgamma, float* dkgamma, float* dbias_table,
                          int use_tf32, float* att_out, unsigned seed, unsigned salt, int drop_thresh, float* work,
                          long long work_elems, cudaStream_t st);
long long attn_gather_bwd_det_workspace_elems(const AttnGeom& g, int reg_per_field);
int attn_gather_bwd_det_run(const float* x, const float* reg, int reg_per_field, const float* film, const float* dtok,
                            const float* dx_out, const float* dreg_res, float reg_scale, float* dx_in, float* dreg_in, float* dfilm,
                            const AttnGeom& g, float eps, float* work, long long work_elems, cudaStream_t st);

}  // namespace vg
