// Launchers of the HBM-bound kernels (see ew_kernels.cu for what each one replaces in the reference).
#pragma once
#include "ptx.cuh"

namespace b2v {

void launch_gn_apply(const __half* y, __half* out, const stat_t* stats_in, const float* gamma, const float* beta,
                     const float* temb, int temb_stride, const __half* res, int B, long long S, int C, int G,
                     float eps, int mode, stat_t* stats_out, int G_out, cudaStream_t st,
                     const int* temb_step = nullptr, long long temb_step_stride = 0);
void launch_splitk_finalize(const float* ws, long long slab, int nsplit, const float* bias, __half* out, stat_t* stats,
                            int B, long long S, int C, int G, cudaStream_t st);
void launch_gn_stats(const __half* x, int B, long long S, int C, int G, stat_t* stats, cudaStream_t st);
void launch_attn_tsum(const __half* x, const stat_t* stats, const float* gamma, const float* beta, __half* s, int B,
                      int T, int P, int C, int G, float eps, cudaStream_t st);
// fused attention-followed ResBlock tail + TemporalAttention (see ew_kernels.cu)
bool attn_fused_supported(int C);
int attn_tsum_splits(int B, int T, int P, int C);
void launch_gn_res_tsum(__half* y, const __half* res, const stat_t* stats_in, const float* gamma, const float* beta,
                        int B, int T, int P, int C, int G, float eps, stat_t* stats_out, int G_out, float* tsum, int TS,
                        cudaStream_t st);
void launch_attn_proj_add(__half* x, const float* tsum, int TS, const stat_t* stats, const float* gamma,
                          const float* beta, const __half* Wt, const float* bias, __half* g_ws, int B, int T, int P,
                          int C, int G, float eps, cudaStream_t st);
void launch_add_bcast_t(__half* x, const __half* y, int B, int T, int P, int C, cudaStream_t st);
void launch_temb(const long long* t_ptr, const float* freqs, const float* W1, const float* b1, const float* W2,
                 const float* b2, float* silu_temb, const float* Wp, const float* bp, float* proj, int rows, int dim,
                 int td, int B, cudaStream_t st);
// device-resident loop state of a sampler graph (one per U-Net program)
struct SamplerCtl {
  int step;                 // loop index: selects the coefficient / noise / time-embedding row; advanced by the graph
  int nan_flag;             // set when one of the reference's NaN/Inf guards fired
  int noise_first;          // loop index of row 0 of `noise`
  int pad;
  const float* noise;       // [rows][numel] per-step N(0,1) draws supplied by the caller, or null
  unsigned long long seed;  // Philox key used by the DDPM update when noise == null
};
struct Coef8 {
  float v[8];
};
// ctl != null: step / noise come from the control block (sampler graphs); else row 0 of coef_table, immediate noise
void launch_ddim_update(float* z, const float* eps, const float* noise, const float* coef_table, const SamplerCtl* ctl,
                        long long n, int* nan_flag, cudaStream_t st);
void launch_ddpm_update(float* z, const float* eps, const float* noise, const float* coef_table, const SamplerCtl* ctl,
                        const Coef8& coef, long long n, cudaStream_t st);
// DPM-Solver++(2M) step: row `step` of coef_table (ctl != null) or coef_table[0..7] with immediate noise (ctl == null)
void launch_dpmpp_update(float* z, float* x0_prev, const float* eps, const float* noise, const float* coef_table,
                         const SamplerCtl* ctl, long long n, int* nan_flag, cudaStream_t st);
void launch_philox_fill(float* out, unsigned long long seed, int step, long long n, cudaStream_t st);
void launch_guard(float* x, long long n, int mode, int* flag, cudaStream_t st);
void launch_or_flag(int* dst, const int* src, cudaStream_t st);  // *dst |= *src
void launch_q_sample(const float* z0, const float* noise, const long long* t, const float* sqrt_ac,
                     const float* sqrt_1m_ac, float* zt, int B, long long per_sample, cudaStream_t st);
size_t eps_mse_ws_bytes(int B);
void launch_eps_mse(const float* pred, const float* noise, const float* mask, int B, long long per_sample, long long HW,
                    double* ws, float* out, cudaStream_t st);
void ew_set_round_bf16(int on);
void launch_advance_step(SamplerCtl* ctl, cudaStream_t st);
void launch_zero(float* p, long long n, cudaStream_t st);
void launch_set_t(long long* t_dev, long long t, int B, cudaStream_t st);
void launch_pack_unet_in(const float* z, const float* c, __half* out, int B, int L, int D, int H, int W,
                         cudaStream_t st);
void launch_pack_vae_dec_in(const float* z, const float* Wpq, const float* bpq, float scaling, __half* out, int B,
                            int L, int D, int H, int W, cudaStream_t st);
void launch_pack_vae_enc_in(const float* v, __half* out, int B, int Cin, int Cpad, int D, int H, int W,
                            cudaStream_t st);
void launch_upsample_depth(const float* in, float* out, int BC, int Din, int Dout, long long HW, cudaStream_t st);
void launch_head_stencil(const float* P, const float* bias, float* out, int N, int cout, int D, int H, int W,
                         long long row_stride, long long slice_stride, int act, cudaStream_t st);
void launch_stitch_accumulate(const float* patch, float* acc, float* wsum, const float* gd, const float* gh,
                              const float* gw, int BC, int pd, int ph, int pw, int D, int H, int W, int d0, int h0,
                              int w0, cudaStream_t st);
void launch_stitch_normalize(float* acc, const float* wsum, long long n, cudaStream_t st);
size_t video_metrics_ws_bytes(int BC, int T, int H, int W);
void launch_video_metrics(const float* a, const float* b, float* out, float* ws, int BC, int T, int H, int W,
                          float max_val, cudaStream_t st);
void launch_extract_patch(const float* vol, float* out, int H, int W, int z0, int n, int y0, int x0, int pd, int ph,
                          int pw, float lo, float hi, float a, float b, cudaStream_t st);
void launch_nc32_to_cl16(const float* in, __half* out, int B, int C, int Cpad, long long S, cudaStream_t st);
void launch_cl16_to_nc32(const __half* in, float* out, int B, int C, int Cpad, long long S, cudaStream_t st);

}  // namespace b2v
