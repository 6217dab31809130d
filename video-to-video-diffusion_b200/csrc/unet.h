// U-Net denoiser object behind b2v_unet (see include/b2v.h)
#pragma once
#include "../../include/b2v.h"
#include "engine.h"

namespace b2v {

struct ResW {  // ResBlock3D (models/unet3d.py:77-133)
  ConvLayer conv1, conv2, res;
  GNW n1, n2;
  bool has_res = false;
  int cin0 = 0, cin1 = 0, cout = 0;
  int temb_off = 0;  // row offset of this block's time_mlp projection in the concatenated table
};
struct AttnW {  // TemporalAttention (models/unet3d.py:136-194): folded (reference mode) or qkv / proj (softmax mode)
  GNW norm;
  ConvLayer pv;
  ConvLayer qkv;   // softmax mode: the qkv 1x1 conv, C -> 3C
  ConvLayer proj;  // softmax mode: dual-source 1x1 conv over (o, x) with weight [Wproj | I_C], bias bproj
  __half* Wt = nullptr;  // [c][co] fp16 transpose of the folded Wp*Wv (fused attn_proj_add path; owned by UNet::ds)
  std::vector<float> u, bp;
  int C = 0;
};
struct ULevel {
  std::vector<ResW> res;
  std::vector<AttnW> attn;
  ConvLayer resample;
  bool has_resample = false;
};

enum { SAMPLER_DDIM = 0, SAMPLER_DDPM = 1, SAMPLER_DPMPP = 2, SAMPLER_KINDS = 3 };  // as b2v_sampler_cfg.sampler
struct UProgram {
  int B = 0, T = 0, h = 0, w = 0;
  long long numel = 0;
  DeviceStore ds;
  Pool pool;
  std::vector<Op> core;
  Program fwd, loop[SAMPLER_KINDS];  // one U-Net evaluation | per sampler: core without time_embed + update + advance
  float *x_in = nullptr, *c_in = nullptr, *eps = nullptr;
  float* x0_prev = nullptr;  // previous step's data prediction (DPM-Solver++), allocated by the first dpmpp_sample
  long long *t_dev = nullptr, *t_table = nullptr;
  SamplerCtl* ctl = nullptr;  // device loop state of the sampler graphs (step counter, NaN flag, noise source)
  int *step_dev = nullptr, *nan_dev = nullptr;  // = &ctl->step, &ctl->nan_flag
  int loop_pos = 0, loop_n = 0;                  // host mirror of ctl->step / loop length of the running sampler
  float *coef_table = nullptr, *silu_temb = nullptr, *proj = nullptr;
  stat_t* stats = nullptr;
  size_t stats_cap = 0;
  TembSource temb;            // set before every run: per-sample table (forward) or all-steps table (loop programs)
  float *silu_all = nullptr, *proj_all = nullptr;  // time embedding of every loop step, computed once per loop
  int all_cap = 0;
  long long stamp = 0;  // last use (least-recently-used program is evicted when the cache is full)
};

enum { ATTN_REFERENCE = 0, ATTN_SOFTMAX = 1 };  // b2v_unet_set_attention modes

struct UNet {
  b2v_unet_desc desc;
  int attention = ATTN_REFERENCE;
  WeightMap wm;
  bool finalized = false;
  DeviceStore ds;
  float *freqs = nullptr, *W1 = nullptr, *B1 = nullptr, *W2 = nullptr, *B2 = nullptr, *Wproj = nullptr,
        *Bproj = nullptr;
  int proj_rows = 0;
  ConvLayer conv_in, conv_out;
  GNW out_norm;
  std::vector<ULevel> enc, dec;
  ResW mid1, mid2;
  AttnW mid_attn;
  std::map<std::string, std::unique_ptr<UProgram>> progs;
  UProgram* last = nullptr;
  UProgram* active = nullptr;
  long long clock = 0;

  int finalize();
  int set_attention(int mode);  // before finalize; validates every attention level's head_dim for softmax mode
  UProgram* program(int B, int T, int h, int w);
  int forward(const float* x, const long long* t, const float* c, float* eps_out, int B, int T, int h, int w,
              cudaStream_t st);
  void forward_temb(UProgram& up) const { up.temb = TembSource{up.proj, proj_rows, nullptr, 0}; }  // before up.fwd
  int sampler_begin(const float* z_init, const float* cond, int B, int T, int h, int w, cudaStream_t st);
  int ddim_sample(const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w,
                  const long long* timesteps, int n, const float* ac, int n_train, float eta, const float* noise,
                  int* nan_flag, cudaStream_t st);
  // DPM-Solver++(2M) over the timesteps (rows from dpmpp_coefficients); sde: noise = DEVICE [n][numel]
  int dpmpp_sample(const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w,
                   const long long* timesteps, int n, const float* ac, int n_train, int order, int sde,
                   const float* noise, int* nan_flag, cudaStream_t st);
  int ddpm_step(long long t, const float* coef, const float* noise, cudaStream_t st);
  // loop steps [first, first + count) of an n-step ancestral loop (step s handles timestep n-1-s)
  int ddpm_run(const float* coef, int n, int first, int count, const float* noise, unsigned long long seed,
               cudaStream_t st);
  int ddpm_sample(const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w, const float* coef,
                  int n, const float* noise, unsigned long long seed, cudaStream_t st);
  int sampler_end(float* z_out, cudaStream_t st);
  ~UNet();
};

// host fp64 coefficient rows of DPM-Solver++(2M) (see b2v_dpmpp_coefficients); no device needed
int dpmpp_coefficients(const long long* timesteps, int n, const float* ac, int n_train, int order, int sde,
                       float* rows);

}  // namespace b2v
