// extern "C" surface of libb2v.so (declared in include/b2v.h)
#include <string.h>

#include "unet.h"
#include "vae.h"

using namespace b2v;

struct b2v_unet {
  UNet u;
  float* gen_ws = nullptr;  // scratch of b2v_generate (input copy, latents), grown on demand
  size_t gen_cap = 0;
  ~b2v_unet() {
    if (gen_ws) cudaFree(gen_ws);
  }
};
struct b2v_vae {
  VAE v;
};
struct b2v_conv {
  ConvLayer L;
  float* ws = nullptr;  // tap-GEMM workspace of narrow heads (grown on demand)
  size_t ws_bytes = 0;
  float* sk = nullptr;  // split-K workspace (zero between uses)
  size_t sk_bytes = 0;
};

static int check_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail("no CUDA device (libb2v has no CPU fallback)");
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return fail("libb2v is built for sm_100a (B200) only; found compute capability major " + std::to_string(major));
  return 0;
}

static int store_weight(WeightMap& wm, bool finalized, const char* key, const float* data, const int64_t* shape,
                        int ndim) {
  if (finalized) return fail("weights already finalized");
  if (!key || !data || ndim < 0 || ndim > 8) return fail("load_weight: bad arguments");
  HostTensor t;
  long long n = 1;
  for (int i = 0; i < ndim; ++i) {
    t.shape.push_back(shape[i]);
    n *= shape[i];
  }
  t.data.assign(data, data + n);
  wm[key] = std::move(t);
  return 0;
}

// The argument checks of b2v_generate / b2v_generate_ensemble, all made before the first device call.
static int check_generate_args(const std::string& who, const b2v_sampler_cfg* cfg, int B, int T_in, int T_out, int H,
                               int W) {
  if (B < 0 || T_in < 1 || T_out < 1 || H < 4 || W < 4 || H % 4 || W % 4) return fail(who + ": bad shape");
  if (cfg->sampler < 0 || cfg->sampler > 4)
    return fail(who + ": unknown sampler (0 = ddim, 1 = ddpm, 2 = dpmpp_2m, 3 = dpmpp_2m_sde, 4 = unipc)");
  if (cfg->sampler == 4) {  // reject a bad UniPC configuration (tables, order, variant) before the encoder is launched
    if (cfg->n < 1 || cfg->n > 4096) return fail(who + ": 1 <= n <= 4096 timesteps");
    std::vector<float> rows((size_t)cfg->n * 16);
    if (unipc_coefficients((const long long*)cfg->timesteps, cfg->n, cfg->alphas_cumprod, cfg->n_train,
                           cfg->unipc_order, cfg->unipc_variant, rows.data()))
      return -1;
  } else if (cfg->sampler >= 2) {  // reject a bad DPM-Solver++ configuration before the encoder is launched
    if (cfg->sampler == 3 && !cfg->noise) return fail(who + ": dpmpp_2m_sde needs the per-step noise draws");
    if (cfg->n < 1 || cfg->n > 4096) return fail(who + ": 1 <= n <= 4096 timesteps");
    std::vector<float> rows((size_t)cfg->n * 8);
    if (dpmpp_coefficients((const long long*)cfg->timesteps, cfg->n, cfg->alphas_cumprod, cfg->n_train, 2,
                           cfg->sampler == 3, rows.data()))
      return -1;
  }
  return 0;
}

// b2v_unet::gen_ws holds at least `need` bytes (grown on demand; the old buffer may be in use by queued work)
static int gen_workspace(b2v_unet* u, size_t need, cudaStream_t st) {
  if (need <= u->gen_cap) return 0;
  B2V_CUDA(cudaStreamSynchronize(st));
  if (u->gen_ws) cudaFree(u->gen_ws);
  u->gen_ws = nullptr;
  u->gen_cap = 0;
  B2V_CUDA(cudaMalloc(&u->gen_ws, need));
  u->gen_cap = need;
  return 0;
}

// The front of generate(), shared by b2v_generate (K = 1) and b2v_generate_ensemble: NaN check of v_in -> encode the B
// inputs -> guard -> depth upsample -> guard -> conditioning repeated K times (k-major) -> the sampler at batch K*B.
// Workspace (floats): vc [n_v] | z_in [n_zi] | cond [K][n_z] | z0 [K][n_z] | flag [2] ints; z0 receives the sampled
// latents, flag[0] the checkpoints so far, flag[1] the sampler's own guards.
struct GenFront {
  float* z0;
  int* flag;
};
static int generate_front(b2v_unet* u, b2v_vae* v, const b2v_sampler_cfg* cfg, const float* v_in, const float* z_init,
                          int K, int B, int T_in, int T_out, int H, int W, size_t extra_bytes, GenFront& g,
                          cudaStream_t st) {
  if (u->u.desc.latent_dim != v->v.desc.latent_dim) return fail("generate: U-Net / VAE latent_dim mismatch");
  const int L = v->v.desc.latent_dim, Cin = v->v.desc.in_channels, h = H / 4, w = W / 4;
  const size_t n_v = (size_t)B * Cin * T_in * H * W, n_zi = (size_t)B * L * T_in * h * w,
               n_z = (size_t)B * L * T_out * h * w;
  if (gen_workspace(u, (n_v + n_zi + 2 * K * n_z) * sizeof(float) + 256 + extra_bytes, st)) return -1;
  float* vc = u->gen_ws;
  float* z_in = vc + n_v;
  float* cond = z_in + n_zi;
  float* z0 = cond + K * n_z;
  int* flag = reinterpret_cast<int*>(z0 + K * n_z);
  B2V_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(int), st));
  B2V_CUDA(cudaMemcpyAsync(vc, v_in, n_v * sizeof(float), cudaMemcpyDeviceToDevice, st));
  launch_guard(vc, (long long)n_v, 0, flag, st);
  if (v->v.encode(vc, z_in, B, T_in, H, W, st)) return -1;
  launch_guard(z_in, (long long)n_zi, 1, flag, st);
  const float* c = z_in;
  if (T_out != T_in) {
    launch_upsample_depth(z_in, cond, B * L, T_in, T_out, (long long)h * w, st);
    launch_guard(cond, (long long)n_z, 1, flag, st);
    g_launches += 2;
    c = cond;
  }
  if (K > 1) {
    for (int k = 0; k < K; ++k)
      if (cond + k * n_z != c)
        B2V_CUDA(cudaMemcpyAsync(cond + k * n_z, c, n_z * sizeof(float), cudaMemcpyDeviceToDevice, st));
    c = cond;
  }
  const int KB = K * B;
  if (cfg->sampler == 0) {
    if (u->u.ddim_sample(z_init, c, z0, KB, T_out, h, w, (const long long*)cfg->timesteps, cfg->n, cfg->alphas_cumprod,
                         cfg->n_train, cfg->eta, cfg->noise, flag + 1, st))
      return -1;
  } else if (cfg->sampler == 1) {
    if (u->u.ddpm_sample(z_init, c, z0, KB, T_out, h, w, cfg->ddpm_coef, cfg->n, cfg->noise,
                         (unsigned long long)cfg->seed, st))
      return -1;
  } else if (cfg->sampler == 2 || cfg->sampler == 3) {
    if (u->u.dpmpp_sample(z_init, c, z0, KB, T_out, h, w, (const long long*)cfg->timesteps, cfg->n, cfg->alphas_cumprod,
                          cfg->n_train, 2, cfg->sampler == 3, cfg->noise, flag + 1, st))
      return -1;
  } else if (cfg->sampler == 4) {
    if (u->u.unipc_sample(z_init, c, z0, KB, T_out, h, w, (const long long*)cfg->timesteps, cfg->n, cfg->alphas_cumprod,
                          cfg->n_train, cfg->unipc_order, cfg->unipc_variant, flag + 1, st))
      return -1;
  }
  g.z0 = z0;
  g.flag = flag;
  return 0;
}

// *nan_flag = flag[0] | flag[1] (the device-side OR of all checkpoints), when the caller asked for it
static int report_nan_flag(int* flag, int* nan_flag, cudaStream_t st) {
  if (!nan_flag) return 0;
  launch_or_flag(flag, flag + 1, st);
  g_launches += 1;
  B2V_CUDA(cudaMemcpyAsync(nan_flag, flag, sizeof(int), cudaMemcpyDeviceToDevice, st));
  return 0;
}

static int write_json(const std::string& js, char* buf, size_t cap) {
  if (js.size() + 1 > cap) return fail("profile: buffer too small (" + std::to_string(js.size() + 1) + " needed)");
  memcpy(buf, js.c_str(), js.size() + 1);
  return 0;
}

#pragma GCC visibility push(default)
extern "C" {

const char* b2v_last_error(void) { return g_err.c_str(); }
int b2v_abi_version(void) { return B2V_ABI_VERSION; }
long long b2v_launch_count(void) { return g_launches.load(); }

// ------------------------------------------------------------------ U-Net
int b2v_unet_create(b2v_unet** out, const b2v_unet_desc* d) {
  if (!out || !d) return fail("unet_create: null argument");
  if (check_device()) return -1;
  if (d->num_levels < 1 || d->num_levels > 8 || d->num_res_blocks < 1) return fail("unet_create: bad descriptor");
  b2v_unet* u = new b2v_unet();
  u->u.desc = *d;
  *out = u;
  return 0;
}
void b2v_unet_destroy(b2v_unet* u) { delete u; }
int b2v_unet_load_weight(b2v_unet* u, const char* key, const float* data, const int64_t* shape, int ndim) {
  if (!u) return fail("unet_load_weight: null handle");
  return store_weight(u->u.wm, u->u.finalized, key, data, shape, ndim);
}
int b2v_unet_set_attention(b2v_unet* u, int mode) {
  if (!u) return fail("unet_set_attention: null handle");
  return u->u.set_attention(mode);
}
int b2v_unet_finalize(b2v_unet* u) {
  if (!u) return fail("unet_finalize: null handle");
  return u->u.finalize();
}
int b2v_unet_forward(b2v_unet* u, const float* x, const int64_t* t, const float* c, float* eps_out, int B, int T,
                     int h, int w, void* stream) {
  if (!u) return fail("unet_forward: null handle");
  return u->u.forward(x, (const long long*)t, c, eps_out, B, T, h, w, (cudaStream_t)stream);
}
int b2v_ddim_sample(b2v_unet* u, const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w,
                    const int64_t* timesteps, int n, const float* alphas_cumprod, int n_train, float eta,
                    const float* noise, int* nan_flag, void* stream) {
  if (!u) return fail("ddim_sample: null handle");
  return u->u.ddim_sample(z_init, cond, z_out, B, T, h, w, (const long long*)timesteps, n, alphas_cumprod, n_train,
                          eta, noise, nan_flag, (cudaStream_t)stream);
}
int b2v_dpmpp_coefficients(const int64_t* timesteps, int n, const float* alphas_cumprod, int n_train, int order, int sde,
                           float* rows) {
  return dpmpp_coefficients((const long long*)timesteps, n, alphas_cumprod, n_train, order, sde, rows);
}
int b2v_dpmpp_sample(b2v_unet* u, const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w,
                     const int64_t* timesteps, int n, const float* alphas_cumprod, int n_train, int order, int sde,
                     const float* noise, int* nan_flag, void* stream) {
  if (!u) return fail("dpmpp_sample: null handle");
  return u->u.dpmpp_sample(z_init, cond, z_out, B, T, h, w, (const long long*)timesteps, n, alphas_cumprod, n_train,
                           order, sde, noise, nan_flag, (cudaStream_t)stream);
}
int b2v_unipc_coefficients(const int64_t* timesteps, int n, const float* alphas_cumprod, int n_train, int order,
                           int variant, float* rows) {
  return unipc_coefficients((const long long*)timesteps, n, alphas_cumprod, n_train, order, variant, rows);
}
int b2v_unipc_sample(b2v_unet* u, const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w,
                     const int64_t* timesteps, int n, const float* alphas_cumprod, int n_train, int order, int variant,
                     int* nan_flag, void* stream) {
  if (!u) return fail("unipc_sample: null handle");
  return u->u.unipc_sample(z_init, cond, z_out, B, T, h, w, (const long long*)timesteps, n, alphas_cumprod, n_train,
                           order, variant, nan_flag, (cudaStream_t)stream);
}
int b2v_sampler_begin(b2v_unet* u, const float* z_init, const float* cond, int B, int T, int h, int w, void* stream) {
  if (!u) return fail("sampler_begin: null handle");
  return u->u.sampler_begin(z_init, cond, B, T, h, w, (cudaStream_t)stream);
}
int b2v_ddpm_step(b2v_unet* u, int64_t t, const float* coef, const float* noise, void* stream) {
  if (!u) return fail("ddpm_step: null handle");
  return u->u.ddpm_step((long long)t, coef, noise, (cudaStream_t)stream);
}
int b2v_sampler_end(b2v_unet* u, float* z_out, void* stream) {
  if (!u) return fail("sampler_end: null handle");
  return u->u.sampler_end(z_out, (cudaStream_t)stream);
}
int b2v_ddpm_sample(b2v_unet* u, const float* z_init, const float* cond, float* z_out, int B, int T, int h, int w,
                    const float* coef, int n, const float* noise, uint64_t seed, void* stream) {
  if (!u) return fail("ddpm_sample: null handle");
  return u->u.ddpm_sample(z_init, cond, z_out, B, T, h, w, coef, n, noise, (unsigned long long)seed,
                          (cudaStream_t)stream);
}
int b2v_ddpm_run(b2v_unet* u, const float* coef, int n, int first, int count, const float* noise, uint64_t seed,
                 void* stream) {
  if (!u) return fail("ddpm_run: null handle");
  return u->u.ddpm_run(coef, n, first, count, noise, (unsigned long long)seed, (cudaStream_t)stream);
}
int b2v_ddim_timesteps(int n_train, int steps, int64_t* out, int cap) {
  if (n_train < 1 || steps < 1 || steps > n_train || !out) return fail("ddim_timesteps: bad arguments");
  const int stride = n_train / steps;  // np.arange(0, n_train, n_train // steps)
  std::vector<int64_t> ts;
  for (int t = 0; t < n_train; t += stride) ts.push_back(t);
  if (ts.back() != n_train - 1) ts.push_back(n_train - 1);
  if ((int)ts.size() > cap) return fail("ddim_timesteps: output buffer too small");
  for (size_t i = 0; i < ts.size(); ++i) out[i] = ts[ts.size() - 1 - i];
  return (int)ts.size();
}
int b2v_philox_normal(float* out, uint64_t seed, int step, long long n, void* stream) {
  if (check_device()) return -1;
  if (n <= 0) return 0;
  launch_philox_fill(out, (unsigned long long)seed, step, n, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("philox_normal");
}

// ------------------------------------------------------------------ end to end (models/model.py:230-343)
int b2v_generate(b2v_unet* u, b2v_vae* v, const b2v_sampler_cfg* cfg, const float* v_in, const float* z_init,
                 float* v_out, int B, int T_in, int T_out, int H, int W, int* nan_flag, void* stream) {
  if (!u || !v || !cfg || !v_in || !z_init || !v_out) return fail("generate: null argument");
  if (check_generate_args("generate", cfg, B, T_in, T_out, H, W)) return -1;
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  GenFront g;
  if (generate_front(u, v, cfg, v_in, z_init, 1, B, T_in, T_out, H, W, 0, g, st)) return -1;
  const int L = v->v.desc.latent_dim, Cin = v->v.desc.in_channels;
  const size_t n_z = (size_t)B * L * T_out * (H / 4) * (W / 4), n_out = (size_t)B * Cin * T_out * H * W;
  launch_guard(g.z0, (long long)n_z, 1, g.flag, st);
  if (v->v.decode(g.z0, v_out, B, T_out, H / 4, W / 4, st)) return -1;
  launch_guard(v_out, (long long)n_out, 1, g.flag, st);
  g_launches += 4;
  if (report_nan_flag(g.flag, nan_flag, st)) return -1;
  return check_launches("generate");
}

int b2v_generate_ensemble(b2v_unet* u, b2v_vae* v, const b2v_sampler_cfg* cfg, const float* v_in, const float* z_init,
                          int K, float* members_out, float* mean_out, float* std_out, int B, int T_in, int T_out, int H,
                          int W, int* nan_flag, void* stream) {
  if (!u || !v || !cfg || !v_in || !z_init || !mean_out || !std_out) return fail("generate_ensemble: null argument");
  if (K < 2) return fail("generate_ensemble: K >= 2 samples per input (the std needs two)");
  if (check_generate_args("generate_ensemble", cfg, B, T_in, T_out, H, W)) return -1;
  if ((long long)K * B > INT32_MAX) return fail("generate_ensemble: K * B too large");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int L = v->v.desc.latent_dim, Cin = v->v.desc.in_channels, h = H / 4, w = W / 4;
  const size_t n_z = (size_t)B * L * T_out * h * w, n_out = (size_t)B * Cin * T_out * H * W;
  // without members_out the decoded members go to the scratch, behind the flags (256-byte aligned)
  GenFront g;
  if (generate_front(u, v, cfg, v_in, z_init, K, B, T_in, T_out, H, W, members_out ? 0 : K * n_out * sizeof(float) + 256,
                     g, st))
    return -1;
  float* members = members_out;
  if (!members) {
    const uintptr_t p = reinterpret_cast<uintptr_t>(g.flag + 2);
    members = reinterpret_cast<float*>((p + 255) & ~(uintptr_t)255);
  }
  launch_guard(g.z0, (long long)(K * n_z), 1, g.flag, st);
  for (int k = 0; k < K; ++k)  // K chunks of B: the batch-B decode program generate() uses
    if (v->v.decode(g.z0 + k * n_z, members + k * n_out, B, T_out, h, w, st)) return -1;
  launch_guard(members, (long long)(K * n_out), 1, g.flag, st);
  launch_ensemble_stats(members, mean_out, std_out, K, (long long)n_out, st);
  g_launches += 5;  // the four guards and the statistics
  if (report_nan_flag(g.flag, nan_flag, st)) return -1;
  return check_launches("generate_ensemble");
}

int b2v_ensemble_stats(const float* members, float* mean, float* stdev, int K, long long n, void* stream) {
  if (!members || !mean || !stdev) return fail("ensemble_stats: null argument");
  if (K < 2) return fail("ensemble_stats: K >= 2 members (the std needs two)");
  if (n < 0) return fail("ensemble_stats: negative n");
  if (check_device()) return -1;
  if (n == 0) return 0;
  launch_ensemble_stats(members, mean, stdev, K, n, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("ensemble_stats");
}

int b2v_q_sample(const float* z0, const float* noise, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac,
                 float* zt, int B, long long per_sample, void* stream) {
  if (check_device()) return -1;
  if (B <= 0 || per_sample <= 0) return 0;
  launch_q_sample(z0, noise, (const long long*)t, sqrt_ac, sqrt_1m_ac, zt, B, per_sample, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("q_sample");
}
size_t b2v_eps_mse_ws_bytes(int B) { return eps_mse_ws_bytes(B < 1 ? 1 : B); }
int b2v_eps_mse(const float* eps_pred, const float* noise, const float* mask, float* out, void* ws, size_t ws_bytes,
                int B, long long per_sample, long long HW, void* stream) {
  if (check_device()) return -1;
  if (B <= 0 || per_sample <= 0) return 0;
  if (HW <= 0 || per_sample % HW) return fail("eps_mse: per_sample must be a multiple of HW");
  if (!ws || ws_bytes < eps_mse_ws_bytes(B)) return fail("eps_mse: workspace too small (b2v_eps_mse_ws_bytes)");
  launch_eps_mse(eps_pred, noise, mask, B, per_sample, HW, (double*)ws, out, (cudaStream_t)stream);
  g_launches += 2;
  return check_launches("eps_mse");
}
int b2v_unet_profile(b2v_unet* u, int iters, char* buf, size_t cap, void* stream) {
  if (!u) return fail("unet_profile: null handle");
  if (!u->u.last) return fail("unet_profile: run a forward first");
  u->u.forward_temb(*u->u.last);
  std::string js;
  if (u->u.last->fwd.profile(iters, (cudaStream_t)stream, js)) return -1;
  return write_json(js, buf, cap);
}

// ------------------------------------------------------------------ VAE
int b2v_vae_create(b2v_vae** out, const b2v_vae_desc* d) {
  if (!out || !d) return fail("vae_create: null argument");
  if (check_device()) return -1;
  b2v_vae* v = new b2v_vae();
  v->v.desc = *d;
  *out = v;
  return 0;
}
void b2v_vae_destroy(b2v_vae* v) { delete v; }
int b2v_vae_load_weight(b2v_vae* v, const char* key, const float* data, const int64_t* shape, int ndim) {
  if (!v) return fail("vae_load_weight: null handle");
  return store_weight(v->v.wm, v->v.finalized, key, data, shape, ndim);
}
int b2v_vae_finalize(b2v_vae* v) {
  if (!v) return fail("vae_finalize: null handle");
  return v->v.finalize();
}
int b2v_vae_encode(b2v_vae* v, const float* x, float* z, int B, int T, int H, int W, void* stream) {
  if (!v) return fail("vae_encode: null handle");
  return v->v.encode(x, z, B, T, H, W, (cudaStream_t)stream);
}
int b2v_vae_decode(b2v_vae* v, const float* z, float* x, int B, int T, int h, int w, void* stream) {
  if (!v) return fail("vae_decode: null handle");
  return v->v.decode(z, x, B, T, h, w, (cudaStream_t)stream);
}
int b2v_vae_profile(b2v_vae* v, int which, int iters, char* buf, size_t cap, void* stream) {
  if (!v) return fail("vae_profile: null handle");
  if (which < 0 || which > 1 || !v->v.last[which]) return fail("vae_profile: run encode/decode first");
  std::string js;
  if (v->v.last[which]->prog.profile(iters, (cudaStream_t)stream, js)) return -1;
  return write_json(js, buf, cap);
}

static Program* debug_prog(void* obj, int prog) {
  if (prog == 0) {
    UNet& u = ((b2v_unet*)obj)->u;
    if (u.last) u.forward_temb(*u.last);
    return u.last ? &u.last->fwd : nullptr;
  }
  VAE& v = ((b2v_vae*)obj)->v;
  return v.last[prog - 1] ? &v.last[prog - 1]->prog : nullptr;
}
long long b2v_debug_op_output(void* obj, int prog, int n_ops, int index, void* dst, size_t cap, void* stream) {
  Program* P = debug_prog(obj, prog);
  if (!P) return fail("debug: run the program once first");
  if (index < 0 || index >= (int)P->ops.size() || index >= n_ops) return fail("debug: bad op index");
  cudaStream_t st = (cudaStream_t)stream;
  for (int i = 0; i < n_ops && i < (int)P->ops.size(); ++i) P->ops[i].run(st);
  const Op& op = P->ops[index];
  if (!op.out) return 0;
  const size_t n = op.out_bytes < cap ? op.out_bytes : cap;
  B2V_CUDA(cudaMemcpyAsync(dst, op.out, n, cudaMemcpyDeviceToDevice, st));
  B2V_CUDA(cudaStreamSynchronize(st));
  return (long long)n;
}
const char* b2v_debug_op_name(void* obj, int prog, int index) {
  Program* P = debug_prog(obj, prog);
  if (!P || index < 0 || index >= (int)P->ops.size()) return "";
  return P->ops[index].name.c_str();
}

// ------------------------------------------------------------------ glue / op level
int b2v_upsample_depth(const float* in, float* out, int BC, int Din, int Dout, int HW, void* stream) {
  if (check_device()) return -1;
  launch_upsample_depth(in, out, BC, Din, Dout, HW, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}

int b2v_stitch_accumulate(const float* patch, float* acc, float* wsum, const float* gd, const float* gh,
                           const float* gw, int BC, int pd, int ph, int pw, int D, int H, int W, int d0, int h0, int w0,
                           void* stream) {
  if (check_device()) return -1;
  if (d0 < 0 || h0 < 0 || w0 < 0 || d0 + pd > D || h0 + ph > H || w0 + pw > W) return fail("stitch: patch outside the volume");
  launch_stitch_accumulate(patch, acc, wsum, gd, gh, gw, BC, pd, ph, pw, D, H, W, d0, h0, w0, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_stitch_normalize(float* acc, const float* wsum, long long n, void* stream) {
  if (check_device()) return -1;
  launch_stitch_normalize(acc, wsum, n, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}

int b2v_video_metrics(const float* a, const float* b, float* out, int BC, int T, int H, int W, float max_val,
                       void* stream) {
  if (check_device()) return -1;
  if (BC <= 0 || T <= 0 || H <= 0 || W <= 0) return fail("video_metrics: empty input");
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = nullptr;  // per-block partials, stream-ordered allocation: freed when the fold kernel has read them
  B2V_CUDA(cudaMallocAsync(&ws, video_metrics_ws_bytes(BC, T, H, W), st));
  launch_video_metrics(a, b, out, ws, BC, T, H, W, max_val, st);
  g_launches += 2;
  B2V_CUDA(cudaFreeAsync(ws, st));
  return check_launches("video_metrics");
}

int b2v_extract_patch(const float* vol, float* out, int D, int H, int W, int z0, int z1, int y0, int x0, int pd, int ph,
                       int pw, float lo, float hi, float a, float b, void* stream) {
  if (check_device()) return -1;
  if (z0 < 0 || z1 > D || z1 <= z0 || y0 < 0 || x0 < 0 || y0 + ph > H || x0 + pw > W || pd < 1)
    return fail("extract_patch: window outside the volume");
  launch_extract_patch(vol, out, H, W, z0, z1 - z0, y0, x0, pd, ph, pw, lo, hi, a, b, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}

int b2v_conv_create(b2v_conv** out, int kind, const float* weight, const float* bias, int cin0, int cin1, int cout) {
  if (check_device()) return -1;
  std::string err;
  if (conv_setup_kernels(err)) return fail(err);
  b2v_conv* c = new b2v_conv();
  if (conv_layer_init(c->L, kind, weight, bias, cin0, cin1, cout, err)) {
    delete c;
    return fail(err);
  }
  *out = c;
  return 0;
}
void b2v_conv_destroy(b2v_conv* c) {
  if (c) {
    conv_layer_free(c->L);
    if (c->ws) cudaFree(c->ws);
    if (c->sk) cudaFree(c->sk);
  }
  delete c;
}
int b2v_conv_forward(b2v_conv* c, const void* in0, const void* in1, void* out, int out_fp32, int64_t* stats, int groups,
                     int act_tanh, int N, int D, int H, int W, void* stream) {
  if (!c) return fail("conv_forward: null handle");
  ConvPlan P;
  std::string err;
  const size_t need_ws = (out_fp32 && !in1 && !stats) ? conv_tap_ws_bytes(c->L, N, D, H, W) : 0;
  if (need_ws > c->ws_bytes) {
    B2V_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (c->ws) cudaFree(c->ws);
    c->ws = nullptr;
    c->ws_bytes = 0;
    B2V_CUDA(cudaMalloc(&c->ws, need_ws));
    c->ws_bytes = need_ws;
  }
  const size_t need_sk = out_fp32 ? 0 : conv_splitk_ws_bytes(c->L, N, D, H, W);
  if (need_sk > c->sk_bytes) {
    B2V_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (c->sk) cudaFree(c->sk);
    c->sk = nullptr;
    c->sk_bytes = 0;
    B2V_CUDA(cudaMalloc(&c->sk, need_sk));
    B2V_CUDA(cudaMemset(c->sk, 0, need_sk));
    c->sk_bytes = need_sk;
  }
  if (conv_plan(P, c->L, (const __half*)in0, (const __half*)in1, N, D, H, W, out, out_fp32 ? OUT_F32 : OUT_CL16, (long long*)stats,
                groups, act_tanh ? ACT_TANH : ACT_NONE, err, need_ws ? c->ws : nullptr, need_sk ? c->sk : nullptr))
    return fail(err);
  conv_launch(P, (cudaStream_t)stream);
  g_launches += (P.tapgemm || P.splitk > 1) ? 2 : 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_nc32_to_cl16(const float* in, void* out, int B, int C, int Cpad, long long S, void* stream) {
  launch_nc32_to_cl16(in, (__half*)out, B, C, Cpad, S, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_cl16_to_nc32(const void* in, float* out, int B, int C, int Cpad, long long S, void* stream) {
  launch_cl16_to_nc32((const __half*)in, out, B, C, Cpad, S, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_gn_apply(const void* y, void* out, const int64_t* stats_in, const float* gamma, const float* beta,
                 const float* temb, const void* res, int B, long long S, int C, int G, int mode, int64_t* stats_out,
                 int G_out, void* stream) {
  if (C % 8 || C / 8 > 256) return fail("gn_apply: C must be a multiple of 8 and <= 2048");
  if (mode < 0 || mode > 2) return fail("gn_apply: mode must be 0, 1 or 2");
  launch_gn_apply((const __half*)y, (__half*)out, (const stat_t*)stats_in, gamma, beta, temb, C, (const __half*)res, B, S,
                  C, G, 1e-5f, mode, (stat_t*)stats_out, G_out, (cudaStream_t)stream, nullptr, 0);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_res_attn_tail(void* y, const void* res, const int64_t* stats_in, const float* gamma2, const float* beta2, int G2,
                      const float* gamma_a, const float* beta_a, int Ga, const void* wt, const float* bias,
                      int64_t* stats_mid, float* tsum_ws, long long tsum_cap, int B, int T, int P, int C, void* stream) {
  if (B < 0 || T < 0 || P < 0) return fail("res_attn_tail: negative extent");
  if (B == 0 || T == 0 || P == 0) return 0;  // empty batch / volume: nothing to do
  if (!attn_fused_supported(C)) return fail("res_attn_tail: unsupported channel count for the fused attention path");
  const int TS = attn_tsum_splits(B, T, P, C);
  if ((long long)B * (TS + 1) * P * C > tsum_cap) return fail("res_attn_tail: depth-sum workspace too small");
  __half* g_ws = (__half*)(tsum_ws + (size_t)B * TS * P * C);  // fp16 [B][P][C] behind the depth sums
  cudaStream_t st = (cudaStream_t)stream;
  launch_gn_res_tsum((__half*)y, (const __half*)res, (const stat_t*)stats_in, gamma2, beta2, B, T, P, C, G2, 1e-5f,
                     (stat_t*)stats_mid, Ga,
                     tsum_ws, TS, st);
  launch_attn_proj_add((__half*)y, tsum_ws, TS, (const stat_t*)stats_mid, gamma_a, beta_a, (const __half*)wt, bias, g_ws, B, T, P, C,
                       Ga, 1e-5f, st);
  g_launches += 3;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_temporal_attention(const void* qkv, void* out, int B, int T, int P, int C, int heads, void* stream) {
  if (check_device()) return -1;
  if (!qkv || !out) return fail("temporal_attention: null argument");
  TAttnPlan plan;
  std::string err;
  if (tattn_plan(plan, (const __half*)qkv, (__half*)out, B, T, P, C, heads, err)) return fail(err);
  tattn_launch(plan, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("temporal_attention");
}
int b2v_gn_stats(const void* x, int B, long long S, int C, int G, int64_t* stats, void* stream) {
  launch_gn_stats((const __half*)x, B, S, C, G, (stat_t*)stats, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_ddpm_update(float* z, const float* eps, const float* noise, const float* coef, long long n, void* stream) {
  if (!z || !eps || !noise || !coef) return fail("ddpm_update: null argument");
  Coef8 c8;
  for (int i = 0; i < 8; ++i) c8.v[i] = coef[i];
  launch_ddpm_update(z, eps, noise, nullptr, nullptr, c8, n, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("ddpm_update");
}
int b2v_ddim_update(float* z, const float* eps, const float* noise, const float* coef, long long n, int* nan_flag,
                    void* stream) {
  launch_ddim_update(z, eps, noise, coef, nullptr, n, nan_flag, (cudaStream_t)stream);
  g_launches += 1;
  B2V_CUDA(cudaGetLastError());
  return 0;
}
int b2v_dpmpp_update(float* z, float* x0_prev, const float* eps, const float* noise, const float* coef, long long n,
                     int* nan_flag, void* stream) {
  if (!z || !x0_prev || !eps || !coef) return fail("dpmpp_update: null argument");
  if (n <= 0) return 0;
  launch_dpmpp_update(z, x0_prev, eps, noise, coef, nullptr, n, nan_flag, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("dpmpp_update");
}
int b2v_unipc_update(float* z, float* xc, float* hist, const float* eps, const float* coef, int step, long long n,
                     int* nan_flag, void* stream) {
  if (!z || !xc || !hist || !eps || !coef) return fail("unipc_update: null argument");
  if (step < 0) return fail("unipc_update: negative step");
  if (n <= 0) return 0;
  launch_unipc_update(z, xc, hist, eps, coef, nullptr, step, n, nan_flag, (cudaStream_t)stream);
  g_launches += 1;
  return check_launches("unipc_update");
}

}  // extern "C"
#pragma GCC visibility pop
