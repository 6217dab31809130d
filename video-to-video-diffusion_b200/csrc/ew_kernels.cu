// HBM-bound kernels of the sampling path: GroupNorm-apply fusions, the (degenerate) temporal-attention
// reduction, time embedding, scheduler updates, layout packs and the depth upsample.
// Activations are NDHWC fp16 ("cl16"); latents / images at the API boundary are NCDHW fp32 ("nc32").
// Every kernel is vectorised to 16-byte accesses along the channel (or w) axis and sized to fill 148 SMs.
#include "ew_kernels.h"

#include <math.h>
#include <stdlib.h>

namespace b2v {

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// Programmatic dependent launch is wired through every kernel but OFF by default: inside the CUDA graphs the
// kernel-to-kernel gap is already negligible and the measured step time was 0.5 % worse with it (16.53 vs 16.44 ms).
void ew_set_round_bf16(int on) { cudaMemcpyToSymbol(c_round_bf16, &on, sizeof(int)); }

bool pdl_enabled() {
  static const bool on = getenv("B2V_PDL") != nullptr;
  return on;
}

// SiLU(x) = x * sigmoid(x) = h + h * tanh(h), h = x/2: one MUFU op (tanh.approx, |err| <= 2^-11 relative, i.e. below
// the fp16 rounding of the stored result) instead of ex2 + IEEE division -- the apply kernels were issue-bound on it
__device__ __forceinline__ float silu_f(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
__device__ __forceinline__ float silu_exact(float x) { return x / (1.0f + expf(-x)); }

struct H8 {
  uint4 u;
};
__device__ __forceinline__ void h8_to_f(const uint4& u, float* f) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 f_to_h8(const float* f) {
  uint4 u;
  __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(operand_round(f[2 * i]), operand_round(f[2 * i + 1]));
  return u;
}

// Per-channel scale / shift of a GroupNorm for the 8 channels c0..c0+7 of sample b: y*sc + sh = gamma*(y-mean)*rstd + beta
__device__ __forceinline__ void gn_scale_shift(const stat_t* __restrict__ stats, const float* __restrict__ gamma,
                                               const float* __restrict__ beta, int b, int G, int cpg, double inv_n,
                                               float eps, int c0, float (&sc)[8], float (&sh)[8]) {
  int gprev = -1;
  float mean = 0.f, rstd = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = c0 + j;
    const int g = c / cpg;
    if (g != gprev) {
      stat_mean_rstd(stats + ((size_t)b * G + g) * 2, inv_n, eps, mean, rstd);
      gprev = g;
    }
    const float ga = gamma[c];
    sc[j] = ga * rstd;
    sh[j] = beta[c] - mean * ga * rstd;
  }
}

// Deterministic block reduction of per-thread partial sums (thread (cv, rr) holds 8 channels of row-slice rr) into the
// per-(sample, group) fixed-point statistics: row slices are folded in index order, then the channels of each group
// in index order, so the CTA's contribution is the same fp32 number in every run; the cross-CTA sum is an integer
// atomic (order-independent).  sm: [(R + 1)][2][C] floats.  All threads of the block must call it.
__device__ __forceinline__ void block_stats_out(const float (&as)[8], const float (&ass)[8], float* sm, int C, int R,
                                                int cv, int rr, int b, int G_out, stat_t* stats_out) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sm[(size_t)(rr * 2) * C + cv * 8 + j] = as[j];
    sm[(size_t)(rr * 2 + 1) * C + cv * 8 + j] = ass[j];
  }
  __syncthreads();
  float* tot = sm + (size_t)R * 2 * C;  // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
    const int m = i / C, c = i - m * C;
    float s = 0.f;
    for (int r = 0; r < R; ++r) s += sm[(size_t)(r * 2 + m) * C + c];
    tot[i] = s;
  }
  __syncthreads();
  const int cpo = C / G_out;
  for (int i = threadIdx.x; i < 2 * G_out; i += blockDim.x) {
    const int g = i >> 1, m = i & 1;
    float s = 0.f;
    for (int j = 0; j < cpo; ++j) s += tot[m * C + g * cpo + j];
    stat_add(stats_out + ((size_t)b * G_out + g) * 2 + m, s);
  }
}

// ------------------------------------------------------------------------------------------------
// GroupNorm apply (+affine) fused with SiLU / time-embedding add / residual add, optional statistics
// of the result for a following GroupNorm.  Reference: Conv3DBlock.forward + ResBlock3D.forward
// (models/unet3d.py:70-74,116-133; models/vae.py:31-35,50-56,72-76,93-97), conv_out[0:2] (unet3d.py:328-330).
//   mode 0: out = silu(gn(y)) + temb[b][c]           (temb may be null)
//   mode 1: out = silu(gn(y) + res)                  (res may be null)
//   mode 2: out = gn(y)                              (out of place: the softmax attention block keeps y for its residual)
// stats_in : [B][G][2] raw (sum, sumsq) over S*cpg elements, produced by the conv epilogue.
// Grid: (blocks, B); block = C8*R threads, each thread owns 8 fixed channels and strides over rows.
// ------------------------------------------------------------------------------------------------
// 3 CTAs of 256 threads per SM need <= 85 registers per thread (allocated in units of 8 -> 80): the launcher sizes the grid
// as ONE resident wave, so a variant that silently drops to 2 CTAs per SM runs a ragged second wave (+33 %)
template <int U, int MODE, bool STATS>
__global__ void __launch_bounds__(256, (!STATS && U <= 4) ? 3 : 2) gn_apply_kernel(const __half* y_, __half* out_, const stat_t* __restrict__ stats_in,
                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                const float* __restrict__ temb, int temb_stride, const int* __restrict__ temb_step,
                                long long temb_step_stride, const __half* res_, long long S, int C, int G, float eps,
                                stat_t* stats_out, int G_out) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // [(R + 1)][2][C] when stats_out
  const int C8 = C >> 3;
  const int R = blockDim.x / C8;
  const int cv = threadIdx.x % C8;
  const int rr = threadIdx.x / C8;
  const int b = blockIdx.y;
  const int c0 = cv * 8;
  const int cpg = C / G;

  // sampler graphs read the time-embedding projections of ALL steps from one table, indexed by the device step counter
  const long long toff = (MODE == 0 && temb_step) ? (long long)(*temb_step) * temb_step_stride : 0;
  float sc[8], sh[8], ta[8];
  gn_scale_shift(stats_in, gamma, beta, b, G, cpg, 1.0 / ((double)S * (double)cpg), eps, c0, sc, sh);
#pragma unroll
  for (int j = 0; j < 8; ++j) ta[j] = (MODE == 0 && temb) ? temb[toff + (size_t)b * temb_stride + c0 + j] : 0.f;
  float as[8], ass[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) as[j] = ass[j] = 0.f;

  const size_t base = (size_t)b * S * C;
  const uint4* y = reinterpret_cast<const uint4*>(y_ + base);
  uint4* out = reinterpret_cast<uint4*>(out_ + base);
  const uint4* res = res_ ? reinterpret_cast<const uint4*>(res_ + base) : nullptr;

  // 4 rows per iteration: all loads are issued before the first use so each thread keeps 4-8 16-byte requests
  // in flight (the kernel is HBM-bound; one request per thread leaves the memory system latency-limited)
  const long long stride = (long long)gridDim.x * R;
  for (long long row0 = (long long)blockIdx.x * R + rr; row0 < S; row0 += U * stride) {
    uint4 yv[U], rv[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const long long row = row0 + k * stride;
      if (row < S) {
        const size_t idx = (size_t)row * C8 + cv;
        yv[k] = y[idx];
        if (MODE == 1 && res) rv[k] = res[idx];
      }
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const long long row = row0 + k * stride;
      if (row >= S) break;
      const size_t idx = (size_t)row * C8 + cv;
      float f[8];
      h8_to_f(yv[k], f);
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j] * sc[j] + sh[j]) + ta[j];
      } else if (MODE == 2) {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = f[j] * sc[j] + sh[j];
      } else {
        float rf[8];
        if (res) {
          h8_to_f(rv[k], rf);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) rf[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j] * sc[j] + sh[j] + rf[j]);
      }
      const uint4 o = f_to_h8(f);
      out[idx] = o;
      if (STATS) {
        float g[8];
        h8_to_f(o, g);  // statistics of the values the consumer will actually read
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          as[j] += g[j];
          ass[j] += g[j] * g[j];
        }
      }
    }
  }
  if (STATS) block_stats_out(as, ass, sm, C, R, cv, rr, b, G_out, stats_out);
}

void launch_gn_apply(const __half* y, __half* out, const stat_t* stats_in, const float* gamma, const float* beta,
                     const float* temb, int temb_stride, const __half* res, int B, long long S, int C, int G,
                     float eps, int mode, stat_t* stats_out, int G_out, cudaStream_t st, const int* temb_step,
                     long long temb_step_stride) {
  const int C8 = C / 8;
  const int R = C8 >= 256 ? 1 : 256 / C8;
  const int threads = C8 * R;
  static const int U = getenv("B2V_GN_UNROLL") ? atoi(getenv("B2V_GN_UNROLL")) : 4;
  long long want = (S + U * R - 1) / (U * R);
  // 3 CTAs per SM over the whole launch = one resident wave (72-80 registers x 256 threads): few long-lived CTAs
  // amortise the per-CTA prologue (statistics -> scale / shift) and leave no ragged last wave.  Measured against 8 per
  // SM: -12 % on the U-Net's GroupNorm-apply total, -3 % on the decoder's (B2V_GN_CTAS_PER_SM overrides for A/B runs).
  static const int per_sm_env = getenv("B2V_GN_CTAS_PER_SM") ? atoi(getenv("B2V_GN_CTAS_PER_SM")) : 0;
  // the statistics-producing variants hold 16 more accumulators and fit 2 CTAs per SM
  const int per_sm = per_sm_env ? per_sm_env : ((stats_out || U > 4) ? 2 : 3);
  long long cap = (148LL * per_sm + B - 1) / B;
  int blocks = (int)(want < cap ? want : cap);
  if (blocks < 1) blocks = 1;
  const size_t smem = stats_out ? (size_t)(R + 1) * 2 * C * sizeof(float) : 0;
#define GN_LAUNCH(UU, MM, SS)                                                                                     \
  launch_k(gn_apply_kernel<UU, MM, SS>, dim3(dim3(blocks, B)), dim3(threads), smem, st, y, out, stats_in, gamma, beta, temb, temb_stride, \
           temb_step, temb_step_stride, res, S, C, G, eps, stats_out, G_out)
#define GN_DISPATCH(UU)                       \
  do {                                        \
    if (mode == 0) {                          \
      if (stats_out) GN_LAUNCH(UU, 0, true);  \
      else GN_LAUNCH(UU, 0, false);           \
    } else if (mode == 2) {                   \
      if (stats_out) GN_LAUNCH(UU, 2, true);  \
      else GN_LAUNCH(UU, 2, false);           \
    } else {                                  \
      if (stats_out) GN_LAUNCH(UU, 1, true);  \
      else GN_LAUNCH(UU, 1, false);           \
    }                                         \
  } while (0)
  if (U == 8) GN_DISPATCH(8);
  else if (U == 2) GN_DISPATCH(2);
  else GN_DISPATCH(4);
#undef GN_DISPATCH
#undef GN_LAUNCH
}

// Split-K epilogue (see conv_igemm.cuh): y = fp16(sum of the k-split slabs in index order + bias), and the
// per-(sample, group) statistics of the fp32 sums.  Deterministic: no atomics on the data path.
__global__ void splitk_finalize_kernel(const float* __restrict__ ws_, long long slab, int nsplit,
                                       const float* __restrict__ bias, __half* out_, stat_t* stats, long long S, int C,
                                       int G) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  const int C8 = C >> 3, R = blockDim.x / C8, cv = threadIdx.x % C8, rr = threadIdx.x / C8, b = blockIdx.y;
  const float4* ws = reinterpret_cast<const float4*>(ws_ + (size_t)b * S * C);
  uint4* out = reinterpret_cast<uint4*>(out_ + (size_t)b * S * C);
  const size_t slab4 = (size_t)slab / 4;
  float bs[8], as[8], ass[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    bs[j] = bias[cv * 8 + j];
    as[j] = ass[j] = 0.f;
  }
  for (long long row = (long long)blockIdx.x * R + rr; row < S; row += (long long)gridDim.x * R) {
    const size_t idx = (size_t)row * C8 + cv;
    float4 a0 = ws[idx * 2], a1 = ws[idx * 2 + 1];
    for (int k = 1; k < nsplit; ++k) {
      const float4 b0 = ws[k * slab4 + idx * 2], b1 = ws[k * slab4 + idx * 2 + 1];
      a0.x += b0.x, a0.y += b0.y, a0.z += b0.z, a0.w += b0.w;
      a1.x += b1.x, a1.y += b1.y, a1.z += b1.z, a1.w += b1.w;
    }
    float f[8] = {a0.x + bs[0], a0.y + bs[1], a0.z + bs[2], a0.w + bs[3],
                  a1.x + bs[4], a1.y + bs[5], a1.z + bs[6], a1.w + bs[7]};
    out[idx] = f_to_h8(f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      as[j] += f[j];
      ass[j] += f[j] * f[j];
    }
  }
  if (stats) block_stats_out(as, ass, sm, C, R, cv, rr, b, G, stats);
}
void launch_splitk_finalize(const float* ws, long long slab, int nsplit, const float* bias, __half* out, stat_t* stats,
                            int B, long long S, int C, int G, cudaStream_t st) {
  const int C8 = C / 8;
  const int R = C8 >= 256 ? 1 : 256 / C8;
  long long want = (S + R - 1) / R;
  long long cap = (148LL * 4 + B - 1) / B;
  int blocks = (int)(want < cap ? want : cap);
  if (blocks < 1) blocks = 1;
  launch_k(splitk_finalize_kernel, dim3(blocks, B), dim3(C8 * R), (size_t)(R + 1) * 2 * C * sizeof(float), st, ws, slab,
           nsplit, bias, out, stats, S, C, G);
}

// Stand-alone statistics pass (used when the producer is not one of our conv / apply kernels, and by tests).
__global__ void gn_stats_kernel(const __half* __restrict__ x_, long long S, int C, int G, stat_t* stats) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  const int C8 = C >> 3, R = blockDim.x / C8, cv = threadIdx.x % C8, rr = threadIdx.x / C8, b = blockIdx.y;
  const uint4* x = reinterpret_cast<const uint4*>(x_ + (size_t)b * S * C);
  float as[8], ass[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) as[j] = ass[j] = 0.f;
  for (long long row = (long long)blockIdx.x * R + rr; row < S; row += (long long)gridDim.x * R) {
    float f[8];
    h8_to_f(x[(size_t)row * C8 + cv], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      as[j] += f[j];
      ass[j] += f[j] * f[j];
    }
  }
  block_stats_out(as, ass, sm, C, R, cv, rr, b, G, stats);
}

void launch_gn_stats(const __half* x, int B, long long S, int C, int G, stat_t* stats, cudaStream_t st) {
  const int C8 = C / 8;
  const int R = C8 >= 256 ? 1 : 256 / C8;
  long long want = (S + R - 1) / R;
  long long cap = (148LL * 8 + B - 1) / B;
  int blocks = (int)(want < cap ? want : cap);
  if (blocks < 1) blocks = 1;
  launch_k(gn_stats_kernel, dim3(dim3(blocks, B)), dim3(C8 * R), (size_t)(R + 1) * 2 * C * sizeof(float), st, x, S, C,
           G, stats);
}

// ------------------------------------------------------------------------------------------------
// TemporalAttention (reference models/unet3d.py:163-194).  The reference's second einsum
// 'bhqk,bhvc->bhqc' sums k and v independently, so out[b,:,t,h,w] = (sum_k softmax) * sum_t V = sum_t V
// for every t.  With V = Wv*GN(x)+bv this is  x + Wp*(Wv * sum_t GN(x) + T*bv) + bp.
// attn_tsum: s[b,p,c] = sum_t GN32(x)[b,t,p,c] = gamma*rstd*(sum_t x - T*mean) + T*beta    (fp16 out)
// (the C x C product Wp*Wv and the folded bias are built once at weight-load time; the tiny GEMM runs on
//  the conv kernel); add_bcast_t: x[b,t,p,:] += y[b,p,:].
// ------------------------------------------------------------------------------------------------
// one block per (sample, spatial position); thread = (8-channel vector, depth split): the T slices are shared
// among blockDim/C8 thread groups (was one thread per column walking all T slices: latency-bound at 1.5 TB/s)
__global__ void attn_tsum_kernel(const __half* __restrict__ x_, const stat_t* __restrict__ stats,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, __half* s_, int T,
                                 int P, int C, int G, float eps) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // [TS][C]
  const int C8 = C >> 3;
  const int TS = blockDim.x / C8;
  const int cv = threadIdx.x % C8, ts = threadIdx.x / C8;
  const int p = blockIdx.x % P, b = blockIdx.x / P;
  const uint4* x = reinterpret_cast<const uint4*>(x_) + ((size_t)b * T * P + p) * C8 + cv;
  const size_t tstride = (size_t)P * C8;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll 4
  for (int t = ts; t < T; t += TS) {
    float f[8];
    h8_to_f(x[t * tstride], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += f[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sm[ts * C + cv * 8 + j] = acc[j];
  __syncthreads();
  if (ts != 0) return;
  for (int k = 1; k < TS; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += sm[k * C + cv * 8 + j];
  const int cpg = C / G;
  float sc[8], sh[8], o[8];
  gn_scale_shift(stats, gamma, beta, b, G, cpg, 1.0 / ((double)T * (double)P * (double)cpg), eps, cv * 8, sc, sh);
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] = fmaf(sc[j], acc[j], (float)T * sh[j]);  // sum_t (sc*x + sh)
  reinterpret_cast<uint4*>(s_)[((size_t)b * P + p) * C8 + cv] = f_to_h8(o);
}

void launch_attn_tsum(const __half* x, const stat_t* stats, const float* gamma, const float* beta, __half* s, int B,
                      int T, int P, int C, int G, float eps, cudaStream_t st) {
  const int C8 = C / 8;
  int TS = 256 / C8;
  if (TS < 1) TS = 1;
  if (TS > T) TS = T;
  launch_k(attn_tsum_kernel, dim3(B * P), dim3(C8 * TS), (size_t)TS * C * sizeof(float), st, x, stats, gamma, beta, s,
           T, P, C, G, eps);
}

__global__ void add_bcast_t_kernel(__half* x_, const __half* __restrict__ y_, int T, int PC8) {
  pdl_trigger();
  pdl_wait();
  // grid.y = sample; 32-bit index math (a 64-bit divide per element made the kernel issue-bound)
  const int b = blockIdx.y;
  uint4* x = reinterpret_cast<uint4*>(x_) + (size_t)b * T * PC8;
  const uint4* y = reinterpret_cast<const uint4*>(y_) + (size_t)b * PC8;
  const int total = T * PC8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    float a[8], c[8];
    h8_to_f(x[i], a);
    h8_to_f(y[i % PC8], c);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += c[j];
    x[i] = f_to_h8(a);
  }
}

void launch_add_bcast_t(__half* x, const __half* y, int B, int T, int P, int C, cudaStream_t st) {
  const int PC8 = P * (C / 8);
  const long long total = (long long)T * PC8;
  int blocks = cdiv(total, 256);
  const int cap = (148 * 16 + B - 1) / B;
  if (blocks > cap) blocks = cap;
  launch_k(add_bcast_t_kernel, dim3(blocks, B), dim3(256), 0, st, x, y, T, PC8);
}

// ------------------------------------------------------------------------------------------------
// Fused form of the attention-followed ResBlock tail + TemporalAttention (the block output is read once less):
//   gn_res_tsum   : y = silu(GN(y) + res) in place (ResBlock3D tail, mode 1 of gn_apply), statistics of the result for
//                   the attention's GroupNorm, and the raw depth sums  tsum[b][ts][p][c] = sum_{t in split ts} y[b,t,p,c]
//                   -- a thread owns one (position, 8-channel vector) and walks the depth axis, so the depth sum is a
//                   register accumulation and doubles as the thread's contribution to the group sums
//   attn_gemm     : s = gamma*rstd*(sum_ts tsum - T*mean) + T*beta ;  g = Wpv*s + (T*u + bp)   on the CUDA cores
//                   (2*C*C FLOP per position, 0.3 GFLOP per block at level 1: the fixed latency of the persistent
//                   tensor-core kernel was 3x its math time); then add_bcast_t: x[b,t,p,:] += g[p,:]
// ------------------------------------------------------------------------------------------------
template <int U>
__global__ void __launch_bounds__(256) gn_res_tsum_kernel(__half* y_, const __half* res_,
                                                          const stat_t* __restrict__ stats_in,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          int T, int P, int C, int G, float eps, stat_t* stats_out,
                                                          int G_out, float* tsum) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // [(PB + 1)][2][C]
  const int C8 = C >> 3;
  const int PB = blockDim.x / C8;
  const int cv = threadIdx.x % C8, pp = threadIdx.x / C8;
  const int b = blockIdx.z, ts = blockIdx.y, TS = gridDim.y;
  const int p = blockIdx.x * PB + pp;
  const int t0 = (int)((long long)ts * T / TS), t1 = (int)((long long)(ts + 1) * T / TS);
  const int cpg = C / G;
  float sc[8], sh[8], acc[8], acc2[8];
  gn_scale_shift(stats_in, gamma, beta, b, G, cpg, 1.0 / ((double)T * (double)P * (double)cpg), eps, cv * 8, sc, sh);
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = acc2[j] = 0.f;
  if (p < P && pp < PB) {
    const size_t tstride = (size_t)P * C8;
    const size_t base = ((size_t)b * T * P + p) * C8 + cv;
    uint4* y = reinterpret_cast<uint4*>(y_) + base;
    const uint4* res = res_ ? reinterpret_cast<const uint4*>(res_) + base : nullptr;
    for (int t = t0; t < t1; t += U) {
      uint4 yv[U], rv[U];
#pragma unroll
      for (int k = 0; k < U; ++k)
        if (t + k < t1) {
          yv[k] = y[(size_t)(t + k) * tstride];
          if (res) rv[k] = res[(size_t)(t + k) * tstride];
        }
#pragma unroll
      for (int k = 0; k < U; ++k) {
        if (t + k >= t1) break;
        float f[8], rf[8];
        h8_to_f(yv[k], f);
        if (res) {
          h8_to_f(rv[k], rf);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) rf[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j] * sc[j] + sh[j] + rf[j]);
        const uint4 o = f_to_h8(f);
        y[(size_t)(t + k) * tstride] = o;
        h8_to_f(o, f);  // sums of the values the consumers will actually read
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[j] += f[j];
          acc2[j] += f[j] * f[j];
        }
      }
    }
    float4* o = reinterpret_cast<float4*>(tsum + (((size_t)b * TS + ts) * P + p) * C + cv * 8);
    o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
  block_stats_out(acc, acc2, sm, C, PB, cv, pp, b, G_out, stats_out);  // threads beyond P contribute zeros
}

// depth splits so that about two waves of CTAs cover (B, P): the small levels have too few positions otherwise
int attn_tsum_splits(int B, int T, int P, int C) {
  const int C8 = C / 8;
  const int PB = 256 / C8 > 0 ? 256 / C8 : 1;
  const long long blocks = (long long)B * ((P + PB - 1) / PB);
  int TS = 1;
  while (blocks * TS < 256 && TS * 2 <= T / 4 && TS < 4) TS *= 2;
  return TS;
}

void launch_gn_res_tsum(__half* y, const __half* res, const stat_t* stats_in, const float* gamma, const float* beta,
                        int B, int T, int P, int C, int G, float eps, stat_t* stats_out, int G_out, float* tsum, int TS,
                        cudaStream_t st) {
  const int C8 = C / 8;
  const int PB = 256 / C8;
  const dim3 grid((P + PB - 1) / PB, TS, B);
  launch_k(gn_res_tsum_kernel<4>, grid, dim3(C8 * PB), (size_t)(PB + 1) * 2 * C * sizeof(float), st, y, res, stats_in, gamma, beta, T, P,
           C, G, eps, stats_out, G_out, tsum);
}

// g[b][p][co] = bias[co] + sum_c Wpv[co][c] * s[b][p][c],  s = gamma*rstd*(sum_ts tsum - T*mean) + T*beta  (fp16 out).
// Tiled CUDA-core GEMM, weight-stationary per CTA: tile = 32 positions x 64 output channels, K chunks of 64 staged in
// shared memory (the s operand is normalised on its way in), next chunk prefetched into registers while the current
// one is multiplied.  Every weight is read ceil(P/32)*B times in total (a per-position-block C x C product re-read the
// whole matrix in every CTA: 74 MB of same-address L2 traffic per launch, ~40 us).
constexpr int AG_P = 32, AG_N = 64, AG_K = 64, AG_T = 128;
template <int TS>
__global__ void __launch_bounds__(AG_T) attn_gemm_kernel(const float* __restrict__ tsum, const stat_t* __restrict__ stats,
                                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                                         const __half* __restrict__ Wt,  // [c][co] = Wpv[co][c]
                                                         const float* __restrict__ bias, __half* g_, int T, int P, int C,
                                                         int G, float eps) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sdyn[];  // per-channel scale / shift of the normalisation: [2][C]
  __shared__ __align__(16) float sS[AG_P][AG_K + 4];  // [position][k]
  __shared__ __align__(16) float sW[AG_K][AG_N];      // [k][output channel]
  float* s_scl = sdyn;
  float* s_shf = sdyn + C;
  const int b = blockIdx.z, p0 = blockIdx.x * AG_P, n0 = blockIdx.y * AG_N;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // register tile: 4 output channels x 4 positions per thread
  // loader roles: s -> (channel sc, positions spg + 2*i: 64 threads read one 256-byte run), w -> (k row wk + 16*i,
  // 8 output channels).  fetch() only ISSUES loads (no arithmetic on the results), so the next chunk's global-memory
  // latency overlaps the multiply of the current one; the normalisation happens when the registers are stashed.
  const int sc = tid & 63, spg = tid >> 6;
  const int wk = tid >> 3, wc = (tid & 7) * 8;
  float rs[TS][16];
  uint4 rw[4];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int ts = 0; ts < TS; ++ts)
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int p = min(p0 + spg + 2 * i, P - 1);  // clamped: rows beyond P are never stored
        rs[ts][i] = tsum[(((size_t)b * TS + ts) * P + p) * C + k0 + sc];
      }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      rw[i] = *reinterpret_cast<const uint4*>(Wt + (size_t)(k0 + wk + 16 * i) * C + n0 + wc);
  };
  auto stash = [&](int k0) {
    const float scl = s_scl[k0 + sc], shf = s_shf[k0 + sc];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float v = rs[0][i];
#pragma unroll
      for (int ts = 1; ts < TS; ++ts) v += rs[ts][i];
      sS[spg + 2 * i][sc] = fmaf(scl, v, shf);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float w[8];
      h8_to_f(rw[i], w);
      float4* d = reinterpret_cast<float4*>(&sW[wk + 16 * i][wc]);
      d[0] = make_float4(w[0], w[1], w[2], w[3]);
      d[1] = make_float4(w[4], w[5], w[6], w[7]);
    }
  };
  fetch(0);
  {
    const int cpg = C / G;
    const double inv_n = 1.0 / ((double)T * (double)P * (double)cpg);
    for (int c = tid; c < C; c += AG_T) {
      const int gi = c / cpg;
      float mean, rstd;
      stat_mean_rstd(stats + ((size_t)b * G + gi) * 2, inv_n, eps, mean, rstd);
      const float scl = gamma[c] * rstd;
      s_scl[c] = scl;
      s_shf[c] = (float)T * (beta[c] - mean * scl);
    }
  }
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < C; k0 += AG_K) {
    __syncthreads();  // previous chunk fully consumed (and, first time, the scale / shift table written)
    stash(k0);
    __syncthreads();
    if (k0 + AG_K < C) fetch(k0 + AG_K);
#pragma unroll 4
    for (int k4 = 0; k4 < AG_K; k4 += 4) {
      float4 sv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) sv[j] = *reinterpret_cast<const float4*>(&sS[ty * 4 + j][k4]);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4 w = *reinterpret_cast<const float4*>(&sW[k4 + kk][tx * 4]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float sj = kk == 0 ? sv[j].x : kk == 1 ? sv[j].y : kk == 2 ? sv[j].z : sv[j].w;
          acc[j][0] = fmaf(w.x, sj, acc[j][0]);
          acc[j][1] = fmaf(w.y, sj, acc[j][1]);
          acc[j][2] = fmaf(w.z, sj, acc[j][2]);
          acc[j][3] = fmaf(w.w, sj, acc[j][3]);
        }
      }
    }
  }
  const float4 bv = *reinterpret_cast<const float4*>(bias + n0 + tx * 4);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int p = p0 + ty * 4 + j;
    if (p >= P) continue;
    const __half2 h0 = __floats2half2_rn(operand_round(acc[j][0] + bv.x), operand_round(acc[j][1] + bv.y));
    const __half2 h1 = __floats2half2_rn(operand_round(acc[j][2] + bv.z), operand_round(acc[j][3] + bv.w));
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t*>(&h0);
    u.y = *reinterpret_cast<const uint32_t*>(&h1);
    *reinterpret_cast<uint2*>(g_ + ((size_t)b * P + p) * C + n0 + tx * 4) = u;
  }
}

bool attn_fused_supported(int C) { return C % 64 == 0 && C >= 64 && C / 8 <= 256; }

// the attention itself: g = Wpv * GN(sum_t x) + bias (attn_gemm), then x[b,t,p,:] += g[b,p,:] (add_bcast_t)
void launch_attn_proj_add(__half* x, const float* tsum, int TS, const stat_t* stats, const float* gamma,
                          const float* beta, const __half* Wt, const float* bias, __half* g_ws, int B, int T, int P,
                          int C, int G, float eps, cudaStream_t st) {
  const dim3 grid((P + AG_P - 1) / AG_P, C / AG_N, B);
  const size_t smem = 2 * (size_t)C * sizeof(float);
#define AG(TT) launch_k(attn_gemm_kernel<TT>, grid, dim3(AG_T), smem, st, tsum, stats, gamma, beta, Wt, bias, g_ws, T, P, C, G, eps)
  if (TS == 1) AG(1);
  else if (TS == 2) AG(2);
  else AG(4);  // attn_tsum_splits returns 1, 2 or 4
#undef AG
  launch_add_bcast_t(x, g_ws, B, T, P, C, st);
}

// ------------------------------------------------------------------------------------------------
// Time embedding (reference models/unet3d.py:18-48 and the per-block time_mlp :88-91,123-125).
//   temb_mlp : sinusoid(t) -> Linear(dim,td) -> SiLU -> Linear(td,td); stores SiLU(temb) (what every block consumes)
//   temb_proj: all ResBlock projections at once: out[b][row] = W[row,:].silu_temb[b,:] + bias[row]
// t comes from t_ptr[b]: one block per sample (forward) or per loop step (the all-steps table of a sampler loop).
// ------------------------------------------------------------------------------------------------
__global__ void temb_mlp_kernel(const long long* __restrict__ t_ptr, const float* __restrict__ freqs,
                                const float* __restrict__ W1, const float* __restrict__ b1,
                                const float* __restrict__ W2, const float* __restrict__ b2, float* silu_temb,
                                int dim, int td) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // emb[dim] | h1[td]
  float* emb = sm;
  float* h1 = sm + dim;
  const int b = blockIdx.x;
  const long long t = t_ptr[b];
  const int half = dim / 2;
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float a = (float)t * freqs[i];
    emb[i] = sinf(a);
    emb[half + i] = cosf(a);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int r = warp; r < td; r += nw) {
    float acc = 0.f;
    for (int k = lane; k < dim; k += 32) acc += W1[(size_t)r * dim + k] * emb[k];
    acc = warp_sum(acc);
    if (lane == 0) h1[r] = silu_exact(acc + b1[r]);
  }
  __syncthreads();
  for (int r = warp; r < td; r += nw) {
    float acc = 0.f;
    for (int k = lane; k < td; k += 32) acc += W2[(size_t)r * td + k] * h1[k];
    acc = warp_sum(acc);
    if (lane == 0) silu_temb[(size_t)b * td + r] = silu_exact(acc + b2[r]);
  }
}

__global__ void temb_proj_kernel(const float* __restrict__ W, const float* __restrict__ bias,
                                 const float* __restrict__ silu_temb, float* out, int rows, int td, int B) {
  pdl_trigger();
  pdl_wait();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  for (int b = 0; b < B; ++b) {
    float acc = 0.f;
    for (int k = lane; k < td; k += 32) acc += W[(size_t)warp * td + k] * silu_temb[(size_t)b * td + k];
    acc = warp_sum(acc);
    if (lane == 0) out[(size_t)b * rows + warp] = acc + bias[warp];
  }
}

void launch_temb(const long long* t_ptr, const float* freqs, const float* W1, const float* b1, const float* W2,
                 const float* b2, float* silu_temb, const float* Wp, const float* bp, float* proj, int rows, int dim,
                 int td, int B, cudaStream_t st) {
  launch_k(temb_mlp_kernel, dim3(B), dim3(512), (dim + td) * sizeof(float), st, t_ptr, freqs, W1, b1, W2, b2, silu_temb,
           dim, td);
  launch_k(temb_proj_kernel, dim3(cdiv((long long)rows * 32, 256)), dim3(256), 0, st, Wp, bp, silu_temb, proj, rows, td, B);
}

// ------------------------------------------------------------------------------------------------
// Scheduler updates, fp32, written with explicit round-to-nearest ops in the reference's operation order so
// the result is bit-identical to the reference's eager elementwise chain for the same eps.
// DDIM: reference inference/sampler.py:286-334.  coef[step] = {c1=sqrt(1-a_t+1e-8), c2=sqrt(a_t+1e-8)+1e-8,
//        c3=sqrt(a_prev+1e-8), c4=sqrt(1-a_prev+1e-8), sigma, 0,0,0}
// DDPM: reference models/diffusion.py:270-338.  coef[step] = {sqrt_1m_ac[t], sqrt_ac[t], coef1[t], coef2[t],
//        (t!=0), exp(0.5*logvar[t]), 0, 0}
// The reference's NaN guards (nan_to_num(nan=0,posinf=1,neginf=-1) when any element is non-finite) are applied
// per element unconditionally -- identical on finite data -- and recorded in *nan_flag instead of a host sync.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float nan_guard(float x, int* flag) {
  if (isnan(x)) {
    *flag = 1;
    return 0.f;
  }
  if (isinf(x)) {
    *flag = 1;
    return x > 0 ? 1.f : -1.f;
  }
  return x;
}

// Loop state of a sampler graph lives on the device (SamplerCtl, ew_kernels.h): the step index that selects the
// coefficient row / time-embedding row, the NaN flag, and where this step's noise comes from.
__device__ __forceinline__ const float* ctl_noise(const SamplerCtl* ctl, int step, long long n) {
  return ctl->noise ? ctl->noise + (long long)(step - ctl->noise_first) * n : nullptr;
}

__global__ void ddim_update_kernel(float* z, const float* __restrict__ eps, const float* __restrict__ noise_imm,
                                   const float* __restrict__ coef_table, const SamplerCtl* __restrict__ ctl,
                                   long long n, int* nan_flag) {
  pdl_trigger();
  pdl_wait();
  const int step = ctl ? ctl->step : 0;
  const float* noise = ctl ? ctl_noise(ctl, step, n) : noise_imm;
  const float* c = coef_table + (size_t)step * 8;
  const float c1 = c[0], c2 = c[1], c3 = c[2], c4 = c[3], sigma = c[4];
  int flag = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float e = nan_guard(eps[i], &flag);
    float z0 = __fdiv_rn(__fsub_rn(z[i], __fmul_rn(c1, e)), c2);
    z0 = nan_guard(z0, &flag);
    z0 = fminf(fmaxf(z0, -10.0f), 10.0f);
    float zn = __fadd_rn(__fmul_rn(c3, z0), __fmul_rn(c4, e));
    if (noise) zn = __fadd_rn(zn, __fmul_rn(sigma, noise[i]));
    z[i] = nan_guard(zn, &flag);
  }
  if (flag && nan_flag) atomicOr(nan_flag, 1);
}

// DPM-Solver++(2M) update (Lu et al. 2022, data prediction; see b2v_dpmpp_coefficients for the rows), in this fp32
// order so that a torch eager chain reproduces it bit for bit:
//   row = {sigma_t, alpha_t, a, b, w0, w1, c, clip}
//   x0 = clamp(guard((z - sigma_t*e) / alpha_t), +-clip);  D = w1 == 0 ? x0 : w0*x0 + w1*x0_prev
//   z = guard(a*z + b*D [+ c*noise]);  x0_prev = x0
// x0_prev is not read when w1 == 0 (it is uninitialised before the first step), noise not when c == 0.
__global__ void dpmpp_update_kernel(float* z, float* x0_prev, const float* __restrict__ eps,
                                    const float* __restrict__ noise_imm, const float* __restrict__ coef_table,
                                    const SamplerCtl* __restrict__ ctl, long long n, int* nan_flag) {
  pdl_trigger();
  pdl_wait();
  const int step = ctl ? ctl->step : 0;
  const float* c = coef_table + (size_t)step * 8;
  const float sig = c[0], alp = c[1], a = c[2], b = c[3], w0 = c[4], w1 = c[5], cn = c[6], clip = c[7];
  const float* noise = cn != 0.f ? (ctl ? ctl_noise(ctl, step, n) : noise_imm) : nullptr;
  int flag = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float e = nan_guard(eps[i], &flag);
    const float zi = z[i];
    float x0 = nan_guard(__fdiv_rn(__fsub_rn(zi, __fmul_rn(sig, e)), alp), &flag);
    x0 = fminf(fmaxf(x0, -clip), clip);
    const float D = (w1 == 0.f) ? x0 : __fadd_rn(__fmul_rn(w0, x0), __fmul_rn(w1, x0_prev[i]));
    float zn = __fadd_rn(__fmul_rn(a, zi), __fmul_rn(b, D));
    if (noise) zn = __fadd_rn(zn, __fmul_rn(cn, noise[i]));
    z[i] = nan_guard(zn, &flag);
    x0_prev[i] = x0;
  }
  if (flag && nan_flag) atomicOr(nan_flag, 1);
}

// Philox4x32-10 (Salmon et al., SC'11; the counter-based generator behind cuRAND / torch CUDA): counter
// (c0..c3), key (k0, k1) -> four 32-bit words.  Used for the DDPM ancestral noise when the caller passes none.
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                       uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}
// four N(0,1) draws for elements 4q..4q+3 of loop step `step`: counter (q lo, q hi, step, 0), key = seed;
// u = (word + 0.5) / 2^32 in (0,1), Box-Muller on the pairs (0,1) and (2,3)
__device__ __forceinline__ void philox_normal4(unsigned long long seed, int step, unsigned long long q, float (&nz)[4]) {
  uint32_t r[4];
  philox4x32_10((uint32_t)q, (uint32_t)(q >> 32), (uint32_t)step, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float u1 = ((float)r[2 * h] + 0.5f) * 2.3283064365386963e-10f;
    const float u2 = ((float)r[2 * h + 1] + 0.5f) * 2.3283064365386963e-10f;
    const float rad = sqrtf(-2.0f * logf(fminf(u1, 0.99999994f)));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    nz[2 * h] = rad * cs;
    nz[2 * h + 1] = rad * sn;
  }
}

// DDPM ancestral update (reference models/diffusion.py:287-338), one thread per 4 consecutive elements
__device__ __forceinline__ float ddpm_one(float zt, float e, float nz, float s1m, float sa, float k1, float k2, float nzc,
                                          float sd) {
  float z0 = __fdiv_rn(__fsub_rn(zt, __fmul_rn(s1m, e)), sa);
  z0 = fminf(fmaxf(z0, -1.0f), 1.0f);
  const float mean = __fadd_rn(__fmul_rn(k1, z0), __fmul_rn(k2, zt));
  return __fadd_rn(mean, __fmul_rn(__fmul_rn(nzc, sd), nz));
}
__global__ void ddpm_update_kernel(float* z, const float* __restrict__ eps, const float* __restrict__ noise_imm,
                                   const float* __restrict__ coef_table, const SamplerCtl* __restrict__ ctl, Coef8 cimm,
                                   long long n) {
  pdl_trigger();
  pdl_wait();
  const int step = ctl ? ctl->step : 0;
  const float* c = ctl ? coef_table + (size_t)step * 8 : cimm.v;
  const float s1m = c[0], sa = c[1], k1 = c[2], k2 = c[3], nzc = c[4], sd = c[5];
  const float* noise = ctl ? ctl_noise(ctl, step, n) : noise_imm;
  const unsigned long long seed = ctl ? ctl->seed : 0ull;
  const long long nq = (n + 3) >> 2;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (long long)gridDim.x * blockDim.x) {
    float nz[4];
    if (!noise) philox_normal4(seed, step, (unsigned long long)q, nz);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long i = q * 4 + j;
      if (i < n) z[i] = ddpm_one(z[i], eps[i], noise ? noise[i] : nz[j], s1m, sa, k1, k2, nzc, sd);
    }
  }
}
// raw generator output (tests: compared with the numpy restatement in oracle/philox.py)
__global__ void philox_fill_kernel(float* out, unsigned long long seed, int step, long long n) {
  const long long nq = (n + 3) >> 2;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (long long)gridDim.x * blockDim.x) {
    float nz[4];
    philox_normal4(seed, step, (unsigned long long)q, nz);
    for (int j = 0; j < 4; ++j)
      if (q * 4 + j < n) out[q * 4 + j] = nz[j];
  }
}
void launch_philox_fill(float* out, unsigned long long seed, int step, long long n, cudaStream_t st) {
  int blocks = cdiv((n + 3) / 4, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(philox_fill_kernel, dim3(blocks), dim3(256), 0, st, out, seed, step, n);
}

__global__ void advance_step_kernel(SamplerCtl* ctl) {
  pdl_trigger();
  pdl_wait();
  ctl->step += 1;
}

void launch_ddim_update(float* z, const float* eps, const float* noise, const float* coef_table, const SamplerCtl* ctl,
                        long long n, int* nan_flag, cudaStream_t st) {
  int blocks = cdiv(n, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(ddim_update_kernel, dim3(blocks), dim3(256), 0, st, z, eps, noise, coef_table, ctl, n, nan_flag);
}
void launch_dpmpp_update(float* z, float* x0_prev, const float* eps, const float* noise, const float* coef_table,
                         const SamplerCtl* ctl, long long n, int* nan_flag, cudaStream_t st) {
  int blocks = cdiv(n, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(dpmpp_update_kernel, dim3(blocks), dim3(256), 0, st, z, x0_prev, eps, noise, coef_table, ctl, n, nan_flag);
}
void launch_ddpm_update(float* z, const float* eps, const float* noise, const float* coef_table, const SamplerCtl* ctl,
                        const Coef8& coef, long long n, cudaStream_t st) {
  int blocks = cdiv((n + 3) / 4, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(ddpm_update_kernel, dim3(blocks), dim3(256), 0, st, z, eps, noise, coef_table, ctl, coef, n);
}

// The reference's NaN/Inf checkpoints of generate() (models/model.py:262-340): nan_to_num(nan=0, posinf=1, neginf=-1)
// when anything is non-finite.  Applied per element unconditionally (identical on finite data), recorded in *flag.
//   mode 0: only NaN -> 0 (the input check, :261-263);  mode 1: NaN -> 0, +inf -> 1, -inf -> -1
__global__ void guard_kernel(float* x, long long n, int mode, int* flag) {
  pdl_trigger();
  pdl_wait();
  int f = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    if (isnan(v)) {
      x[i] = 0.f;
      f = 1;
    } else if (mode == 1 && isinf(v)) {
      x[i] = v > 0 ? 1.f : -1.f;
      f = 1;
    }
  }
  if (f && flag) atomicOr(flag, 1);
}
__global__ void or_flag_kernel(int* dst, const int* src) { *dst |= *src; }
void launch_or_flag(int* dst, const int* src, cudaStream_t st) { launch_k(or_flag_kernel, dim3(1), dim3(1), 0, st, dst, src); }
void launch_guard(float* x, long long n, int mode, int* flag, cudaStream_t st) {
  int blocks = cdiv(n, 1024);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  launch_k(guard_kernel, dim3(blocks), dim3(256), 0, st, x, n, mode, flag);
}

// ------------------------------------------------------------------------------------------------
// Training forward (reference models/diffusion.py:81-190), forward only:
//   q_sample : z_t = sqrt_ac[t_b] * z_0 + sqrt_1m_ac[t_b] * noise          (per-sample timestep, fp32, reference op order)
//   eps_mse  : per sample, sum of mask * (eps_pred - noise)^2 and sum of mask (mask (B, C, T) broadcast over H, W, or
//              null); the Min-SNR-5 weighting and the batch mean are B-element host math in the mirror.
// eps_mse is a two-stage, fixed-order reduction (per-block partials, then one block folds them): deterministic.
// ------------------------------------------------------------------------------------------------
__global__ void q_sample_kernel(const float* __restrict__ z0, const float* __restrict__ noise,
                                const long long* __restrict__ t, const float* __restrict__ sqrt_ac,
                                const float* __restrict__ sqrt_1m_ac, float* zt, long long per_sample) {
  const int b = blockIdx.y;
  const float a = sqrt_ac[t[b]], s = sqrt_1m_ac[t[b]];
  const size_t base = (size_t)b * per_sample;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_sample;
       i += (long long)gridDim.x * blockDim.x)
    zt[base + i] = __fadd_rn(__fmul_rn(a, z0[base + i]), __fmul_rn(s, noise[base + i]));
}
void launch_q_sample(const float* z0, const float* noise, const long long* t, const float* sqrt_ac,
                     const float* sqrt_1m_ac, float* zt, int B, long long per_sample, cudaStream_t st) {
  int blocks = cdiv(per_sample, 256);
  if (blocks > 148 * 4) blocks = 148 * 4;
  launch_k(q_sample_kernel, dim3(blocks, B), dim3(256), 0, st, z0, noise, t, sqrt_ac, sqrt_1m_ac, zt, per_sample);
}

constexpr int MSE_BLOCKS = 128;
__global__ void __launch_bounds__(256) eps_mse_partial_kernel(const float* __restrict__ pred,
                                                              const float* __restrict__ noise,
                                                              const float* __restrict__ mask, long long per_sample,
                                                              long long HW, double* partial /*[B][MSE_BLOCKS][2]*/) {
  __shared__ double sh[2][256];
  const int b = blockIdx.y;
  const size_t base = (size_t)b * per_sample;
  double se = 0.0, sm = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_sample;
       i += (long long)gridDim.x * blockDim.x) {
    const float m = mask ? mask[(size_t)b * (per_sample / HW) + i / HW] : 1.0f;
    const float d = __fsub_rn(pred[base + i], noise[base + i]);
    se += (double)__fmul_rn(__fmul_rn(d, d), m);
    sm += (double)m;
  }
  sh[0][threadIdx.x] = se;
  sh[1][threadIdx.x] = sm;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {  // fixed tree
    if ((int)threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
      sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[((size_t)b * gridDim.x + blockIdx.x) * 2] = sh[0][0];
    partial[((size_t)b * gridDim.x + blockIdx.x) * 2 + 1] = sh[1][0];
  }
}
__global__ void eps_mse_final_kernel(const double* __restrict__ partial, int nblk, float* out /*[B][2]*/) {
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    double se = 0.0, sm = 0.0;
    for (int k = 0; k < nblk; ++k) {
      se += partial[((size_t)b * nblk + k) * 2];
      sm += partial[((size_t)b * nblk + k) * 2 + 1];
    }
    out[b * 2] = (float)se;
    out[b * 2 + 1] = (float)sm;
  }
}
size_t eps_mse_ws_bytes(int B) { return (size_t)B * MSE_BLOCKS * 2 * sizeof(double); }
void launch_eps_mse(const float* pred, const float* noise, const float* mask, int B, long long per_sample, long long HW,
                    double* ws, float* out, cudaStream_t st) {
  launch_k(eps_mse_partial_kernel, dim3(MSE_BLOCKS, B), dim3(256), 0, st, pred, noise, mask, per_sample, HW, ws);
  launch_k(eps_mse_final_kernel, dim3(B), dim3(32), 0, st, (const double*)ws, MSE_BLOCKS, out);
}

__global__ void zero_kernel(float* p, long long n) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = 0.f;
}
void launch_zero(float* p, long long n, cudaStream_t st) {
  int blocks = cdiv(n, 256);
  if (blocks > 148) blocks = 148;
  launch_k(zero_kernel, dim3(blocks), dim3(256), 0, st, p, n);
}
void launch_advance_step(SamplerCtl* ctl, cudaStream_t st) { launch_k(advance_step_kernel, dim3(1), dim3(1), 0, st, ctl); }

// t_dev[b] = t for every sample (step-wise DDPM)
__global__ void set_t_kernel(long long* t_dev, long long t, int B) {
  pdl_trigger();
  pdl_wait();
  const int b = threadIdx.x;
  if (b < B) t_dev[b] = t;
}
void launch_set_t(long long* t_dev, long long t, int B, cudaStream_t st) {
  const int threads = B < 64 ? 64 : B;
  launch_k(set_t_kernel, dim3(1), dim3(threads), 0, st, t_dev, t, B);
}

// ------------------------------------------------------------------------------------------------
// Input packs.  Tiny-channel inputs (latents: 2L or 8 channels, CT slices: 1 channel) are expanded so that
// the filter taps along w (or all 27 taps) sit in the 64-wide channel slot of one cl16 row; the remaining
// taps are then ordinary shifted TMA boxes of the conv kernel.
// ------------------------------------------------------------------------------------------------
// U-Net conv_in input: cat([z, c], 1) (reference models/unet3d.py:372), slot = kw*(2L) + ch
// One block = PK_SPAN consecutive positions of one sample: the 2L input rows (+1 halo element each side) are staged in
// shared memory with coalesced fp32 loads (the per-thread gather of the first version ran at 1.2 TB/s), then every
// thread assembles 16-byte output segments from them.
constexpr int PK_SPAN = 128;
__global__ void __launch_bounds__(256) pack_unet_in_kernel(const float* __restrict__ z, const float* __restrict__ c,
                                                           __half* out, int L, int W, long long S) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // [2L][PK_SPAN + 2]
  const int b = blockIdx.y;
  const long long p0 = (long long)blockIdx.x * PK_SPAN;
  const int C2 = 2 * L, pitch = PK_SPAN + 2;
  for (int i = threadIdx.x; i < C2 * pitch; i += blockDim.x) {
    const int ch = i / pitch, k = i - ch * pitch;
    const long long sp = p0 + k - 1;
    const float* src = (ch < L) ? z : c;
    const int cc = (ch < L) ? ch : ch - L;
    sm[i] = (sp >= 0 && sp < S) ? src[((size_t)b * L + cc) * S + sp] : 0.f;
  }
  __syncthreads();
  uint4* o = reinterpret_cast<uint4*>(out) + ((size_t)b * S + p0) * 8;
  // a thread keeps its segment (blockDim is a multiple of 8): the slot -> (tap, channel) map is computed once, and the
  // w coordinate advances by 32 positions per iteration -- no integer division in the loop (the first version spent
  // its time there: 72 us for 85 MB)
  const int seg = threadIdx.x & 7;
  int koff[8], kws[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int slot = seg * 8 + j;
    const int kw = slot / C2, ch = slot - kw * C2;
    kws[j] = kw;
    koff[j] = ch * pitch + kw;
  }
  const int step = blockDim.x >> 3;  // positions per iteration
  int pl = threadIdx.x >> 3;
  int w = (int)((p0 + pl) % W);
  const int wstep = step % W;
  const int n_valid = (S - p0 < PK_SPAN) ? (int)(S - p0) : PK_SPAN;
  for (; pl < n_valid; pl += step) {
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ww = w + kws[j] - 1;
      f[j] = (kws[j] < 3 && ww >= 0 && ww < W) ? sm[koff[j] + pl] : 0.f;
    }
    o[pl * 8 + seg] = f_to_h8(f);
    w += wstep;
    if (w >= W) w -= W;
  }
}
void launch_pack_unet_in(const float* z, const float* c, __half* out, int B, int L, int D, int H, int W,
                         cudaStream_t st) {
  const long long S = (long long)D * H * W;
  launch_k(pack_unet_in_kernel, dim3(cdiv(S, PK_SPAN), B), dim3(256), (size_t)2 * L * (PK_SPAN + 2) * sizeof(float), st,
           z, c, out, L, W, S);
}

// VAE decoder input: u = post_quant_conv(z / scaling_factor) (reference models/vae.py:259,192), 8 channels,
// slot = kw*8 + co
__global__ void pack_vae_dec_in_kernel(const float* __restrict__ z, const float* __restrict__ Wpq,
                                       const float* __restrict__ bpq, float scaling, __half* out, int L, int D, int H,
                                       int W, long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (b, sp, seg)
  if (i >= total) return;
  const int seg = (int)(i & 7);
  const long long pos = i >> 3;
  const long long S = (long long)D * H * W;
  const long long b = pos / S, sp = pos % S;
  const int w = (int)(pos % W);
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = 0.f;
  const int ww = w + seg - 1;
  if (seg < 3 && ww >= 0 && ww < W) {
    for (int co = 0; co < 8; ++co) f[co] = bpq[co];
    for (int ci = 0; ci < L; ++ci) {
      const float v = __fdiv_rn(z[((size_t)b * L + ci) * S + sp + (seg - 1)], scaling);
      for (int co = 0; co < 8; ++co) f[co] += Wpq[co * L + ci] * v;
    }
  }
  reinterpret_cast<uint4*>(out)[i] = f_to_h8(f);
}
void launch_pack_vae_dec_in(const float* z, const float* Wpq, const float* bpq, float scaling, __half* out, int B,
                            int L, int D, int H, int W, cudaStream_t st) {
  const long long total = (long long)B * D * H * W * 8;
  launch_k(pack_vae_dec_in_kernel, dim3(cdiv(total, 256)), dim3(256), 0, st, z, Wpq, bpq, scaling, out, L, D, H, W, total);
}

// VAE encoder input: all 27 taps of the Cin-channel volume, slot = tap*Cin + ci, tap=(kd*3+kh)*3+kw
__global__ void pack_vae_enc_in_kernel(const float* __restrict__ v, __half* out, int Cin, int Cpad, int D, int H,
                                       int W, long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (b, sp, seg)
  if (i >= total) return;
  const int nseg = Cpad / 8;
  const int seg = (int)(i % nseg);
  const long long pos = i / nseg;
  const long long S = (long long)D * H * W;
  const long long b = pos / S, sp = pos % S;
  const int w = (int)(sp % W), h = (int)((sp / W) % H), d = (int)(sp / ((long long)W * H));
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int slot = seg * 8 + j;
    const int tap = slot / Cin, ci = slot % Cin;
    float x = 0.f;
    if (tap < 27) {
      const int dd = d + tap / 9 - 1, hh = h + (tap / 3) % 3 - 1, ww = w + tap % 3 - 1;
      if (dd >= 0 && dd < D && hh >= 0 && hh < H && ww >= 0 && ww < W)
        x = v[((size_t)b * Cin + ci) * S + ((size_t)dd * H + hh) * W + ww];
    }
    f[j] = x;
  }
  reinterpret_cast<uint4*>(out)[i] = f_to_h8(f);
}
void launch_pack_vae_enc_in(const float* v, __half* out, int B, int Cin, int Cpad, int D, int H, int W,
                            cudaStream_t st) {
  const long long total = (long long)B * D * H * W * (Cpad / 8);
  launch_k(pack_vae_enc_in_kernel, dim3(cdiv(total, 256)), dim3(256), 0, st, v, out, Cin, Cpad, D, H, W, total);
}

// ------------------------------------------------------------------------------------------------
// Depth-only trilinear resample of the conditioning latent (reference models/model.py:284-289:
// F.interpolate(mode='trilinear', align_corners=False) with H, W unchanged), nc32 -> nc32.
// ------------------------------------------------------------------------------------------------
__global__ void upsample_depth_kernel(const float* __restrict__ in, float* out, int Din, int Dout, long long HW,
                                      long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (bc, dout, hw)
  if (i >= total) return;
  const long long hw = i % HW;
  const int d = (int)((i / HW) % Dout);
  const long long bc = i / (HW * Dout);
  const float scale = (float)Din / (float)Dout;
  float src = scale * ((float)d + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  const int d0 = (int)src;
  const int d1 = d0 + ((d0 < Din - 1) ? 1 : 0);
  const float l1 = src - (float)d0, l0 = 1.0f - l1;
  const float* p = in + bc * Din * HW + hw;
  out[i] = l0 * p[(size_t)d0 * HW] + l1 * p[(size_t)d1 * HW];
}
void launch_upsample_depth(const float* in, float* out, int BC, int Din, int Dout, long long HW, cudaStream_t st) {
  const long long total = (long long)BC * Dout * HW;
  launch_k(upsample_depth_kernel, dim3(cdiv(total, 256)), dim3(256), 0, st, in, out, Din, Dout, HW, total);
}

// ------------------------------------------------------------------------------------------------
// Narrow 3x3x3 heads (Cout <= 16: U-Net conv_out, VAE encoder/decoder conv_out), second half: the tap GEMM summed
// the three depth taps and wrote P[(kh*3+kw)*Cout+co][n][d][hw (padded to slice_stride)];
// out[n,co,d,h,w] = bias[co] + sum_{kh,kw} P[(kh*3+kw)*Cout+co][n,d,(h+kh-1)*W + w+kw-1] over the in-bounds taps
// (zero padding), optional tanh, fp32 NCDHW.  Every P element is read exactly once.
// ------------------------------------------------------------------------------------------------
__global__ void head_stencil_kernel(const float* __restrict__ P, const float* __restrict__ bias, float* out,
                                    int cout, int D, int H, int W, long long row_stride, long long slice_stride,
                                    int act, int planes) {
  pdl_trigger();
  pdl_wait();
  // grid.y walks the (n, co, d) planes, grid.x * block = position in the plane: only 32-bit index math per thread
  const int hw = blockIdx.x * blockDim.x + threadIdx.x;
  if (hw >= H * W) return;
  const int h = hw / W, w = hw - h * W;
  const long long tap_stride = (long long)cout * row_stride;
  for (int plane = blockIdx.y; plane < planes; plane += gridDim.y) {  // plane = (n * cout + co) * D + d
    const int d = plane % D;
    const int co = (plane / D) % cout;
    const int n = plane / (D * cout);
    const float* base = P + (long long)co * row_stride + ((long long)n * D + d) * slice_stride + hw;
    float acc = bias[co];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int dh = t / 3 - 1, dw = t % 3 - 1;
      if ((unsigned)(h + dh) < (unsigned)H && (unsigned)(w + dw) < (unsigned)W)
        acc += base[t * tap_stride + (long long)(dh * W + dw)];
    }
    out[(size_t)plane * H * W + hw] = act ? tanhf(acc) : acc;
  }
}
void launch_head_stencil(const float* P, const float* bias, float* out, int N, int cout, int D, int H, int W,
                         long long row_stride, long long slice_stride, int act, cudaStream_t st) {
  const int planes = N * cout * D;
  launch_k(head_stencil_kernel, dim3(cdiv((long long)H * W, 256), planes < 65535 ? planes : 65535), dim3(256), 0, st, P,
           bias, out, cout, D, H, W, row_stride, slice_stride, act, planes);
}

// ------------------------------------------------------------------------------------------------
// Sliding-window stitching (reference inference/sampler.py:379-451): every decoded patch is blended into the full
// volume with a separable Gaussian window (sigma = size/6), then the accumulator is divided by the summed weights.
//   acc[b,c,d0+d,h0+h,w0+w] += patch[b,c,d,h,w] * gd[d]*gh[h]*gw[w] ;  wsum[...] += gd[d]*gh[h]*gw[w]
// Patches of one launch must not overlap each other (the caller batches non-overlapping windows or launches
// one patch at a time); both tensors are nc32.
// ------------------------------------------------------------------------------------------------
__global__ void stitch_accumulate_kernel(const float* __restrict__ patch, float* acc, float* wsum,
                                         const float* __restrict__ gd, const float* __restrict__ gh,
                                         const float* __restrict__ gw, int C, int pd, int ph, int pw, int D, int H,
                                         int W, int d0, int h0, int w0, long long total) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(i % pw);
    const int h = (int)((i / pw) % ph);
    const int d = (int)((i / ((long long)pw * ph)) % pd);
    const long long bc = i / ((long long)pw * ph * pd);
    const float wt = __fmul_rn(__fmul_rn(gd[d], gh[h]), gw[w]);  // the reference's outer-product order
    const size_t o = ((size_t)bc * D + (d0 + d)) * H * W + (size_t)(h0 + h) * W + (w0 + w);
    acc[o] = __fadd_rn(acc[o], __fmul_rn(patch[i], wt));
    wsum[o] = __fadd_rn(wsum[o], wt);
  }
}
void launch_stitch_accumulate(const float* patch, float* acc, float* wsum, const float* gd, const float* gh,
                              const float* gw, int BC, int pd, int ph, int pw, int D, int H, int W, int d0, int h0,
                              int w0, cudaStream_t st) {
  const long long total = (long long)BC * pd * ph * pw;
  int blocks = cdiv(total, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(stitch_accumulate_kernel, dim3(blocks), dim3(256), 0, st, patch, acc, wsum, gd, gh, gw, BC, pd, ph, pw, D,
           H, W, d0, h0, w0, total);
}
__global__ void stitch_normalize_kernel(float* acc, const float* __restrict__ wsum, long long n) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc[i] = __fdiv_rn(acc[i], __fadd_rn(wsum[i], 1e-8f));
}
void launch_stitch_normalize(float* acc, const float* wsum, long long n, cudaStream_t st) {
  int blocks = cdiv(n, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(stitch_normalize_kernel, dim3(blocks), dim3(256), 0, st, acc, wsum, n);
}

// ------------------------------------------------------------------------------------------------
// Caller-side quality metrics (reference utils/metrics.py:14-193, what Trainer.validate* runs after generate()):
// per depth slice t, over all (b, c, h, w):  sum of squared error  and  sum of the box-filter SSIM map
//   mu = avg_pool2d(x, 11, stride 1, pad 5) (zero padding, divisor 121), sigma^2 = E[x^2]-mu^2 clamped at 0,
//   ssim = clamp(((2 mu1 mu2 + C1)(2 s12 + C2)) / ((mu1^2 + mu2^2 + C1)(s1 + s2 + C2) + 1e-8), 0, 1)
// One block = a 32x32 output tile of one (b, c, t) plane; the 42x42 halo tiles of both images sit in shared memory,
// the 11x11 box sums of the five moments are separable.  out[t] += (sq_err, ssim) with one atomic pair per block;
// the reference does two .item() host syncs per slice instead.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) video_metrics_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                            float* part, int T, int H, int W, float C1, float C2) {
  pdl_trigger();
  pdl_wait();
  constexpr int TS = 32, R = 5, IN = TS + 2 * R;  // 42
  __shared__ float sa[IN][IN + 1], sb[IN][IN + 1];
  __shared__ float hs[5][IN][TS + 1];
  __shared__ float red[2][8];
  const int plane = blockIdx.z;  // (b*C + c)*T + t
  const int t = plane % T;
  const float* pa = a + (size_t)plane * H * W;
  const float* pb = b + (size_t)plane * H * W;
  const int x0 = blockIdx.x * TS, y0 = blockIdx.y * TS;
  for (int i = threadIdx.x; i < IN * IN; i += 256) {
    const int ly = i / IN, lx = i % IN;
    const int gy = y0 + ly - R, gx = x0 + lx - R;
    const bool in = (gy >= 0 && gy < H && gx >= 0 && gx < W);
    sa[ly][lx] = in ? pa[(size_t)gy * W + gx] : 0.f;
    sb[ly][lx] = in ? pb[(size_t)gy * W + gx] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < IN * TS; i += 256) {  // horizontal 11-tap sums of x, y, xx, yy, xy
    const int ly = i / TS, lx = i % TS;
    float s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0;
#pragma unroll
    for (int k = 0; k < 2 * R + 1; ++k) {
      const float u = sa[ly][lx + k], v = sb[ly][lx + k];
      s0 += u;
      s1 += v;
      s2 += u * u;
      s3 += v * v;
      s4 += u * v;
    }
    hs[0][ly][lx] = s0;
    hs[1][ly][lx] = s1;
    hs[2][ly][lx] = s2;
    hs[3][ly][lx] = s3;
    hs[4][ly][lx] = s4;
  }
  __syncthreads();
  float se = 0.f, ssim = 0.f;
  for (int i = threadIdx.x; i < TS * TS; i += 256) {
    const int ly = i / TS, lx = i % TS;
    if (y0 + ly < H && x0 + lx < W) {
      float m[5] = {0, 0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < 2 * R + 1; ++k)
#pragma unroll
        for (int q = 0; q < 5; ++q) m[q] += hs[q][ly + k][lx];
      const float inv = 1.0f / 121.0f;
      const float mu1 = m[0] * inv, mu2 = m[1] * inv;
      const float s1 = fmaxf(m[2] * inv - mu1 * mu1, 0.f), s2 = fmaxf(m[3] * inv - mu2 * mu2, 0.f);
      const float s12 = m[4] * inv - mu1 * mu2;
      const float num = (2.f * mu1 * mu2 + C1) * (2.f * s12 + C2);
      const float den = (mu1 * mu1 + mu2 * mu2 + C1) * (s1 + s2 + C2) + 1e-8f;
      ssim += fminf(fmaxf(num / den, 0.f), 1.f);
      const float d = sa[ly + R][lx + R] - sb[ly + R][lx + R];
      se += d * d;
    }
  }
  se = warp_sum(se);
  ssim = warp_sum(ssim);
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = se;
    red[1][threadIdx.x >> 5] = ssim;
  }
  __syncthreads();
  if (threadIdx.x < 2) {  // one partial per block (no atomics: the second pass folds them in a fixed order)
    float s = 0.f;
    for (int k = 0; k < 8; ++k) s += red[threadIdx.x][k];
    (void)t;
    part[(((size_t)plane * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 2 + threadIdx.x] = s;
  }
}
// out[t] = sum over (bc, tile) of the block partials of slice t, in index order (fp64 accumulation): deterministic
__global__ void video_metrics_fold_kernel(const float* __restrict__ part, float* out, int BC, int T, int tiles) {
  const int t = blockIdx.x, m = threadIdx.x;
  if (m >= 2) return;
  double s = 0.0;
  for (int bc = 0; bc < BC; ++bc) {
    const float* p = part + ((size_t)(bc * T + t) * tiles) * 2 + m;
    for (int k = 0; k < tiles; ++k) s += (double)p[(size_t)k * 2];
  }
  out[t * 2 + m] = (float)s;
}
size_t video_metrics_ws_bytes(int BC, int T, int H, int W) {
  return (size_t)BC * T * ((W + 31) / 32) * ((H + 31) / 32) * 2 * sizeof(float);
}
void launch_video_metrics(const float* a, const float* b, float* out, float* ws, int BC, int T, int H, int W,
                          float max_val, cudaStream_t st) {
  const float C1 = (0.01f * max_val) * (0.01f * max_val), C2 = (0.03f * max_val) * (0.03f * max_val);
  const dim3 grid((W + 31) / 32, (H + 31) / 32, BC * T);
  launch_k(video_metrics_kernel, grid, dim3(256), 0, st, a, b, ws, T, H, W, C1, C2);
  launch_k(video_metrics_fold_kernel, dim3(T), dim3(32), 0, st, (const float*)ws, out, BC, T, (int)(grid.x * grid.y));
}

// ------------------------------------------------------------------------------------------------
// Input side (reference data/slice_interpolation_dataset.py:575-592 CT windowing, and
// data/patch_slice_interpolation_dataset.py:163-181 aligned crop + depth resample of the thick sub-volume):
//   out[d,h,w] = lerp_depth( f(vol[z0 + i, y0 + h, x0 + w]) ),  f(v) = a * clip(v, lo, hi) + b
// with the depth source index of F.interpolate(trilinear, align_corners=False): src = n/pd * (d + 0.5) - 0.5 (>= 0).
// One pass, coalesced along w; feeds the encoder directly on the device.
// ------------------------------------------------------------------------------------------------
__global__ void extract_patch_kernel(const float* __restrict__ vol, float* out, int H, int W, int z0, int n, int y0,
                                     int x0, int pd, int ph, int pw, float lo, float hi, float a, float b,
                                     long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int w = (int)(i % pw), h = (int)((i / pw) % ph), d = (int)(i / ((long long)pw * ph));
  const float scale = (float)n / (float)pd;
  float src = scale * ((float)d + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  const int i0 = (int)src;
  const int i1 = i0 + ((i0 < n - 1) ? 1 : 0);
  const float l1 = src - (float)i0, l0 = 1.0f - l1;
  const size_t plane = (size_t)H * W, off = (size_t)(y0 + h) * W + (x0 + w);
  const float v0 = fminf(fmaxf(vol[(size_t)(z0 + i0) * plane + off], lo), hi) * a + b;
  const float v1 = fminf(fmaxf(vol[(size_t)(z0 + i1) * plane + off], lo), hi) * a + b;
  out[i] = l0 * v0 + l1 * v1;
}
void launch_extract_patch(const float* vol, float* out, int H, int W, int z0, int n, int y0, int x0, int pd, int ph,
                          int pw, float lo, float hi, float a, float b, cudaStream_t st) {
  const long long total = (long long)pd * ph * pw;
  launch_k(extract_patch_kernel, dim3(cdiv(total, 256)), dim3(256), 0, st, vol, out, H, W, z0, n, y0, x0, pd, ph, pw,
           lo, hi, a, b, total);
}

// ------------------------------------------------------------------------------------------------
// Layout casts for the op-level API and tests
// ------------------------------------------------------------------------------------------------
__global__ void nc32_to_cl16_kernel(const float* __restrict__ in, __half* out, int C, int Cpad, long long S,
                                    long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (b, sp, c)
  if (i >= total) return;
  const int c = (int)(i % Cpad);
  const long long sp = (i / Cpad) % S, b = i / (Cpad * S);
  out[i] = __float2half_rn(operand_round(c < C ? in[((size_t)b * C + c) * S + sp] : 0.f));
}
__global__ void cl16_to_nc32_kernel(const __half* __restrict__ in, float* out, int C, int Cpad, long long S,
                                    long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (b, c, sp)
  if (i >= total) return;
  const long long sp = i % S;
  const int c = (int)((i / S) % C);
  const long long b = i / (S * C);
  out[i] = __half2float(in[((size_t)b * S + sp) * Cpad + c]);
}
void launch_nc32_to_cl16(const float* in, __half* out, int B, int C, int Cpad, long long S, cudaStream_t st) {
  const long long total = (long long)B * S * Cpad;
  launch_k(nc32_to_cl16_kernel, dim3(cdiv(total, 256)), dim3(256), 0, st, in, out, C, Cpad, S, total);
}
void launch_cl16_to_nc32(const __half* in, float* out, int B, int C, int Cpad, long long S, cudaStream_t st) {
  const long long total = (long long)B * S * C;
  launch_k(cl16_to_nc32_kernel, dim3(cdiv(total, 256)), dim3(256), 0, st, in, out, C, Cpad, S, total);
}

}  // namespace b2v
