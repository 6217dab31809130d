#include "conv_host.h"

#include "conv_igemm_t.cuh"
#include "ew_kernels.h"
#include "temporal_attention.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

namespace b2v {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

static int encode_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                      const cuuint32_t* box, std::string& err) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    err = "cuTensorMapEncodeTiled entry point not available";
    return -1;
  }
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box,
                   es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (%d): rank %d dims %llu %llu %llu box %u %u %u", (int)r,
             rank, (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2], box[0],
             box[1], box[2]);
    err = buf;
    return -1;
  }
  return 0;
}

static int g_sms = 0;
int device_sm_count() {
  if (!g_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_sms <= 0) g_sms = 148;
  }
  return g_sms;
}

// B2V_OPERANDS=bf16: operand-precision study (see ptx.cuh); weights are rounded to BF16 precision at pack time
static bool operands_bf16() {
  static const bool on = getenv("B2V_OPERANDS") && std::string(getenv("B2V_OPERANDS")) == "bf16";
  return on;
}
static inline __half to_operand(float x) {
  if (operands_bf16()) {
    uint32_t u;
    memcpy(&u, &x, 4);
    u += 0x7FFFu + ((u >> 16) & 1u);
    u &= 0xFFFF0000u;
    memcpy(&x, &u, 4);
  }
  return __float2half_rn(x);
}

__half conv_operand(float x) { return to_operand(x); }

int conv_setup_kernels(std::string& err) {
  cudaError_t e;
  {
    const int on = operands_bf16() ? 1 : 0;
    cudaMemcpyToSymbol(c_round_bf16, &on, sizeof(int));
    ew_set_round_bf16(on);
  }
  e = cudaFuncSetAttribute(conv_igemm_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<16>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(conv_igemm_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<64>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(conv_igemm_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<128>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(conv_igemm_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<256>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(conv_igemm_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             ConvCfg<256, true>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(conv_igemm_t_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfgT::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(conv_igemm_t_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfgT::SMEM);
  if (e != cudaSuccess) {
    err = std::string("cudaFuncSetAttribute(conv_igemm): ") + cudaGetErrorString(e);
    return -1;
  }
  return 0;
}

static inline int32_t enc_tap(int map, int dd, int dh, int dw) {
  return (map << 24) | ((dd + 8) << 16) | ((dh + 8) << 8) | (dw + 8);
}
static inline int pad64(int c) { return (c + 63) / 64 * 64; }

int conv_layer_init(ConvLayer& L, int kind, const float* w, const float* b, int cin0, int cin1, int cout,
                    std::string& err) {
  L = ConvLayer();
  L.kind = kind;
  L.cin0 = cin0;
  L.cin1 = cin1;
  L.cout = cout;
  if (cout <= 16) L.bn = 16;
  else if (cout % 256 == 0) L.bn = 256;
  else if (cout % 128 == 0) L.bn = 128;
  else if (cout % 64 == 0) L.bn = 64;
  else {
    err = "conv: Cout must be <= 16 or a multiple of 64";
    return -1;
  }
  L.cout_pad = (cout + L.bn - 1) / L.bn * L.bn;
  const bool packed = (kind == CONV_K3_PACKW || kind == CONV_K3_PACKALL);
  if (packed) {
    if (cin1) {
      err = "conv: packed kinds are single-source";
      return -1;
    }
    L.cin0_pad = pad64(cin0 * (kind == CONV_K3_PACKW ? 3 : 27));
  } else {
    if (cin0 % 64 || cin1 % 64) {
      err = "conv: Cin must be a multiple of 64 (use a packed kind for small Cin)";
      return -1;
    }
    L.cin0_pad = cin0;
    L.cin1_pad = cin1;
  }
  const int cin = cin0 + cin1;
  const int K = L.cin0_pad + L.cin1_pad;
  int kd_n = 3, kh_n = 3, kw_n = 3;
  switch (kind) {
    case CONV_K3: L.ntaps = 27; break;
    case CONV_K1: L.ntaps = 1; kd_n = kh_n = kw_n = 1; break;
    case CONV_DOWN: L.ntaps = 48; kh_n = kw_n = 4; break;
    case CONV_UPT: L.ntaps = 12; L.nclass = 4; kh_n = kw_n = 4; break;
    case CONV_K3_PACKW: L.ntaps = 9; break;
    case CONV_K3_PACKALL: L.ntaps = 1; break;
    default: err = "conv: unknown kind"; return -1;
  }
  const int nt = L.ntaps * L.nclass;
  std::vector<__half> wp((size_t)nt * L.cout_pad * K, __float2half(0.f));
  auto W = [&](int t, int co, int k) -> __half& { return wp[((size_t)t * L.cout_pad + co) * K + k]; };
  // torch Conv3d weight index [co][ci][kd][kh][kw]
  auto wc = [&](int co, int ci, int kd, int kh, int kw) {
    return w[((((size_t)co * cin + ci) * kd_n + kd) * kh_n + kh) * kw_n + kw];
  };
  if (kind == CONV_K3 || kind == CONV_K1) {
    for (int kd = 0; kd < kd_n; ++kd)
      for (int kh = 0; kh < kh_n; ++kh)
        for (int kw = 0; kw < kw_n; ++kw) {
          const int t = (kd * kh_n + kh) * kw_n + kw;
          L.taps[t] = (kind == CONV_K1) ? enc_tap(0, 0, 0, 0) : enc_tap(0, kd - 1, kh - 1, kw - 1);
          for (int co = 0; co < cout; ++co)
            for (int ci = 0; ci < cin; ++ci) W(t, co, ci) = to_operand(wc(co, ci, kd, kh, kw));
        }
  } else if (kind == CONV_DOWN) {
    // input index 2*o + k - 1  ->  parity view p, offset dlt:  k=0:(1,-1) 1:(0,0) 2:(1,0) 3:(0,+1)
    static const int par[4] = {1, 0, 1, 0}, dlt[4] = {-1, 0, 0, 1};
    for (int kd = 0; kd < 3; ++kd)
      for (int kh = 0; kh < 4; ++kh)
        for (int kw = 0; kw < 4; ++kw) {
          const int t = (kd * 4 + kh) * 4 + kw;
          L.taps[t] = enc_tap(par[kh] * 2 + par[kw], kd - 1, dlt[kh], dlt[kw]);
          for (int co = 0; co < cout; ++co)
            for (int ci = 0; ci < cin; ++ci) W(t, co, ci) = to_operand(wc(co, ci, kd, kh, kw));
        }
  } else if (kind == CONV_UPT) {
    // out(od, 2j+ph, 2i+pw) = sum in(od+1-kd, j+dh, i+dw) * w[ci][co][kd][kh][kw]
    //   ph=0: kh in {1 (dh 0), 3 (dh -1)};  ph=1: kh in {0 (dh +1), 2 (dh 0)}
    static const int ks[2][2] = {{1, 3}, {0, 2}}, ds[2][2] = {{0, -1}, {1, 0}};
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw)
        for (int kd = 0; kd < 3; ++kd)
          for (int a = 0; a < 2; ++a)
            for (int c2 = 0; c2 < 2; ++c2) {
              const int cls = ph * 2 + pw;
              const int t = cls * 12 + (kd * 2 + a) * 2 + c2;
              const int kh = ks[ph][a], kw = ks[pw][c2];
              L.taps[t] = enc_tap(0, 1 - kd, ds[ph][a], ds[pw][c2]);
              for (int co = 0; co < cout; ++co)
                for (int ci = 0; ci < cin; ++ci)
                  W(t, co, ci) = to_operand(w[((((size_t)ci * cout + co) * 3 + kd) * 4 + kh) * 4 + kw]);
            }
  } else if (kind == CONV_K3_PACKW) {
    for (int kd = 0; kd < 3; ++kd)
      for (int kh = 0; kh < 3; ++kh) {
        const int t = kd * 3 + kh;
        L.taps[t] = enc_tap(0, kd - 1, kh - 1, 0);
        for (int co = 0; co < cout; ++co)
          for (int kw = 0; kw < 3; ++kw)
            for (int ci = 0; ci < cin; ++ci) W(t, co, kw * cin + ci) = to_operand(wc(co, ci, kd, kh, kw));
      }
  } else {  // PACKALL
    L.taps[0] = enc_tap(0, 0, 0, 0);
    for (int co = 0; co < cout; ++co)
      for (int tp = 0; tp < 27; ++tp)
        for (int ci = 0; ci < cin; ++ci)
          W(0, co, tp * cin + ci) = to_operand(wc(co, ci, tp / 9, (tp / 3) % 3, tp % 3));
  }
  std::vector<float> bp(L.cout_pad, 0.f);
  if (b)
    for (int i = 0; i < cout; ++i) bp[i] = b[i];
  cudaError_t e = cudaMalloc(&L.w, wp.size() * sizeof(__half));
  if (e == cudaSuccess) e = cudaMalloc(&L.bias, bp.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(L.w, wp.data(), wp.size() * sizeof(__half), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(L.bias, bp.data(), bp.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    err = std::string("conv weights upload: ") + cudaGetErrorString(e);
    return -1;
  }
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)L.cout_pad, (cuuint64_t)nt};
  cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)K * L.cout_pad * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)L.bn, 1};
  if (encode_map(&L.tmB, L.w, 3, dims, strides, box, err)) return -1;
  cuuint32_t box2[3] = {64, (cuuint32_t)(L.bn >= 32 ? L.bn / 2 : L.bn), 1};
  if (encode_map(&L.tmB2, L.w, 3, dims, strides, box2, err)) return -1;
  if (kind == CONV_K3 && cout <= 16 && cin1 == 0) {
    // tap-GEMM layout: [kd][row][cin], row (kh*3+kw)*Cout + co holds w[co][:, kd, kh, kw] -- the depth taps are
    // accumulated inside the GEMM (three depth-shifted loads), the 3x3 in-plane taps stay separate rows
    L.tap_row_tiles = (9 * cout + 127) / 128;
    const int rows = L.tap_row_tiles * 128;
    std::vector<__half> wg((size_t)3 * rows * cin, __float2half(0.f));
    for (int t = 0; t < 27; ++t)
      for (int co = 0; co < cout; ++co)
        for (int ci = 0; ci < cin; ++ci)
        {
          // logical row r lives in UMMA row (r % 4) * 32 + r / 4 of its 128-row tile (see MODE 1 epilogue)
          const int kd = t / 9, r = (t % 9) * cout + co, tile = r / 128, rl = r % 128;
          const int phys = tile * 128 + (rl % 4) * 32 + rl / 4;
          wg[((size_t)kd * rows + phys) * cin + ci] = to_operand(wc(co, ci, kd, (t / 3) % 3, t % 3));
        }
    e = cudaMalloc(&L.wg, wg.size() * sizeof(__half));
    if (e == cudaSuccess) e = cudaMemcpy(L.wg, wg.data(), wg.size() * sizeof(__half), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      err = std::string("conv tap-gemm weights upload: ") + cudaGetErrorString(e);
      return -1;
    }
    cuuint64_t gd[3] = {(cuuint64_t)cin, (cuuint64_t)rows, 3};
    cuuint64_t gs[2] = {(cuuint64_t)cin * 2, (cuuint64_t)cin * rows * 2};
    cuuint32_t gb[3] = {64, 128, 1};
    if (encode_map(&L.tmBg, L.wg, 3, gd, gs, gb, err)) return -1;
    L.tapgemm = true;
  }
  return 0;
}

void conv_layer_free(ConvLayer& L) {
  if (L.w) cudaFree(L.w);
  if (L.bias) cudaFree(L.bias);
  if (L.wg) cudaFree(L.wg);
  L.wg = nullptr;
  L.w = nullptr;
  L.bias = nullptr;
}

// choose the (bw,bh,bd) box of <=128 positions that covers the WxHxD grid with the fewest tiles
static void choose_box(int W, int H, int D, int& bw, int& bh, int& bd) {
  long long best = -1;
  for (int w = 1; w <= 128 && w <= W; ++w)
    for (int h = 1; h * w <= 128 && h <= H; ++h) {
      int d = 128 / (w * h);
      if (d > D) d = D;
      if (d < 1) continue;
      const long long tiles = (long long)((W + w - 1) / w) * ((H + h - 1) / h) * ((D + d - 1) / d);
      const long long score = tiles * 4096 - w * 8 - h;  // fewer tiles, then longer contiguous runs
      if (best < 0 || score < best) {
        best = score;
        bw = w;
        bh = h;
        bd = d;
      }
    }
}

static void out_grid(const ConvLayer& L, int D, int H, int W, int& gD, int& gH, int& gW) {
  gD = D;
  gH = (L.kind == CONV_DOWN) ? H / 2 : H;
  gW = (L.kind == CONV_DOWN) ? W / 2 : W;
}

int conv_splitk_factor(const ConvLayer& L, int N, int D, int H, int W) {
  static const bool off = getenv("B2V_NO_SPLITK") != nullptr;
  if (off || L.bn < 64 || L.kind == CONV_UPT || L.cout % 8) return 1;
  int gD, gH, gW, bw, bh, bd;
  out_grid(L, D, H, W, gD, gH, gW);
  choose_box(gW, gH, gD, bw, bh, bd);
  const long long m_tiles = (long long)((gW + bw - 1) / bw) * ((gH + bh - 1) / bh) * ((gD + bd - 1) / bd) * N;
  const long long tiles = m_tiles * (L.cout_pad / L.bn);
  const int ksteps = L.ntaps * (L.cin0_pad + L.cin1_pad) / 64;
  const int sms = device_sm_count();
  if (ksteps < 32) return 1;
  if (tiles * 2 <= sms) {
    int S = (int)(sms / tiles);
    if (S > ksteps / 16) S = ksteps / 16;
    if (S > 8) S = 8;
    return S < 2 ? 1 : S;
  }
  // a partially filled single wave is NOT split (tried: the 6x6 level at batch 4, 56 CTA-pair units on 74 clusters cut
  // into 5 k-slices -- the atomics and the finalize pass cost more than the idle SMs: 947 vs 932 ms per batch)
  return 1;
}
size_t conv_splitk_ws_bytes(const ConvLayer& L, int N, int D, int H, int W) {
  if (conv_splitk_factor(L, N, D, H, W) < 2) return 0;
  int gD, gH, gW;
  out_grid(L, D, H, W, gD, gH, gW);
  return (size_t)conv_splitk_factor(L, N, D, H, W) * N * gD * gH * gW * L.cout * sizeof(float);  // one slab per split
}

// tap-GEMM position tiles: 128 consecutive (h, w) positions of one depth slice; slices are padded to whole tiles
static inline long long tap_slice_tiles(int H, int W) { return ((long long)H * W + 127) / 128; }
static inline long long tap_pairs(int N, int D, int H, int W) { return (tap_slice_tiles(H, W) * D * N + 1) / 2; }

size_t conv_tap_ws_bytes(const ConvLayer& L, int N, int D, int H, int W) {
  static const bool off = getenv("B2V_NO_TAPGEMM") != nullptr;
  if (!L.tapgemm || off) return 0;
  return (size_t)9 * L.cout * (size_t)(tap_pairs(N, D, H, W) * 256) * sizeof(float);
}

// GEMM over depth-slice tiles: P[(kh,kw,co)][n,d,hw] = sum_kd sum_c w[co][c][kd,kh,kw] * x[n][d+kd-1][hw][c]
// (out-of-range depths are zero-filled by TMA = the conv padding along d)
static int plan_tapgemm(ConvPlan& P, const ConvLayer& L, const __half* in0, int N, int D, int H, int W, void* out,
                        int act, std::string& err, float* ws) {
  ConvParams& p = P.p;
  p.splitk = 1;
  const long long pos = (long long)N * D * H * W;
  const long long hw = (long long)H * W;
  const long long pairs = tap_pairs(N, D, H, W);
  p.bw = 128;
  p.bh = p.bd = 1;
  p.rows_valid = 128;
  p.tiles_w = (int)tap_slice_tiles(H, W);
  p.tiles_h = 1;
  p.tiles_d = D;
  p.batch = N;
  p.n_tiles = L.tap_row_tiles;
  p.nclass = 1;
  p.ntaps = 3;
  p.src_chunks0 = L.cin0_pad / 64;
  p.src_chunks1 = 0;
  for (int kd = 0; kd < 3; ++kd) p.taps[kd] = enc_tap(0, kd - 1, 0, 0);
  p.tmB = L.tmBg;
  p.W = (int)hw;
  p.H = 1;
  p.D = D;
  p.cpg = 1;
  p.cout_valid = 9 * L.cout;
  p.out = ws;
  p.sC = pairs * 256;
  const cuuint64_t C = L.cin0_pad;
  cuuint64_t dims[5] = {C, (cuuint64_t)hw, 1, (cuuint64_t)D, (cuuint64_t)N};
  cuuint64_t st[4] = {C * 2, (cuuint64_t)hw * C * 2, (cuuint64_t)hw * C * 2, (cuuint64_t)D * hw * C * 2};
  cuuint32_t box[5] = {64, 128, 1, 1, 1};
  if (encode_map(&p.tmA[0], in0, 5, dims, st, box, err)) return -1;
  P.tapgemm = true;
  P.st.P = ws;
  P.st.bias = L.bias;
  P.st.out = (float*)out;
  P.st.N = N;
  P.st.cout = L.cout;
  P.st.D = D;
  P.st.H = H;
  P.st.W = W;
  P.st.act = act;
  P.st.row_stride = pairs * 256;
  P.st.slice_stride = tap_slice_tiles(H, W) * 128;
  const long long total = pairs * L.tap_row_tiles;
  const int sms = device_sm_count();
  P.grid = (int)(total < sms ? total : sms);
  P.flops = 2.0 * (double)pos * 27.0 * (double)L.cin0 * (double)L.cout;
  return 0;
}

int conv_plan(ConvPlan& P, const ConvLayer& L, const __half* in0, const __half* in1, int N, int D, int H, int W,
              void* out, int out_mode, long long* stats, int groups, int act, std::string& err, float* tap_ws,
              float* splitk_ws) {
  P = ConvPlan();
  ConvParams& p = P.p;
  P.bn = L.bn;
  P.splitk = 1;
  p.splitk = 1;
  if (tap_ws && out_mode == OUT_F32 && !in1 && !stats && conv_tap_ws_bytes(L, N, D, H, W))
    return plan_tapgemm(P, L, in0, N, D, H, W, out, act, err, tap_ws);
  if ((L.cin1 != 0) != (in1 != nullptr)) {
    err = "conv_plan: second source mismatch";
    return -1;
  }
  if (out_mode == OUT_CL16 && L.bn == 16) {
    err = "conv_plan: Cout<=16 layers write fp32";
    return -1;
  }
  int gW = W, gH = H, gD = D;  // grid of logical output positions
  if (L.kind == CONV_DOWN) {
    if ((W | H) & 1) {
      err = "conv_plan: strided conv needs even H, W";
      return -1;
    }
    gW = W / 2;
    gH = H / 2;
  }
  p.W = gW;
  p.H = gH;
  p.D = gD;
  choose_box(gW, gH, gD, p.bw, p.bh, p.bd);
  p.rows_valid = p.bw * p.bh * p.bd;
  p.tiles_w = (gW + p.bw - 1) / p.bw;
  p.tiles_h = (gH + p.bh - 1) / p.bh;
  p.tiles_d = (gD + p.bd - 1) / p.bd;
  p.batch = N;
  p.n_tiles = L.cout_pad / L.bn;
  p.nclass = L.nclass;
  p.ntaps = L.ntaps;
  p.src_chunks0 = L.cin0_pad / 64;
  p.src_chunks1 = L.cin1_pad / 64;
  memcpy(p.taps, L.taps, sizeof(p.taps));
  p.tmB = L.tmB;
  p.tmB2 = L.tmB2;
  p.bias = L.bias;
  p.stats = stats;
  p.groups = groups;
  p.cpg = groups ? L.cout / groups : 1;
  if (stats && (p.cpg < 2 || (p.cpg & (p.cpg - 1)) || (L.bn + p.cpg - 1) / p.cpg > 64)) {
    err = "conv_plan: channels per group must be a power of two >= 2 (and <= 64 groups per N tile)";
    return -1;
  }
  p.cout_valid = L.cout;
  p.out_mode = out_mode;
  p.act = act;
  p.out = out;

  // A tensor maps
  cuuint32_t box[5] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bh, (cuuint32_t)p.bd, 1};
  const __half* srcs[2] = {in0, in1};
  const int cpads[2] = {L.cin0_pad, L.cin1_pad};
  if (L.kind == CONV_DOWN) {
    const cuuint64_t C = cpads[0];
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) {
        cuuint64_t dims[5] = {C, (cuuint64_t)gW, (cuuint64_t)gH, (cuuint64_t)D, (cuuint64_t)N};
        cuuint64_t st[4] = {2 * C * 2, 2 * (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2,
                            (cuuint64_t)D * H * W * C * 2};
        const __half* base = in0 + ((size_t)ph * W + pw) * C;
        if (encode_map(&p.tmA[ph * 2 + pw], base, 5, dims, st, box, err)) return -1;
      }
  } else {
    for (int s = 0; s < 2; ++s) {
      if (!srcs[s]) continue;
      const cuuint64_t C = cpads[s];
      cuuint64_t dims[5] = {C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
      cuuint64_t st[4] = {C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2, (cuuint64_t)D * H * W * C * 2};
      if (encode_map(&p.tmA[s], srcs[s], 5, dims, st, box, err)) return -1;
    }
  }

  // output strides (elements)
  const long long oW = (L.kind == CONV_UPT) ? 2LL * W : gW, oH = (L.kind == CONV_UPT) ? 2LL * H : gH, oD = gD;
  const long long up = (L.kind == CONV_UPT) ? 2 : 1;
  if (out_mode == OUT_CL16) {
    const long long C = L.cout;
    p.sC = 1;
    p.sW = up * C;
    p.sH = up * oW * C;
    p.sD = oH * oW * C;
    p.sN = oD * oH * oW * C;
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) p.cls_off[ph * 2 + pw] = (ph * oW + pw) * C;
  } else {
    p.sC = oD * oH * oW;
    p.sW = up;
    p.sH = up * oW;
    p.sD = oH * oW;
    p.sN = (long long)L.cout * oD * oH * oW;
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) p.cls_off[ph * 2 + pw] = ph * oW + pw;
  }
  long long total = (long long)p.tiles_w * p.tiles_h * p.tiles_d * N * p.nclass * p.n_tiles;
  const int sms = device_sm_count();
  static const bool no_swap = getenv("B2V_NO_SWAP") != nullptr;
  const int tiles_per_sample = p.tiles_w * p.tiles_h * p.tiles_d;
  P.swapped = !no_swap && L.cout == 128 && L.bn == 128 && out_mode == OUT_CL16 && act == ACT_NONE &&
              (tiles_per_sample % 2 == 0) && (!stats || p.cpg <= 32);
  if (P.swapped) total /= 2;
  if (splitk_ws && !P.swapped && out_mode == OUT_CL16 && act == ACT_NONE) {
    const int S = conv_splitk_factor(L, N, D, H, W);
    if (S > 1) {
      P.splitk = p.splitk = S;
      p.ws = splitk_ws;
      p.ws_slab = (long long)N * gD * gH * gW * L.cout;
      total *= S;
      P.fin.ws = splitk_ws;
      P.fin.slab = p.ws_slab;
      P.fin.bias = L.bias;
      P.fin.out = (__half*)out;
      P.fin.stats = stats;
      P.fin.S = (long long)gD * gH * gW;
      P.fin.C = L.cout;
      P.fin.G = groups ? groups : 1;
      P.fin.B = N;
    }
  }
  // CTA pairs (cta_group::2) for the wide layers: a work unit is two consecutive m-tiles of one (class, n-tile)
  static const bool no_pair = getenv("B2V_NO_PAIR") != nullptr;
  P.pair = !no_pair && !P.swapped && L.bn == 256 && sms >= 2;
  if (P.pair) {
    const long long m_tiles = (long long)p.tiles_w * p.tiles_h * p.tiles_d * N;
    total = ((m_tiles + 1) / 2) * p.nclass * p.n_tiles * P.splitk;
    const long long clusters = total < sms / 2 ? total : sms / 2;
    P.grid = (int)(2 * clusters);
  } else {
    P.grid = (int)(total < sms ? total : sms);
  }
  const double taps_real = (L.kind == CONV_K1) ? 1 : (L.kind == CONV_DOWN || L.kind == CONV_UPT) ? 48 : 27;
  const double pos = (L.kind == CONV_UPT) ? (double)N * D * H * W : (double)N * gD * gH * gW;
  P.flops = 2.0 * pos * taps_real * (double)(L.cin0 + L.cin1) * (double)L.cout;
  return 0;
}

void conv_launch(const ConvPlan& P, cudaStream_t st) {
  if (P.tapgemm) {
    static const int dbg = getenv("B2V_TAP_DEBUG") ? atoi(getenv("B2V_TAP_DEBUG")) : 0;  // 1: GEMM only, 2: stencil only
    if (dbg != 2) launch_k(conv_igemm_t_kernel<1>, dim3(P.grid), dim3(ConvCfgT::threads(1)), ConvCfgT::SMEM, st, P.p);
    if (dbg != 1) launch_head_stencil(P.st.P, P.st.bias, P.st.out, P.st.N, P.st.cout, P.st.D, P.st.H, P.st.W, P.st.row_stride,
                        P.st.slice_stride, P.st.act, st);
    return;
  }
  if (P.swapped) {
    launch_k(conv_igemm_t_kernel<0>, dim3(P.grid), dim3(ConvCfgT::threads(0)), ConvCfgT::SMEM, st, P.p);
    return;
  }
  if (P.splitk > 1) {
    if (P.pair) launch_k_pair(conv_igemm_kernel<256, true>, dim3(P.grid), dim3(ConvCfg<256, true>::THREADS), ConvCfg<256, true>::SMEM, st, P.p);
    else switch (P.bn) {
      case 64: launch_k(conv_igemm_kernel<64>, dim3(P.grid), dim3(ConvCfg<64>::THREADS), ConvCfg<64>::SMEM, st, P.p); break;
      case 128: launch_k(conv_igemm_kernel<128>, dim3(P.grid), dim3(ConvCfg<128>::THREADS), ConvCfg<128>::SMEM, st, P.p); break;
      default: launch_k(conv_igemm_kernel<256>, dim3(P.grid), dim3(ConvCfg<256>::THREADS), ConvCfg<256>::SMEM, st, P.p); break;
    }
    launch_splitk_finalize(P.fin.ws, P.fin.slab, P.splitk, P.fin.bias, P.fin.out, P.fin.stats, P.fin.B, P.fin.S,
                           P.fin.C, P.fin.G, st);
    return;
  }
  if (P.pair) {
    launch_k_pair(conv_igemm_kernel<256, true>, dim3(P.grid), dim3(ConvCfg<256, true>::THREADS), ConvCfg<256, true>::SMEM, st, P.p);
    return;
  }
  switch (P.bn) {
    case 16: launch_k(conv_igemm_kernel<16>, dim3(P.grid), dim3(ConvCfg<16>::THREADS), ConvCfg<16>::SMEM, st, P.p); break;
    case 64: launch_k(conv_igemm_kernel<64>, dim3(P.grid), dim3(ConvCfg<64>::THREADS), ConvCfg<64>::SMEM, st, P.p); break;
    case 128: launch_k(conv_igemm_kernel<128>, dim3(P.grid), dim3(ConvCfg<128>::THREADS), ConvCfg<128>::SMEM, st, P.p); break;
    default: launch_k(conv_igemm_kernel<256>, dim3(P.grid), dim3(ConvCfg<256>::THREADS), ConvCfg<256>::SMEM, st, P.p); break;
  }
}

// ------------------------------------------------------------------ softmax temporal attention (temporal_attention.cuh)
bool tattn_head_dim_ok(int hd) { return hd >= 16 && hd <= 128 && hd % 16 == 0; }

int tattn_plan(TAttnPlan& P, const __half* qkv, __half* out, int B, int T, int Pn, int C, int heads, std::string& err) {
  P = TAttnPlan();
  if (B < 1 || T < 1 || Pn < 1 || heads < 1 || C % heads) {
    err = "temporal_attention: bad shape (B, T, P >= 1 and C divisible by heads)";
    return -1;
  }
  const int hd = C / heads;
  if (!tattn_head_dim_ok(hd)) {
    err = "temporal_attention: head_dim = C / heads = " + std::to_string(hd) +
          " is not supported (a multiple of 16 in [16, 128])";
    return -1;
  }
  TAttnParams& p = P.p;
  p.out = out;
  p.T = T;
  p.P = Pn;
  p.C = C;
  p.heads = heads;
  p.hd = hd;
  p.TT = T >= 128 ? 128 : (T + 15) / 16 * 16;
  p.nkt = (T + p.TT - 1) / p.TT;
  p.chunks = (hd + 63) / 64;
  p.pch = (p.TT + 63) / 64;
  p.units = (long long)B * Pn * heads * p.nkt;
  p.o_col = (p.TT + 31) / 32 * 32;
  p.tm_cols = 32;
  while (p.tm_cols < p.o_col + hd) p.tm_cols *= 2;
  p.scale_log2 = (float)(1.4426950408889634 / sqrt((double)hd));
  // shared memory: Q ring, K ring, V ring, P, the overread slack of the M = 128 operand reads, barriers, alignment
  const size_t CB = (size_t)p.TT * 128, tile = CB * p.chunks;
  const size_t kMaxSmem = 232448;  // 227 KB per block
  auto need = [&](int nq, int nkv) {
    return (nq + 2 * nkv) * tile + p.pch * CB + (size_t)(128 - p.TT) * 128 + 128 + 1024;
  };
  const int rings[4][2] = {{2, 2}, {1, 2}, {2, 1}, {1, 1}};
  int pick = -1;
  for (int i = 0; i < 4 && pick < 0; ++i)
    if (need(rings[i][0], rings[i][1]) <= kMaxSmem) pick = i;
  if (pick < 0) {
    err = "temporal_attention: tile does not fit in shared memory";
    return -1;
  }
  p.nq = rings[pick][0];
  p.nkv = rings[pick][1];
  const size_t smem = need(p.nq, p.nkv);
  cudaError_t e = cudaFuncSetAttribute(temporal_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
  int occ = 0;
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, temporal_attention_kernel, TATTN_THREADS, smem);
  if (e != cudaSuccess) {
    err = std::string("temporal_attention: ") + cudaGetErrorString(e);
    return -1;
  }
  // co-resident CTAs share the SM's 512 TMEM columns: request enough shared memory that no more than that fit
  int cps = occ < 512 / p.tm_cols ? occ : 512 / p.tm_cols;
  if (cps < 1) cps = 1;
  const size_t fence = 233472 / (size_t)(cps + 1) - 1024 + 128;  // (cps + 1) blocks of this size exceed the SM
  P.smem = smem > fence ? smem : (fence > kMaxSmem ? kMaxSmem : fence);
  const long long slots = (long long)device_sm_count() * cps;
  P.grid = (int)(p.units < slots ? p.units : slots);
  // (3C, P, T, B) view of the qkv tensor; a box is 64 channels of TT consecutive depths at one position
  const cuuint64_t C3 = 3 * (cuuint64_t)C;
  cuuint64_t dims[4] = {C3, (cuuint64_t)Pn, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[3] = {C3 * 2, C3 * Pn * 2, C3 * Pn * T * 2};
  cuuint32_t box[4] = {64, 1, (cuuint32_t)p.TT, 1};
  if (encode_map(&p.tm, qkv, 4, dims, strides, box, err)) return -1;
  P.flops = 4.0 * B * Pn * (double)T * T * C;  // Q K^T and P V
  P.bytes = (double)B * T * Pn * (3.0 * C + C) * 2.0;
  return 0;
}

void tattn_launch(const TAttnPlan& P, cudaStream_t st) {
  launch_k(temporal_attention_kernel, dim3(P.grid), dim3(TATTN_THREADS), P.smem, st, P.p);
}

}  // namespace b2v
