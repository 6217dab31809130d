// Host side of the implicit-GEMM convolution: weight repacking, TMA tensor maps, tile geometry, launch.
#pragma once
#include <string>

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "conv_params.h"

namespace b2v {

enum ConvKind {
  CONV_K3 = 0,        // 3x3x3, stride 1, pad 1                     (torch Conv3d weight [Co][Ci][3][3][3])
  CONV_K1 = 1,        // 1x1x1                                      ([Co][Ci][1][1][1])
  CONV_DOWN = 2,      // (3,4,4) stride (1,2,2) pad 1               ([Co][Ci][3][4][4])
  CONV_UPT = 3,       // ConvTranspose3d (3,4,4) stride (1,2,2) p1  ([Ci][Co][3][4][4])
  CONV_K3_PACKW = 4,  // 3x3x3 on an input whose 3 w-taps are packed into the channel slot (slot = kw*Ci + ci)
  CONV_K3_PACKALL = 5 // 3x3x3 on an input whose 27 taps are packed into the channel slot (slot = tap*Ci + ci)
};

struct ConvLayer {
  int kind = 0;
  int cin0 = 0, cin1 = 0;          // real input channels per source (cin1 = 0: single source)
  int cin0_pad = 0, cin1_pad = 0;  // channels of the A tensors (multiples of 64)
  int cout = 0, cout_pad = 0, bn = 0;
  int ntaps = 0, nclass = 1;
  __half* w = nullptr;   // device [nclass*ntaps][cout_pad][cin0_pad+cin1_pad]
  float* bias = nullptr; // device [cout_pad]
  CUtensorMap tmB, tmB2;  // full-tile / half-tile (CTA pair) boxes
  int32_t taps[48];
  // narrow 3x3x3 heads (Cout <= 16, Cin % 64 == 0): second weight layout for the tap-GEMM path
  bool tapgemm = false;
  int tap_row_tiles = 0;    // ceil(9*Cout / 128)
  __half* wg = nullptr;     // device [kd][tap_row_tiles*128][Cin]: row = (kh*3+kw)*Cout + co
  CUtensorMap tmBg;
};

struct ConvPlan {
  ConvParams p;
  int bn = 0;
  int grid = 0;
  bool swapped = false;  // Cout == 128: operand-swapped kernel (conv_igemm_t.cuh)
  bool pair = false;     // BN == 256: CTA-pair kernel (cta_group::2, M = 256 per cluster)
  // tap-GEMM head: p describes the GEMM, the stencil pass below turns its rows into the NCDHW fp32 output
  bool tapgemm = false;
  struct {
    const float* P;
    const float* bias;
    float* out;
    int N, cout, D, H, W, act;
    long long row_stride, slice_stride;
  } st;
  // split-K (small-M layers): the conv kernel stores fp32 partial tiles into per-split slabs of fin.ws, fin describes the
  // finalize pass that sums them
  int splitk = 1;
  struct {
    float* ws;
    long long slab;
    const float* bias;
    __half* out;
    long long* stats;
    long long S;
    int C, G, B;
  } fin;
  double flops = 0;  // algorithmic 2*MAC of the reference convolution (no padding / packing waste)
};

// w_host / b_host: fp32 host arrays in the torch layout of `kind`; b_host may be null (zero bias)
int conv_layer_init(ConvLayer& L, int kind, const float* w_host, const float* b_host, int cin0, int cin1, int cout,
                    std::string& err);
void conv_layer_free(ConvLayer& L);

// in0/in1: NDHWC fp16 [N][D][H][W][cin*_pad]; (D,H,W) are the INPUT dims.
// out_mode OUT_CL16: out is NDHWC fp16 with cout channels; OUT_F32: out is NCDHW fp32 with cout channels.
int conv_plan(ConvPlan& P, const ConvLayer& L, const __half* in0, const __half* in1, int N, int D, int H, int W,
              void* out, int out_mode, long long* stats, int groups, int act, std::string& err, float* tap_ws = nullptr,
              float* splitk_ws = nullptr);
// k-split factor the planner would use for this layer / input (1 = none) and the fp32 workspace it needs
int conv_splitk_factor(const ConvLayer& L, int N, int D, int H, int W);
size_t conv_splitk_ws_bytes(const ConvLayer& L, int N, int D, int H, int W);
// bytes of fp32 workspace the tap-GEMM path of a narrow head needs for this input (0: layer has no such path)
size_t conv_tap_ws_bytes(const ConvLayer& L, int N, int D, int H, int W);
void conv_launch(const ConvPlan& P, cudaStream_t st);
int conv_setup_kernels(std::string& err);  // opt-in to large dynamic shared memory; call once per device
int device_sm_count();
__half conv_operand(float x);  // fp32 -> MMA operand (fp16; BF16-rounded first under B2V_OPERANDS=bf16)

// softmax temporal attention (temporal_attention.cuh): qkv NDHWC fp16 [B][T][P][3C] -> out [B][T][P][C]
struct TAttnPlan {
  TAttnParams p;
  int grid = 0;
  size_t smem = 0;
  double flops = 0, bytes = 0;  // algorithmic: Q K^T + P V; qkv read once, o written once
};
bool tattn_head_dim_ok(int hd);  // a multiple of 16 in [16, 128]
int tattn_plan(TAttnPlan& P, const __half* qkv, __half* out, int B, int T, int Pn, int C, int heads, std::string& err);
void tattn_launch(const TAttnPlan& P, cudaStream_t st);

}  // namespace b2v
