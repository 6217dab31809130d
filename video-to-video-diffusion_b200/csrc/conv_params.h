// Kernel parameter block shared by the implicit-GEMM convolution kernels and their host-side planner.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace b2v {

enum { OUT_CL16 = 0, OUT_F32 = 1 };
enum { ACT_NONE = 0, ACT_TANH = 1 };

struct ConvParams {
  CUtensorMap tmA[4];
  CUtensorMap tmB;
  CUtensorMap tmB2;       // weight map with a half-height box (BN/2 rows): CTA-pair kernels load half a tile each
  int32_t taps[48];       // per (class, tap): (map << 24) | ((dd+8) << 16) | ((dh+8) << 8) | (dw+8)
  long long cls_off[4];   // output element offset of each class
  long long sN, sD, sH, sW, sC;  // output strides (elements)
  void* out;
  const float* bias;      // [n_tiles*BN]
  long long* stats;       // [batch][groups][2] (sum, sumsq) as Q43.20 fixed point (stat_t, ptx.cuh) or nullptr
  int bw, bh, bd, rows_valid;
  int tiles_w, tiles_h, tiles_d, batch;
  int n_tiles, nclass, ntaps;
  int src_chunks0, src_chunks1;
  int W, H, D;            // logical grid of output positions per sample and class
  int groups, cpg, cout_valid, out_mode, act;
  int splitk;             // k-splits per output tile (1 = off)
  float* ws;              // split-K fp32 workspace: splitk slabs, each NDHWC like the output
  long long ws_slab;      // elements per slab
};

// softmax temporal attention (temporal_attention.cuh)
struct TAttnParams {
  CUtensorMap tm;  // (3C, P, T, B) view of qkv, box (64, 1, TT, 1), 128-byte swizzle
  void* out;             // __half [B][T][P][C]
  long long units;
  int T, P, C, heads, hd;
  int TT;            // query / key tile rows
  int nkt;           // key tiles (= query tiles) per (b, position, head)
  int chunks;        // 64-channel chunks of one head (ceil(hd / 64))
  int pch;           // 64-key chunks of the P tile (ceil(TT / 64))
  int nq, nkv;       // depths of the Q and K/V rings (1 or 2)
  int o_col;         // first TMEM column of O (S occupies columns [0, TT))
  int tm_cols;       // TMEM columns allocated
  float scale_log2;  // log2(e) / sqrt(hd)
};

}  // namespace b2v
