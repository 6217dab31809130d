// Softmax temporal attention for sm_100a: o = softmax(q k^T / sqrt(hd)) v over the T depth tokens of every
// (sample, spatial position, head) -- the corrected form of the reference TemporalAttention (models/unet3d.py:163-194,
// with 'bhqk,bhkc->bhqc' as the second contraction), used by the U-Net's opt-in "softmax" attention mode.
//
//   input  : the qkv 1x1 conv's NDHWC fp16 output [B][T][P][3C]; q, k, v of head h are channels h*hd, C + h*hd, 2C + h*hd
//   output : o, NDHWC fp16 [B][T][P][C]
//   unit   : one (b, position, head, 128-query tile); its Q, K and V are T rows P*3C elements apart, fetched by one 4-D
//            TMA box (64 channels, 1, TT rows, 1) per 64-channel chunk over the (3C, P, T, B) view of the qkv tensor;
//            TMA zero-fills rows past T.  TT = min(128, T rounded up to 16) is both the query and the key tile.
//   MMA    : tcgen05.mma kind::f16, M = 128 with fp32 accumulators in TMEM.  The query tile is padded to 128 rows:
//            rows >= TT read whatever follows the tile in shared memory and only ever reach their own (discarded)
//            output rows, since row r of S = Q K^T and of O = P V depends on row r of Q / P alone.
//              S = Q K^T   A = Q (K-major), B = K (K-major), N = TT
//              O += P V    A = P (K-major, written by the softmax warps), B = V (MN-major: d is contiguous), N = hd
//   softmax: fp32 in registers after tcgen05.ld, one thread per query row, keys >= T masked; online over key tiles
//            (running max / sum, O rescaled in TMEM when the max grows); O is normalised once at the end.
//   warps  : 0 TMA producer, 1 MMA issuer, 2..5 softmax + epilogue (one TMEM lane quarter each).
// Persistent: every CTA walks units blockIdx.x, +gridDim.x, ...; Q and K/V sit in two-deep rings, so the loads of the
// next unit run under the current one's math.  No atomics and a fixed summation order: results are bitwise
// reproducible.
#pragma once
#include "conv_params.h"
#include "ptx.cuh"

namespace b2v {

constexpr int TATTN_THREADS = 192;

__device__ __forceinline__ void tattn_unit(long long u, const TAttnParams& p, int& b, int& pos, int& head, int& qt) {
  head = (int)(u % p.heads);
  long long r = u / p.heads;
  qt = (int)(r % p.nkt);
  r /= p.nkt;
  pos = (int)(r % p.P);
  b = (int)(r / p.P);
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__global__ void __launch_bounds__(TATTN_THREADS, 1) temporal_attention_kernel(const __grid_constant__ TAttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t CB = (uint32_t)p.TT * 128u;  // one 64-channel chunk of a TT-row tile (multiple of 2048 B)
  const uint32_t tile = CB * (uint32_t)p.chunks;
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + p.nq * tile;
  uint8_t* sV = sK + p.nkv * tile;
  uint8_t* sP = sV + p.nkv * tile;
  // the M = 128 reads of the last P chunk run (128 - TT) rows past it: that slack precedes the barriers
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + p.pch * CB + (128 - p.TT) * 128);
  uint64_t* q_full = bars;
  uint64_t* q_empty = bars + 2;
  uint64_t* kv_full = bars + 4;
  uint64_t* kv_empty = bars + 6;
  uint64_t* s_full = bars + 8;   // S = Q K^T of the current key tile is in TMEM
  uint64_t* p_full = bars + 9;   // P is in shared memory and O is rescaled (S may be overwritten)
  uint64_t* pv_done = bars + 10; // O += P V has completed (P may be overwritten, O may be read)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 11);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tm);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 4);
    mbar_init(pv_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tm_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      long long n = 0, m = 0;  // units / key tiles issued by this CTA
      for (long long u = blockIdx.x; u < p.units; u += gridDim.x, ++n) {
        int b, pos, head, qt;
        tattn_unit(u, p, b, pos, head, qt);
        const int qs = (int)(n % p.nq);
        mbar_wait(&q_empty[qs], (uint32_t)((n / p.nq) & 1) ^ 1u);
        mbar_arrive_expect_tx(&q_full[qs], tile);
        for (int c = 0; c < p.chunks; ++c)
          tma_load_4d(sQ + qs * tile + c * CB, &p.tm, &q_full[qs], head * p.hd + c * 64, pos, qt * p.TT, b);
        for (int j = 0; j < p.nkt; ++j, ++m) {
          const int ks = (int)(m % p.nkv);
          mbar_wait(&kv_empty[ks], (uint32_t)((m / p.nkv) & 1) ^ 1u);
          mbar_arrive_expect_tx(&kv_full[ks], 2u * tile);
          for (int c = 0; c < p.chunks; ++c) {
            tma_load_4d(sK + ks * tile + c * CB, &p.tm, &kv_full[ks], p.C + head * p.hd + c * 64, pos, j * p.TT, b);
            tma_load_4d(sV + ks * tile + c * CB, &p.tm, &kv_full[ks], 2 * p.C + head * p.hd + c * 64, pos, j * p.TT, b);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc_s = umma_idesc_f16(128, p.TT, 0);
      const uint32_t idesc_o = umma_idesc_f16(128, p.hd, 0) | (1u << 16);  // B (= V) MN-major
      const uint32_t tS = tmem, tO = tmem + (uint32_t)p.o_col;
      long long n = 0, m = 0;
      for (long long u = blockIdx.x; u < p.units; u += gridDim.x, ++n) {
        const int qs = (int)(n % p.nq);
        mbar_wait(&q_full[qs], (uint32_t)((n / p.nq) & 1));
        tc_fence_after();
        const uint32_t qa = smem_u32(sQ + qs * tile);
        for (int j = 0; j < p.nkt; ++j, ++m) {
          const int ks = (int)(m % p.nkv);
          mbar_wait(&kv_full[ks], (uint32_t)((m / p.nkv) & 1));
          tc_fence_after();
          const uint32_t ka = smem_u32(sK + ks * tile), va = smem_u32(sV + ks * tile);
          for (int kk = 0; kk < p.hd / 16; ++kk) {  // K = 16 steps: 32 B along the swizzled 128 B row
            const uint32_t off = (uint32_t)(kk >> 2) * CB;
            umma_f16(tS, umma_desc_sw128(qa + off) + (uint64_t)((kk & 3) * 2),
                     umma_desc_sw128(ka + off) + (uint64_t)((kk & 3) * 2), idesc_s, kk > 0 ? 1u : 0u);
          }
          umma_commit(s_full);
          if (j == p.nkt - 1) umma_commit(&q_empty[qs]);
          mbar_wait(p_full, (uint32_t)(m & 1));  // P written; the previous unit's O has been read out
          tc_fence_after();
          const uint32_t pa = smem_u32(sP);
          for (int kk = 0; kk < p.TT / 16; ++kk)  // K = 16 keys: 32 B along P's rows, 16 rows (2048 B) of V
            umma_f16(tO, umma_desc_sw128(pa + (uint32_t)(kk >> 2) * CB) + (uint64_t)((kk & 3) * 2),
                     umma_desc_sw128_mn(va + (uint32_t)kk * 2048u, CB), idesc_o, (j > 0 || kk > 0) ? 1u : 0u);
          umma_commit(&kv_empty[ks]);
          umma_commit(pv_done);
        }
      }
    }
  } else {
    // ------------------------------------------------------------ softmax + epilogue (warps 2..5)
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;  // query row of the tile
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const uint32_t tS = tmem + lane_off, tO = tmem + lane_off + (uint32_t)p.o_col;
    const uint32_t prow = smem_u32(sP) + (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;
    const bool prow_ok = r < p.TT;  // rows >= TT would land in the next P chunk
    long long m = 0;
    for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
      int b, pos, head, qt;
      tattn_unit(u, p, b, pos, head, qt);
      float mrun = -INFINITY, l = 0.f;
      for (int j = 0; j < p.nkt; ++j, ++m) {
        mbar_wait(s_full, (uint32_t)(m & 1));
        tc_fence_after();
        const int kv = p.T - j * p.TT;  // valid keys in this tile (columns >= kv are masked)
        float mt = -INFINITY;
        for (int c0 = 0; c0 < p.TT; c0 += 16) {
          float v[16];
          tmem_ld_32x16(tS + (uint32_t)c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (c0 + i < kv) mt = fmaxf(mt, v[i]);
        }
        const float mnew = fmaxf(mrun, mt * p.scale_log2);
        const float alpha = exp2f(mrun - mnew);  // 0 on the first tile
        mrun = mnew;
        if (j > 0) {  // the previous P V must be done before P is overwritten and O rescaled
          mbar_wait(pv_done, (uint32_t)((m - 1) & 1));
          tc_fence_after();
        }
        float ls = 0.f;
        for (int c0 = 0; c0 < p.TT; c0 += 16) {
          float v[16];
          tmem_ld_32x16(tS + (uint32_t)c0, v);
          tmem_ld_wait();
          uint32_t h[8];
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const float e0 = (c0 + i < kv) ? exp2f(fmaf(v[i], p.scale_log2, -mnew)) : 0.f;
            const float e1 = (c0 + i + 1 < kv) ? exp2f(fmaf(v[i + 1], p.scale_log2, -mnew)) : 0.f;
            ls += e0;
            ls += e1;
            __half2 hh = __floats2half2_rn(e0, e1);
            h[i / 2] = *reinterpret_cast<uint32_t*>(&hh);
          }
          if (prow_ok) {  // 128-byte swizzle: 16-byte piece k of row r sits at piece k ^ (r % 8)
            const uint32_t a = prow + (uint32_t)(c0 >> 6) * CB;
            const uint32_t k = (uint32_t)((c0 & 63) >> 3);
            st_shared_v4(a + ((k ^ (uint32_t)(r & 7)) << 4), h[0], h[1], h[2], h[3]);
            st_shared_v4(a + (((k + 1) ^ (uint32_t)(r & 7)) << 4), h[4], h[5], h[6], h[7]);
          }
        }
        l = l * alpha + ls;
        if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
          for (int d0 = 0; d0 < p.hd; d0 += 16) {
            float v[16];
            tmem_ld_32x16(tO + (uint32_t)d0, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] *= alpha;
            tmem_st_32x16(tO + (uint32_t)d0, v);
          }
          tmem_st_wait();
        }
        fence_proxy_async_smem();  // P (generic stores) -> tensor core (async proxy)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
      }
      mbar_wait(pv_done, (uint32_t)((m - 1) & 1));
      tc_fence_after();
      const float inv = 1.f / l;
      const int t = qt * p.TT + r;
      const bool ok = prow_ok && t < p.T;
      __half* o = reinterpret_cast<__half*>(p.out) + (((size_t)b * p.T + (ok ? t : 0)) * p.P + pos) * p.C + head * p.hd;
      for (int d0 = 0; d0 < p.hd; d0 += 16) {
        float v[16];
        tmem_ld_32x16(tO + (uint32_t)d0, v);
        tmem_ld_wait();
        if (ok) {
          uint32_t h[8];
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            __half2 hh = __floats2half2_rn(v[i] * inv, v[i + 1] * inv);
            h[i / 2] = *reinterpret_cast<uint32_t*>(&hh);
          }
          uint4* dst = reinterpret_cast<uint4*>(o + d0);
          dst[0] = make_uint4(h[0], h[1], h[2], h[3]);
          dst[1] = make_uint4(h[4], h[5], h[6], h[7]);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, (uint32_t)p.tm_cols);
}

}  // namespace b2v
