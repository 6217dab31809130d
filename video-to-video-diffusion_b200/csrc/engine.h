// Host runtime shared by the U-Net and VAE objects: weight store, device buffer pool, op lists that are
// captured into CUDA graphs, per-op CUDA-event profiling.
#pragma once
#include <atomic>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "conv_host.h"
#include "ew_kernels.h"

namespace b2v {

extern thread_local std::string g_err;
extern std::atomic<long long> g_launches;
int fail(const std::string& msg);  // sets g_err, returns -1
int check_launches(const char* what);  // first failed launch since the last check / cudaGetLastError -> fail()
#define B2V_CUDA(x)                                                                       \
  do {                                                                                    \
    cudaError_t e__ = (x);                                                                \
    if (e__ != cudaSuccess) return fail(std::string(#x ": ") + cudaGetErrorString(e__)); \
  } while (0)

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
  long long numel() const {
    long long n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};
using WeightMap = std::map<std::string, HostTensor>;
// returns nullptr and sets g_err if missing or (when numel > 0) of the wrong size
const HostTensor* need(const WeightMap& wm, const std::string& key, long long numel);

// device arrays owned by an object
struct DeviceStore {
  std::vector<void*> ptrs;
  float* upload(const float* h, size_t n);
  float* upload(const std::vector<float>& h) { return upload(h.data(), h.size()); }
  void* alloc(size_t bytes);   // zero-initialised; nullptr (and g_err) on failure
  void release(void* p);       // free one array early (tables that are re-grown)
  ~DeviceStore();
};

// caching device allocator for the activations of one program (all requests happen at build time)
struct Pool {
  struct Blk {
    void* p;
    size_t sz;
    bool used;
  };
  std::vector<Blk> blks;
  void* get(size_t bytes);
  void put(void* p);
  size_t total() const;
  ~Pool();
};

struct Op {
  std::string name;
  double flops = 0, bytes = 0;
  int launches = 1;
  void* out = nullptr;      // primary output of the op (debug / bisecting)
  size_t out_bytes = 0;
  std::function<void(cudaStream_t)> run;
};

// a fixed op list, replayed as one CUDA graph
struct Program {
  std::vector<Op> ops;
  cudaGraphExec_t exec = nullptr;
  int launches = 0;
  int run(cudaStream_t st);                                        // capture on first use, then graph launch
  int run_eager(cudaStream_t st);                                  // plain launches (debug)
  int profile(int iters, cudaStream_t st, std::string& json) const; // per-op event timing
  ~Program();
};

struct GNW {
  float* gamma = nullptr;
  float* beta = nullptr;
  int C = 0, G = 0;
};
int load_gn(GNW& g, const WeightMap& wm, const std::string& prefix, int C, int G, DeviceStore& ds);
int load_conv(ConvLayer& L, int kind, const WeightMap& wm, const std::string& prefix, int cin0, int cin1, int cout);
int groups32(int C);  // reference _get_num_groups: largest of 32,16,8,4,2,1 dividing C

// where gn_apply finds the per-block time-embedding projections; read at launch (= graph capture) time
struct TembSource {
  const float* base = nullptr;   // [sample or step][rows]
  int sample_stride = 0;         // per-sample stride (0: all samples share one row)
  const int* step_ptr = nullptr; // device step counter selecting the row block (sampler graphs), or null
  long long step_stride = 0;
};

// activation handle (batch is a property of the program)
struct Act {
  __half* p = nullptr;
  int C = 0, D = 0, H = 0, W = 0;
  long long S() const { return (long long)D * H * W; }
};

// op-list builder shared by the U-Net and VAE programs
struct Builder {
  std::vector<Op>& ops;
  Pool& pool;
  int B;
  stat_t* stats_base;  // Q43.20 fixed-point (sum, sumsq) pairs, see ptx.cuh
  size_t stats_cap, stats_used = 0;
  bool ok = true;
  const TembSource* temb_src = nullptr;  // U-Net programs only
  DeviceStore* ds = nullptr;             // owner of the zero-initialised split-K workspace
  float* sk_ws = nullptr;
  size_t sk_cap = 0;
  Builder(std::vector<Op>& o, Pool& p, int b, stat_t* sb, size_t sc) : ops(o), pool(p), B(b), stats_base(sb), stats_cap(sc) {}
  Act alloc(int C, int D, int H, int W);
  void free(Act& a);
  stat_t* new_stats(int G);
  // out_fp32 != nullptr: NCDHW fp32 head; otherwise returns a fresh cl16 activation
  Act conv(const std::string& name, const ConvLayer& L, const Act& in0, const Act* in1, stat_t* stats, int groups,
           float* out_fp32 = nullptr, int act = ACT_NONE);
  // temb_off >= 0: add row offset temb_off of the time-embedding table (*temb_src) after the SiLU (mode 0)
  void gn_apply(const std::string& name, Act& y, const stat_t* stats_in, const GNW& g, int temb_off, const Act* res,
                int mode, stat_t* stats_out, int G_out);
};

}  // namespace b2v
