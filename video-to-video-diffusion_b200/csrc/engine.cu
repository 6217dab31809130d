#include "engine.h"

#include <stdio.h>
#include <stdlib.h>

namespace b2v {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

int fail(const std::string& msg) {
  g_err = msg;
  return -1;
}

static thread_local cudaError_t g_launch_err = cudaSuccess;
void note_launch_error(cudaError_t e) {
  if (g_launch_err == cudaSuccess) g_launch_err = e;
}
cudaError_t take_launch_error() {
  const cudaError_t e = g_launch_err;
  g_launch_err = cudaSuccess;
  return e;
}
// status of everything launched since the last check: a failed cudaLaunchKernelEx first, then the runtime's last error
int check_launches(const char* what) {
  cudaError_t e = take_launch_error();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return fail(std::string(what) + ": " + cudaGetErrorString(e));
  return 0;
}

const HostTensor* need(const WeightMap& wm, const std::string& key, long long numel) {
  auto it = wm.find(key);
  if (it == wm.end()) {
    fail("missing state_dict key: " + key);
    return nullptr;
  }
  if (numel > 0 && it->second.numel() != numel) {
    fail("state_dict key " + key + " has " + std::to_string(it->second.numel()) + " elements, expected " +
         std::to_string(numel));
    return nullptr;
  }
  return &it->second;
}

float* DeviceStore::upload(const float* h, size_t n) {
  float* d = nullptr;
  cudaError_t e = cudaMalloc(&d, (n ? n : 1) * sizeof(float));
  if (e == cudaSuccess && n) e = cudaMemcpy(d, h, n * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {  // a failed upload must not leave uninitialised weights behind a success code
    if (d) cudaFree(d);
    fail(std::string("device upload failed: ") + cudaGetErrorString(e));
    return nullptr;
  }
  ptrs.push_back(d);
  return d;
}
void* DeviceStore::alloc(size_t bytes) {
  void* d = nullptr;
  cudaError_t e = cudaMalloc(&d, bytes ? bytes : 1);
  if (e == cudaSuccess && bytes) e = cudaMemset(d, 0, bytes);
  if (e != cudaSuccess) {
    if (d) cudaFree(d);
    fail(std::string("device allocation failed: ") + cudaGetErrorString(e));
    return nullptr;
  }
  ptrs.push_back(d);
  return d;
}
void DeviceStore::release(void* p) {
  for (size_t i = 0; i < ptrs.size(); ++i)
    if (ptrs[i] == p) {
      cudaFree(p);
      ptrs.erase(ptrs.begin() + i);
      return;
    }
}
DeviceStore::~DeviceStore() {
  for (void* p : ptrs) cudaFree(p);
}

void* Pool::get(size_t bytes) {
  bytes = (bytes + 1023) / 1024 * 1024;
  int best = -1;
  for (int i = 0; i < (int)blks.size(); ++i)
    if (!blks[i].used && blks[i].sz >= bytes && (best < 0 || blks[i].sz < blks[best].sz)) best = i;
  if (best >= 0 && blks[best].sz <= bytes * 2) {
    blks[best].used = true;
    return blks[best].p;
  }
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    fail("out of device memory in activation pool (" + std::to_string(bytes) + " bytes)");
    return nullptr;
  }
  blks.push_back({p, bytes, true});
  return p;
}
void Pool::put(void* p) {
  for (auto& b : blks)
    if (b.p == p) b.used = false;
}
size_t Pool::total() const {
  size_t t = 0;
  for (auto& b : blks) t += b.sz;
  return t;
}
Pool::~Pool() {
  for (auto& b : blks) cudaFree(b.p);
}

Program::~Program() {
  if (exec) cudaGraphExecDestroy(exec);
}

int Program::run_eager(cudaStream_t st) {
  for (auto& op : ops) op.run(st);
  g_launches += launches;
  return check_launches("program launch");
}

int Program::run(cudaStream_t st) {
  static const bool eager = getenv("B2V_EAGER") != nullptr;  // debugging aid: plain launches instead of a graph
  if (eager) {
    if (!launches)
      for (auto& op : ops) launches += op.launches;
    return run_eager(st);
  }
  if (!exec) {
    launches = 0;
    for (auto& op : ops) launches += op.launches;
    cudaStream_t cs;
    B2V_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
    if (e == cudaSuccess) {
      for (auto& op : ops) op.run(cs);
      e = cudaStreamEndCapture(cs, &g);
      const cudaError_t le = take_launch_error();
      if (e == cudaSuccess) e = le;
    }
    if (e == cudaSuccess) e = cudaGraphInstantiate(&exec, g, 0);
    if (g) cudaGraphDestroy(g);
    cudaStreamDestroy(cs);
    if (e != cudaSuccess) {
      exec = nullptr;
      return fail(std::string("CUDA graph capture failed: ") + cudaGetErrorString(e));
    }
  }
  B2V_CUDA(cudaGraphLaunch(exec, st));
  g_launches += launches;
  return 0;
}

int Program::profile(int iters, cudaStream_t st, std::string& json) const {
  cudaEvent_t e0, e1;
  B2V_CUDA(cudaEventCreate(&e0));
  B2V_CUDA(cudaEventCreate(&e1));
  std::vector<float> ms(ops.size(), 0.f);
  for (int it = 0; it < iters + 1; ++it) {  // first pass is warm-up
    for (size_t i = 0; i < ops.size(); ++i) {
      cudaEventRecord(e0, st);
      ops[i].run(st);
      cudaEventRecord(e1, st);
      cudaEventSynchronize(e1);
      float t = 0;
      cudaEventElapsedTime(&t, e0, e1);
      if (it > 0) ms[i] += t / iters;
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (check_launches("profile")) return -1;
  json = "[";
  char buf[512];
  for (size_t i = 0; i < ops.size(); ++i) {
    snprintf(buf, sizeof buf, "%s{\"name\": \"%s\", \"ms\": %.6f, \"flops\": %.6e, \"bytes\": %.6e}", i ? ", " : "",
             ops[i].name.c_str(), ms[i], ops[i].flops, ops[i].bytes);
    json += buf;
  }
  json += "]";
  return 0;
}

int groups32(int C) {
  const int cand[6] = {32, 16, 8, 4, 2, 1};
  for (int g : cand)
    if (C % g == 0) return g;
  return 1;
}

int load_gn(GNW& g, const WeightMap& wm, const std::string& prefix, int C, int G, DeviceStore& ds) {
  const HostTensor* w = need(wm, prefix + ".weight", C);
  const HostTensor* b = need(wm, prefix + ".bias", C);
  if (!w || !b) return -1;
  g.gamma = ds.upload(w->data);
  g.beta = ds.upload(b->data);
  g.C = C;
  g.G = G;
  return (g.gamma && g.beta) ? 0 : fail("device alloc failed for " + prefix);
}

int load_conv(ConvLayer& L, int kind, const WeightMap& wm, const std::string& prefix, int cin0, int cin1, int cout) {
  const int cin = cin0 + cin1;
  long long taps = 27;
  if (kind == CONV_K1) taps = 1;
  if (kind == CONV_DOWN || kind == CONV_UPT) taps = 48;
  const HostTensor* w = need(wm, prefix + ".weight", (long long)cout * cin * taps);
  const HostTensor* b = need(wm, prefix + ".bias", cout);
  if (!w || !b) return -1;
  std::string err;
  if (conv_layer_init(L, kind, w->data.data(), b->data.data(), cin0, cin1, cout, err)) return fail(prefix + ": " + err);
  return 0;
}

Act Builder::alloc(int C, int D, int H, int W) {
  Act a;
  a.C = C;
  a.D = D;
  a.H = H;
  a.W = W;
  a.p = (__half*)pool.get((size_t)B * D * H * W * C * sizeof(__half));
  if (!a.p) ok = false;
  return a;
}
void Builder::free(Act& a) {
  if (a.p) pool.put(a.p);
  a.p = nullptr;
}
stat_t* Builder::new_stats(int G) {
  const size_t n = (size_t)B * G * 2;
  if (stats_used + n > stats_cap) {
    fail("statistics arena exhausted");
    ok = false;
    return stats_base;
  }
  stat_t* s = stats_base + stats_used;
  stats_used += n;
  return s;
}

Act Builder::conv(const std::string& name, const ConvLayer& L, const Act& in0, const Act* in1, stat_t* stats,
                  int groups, float* out_fp32, int act) {
  Act out;
  int oD = in0.D, oH = in0.H, oW = in0.W;
  if (L.kind == CONV_DOWN) {
    oH /= 2;
    oW /= 2;
  } else if (L.kind == CONV_UPT) {
    oH *= 2;
    oW *= 2;
  }
  if (!out_fp32) out = alloc(L.cout, oD, oH, oW);
  if (!ok) return out;
  if (in0.C != L.cin0_pad || (in1 && in1->C != L.cin1_pad)) {
    fail(name + ": input channel mismatch");
    ok = false;
    return out;
  }
  ConvPlan P;
  std::string err;
  float* ws = nullptr;
  const size_t ws_bytes = (out_fp32 && !in1 && !stats) ? conv_tap_ws_bytes(L, B, in0.D, in0.H, in0.W) : 0;
  if (ws_bytes) {
    ws = (float*)pool.get(ws_bytes);  // live only during this op: returned to the pool right after planning
    if (!ws) {
      ok = false;
      return out;
    }
  }
  // split-K workspace: persistent and zero between uses (the finalize pass re-zeroes it), so not from the pool
  const size_t sk_bytes = (!out_fp32 && ds) ? conv_splitk_ws_bytes(L, B, in0.D, in0.H, in0.W) : 0;
  if (sk_bytes > sk_cap) {
    sk_ws = (float*)ds->alloc(sk_bytes);
    sk_cap = sk_ws ? sk_bytes : 0;
  }
  // the conv epilogue folds statistics with power-of-two shuffles; other group widths (e.g. model_channels 192 ->
  // 24 channels per group) take a separate statistics pass over the fp16 output
  const int cpg = (stats && groups > 0) ? L.cout / groups : 0;
  const bool epi_stats = stats && cpg >= 2 && !(cpg & (cpg - 1)) && (L.bn + cpg - 1) / cpg <= 64 && !out_fp32;
  const int rc = conv_plan(P, L, in0.p, in1 ? in1->p : nullptr, B, in0.D, in0.H, in0.W,
                           out_fp32 ? (void*)out_fp32 : (void*)out.p, out_fp32 ? OUT_F32 : OUT_CL16,
                           epi_stats ? stats : nullptr, epi_stats ? groups : 0, act, err, ws,
                           (sk_bytes && sk_ws) ? sk_ws : nullptr);
  if (ws) pool.put(ws);
  if (rc) {
    fail(name + ": " + err);
    ok = false;
    return out;
  }
  Op op;
  op.name = name;
  op.flops = P.flops;
  op.bytes = 0;
  op.launches = (P.tapgemm || P.splitk > 1) ? 2 : 1;
  op.out = out_fp32 ? (void*)out_fp32 : (void*)out.p;
  op.out_bytes = out_fp32 ? (size_t)B * L.cout * oD * oH * oW * 4 : (size_t)B * oD * oH * oW * L.cout * 2;
  op.run = [P](cudaStream_t st) { conv_launch(P, st); };
  ops.push_back(std::move(op));
  if (stats && !epi_stats && !out_fp32) {
    const __half* xp = out.p;
    const long long S = out.S();
    const int C = out.C, Bc = B;
    Op so;
    so.name = name + ".stats";
    so.bytes = (double)B * S * C * 2.0;
    so.run = [=](cudaStream_t st) { launch_gn_stats(xp, Bc, S, C, groups, stats, st); };
    ops.push_back(std::move(so));
  }
  return out;
}

void Builder::gn_apply(const std::string& name, Act& y, const stat_t* stats_in, const GNW& g, int temb_off,
                       const Act* res, int mode, stat_t* stats_out, int G_out) {
  const int Bc = B;
  const long long S = y.S();
  const int C = y.C;
  __half* yp = y.p;
  const __half* rp = res ? res->p : nullptr;
  const float *ga = g.gamma, *be = g.beta;
  const int G = g.G;
  const TembSource* ts = (temb_off >= 0) ? temb_src : nullptr;
  Op op;
  op.name = name;
  op.bytes = (double)Bc * S * C * 2.0 * (res ? 3.0 : 2.0);
  op.out = yp;
  op.out_bytes = (size_t)Bc * S * C * 2;
  op.run = [=](cudaStream_t st) {
    const float* tp = ts ? ts->base + temb_off : nullptr;
    launch_gn_apply(yp, yp, stats_in, ga, be, tp, ts ? ts->sample_stride : 0, rp, Bc, S, C, G, 1e-5f, mode, stats_out,
                    G_out, st, ts ? ts->step_ptr : nullptr, ts ? ts->step_stride : 0);
  };
  ops.push_back(std::move(op));
}

}  // namespace b2v
