// Library-wide plumbing: thread-local error message, version, device queries.
#include <stdarg.h>
#include <stdio.h>

#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"

namespace dss {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* last_error() { return g_err; }

int device_sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return -1;
  if (cached[dev] > 0) return cached[dev];
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  cached[dev] = n;
  return n;
}

cudaError_t allow_dynamic_smem(const void* kernel, int bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, int> allowed;   // (kernel, device) -> bytes
  std::lock_guard<std::mutex> lk(mu);
  int& have = allowed[{kernel, dev}];
  if (bytes <= have) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) have = bytes;
  return e;
}

// ---- launch counter + optional per-class event timing
static std::atomic<long long> g_launches{0};
static bool g_prof_on = false;
struct ProfRec { cudaEvent_t a, b; int cls; };
static std::vector<ProfRec> g_recs;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_pool;
static std::mutex g_prof_mu;

LaunchScope::LaunchScope(cudaStream_t stream, int kernel_class) : st(stream), slot(-1) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  ProfRec r;
  if (!g_pool.empty()) {
    r.a = g_pool.back().first; r.b = g_pool.back().second; g_pool.pop_back();
  } else {
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  }
  r.cls = kernel_class;
  cudaEventRecord(r.a, st);
  g_recs.push_back(r);
  slot = (int)g_recs.size() - 1;
}
LaunchScope::~LaunchScope() {
  if (slot < 0) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  cudaEventRecord(g_recs[slot].b, st);
}

static const char* kClassNames[KC_COUNT] = {"im2col", "gemm_patch", "cls_row", "layernorm", "gemm_qkv", "attention",
                                            "gemm_proj", "gemm_fc1", "gemm_fc2", "gemm_kproj", "gemm_other",
                                            "rownorm", "affinity", "knn", "eigsh", "misc"};

}  // namespace dss

extern "C" long long dss_kernel_launch_count(void) { return dss::g_launches.load(); }

extern "C" void dss_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(dss::g_prof_mu);
  for (auto& r : dss::g_recs) dss::g_pool.push_back({r.a, r.b});
  dss::g_recs.clear();
  dss::g_prof_on = on != 0;
}

extern "C" int dss_profile_read(dss_profile_entry* out, int max_entries) {
  using namespace dss;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double ms[KC_COUNT] = {0};
  long long n[KC_COUNT] = {0};
  for (auto& r : g_recs) {
    if (cudaEventSynchronize(r.b) != cudaSuccess) { set_error("profile_read: event sync failed"); return DSS_ERR_CUDA; }
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) != cudaSuccess) { set_error("profile_read: elapsed failed"); return DSS_ERR_CUDA; }
    ms[r.cls] += t; n[r.cls] += 1;
  }
  int k = 0;
  for (int c = 0; c < KC_COUNT && k < max_entries; ++c) {
    if (!n[c]) continue;
    out[k].name = kClassNames[c]; out[k].launches = n[c]; out[k].total_ms = ms[c];
    ++k;
  }
  return k;
}

extern "C" const char* dss_last_error(void) { return dss::last_error(); }
extern "C" int dss_version(void) { return 1; }
extern "C" int dss_device_sm_count(void) {
  const int n = dss::device_sm_count();
  if (n < 0) dss::set_error("no CUDA device available");
  return n;
}
