// capi_common.cu — error reporting, build info and the launch counter of libgsicp_b200.so.
#include <cstring>
#include <mutex>
#include <utility>
#include <vector>
#include "host_common.h"

#include <cstdlib>
namespace gsicp {
std::atomic<uint64_t> g_launches{0};
int g_debug_sync = [] { const char* e = std::getenv("GSICP_DEBUG_SYNC"); return (e && e[0] == '1') ? 1 : 0; }();
void debug_sync_report(const char* kernel, cudaStream_t stream) {
  const cudaError_t e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess) fprintf(stderr, "[gsicp debug] kernel %s failed: %s\n", kernel, cudaGetErrorString(e));
}
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int HostMailbox::ensure(size_t bytes) {
  if (host) return GSICP_OK;
  GSICP_CUDA(cudaHostAlloc((void**)&host, bytes, cudaHostAllocMapped));
  std::memset(host, 0, bytes);
  const cudaError_t e = cudaHostGetDevicePointer((void**)&dev, host, 0);
  if (e != cudaSuccess) {
    release();
    set_error("cudaHostGetDevicePointer failed: %s", cudaGetErrorString(e));
    return GSICP_ECUDA;
  }
  return GSICP_OK;
}

int HostMailbox::wait(size_t word, unsigned long long s, cudaStream_t stream, const char* what) const {
  const volatile unsigned long long* p = host + word;
  long spins = 0;
  while (*p != s) {
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
    if ((++spins & 0xfffff) == 0) {
      const cudaError_t q = cudaStreamQuery(stream);
      if (q != cudaSuccess && q != cudaErrorNotReady) {
        set_error("%s failed: %s", what, cudaGetErrorString(q));
        return GSICP_ECUDA;
      }
      if (q == cudaSuccess && *p != s) {
        set_error("%s was not published", what);
        return GSICP_ECUDA;
      }
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);  // the caller's reads of the published words come after this one
  return GSICP_OK;
}

void HostMailbox::release() {
  if (host) cudaFreeHost(host);
  host = dev = nullptr;
}
}  // namespace gsicp

namespace gsicp {
bool g_prof_on = false;
namespace {
struct ProfSlot {
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
  cudaEvent_t open = nullptr;
  double total_ms = 0.0;
  long count = 0;
};
ProfSlot g_prof[kProfCount];
std::vector<cudaEvent_t> g_event_pool;
std::mutex g_prof_mu;
cudaEvent_t take_event() {
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
void resolve(ProfSlot& p) {
  for (auto& pr : p.pending) {
    cudaEventSynchronize(pr.second);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
      p.total_ms += ms;
      p.count++;
    }
    g_event_pool.push_back(pr.first);
    g_event_pool.push_back(pr.second);
  }
  p.pending.clear();
}
}  // namespace
void prof_begin(int k, cudaStream_t s) {
  std::lock_guard<std::mutex> l(g_prof_mu);
  ProfSlot& p = g_prof[k];
  p.open = take_event();
  cudaEventRecord(p.open, s);
}
void prof_end(int k, cudaStream_t s) {
  std::lock_guard<std::mutex> l(g_prof_mu);
  ProfSlot& p = g_prof[k];
  if (!p.open) return;
  cudaEvent_t e = take_event();
  cudaEventRecord(e, s);
  p.pending.emplace_back(p.open, e);
  p.open = nullptr;
  if (p.pending.size() > 4096) resolve(p);
}
}  // namespace gsicp

static const char* kProfNames[gsicp::kProfCount] = {"preprocess", "tile_scan", "emit_instances", "tile_sort",
                                                    "render_forward", "render_backward", "gaussian_backward",
                                                    "gicp_covariance", "gicp_linearize", "gicp_error", "grid_build",
                                                    "dist2", "loss_forward", "loss_backward", "moment_exchange"};

extern "C" void gsicp_prof_enable(int on) { gsicp::g_prof_on = on != 0; }
extern "C" void gsicp_prof_reset(void) {
  std::lock_guard<std::mutex> l(gsicp::g_prof_mu);
  for (auto& p : gsicp::g_prof) {
    gsicp::resolve(p);
    p.total_ms = 0.0;
    p.count = 0;
  }
}
extern "C" int gsicp_prof_count(void) { return gsicp::kProfCount; }
extern "C" const char* gsicp_prof_name(int k) { return (k >= 0 && k < gsicp::kProfCount) ? kProfNames[k] : ""; }
extern "C" int gsicp_prof_read(int k, double* total_ms, long* count) {
  if (k < 0 || k >= gsicp::kProfCount) return GSICP_EINVAL;
  std::lock_guard<std::mutex> l(gsicp::g_prof_mu);
  gsicp::resolve(gsicp::g_prof[k]);
  if (total_ms) *total_ms = gsicp::g_prof[k].total_ms;
  if (count) *count = gsicp::g_prof[k].count;
  return GSICP_OK;
}

extern "C" const char* gsicp_last_error(void) { return gsicp::g_err; }

#define GSICP_STR2(x) #x
#define GSICP_STR(x) GSICP_STR2(x)
extern "C" const char* gsicp_build_info(void) {
  return "libgsicp_b200 sm_100a (CUDA " GSICP_STR(CUDART_VERSION) ", built " __DATE__ ")";
}

extern "C" uint64_t gsicp_launch_count(void) { return gsicp::g_launches.load(); }
