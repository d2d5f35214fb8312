// host_common.h — host-side helpers shared by every translation unit of libgsicp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdint>
#include "../../include/gsicp_b200.h"

namespace gsicp {

extern std::atomic<uint64_t> g_launches;
void set_error(const char* fmt, ...);

// Counts every kernel launch of ours; bench.py reports it as gpu_launches.  With GSICP_DEBUG_SYNC=1 in the environment every
// launch is followed by a stream synchronize and the first failing kernel is named on stderr (debugging aid only).
extern int g_debug_sync;
void debug_sync_report(const char* kernel, cudaStream_t stream);
#define GSICP_LAUNCH(kernel, grid, block, smem, stream, ...)          \
  do {                                                                \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);       \
    ::gsicp::g_launches.fetch_add(1, std::memory_order_relaxed);      \
    if (::gsicp::g_debug_sync) ::gsicp::debug_sync_report(#kernel, (stream)); \
  } while (0)

#define GSICP_CUDA(expr)                                                                  \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::gsicp::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return GSICP_ECUDA;                                                                 \
    }                                                                                     \
  } while (0)

// Optional per-kernel device timing (bench.py roofline leg): when enabled, the hot kernels are bracketed by
// CUDA events recorded on the launching stream; totals are resolved when read.  Off by default.
enum ProfKernel {
  kProfPreprocess = 0, kProfDepthSort, kProfEmit, kProfTileSort, kProfRenderFwd, kProfRenderBwd, kProfGaussBwd,
  kProfCovariance, kProfLinearize, kProfError, kProfGridBuild, kProfDist2, kProfLossFwd, kProfLossBwd, kProfExchange, kProfCount
};
extern bool g_prof_on;
void prof_begin(int k, cudaStream_t s);
void prof_end(int k, cudaStream_t s);
struct ProfScope {
  int k; cudaStream_t s;
  ProfScope(int kk, cudaStream_t ss) : k(kk), s(ss) { if (g_prof_on) prof_begin(k, s); }
  ~ProfScope() { if (g_prof_on) prof_end(k, s); }
};

// Grow-only device scratch buffer (library-internal workspace that backward does not need).
struct Scratch {
  void* ptr = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return GSICP_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&ptr, want);
    if (e != cudaSuccess) {
      set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
      return GSICP_ECUDA;
    }
    cap = want;
    return GSICP_OK;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(ptr); }
};

// Mapped pinned words a kernel publishes a small result into (a count, a reduction, the LM result), then a sequence word
// the host spins on.  The host gets the result without a D2H memcpy + cudaStreamSynchronize round trip (two driver calls
// and a thread wake-up per result otherwise).  Not thread-safe: each owner serialises its launches and waits itself.
struct HostMailbox {
  unsigned long long* host = nullptr;  // mapped pinned, zeroed on first use
  unsigned long long* dev = nullptr;   // device alias of host
  unsigned long long seq = 0;          // last sequence number handed out
  int ensure(size_t bytes);
  // Spins until host[word] == s.  The fast path makes no driver call; every ~1M spins the stream is queried so that a
  // failed kernel ("<what> failed: ...") or a finished stream that never published s ("<what> was not published")
  // returns GSICP_ECUDA instead of hanging.
  int wait(size_t word, unsigned long long s, cudaStream_t stream, const char* what) const;
  void release();
};

}  // namespace gsicp
