// Shared host/device utilities of the linetr_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

namespace ltr {

// ---------------------------------------------------------------- error reporting
extern thread_local std::string g_last_error;
int set_error(int code, const std::string& msg);

#define LTR_CUDA_TRY(expr)                                                              \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return ::ltr::set_error(-2, std::string(#expr) + ": " + cudaGetErrorString(_e));  \
  } while (0)

// ---------------------------------------------------------------- instrumentation
// Kernel classes for launch counting and per-class CUDA-event timing (ltr_profile_*).
enum KernelClass : int {
  KC_SMALL_MLP = 0,
  KC_LINEAR,
  KC_IMG_CONVERT,
  KC_SIG_ATTN,
  KC_FINAL_NORM,
  KC_DIST,
  KC_SEGMEAN,
  KC_ARGMIN,
  KC_MUTUAL,
  KC_TOKEN_FUSED,
  KC_TOKENIZE,
  KC_DESC_TILES,
  KC_MATCH_TC,
  KC_MATCH_TAIL,
  KC_MATCH_EXACT,
  KC_COUNT
};
const char* kernel_class_name(int kc);

extern std::atomic<int64_t> g_launches;

// Threading contract of the C ABI: any number of host threads may call into the library
// concurrently (e.g. one thread per GPU); the process-wide state below is guarded by g_state_mutex.
// Per-class profiling (ltr_profile_*) is a process-wide switch: arm it, run, read it - from one thread.
extern std::mutex g_state_mutex;

struct Profiler {
  std::atomic<bool> on{false};
  struct Rec { int kc; cudaEvent_t a, b; };
  std::vector<Rec> recs;          // guarded by g_state_mutex
  std::vector<cudaEvent_t> pool;  // guarded by g_state_mutex
  cudaEvent_t get();
};
extern Profiler g_prof;

// RAII bracket around one kernel launch: counts it, and when profiling is armed records
// CUDA events on the launching stream (so the measurement sees exactly that kernel).
struct LaunchScope {
  cudaStream_t s;
  cudaEvent_t end = nullptr;
  LaunchScope(int kc, cudaStream_t stream) : s(stream) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (g_prof.on.load(std::memory_order_relaxed)) {
      std::lock_guard<std::mutex> lk(g_state_mutex);
      Profiler::Rec r{kc, g_prof.get(), g_prof.get()};
      cudaEventRecord(r.a, s);
      g_prof.recs.push_back(r);
      end = r.b;
    }
  }
  ~LaunchScope() {
    if (end) cudaEventRecord(end, s);
  }
};

// ---------------------------------------------------------------- programmatic dependent launch (PDL)
// Every kernel of the path is launched with programmaticStreamSerialization: its CTAs may become
// resident as soon as SMs free up at the tail of the previous kernel and run their prologue
// (barrier init, TMEM allocation, constant staging) there; pdl_wait() then blocks until the
// previous grid has completed and flushed, BEFORE anything it produced is read or anything it
// still reads is overwritten.  pdl_launch_dependents() at kernel entry lets the next kernel do
// the same behind this one.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------- debug tracing (clock64 stamps of CTA 0)
__device__ unsigned long long g_dbg_trace[128];
__device__ int g_dbg_on = 0;
#define LTR_DBG_STAMP(slot)                                            \
  do {                                                                 \
    if (g_dbg_on && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) g_dbg_trace[slot] = clock64(); \
  } while (0)
// host side: trace only the n-th chained GEMM launch after arming (ltr_debug_trace_arm(100 + n)); -1 = no selection
inline int& dbg_chain_sel() { static int v = -1; return v; }
inline int& dbg_chain_cnt() { static int v = 0; return v; }

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Lines of image i: [begin, end).  cu == nullptr means a uniform batch of lpi lines/image.
__device__ __forceinline__ void image_range(const int* __restrict__ cu, int lpi, int i, int& b, int& e) {
  if (cu) { b = cu[i]; e = cu[i + 1]; } else { b = i * lpi; e = b + lpi; }
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device AND per kernel: remember the
// (kernel address, device) pairs already configured.  (Kernels sharing a signature share the
// template instantiation below, so the cache must be keyed by the function pointer.)
extern std::vector<std::pair<const void*, int>> g_smem_configured;   // guarded by g_state_mutex
template <typename K>
inline cudaError_t ensure_dynamic_smem(K kernel, int bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const void* key = reinterpret_cast<const void*>(kernel);
  std::lock_guard<std::mutex> lk(g_state_mutex);
  auto& done = g_smem_configured;
  for (auto& d : done)
    if (d.first == key && d.second == dev) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done.emplace_back(key, dev);
  return e;
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

}  // namespace ltr
