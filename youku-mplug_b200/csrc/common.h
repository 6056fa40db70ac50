// Host-side helpers shared by every translation unit of libymp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/ymp.h"

namespace ymp {

int set_error(int code, const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
inline void count_launch(uint64_t n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int num_sms();  // SM count of the current device (cached)

// Programmatic dependent launch (PDL) for the latency-bound decoding step: when on (ymp_set_pdl, thread-local), launch_k
// adds cudaLaunchAttributeProgrammaticStreamSerialization, so the kernel may start while its predecessor in the stream is
// still draining; the kernels launched this way call griddep_wait() (ptx.cuh) before they touch anything the predecessor
// wrote and griddep_launch() as early as possible.  Off: an ordinary launch (the two instructions are then no-ops).
extern thread_local int g_pdl;
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = g_pdl ? 1 : 0;
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);  // errors surface in YMP_LAUNCH_CHECK
}

#define YMP_CHECK_ARG(cond, ...)                                   \
  do {                                                             \
    if (!(cond)) return ymp::set_error(YMP_EINVAL, __VA_ARGS__);   \
  } while (0)

#define YMP_CUDA(expr)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return ymp::set_error(YMP_ECUDA, "%s failed: %s (%s:%d)", #expr,                  \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                \
  } while (0)

#define YMP_LAUNCH_CHECK()                                                              \
  do {                                                                                  \
    cudaError_t _e = cudaPeekAtLastError();                                             \
    if (_e != cudaSuccess) {                                                            \
      cudaGetLastError();                                                               \
      return ymp::set_error(YMP_ECUDA, "kernel launch failed: %s (%s:%d)",              \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                \
    }                                                                                   \
    ymp::count_launch();                                                                \
  } while (0)

// Per-device "done once" flag for cudaFuncSetAttribute (function attributes belong to the device's context: a process
// that drives several GPUs must set them on each).  Usage: static DeviceOnce once; if (once.first()) { ...set... }
struct DeviceOnce {
  bool done[64] = {};
  bool first() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
    if (done[dev]) return false;
    done[dev] = true;
    return true;
  }
};

// Per-device running maximum (dynamic shared-memory opt-in that grows with the problem size).
struct DeviceMax {
  int cur[64] = {};
  bool raise(int v) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
    if (v <= cur[dev]) return false;
    cur[dev] = v;
    return true;
  }
};

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Deterministic reductions.  A kernel whose blocks (or split-K slices) each produce a partial sum of the same outputs
// writes the partials to scratch memory instead of adding them with atomics, whose order depends on scheduling; a
// second kernel then adds the partials in an order fixed by the shapes alone, so a run gives the same bits every time.
// The scratch is stream-ordered (cudaMallocFromPoolAsync / cudaFreeAsync on the caller's stream, from a memory pool
// of the library's own that keeps freed blocks for the next call), which also holds inside CUDA-graph capture, where
// it becomes a graph allocation node.  A Scratch gives its block back when it goes out of scope, so every return path,
// error returns included, frees it; release() frees it early and reports the status.
struct Scratch {
  void* p = nullptr;
  cudaStream_t st = nullptr;
  int alloc(size_t bytes, cudaStream_t stream);
  int release();
  ~Scratch() { if (p) cudaFreeAsync(p, st); }
};
// out[c] += sum over b = 0 .. nblk-1 of part[b * ldp + c], c < C (fp32); with out2, columns c >= C1 go to out2[c - C1]
int reduce_partials(const float* part, int nblk, long ldp, int C, float* out, cudaStream_t st, float* out2 = nullptr,
                    int C1 = 0);

}  // namespace ymp
