#include "common.h"

#include <string.h>

namespace ymp {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
thread_local int g_pdl = 0;

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

int Scratch::alloc(size_t bytes, cudaStream_t stream) {
  // one pool per device, owned by the library (the device's default pool is left as it is); it keeps freed blocks
  // across synchronisations, so the reductions of every step reuse the same memory
  static cudaMemPool_t pools[64] = {};
  int dev = 0;
  YMP_CUDA(cudaGetDevice(&dev));
  YMP_CHECK_ARG(dev >= 0 && dev < 64, "scratch: device index %d out of range", dev);
  if (!pools[dev]) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool;
    YMP_CUDA(cudaMemPoolCreate(&pool, &props));
    uint64_t keep = UINT64_MAX;
    YMP_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    pools[dev] = pool;
  }
  st = stream;
  YMP_CUDA(cudaMallocFromPoolAsync(&p, bytes, pools[dev], stream));
  return YMP_OK;
}

int Scratch::release() {
  void* q = p;
  p = nullptr;
  YMP_CUDA(cudaFreeAsync(q, st));
  return YMP_OK;
}

// lane = column, warp w adds partials w, w + 32, w + 64, ... in turn, then warp 0 adds the 32 warp sums in warp order
__global__ void __launch_bounds__(1024) reduce_partials_kernel(const float* __restrict__ part, int nblk, long ldp, int C,
                                                              float* __restrict__ out, float* __restrict__ out2, int C1) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < C) {
#pragma unroll 4
    for (int b = warp; b < nblk; b += 32) s += part[(size_t)b * ldp + c];
  }
  __shared__ float red[32][33];
  red[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && c < C) {
    float t = red[0][lane];
#pragma unroll
    for (int w = 1; w < 32; ++w) t += red[w][lane];
    if (out2 && c >= C1) out2[c - C1] += t;
    else out[c] += t;
  }
}

int reduce_partials(const float* part, int nblk, long ldp, int C, float* out, cudaStream_t st, float* out2, int C1) {
  reduce_partials_kernel<<<(C + 31) / 32, 1024, 0, st>>>(part, nblk, ldp, C, out, out2, C1);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

}  // namespace ymp

extern "C" {
const char* ymp_last_error(void) { return ymp::g_err; }
int ymp_abi_version(void) { return 3; }
uint64_t ymp_launch_count(void) { return ymp::g_launches.load(std::memory_order_relaxed); }
int ymp_set_pdl(int on) { const int prev = ymp::g_pdl; ymp::g_pdl = on ? 1 : 0; return prev; }
}
