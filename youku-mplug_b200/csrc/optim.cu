// Optimizer step on flat buffers: global grad-norm (sum of squares) and fused AdamW with the clip
// coefficient read from device memory (no host sync).  Replaces DeepSpeed FusedAdam + clip
// (reference utils.py:490-526, run_pretrain_distributed_gpt3.py:136-137).  HBM-bound.
#include "common.h"
#include "ptx.cuh"

namespace ymp {

// one partial sum per block (part[blockIdx.x]); reduce_partials adds them in block order
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, long n, float* __restrict__ part) {
  float acc = 0.f;
  const long n4 = n >> 2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  for (long i = (n4 << 2) + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    acc += g[i] * g[i];
  acc = warp_sum(acc);
  __shared__ float s[8];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    float v = s[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffu, v, o);
    if (threadIdx.x == 0) part[blockIdx.x] = v;
  }
}

struct AdamParams {
  float* master;
  __nv_bfloat16* param;
  const float* grad;
  float* m;
  float* v;
  const float* sumsq;  // device scalar: sum of squares of the (unscaled) global gradient, or NULL
  const float* hyper;  // optional device array {lr, weight_decay, bc1, bc2}: overrides the by-value fields
  long n;
  float lr, beta1, beta2, eps, wd, grad_scale, max_norm, bc1, bc2;
  int vec;        // all five arrays 16-byte aligned (bf16 param: 8-byte): 4 parameters per thread
  int zero_grad;  // write zeros back to grad (the accumulator of the next step) instead of a separate memset
};

__global__ void __launch_bounds__(256) adamw_kernel(const AdamParams p) {
  float coef = p.grad_scale;
  if (p.sumsq && p.max_norm > 0.f) {
    const float norm = sqrtf(*p.sumsq) * p.grad_scale;
    coef *= fminf(1.f, p.max_norm / (norm + 1e-6f));
  }
  float lr = p.lr, wd = p.wd, bc1 = p.bc1, bc2 = p.bc2;
  if (p.hyper) { lr = p.hyper[0]; wd = p.hyper[1]; bc1 = p.hyper[2]; bc2 = p.hyper[3]; }
  const float step = lr / bc1;
  const float inv_bc2 = rsqrtf(bc2);
  const float decay = 1.f - lr * wd;
  // 4 parameters per thread and iteration: 128-bit loads / stores of grad, m, v, master (fp32) and one 64-bit store of
  // the refreshed bf16 weights; 26 bytes of HBM traffic per parameter (the gradient is zeroed in the same pass)
  const long n4 = p.vec ? (p.n >> 2) : 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 g = reinterpret_cast<const float4*>(p.grad)[i];
    float4 m = reinterpret_cast<float4*>(p.m)[i], v = reinterpret_cast<float4*>(p.v)[i], w = reinterpret_cast<float4*>(p.master)[i];
    float* gp = &g.x; float* mp = &m.x; float* vp = &v.x; float* wp = &w.x;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float ge = gp[e] * coef;
      mp[e] = p.beta1 * mp[e] + (1.f - p.beta1) * ge;
      vp[e] = p.beta2 * vp[e] + (1.f - p.beta2) * ge * ge;
      wp[e] = wp[e] * decay - step * mp[e] / (sqrtf(vp[e]) * inv_bc2 + p.eps);
    }
    reinterpret_cast<float4*>(p.m)[i] = m;
    reinterpret_cast<float4*>(p.v)[i] = v;
    reinterpret_cast<float4*>(p.master)[i] = w;
    reinterpret_cast<uint2*>(p.param)[i] = make_uint2(pack_bf16(w.x, w.y), pack_bf16(w.z, w.w));
    if (p.zero_grad) reinterpret_cast<float4*>(const_cast<float*>(p.grad))[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long i = (n4 << 2) + (long)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += (long)gridDim.x * blockDim.x) {
    const float g = p.grad[i] * coef;
    const float m = p.beta1 * p.m[i] + (1.f - p.beta1) * g;
    const float v = p.beta2 * p.v[i] + (1.f - p.beta2) * g * g;
    float w = p.master[i];
    w = w * decay - step * m / (sqrtf(v) * inv_bc2 + p.eps);
    p.m[i] = m; p.v[i] = v; p.master[i] = w;
    p.param[i] = __float2bfloat16(w);
    if (p.zero_grad) const_cast<float*>(p.grad)[i] = 0.f;
  }
}

}  // namespace ymp

using namespace ymp;

extern "C" int ymp_sumsq(const float* g, int64_t n, float* out, void* stream) {
  YMP_CHECK_ARG(g && out && n > 0, "ymp_sumsq: bad args");
  YMP_CHECK_ARG(aligned16(g), "ymp_sumsq: g must be 16-byte aligned");
  const int blocks = (int)min((long)((n / 4 + 255) / 256) + 1, (long)num_sms() * 8);
  cudaStream_t st = (cudaStream_t)stream;
  Scratch part;
  int rc = part.alloc(sizeof(float) * blocks, st);
  if (rc) return rc;
  sumsq_kernel<<<blocks, 256, 0, st>>>(g, (long)n, (float*)part.p);
  YMP_LAUNCH_CHECK();
  rc = reduce_partials((const float*)part.p, blocks, 1, 1, out, st);
  if (rc) return rc;
  return part.release();
}

extern "C" int ymp_adamw(const ymp_adamw_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->master && a->param && a->grad && a->m && a->v && a->n > 0, "ymp_adamw: bad args");
  YMP_CHECK_ARG(a->step >= 1 || a->hyper, "ymp_adamw: step must be >= 1 (or pass hyper)");
  AdamParams p;
  p.master = a->master; p.param = (__nv_bfloat16*)a->param; p.grad = a->grad; p.m = a->m; p.v = a->v;
  p.sumsq = a->sumsq; p.hyper = a->hyper; p.n = a->n;
  p.lr = a->lr; p.beta1 = a->beta1; p.beta2 = a->beta2; p.eps = a->eps; p.wd = a->weight_decay;
  p.grad_scale = a->grad_scale; p.max_norm = a->max_grad_norm;
  p.bc1 = 1.f - powf(a->beta1, (float)a->step);
  p.bc2 = 1.f - powf(a->beta2, (float)a->step);
  p.vec = aligned16(a->master) && aligned16(a->grad) && aligned16(a->m) && aligned16(a->v) && (reinterpret_cast<uintptr_t>(a->param) & 7) == 0;
  p.zero_grad = a->zero_grad ? 1 : 0;
  const int blocks = (int)min((long)((a->n / 4 + 255) / 256) + 1, (long)num_sms() * 8);
  adamw_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(p);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}
