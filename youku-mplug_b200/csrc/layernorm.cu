// LayerNorm forward / backward: one warp per row, 128-bit coalesced loads, fp32 statistics,
// warp-shuffle reductions.  HBM-bound (reads x once, writes y once).
#include "common.h"
#include "philox.cuh"
#include "ptx.cuh"

namespace ymp {

constexpr int LN_WARPS = 8;

struct LnParams {
  const void* x;  // bf16 or fp32 (XF32)
  const __nv_bfloat16* gamma;
  const __nv_bfloat16* beta;
  void* y;        // bf16 or fp32 (y_f32)
  int y_f32;
  float* mean;
  float* rstd;
  const int32_t* in_rows;
  int rows, D, ldx, ldy;
  float eps;
};

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  f[0] = bf16_lo(u.x); f[1] = bf16_hi(u.x); f[2] = bf16_lo(u.y); f[3] = bf16_hi(u.y);
  f[4] = bf16_lo(u.z); f[5] = bf16_hi(u.z); f[6] = bf16_lo(u.w); f[7] = bf16_hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16(f[0], f[1]); u.y = pack_bf16(f[2], f[3]);
  u.z = pack_bf16(f[4], f[5]); u.w = pack_bf16(f[6], f[7]);
  return u;
}

// 8 consecutive elements of row `row` (vector index vi) as floats, from bf16 or fp32 storage
template <bool XF32>
__device__ __forceinline__ void load8(const void* base, size_t row, int ld, int vi, float (&f)[8]) {
  if (XF32) {
    const float4* p4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + row * ld) + 2 * vi;
    const float4 a = __ldg(p4), b = __ldg(p4 + 1);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  } else {
    unpack8(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + row * ld) + vi), f);
  }
}

// VPL = 8-element vectors per lane (D <= VPL*256)
template <int VPL, bool XF32>
__global__ void __launch_bounds__(LN_WARPS * 32) ln_fwd_kernel(const LnParams p) {
  griddep_launch();   // (programmatic dependent launch in the decoding step; no-ops for an ordinary launch)
  griddep_wait();
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nvec = p.D >> 3;
  for (int row = blockIdx.x * LN_WARPS + warp; row < p.rows; row += gridDim.x * LN_WARPS) {
    const int irow = p.in_rows ? p.in_rows[row] : row;
    if (irow < 0) {  // padding slot: emit a zero row (the caller overwrites it), no statistics
      uint4* yz = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.y) + (size_t)row * p.ldy);
      for (int vi = lane; vi < nvec; vi += 32) yz[vi] = make_uint4(0, 0, 0, 0);  // (bf16 outputs only)
      if (lane == 0) {
        if (p.mean) p.mean[row] = 0.f;
        if (p.rstd) p.rstd[row] = 0.f;
      }
      continue;
    }
    float v[VPL][8];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int vi = j * 32 + lane;
      if (vi < nvec) {
        load8<XF32>(p.x, (size_t)irow, p.ldx, vi, v[j]);
#pragma unroll
        for (int e = 0; e < 8; ++e) s += v[j][e];
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[j][e] = 0.f;
      }
    }
    const float mu = warp_sum(s) / (float)p.D;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      if (j * 32 + lane < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) { float d = v[j][e] - mu; q += d * d; }
      }
    }
    const float rs = rsqrtf(warp_sum(q) / (float)p.D + p.eps);
    if (lane == 0) {
      if (p.mean) p.mean[row] = mu;
      if (p.rstd) p.rstd[row] = rs;
    }
    const uint4* g4 = reinterpret_cast<const uint4*>(p.gamma);
    const uint4* b4 = reinterpret_cast<const uint4*>(p.beta);
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int vi = j * 32 + lane;
      if (vi < nvec) {
        float g[8], b[8], o[8];
        unpack8(__ldg(g4 + vi), g);
        unpack8(__ldg(b4 + vi), b);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = fmaf((v[j][e] - mu) * rs, g[e], b[e]);
        if (p.y_f32) {
          float4* yr = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.y) + (size_t)row * p.ldy) + 2 * vi;
          yr[0] = make_float4(o[0], o[1], o[2], o[3]);
          yr[1] = make_float4(o[4], o[5], o[6], o[7]);
        } else {
          reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.y) + (size_t)row * p.ldy)[vi] = pack8(o);
        }
      }
    }
  }
}

struct LnBwdParams {
  const __nv_bfloat16* dy;
  const void* x;  // bf16 or fp32 (XF32)
  const __nv_bfloat16* gamma;
  const float* mean;
  const float* rstd;
  const __nv_bfloat16* add;  // optional gradient of the residual branch, added to dx
  __nv_bfloat16* dx;
  float* dgamma;  // fp32 [D], accumulated (caller zeroes); NULL = frozen
  float* dbeta;
  float* wpart;   // with dgamma: per-block partials, row b = [dgamma part (D) | dbeta part (D)], added by reduce_partials
  const int32_t* in_rows;
  int rows, D, ldx, lddy, ldadd;
  __nv_bfloat16* dx_drop;  // optional: dx with the dropout mask of the site that produced x applied
  DropSpec drop;
};

template <int VPL, bool WGRAD, bool XF32, bool DROP>
__global__ void __launch_bounds__(LN_WARPS * 32, WGRAD ? (VPL <= 4 ? 3 : 1) : (DROP ? 2 : 4)) ln_bwd_kernel(const LnBwdParams p) {
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nvec = p.D >> 3;
  float dg[WGRAD ? VPL : 1][8], db[WGRAD ? VPL : 1][8];
  if (WGRAD) {
#pragma unroll
    for (int j = 0; j < VPL; ++j)
#pragma unroll
      for (int e = 0; e < 8; ++e) { dg[j][e] = 0.f; db[j][e] = 0.f; }
  }
  const uint4* g4 = reinterpret_cast<const uint4*>(p.gamma);
  DropState ds = {};
  if (DROP) ds = drop_state(p.drop);
  for (int row = blockIdx.x * LN_WARPS + warp; row < p.rows; row += gridDim.x * LN_WARPS) {
    const int irow = p.in_rows ? p.in_rows[row] : row;
    if (irow < 0) continue;  // padding slot of the forward: no input row behind it
    const uint4* dyr = reinterpret_cast<const uint4*>(p.dy + (size_t)row * p.lddy);
    const float mu = p.mean[row], rs = p.rstd[row];
    // Two passes over the row keep the register footprint small (high occupancy for an HBM-bound
    // kernel); the second pass re-reads the 3-8 KB row from L1/L2, not from HBM.
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int vi = j * 32 + lane;
      if (vi < nvec) {
        float xv[8], dyv[8], g[8];
        load8<XF32>(p.x, (size_t)irow, p.ldx, vi, xv);
        unpack8(__ldg(dyr + vi), dyv);
        unpack8(__ldg(g4 + vi), g);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float xh = (xv[e] - mu) * rs, gy = dyv[e] * g[e];
          s1 += gy;
          s2 += gy * xh;
          if (WGRAD) { dg[j][e] += dyv[e] * xh; db[j][e] += dyv[e]; }
        }
      }
    }
    s1 = warp_sum(s1) / (float)p.D;
    s2 = warp_sum(s2) / (float)p.D;
    uint4* dxr = reinterpret_cast<uint4*>(p.dx + (size_t)irow * p.ldx);
    const uint4* ar = p.add ? reinterpret_cast<const uint4*>(p.add + (size_t)irow * p.ldadd) : nullptr;
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int vi = j * 32 + lane;
      if (vi < nvec) {
        float xv[8], dyv[8], g[8], o[8];
        load8<XF32>(p.x, (size_t)irow, p.ldx, vi, xv);
        unpack8(__ldg(dyr + vi), dyv);
        unpack8(__ldg(g4 + vi), g);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = rs * (dyv[e] * g[e] - s1 - (xv[e] - mu) * rs * s2);
        if (ar) {
          float a[8];
          unpack8(__ldg(ar + vi), a);
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] += a[e];
        }
        dxr[vi] = pack8(o);
        if (DROP) {  // gradient w.r.t. the pre-dropout branch output: same mask bits as the forward epilogue
          drop4(ds, (uint32_t)irow, (uint32_t)(vi * 8), o[0], o[1], o[2], o[3]);
          drop4(ds, (uint32_t)irow, (uint32_t)(vi * 8 + 4), o[4], o[5], o[6], o[7]);
          reinterpret_cast<uint4*>(p.dx_drop + (size_t)irow * p.ldx)[vi] = pack8(o);
        }
      }
    }
  }
  if (WGRAD) {
    // block-level reduce across the 8 warps, then this block's partials go to its row of p.wpart
    __shared__ float red[LN_WARPS][32 * 8 + 1];
    for (int j = 0; j < VPL; ++j) {
      for (int pass = 0; pass < 2; ++pass) {
        __syncthreads();
#pragma unroll
        for (int e = 0; e < 8; ++e) red[warp][lane * 8 + e] = pass == 0 ? dg[j][e] : db[j][e];
        __syncthreads();
        // 256 columns per (j, pass): thread t < 64 owns 4 consecutive columns -> one 16-byte reduction
        if (threadIdx.x < 64) {
          float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int w = 0; w < LN_WARPS; ++w)
#pragma unroll
            for (int e = 0; e < 4; ++e) s[e] += red[w][threadIdx.x * 4 + e];
          const int col = j * 256 + threadIdx.x * 4;
          float* dst = p.wpart + (size_t)blockIdx.x * 2 * p.D + pass * p.D + col;
          if (col + 3 < p.D) {
            *reinterpret_cast<float4*>(dst) = make_float4(s[0], s[1], s[2], s[3]);
          } else {
            for (int e = 0; e < 4; ++e)
              if (col + e < p.D) dst[e] = s[e];
          }
        }
      }
    }
  }
}

}  // namespace ymp

extern "C" int ymp_layernorm_fwd(const ymp_layernorm_args* a, void* stream) {
  using namespace ymp;
  YMP_CHECK_ARG(a && a->x && a->y && a->gamma && a->beta, "ymp_layernorm_fwd: null pointer");
  YMP_CHECK_ARG(a->rows > 0 && a->D > 0 && a->D % 8 == 0 && a->D <= 4096, "ymp_layernorm_fwd: D=%d must be a multiple of 8 and <= 4096", a->D);
  YMP_CHECK_ARG(a->ldx % 8 == 0 && a->ldy % 8 == 0 && a->ldx >= a->D && a->ldy >= a->D, "ymp_layernorm_fwd: bad ld");
  YMP_CHECK_ARG(aligned16(a->x) && aligned16(a->y) && aligned16(a->gamma) && aligned16(a->beta), "ymp_layernorm_fwd: 16-byte alignment required");
  YMP_CHECK_ARG(!(a->in_rows && a->y_dtype == YMP_DT_F32), "ymp_layernorm_fwd: row gather supports bf16 outputs only");
  LnParams p;
  p.x = a->x; p.gamma = (const __nv_bfloat16*)a->gamma; p.beta = (const __nv_bfloat16*)a->beta;
  p.y = a->y; p.y_f32 = (a->y_dtype == YMP_DT_F32); p.mean = a->mean; p.rstd = a->rstd; p.in_rows = a->in_rows;
  p.rows = a->rows; p.D = a->D; p.ldx = a->ldx; p.ldy = a->ldy; p.eps = a->eps;
  const int blocks = min((a->rows + LN_WARPS - 1) / LN_WARPS, num_sms() * 8);
  cudaStream_t st = (cudaStream_t)stream;
  const int vpl = (a->D / 8 + 31) / 32;
  const int thr = LN_WARPS * 32;
  if (a->x_dtype == YMP_DT_F32) {
    if (vpl <= 3) launch_k(ln_fwd_kernel<3, true>, dim3(blocks), dim3(thr), 0, st, p);
    else if (vpl <= 8) launch_k(ln_fwd_kernel<8, true>, dim3(blocks), dim3(thr), 0, st, p);
    else launch_k(ln_fwd_kernel<16, true>, dim3(blocks), dim3(thr), 0, st, p);
  } else {
    if (vpl <= 3) launch_k(ln_fwd_kernel<3, false>, dim3(blocks), dim3(thr), 0, st, p);
    else if (vpl <= 8) launch_k(ln_fwd_kernel<8, false>, dim3(blocks), dim3(thr), 0, st, p);
    else launch_k(ln_fwd_kernel<16, false>, dim3(blocks), dim3(thr), 0, st, p);
  }
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_layernorm_bwd(const ymp_layernorm_bwd_args* a, void* stream) {
  using namespace ymp;
  YMP_CHECK_ARG(a && a->dy && a->x && a->gamma && a->mean && a->rstd && a->dx, "ymp_layernorm_bwd: null pointer");
  YMP_CHECK_ARG(a->rows > 0 && a->D > 0 && a->D % 8 == 0 && a->D <= 4096, "ymp_layernorm_bwd: bad D=%d", a->D);
  YMP_CHECK_ARG((a->dgamma == nullptr) == (a->dbeta == nullptr), "ymp_layernorm_bwd: dgamma/dbeta must both be set or both NULL");
  YMP_CHECK_ARG(!a->dgamma || (aligned16(a->dgamma) && aligned16(a->dbeta)), "ymp_layernorm_bwd: dgamma/dbeta must be 16-byte aligned");
  YMP_CHECK_ARG(a->ldx % 8 == 0 && a->lddy % 8 == 0 && (!a->add || a->ldadd % 8 == 0), "ymp_layernorm_bwd: bad ld");
  LnBwdParams p;
  p.dy = (const __nv_bfloat16*)a->dy; p.x = a->x; p.gamma = (const __nv_bfloat16*)a->gamma;
  p.mean = a->mean; p.rstd = a->rstd; p.add = (const __nv_bfloat16*)a->add; p.dx = (__nv_bfloat16*)a->dx;
  p.dgamma = a->dgamma; p.dbeta = a->dbeta; p.in_rows = a->in_rows;
  p.rows = a->rows; p.D = a->D; p.ldx = a->ldx; p.lddy = a->lddy; p.ldadd = a->ldadd;
  const bool dropped = a->dx_drop && a->drop.rng && a->drop.p > 0.f;
  YMP_CHECK_ARG(!a->dx_drop || (dropped && a->drop.p < 1.f && aligned16(a->dx_drop)), "ymp_layernorm_bwd: dx_drop needs a dropout spec with 0 < p < 1");
  p.dx_drop = dropped ? (__nv_bfloat16*)a->dx_drop : nullptr;
  p.drop.rng = a->drop.rng; p.drop.site = a->drop.site; p.drop.p = a->drop.p;
  cudaStream_t st = (cudaStream_t)stream;
  const int vpl = (a->D / 8 + 31) / 32;
  const bool wg = a->dgamma != nullptr;
  // resident blocks per SM: 3 with weight grads (80 registers at D <= 1024), 4 without; the grid is a whole
  // number of such waves so that the row loop stays balanced
  const int cap = wg ? num_sms() * (a->D <= 1024 ? 3 : 2) : num_sms() * 8;
  const int blocks = min((a->rows + LN_WARPS - 1) / LN_WARPS, cap);
  const int thr = LN_WARPS * 32;
  const bool xf = (a->x_dtype == YMP_DT_F32);
#define YMP_LN_BWD(V, W, X) do { if (p.dx_drop) ln_bwd_kernel<V, W, X, true><<<blocks, thr, 0, st>>>(p); else ln_bwd_kernel<V, W, X, false><<<blocks, thr, 0, st>>>(p); } while (0)
#define YMP_LN_BWD_V(W, X) do { if (vpl <= 3) YMP_LN_BWD(3, W, X); else if (vpl <= 8) YMP_LN_BWD(8, W, X); else YMP_LN_BWD(16, W, X); } while (0)
  Scratch part;
  p.wpart = nullptr;
  if (wg) {
    const int rc = part.alloc(sizeof(float) * 2 * (size_t)a->D * blocks, st);
    if (rc) return rc;
    p.wpart = (float*)part.p;
  }
  if (wg) { if (xf) YMP_LN_BWD_V(true, true); else YMP_LN_BWD_V(true, false); }
  else { if (xf) YMP_LN_BWD_V(false, true); else YMP_LN_BWD_V(false, false); }
#undef YMP_LN_BWD_V
#undef YMP_LN_BWD
  YMP_LAUNCH_CHECK();
  if (!wg) return YMP_OK;
  const int rc = reduce_partials(p.wpart, blocks, 2L * a->D, 2 * a->D, a->dgamma, st, a->dbeta, a->D);
  if (rc) return rc;
  return part.release();
}
