// Skinny GEMM for single-token decoding (SURVEY.md 8f N2): y[M, N] = epilogue(x[M, K] . w[N, K]^T) with M <= 8 rows
// (beam width / decode batch).  Replaces the GPT-3 layer's linears at the KV-cache step of
// models/modeling_distributed_gpt3.py:868-938,580-595,1348-1350.  With a handful of rows the work is one pass over
// the weight matrix: HBM-bound.  A 128-row tcgen05 tile would occupy N/128 CTAs (16 for N = 2048) and stream the
// weights at a fraction of the memory bandwidth; a CUDA-core dot product needs ~2.5 issue slots per weight byte-pair
// (bf16 -> fp32 converts + FMAs for every row) and is issue-bound at a quarter of the bandwidth.  So:
//   * a warp owns 8 output columns and one K slice and feeds mma.sync.m16n8k16 (bf16, fp32 accumulate) STRAIGHT FROM
//     GLOBAL MEMORY: lane (g, t) loads 16 bytes (8 consecutive k) of weight row n0+g and of activation row g.  The
//     tensor-core fragment wants k = {2t, 2t+1, 2t+8, 2t+9} per lane - but a dot product does not care in which order
//     k is summed as long as both operands use the same order, so the 8 consecutive elements are simply declared to be
//     those positions of two k-steps (a k permutation inside each 32-element block).  No shared memory, no converts:
//     two loads and two MMAs per 16 weight bytes per lane.  x is the A operand (rows >= M are zero registers);
//   * the 8 warps of a CTA are `ksplit` K-slices x (8 / ksplit) column tiles; every lane keeps UNROLL k-blocks
//     (UNROLL x 16 bytes of weights) in flight, ~8 CTAs resident per SM;
//   * partial sums meet in shared memory; lane (g, t) of the slice-0 warp owns (row g, columns n0+2t, n0+2t+1) and applies
//       v = acc + bias[n] ; v = gelu(v) (optional) ; v += residual[m, n] (bf16 or fp32) ; store bf16 or fp32
//     (+ an optional second bf16 copy at a device-side row offset: the KV-cache row of the new token).
// 9..64 rows (batched beam search) run on gemm_skinny_wide_kernel below: the same layout with up to four m16 row tiles.
// Algorithmic bytes per call: N*K*2 (weights) + M*(K + N)*2..4.
#include "common.h"
#include "ptx.cuh"

namespace ymp {

constexpr int SK_MAXM = 8, SK_TILE_N = 8, SK_WARPS = 8;

struct SkinnyParams {
  const __nv_bfloat16* x;
  const __nv_bfloat16* w;
  const __nv_bfloat16* bias;
  const void* residual;
  void* y;
  __nv_bfloat16* y2;
  const long long* y2_off;
  long long ldy2, y2_stride;
  int M, N, K, ldx, ldw, ldr, ldy;
  int act, res_f32, out_f32, ksplit;
  const __nv_bfloat16* ln_gamma;
  const __nv_bfloat16* ln_beta;
  __nv_bfloat16* ln_out;
  unsigned int* ln_counter;
  int ld_ln;
  float ln_eps;
};

// LayerNorm of all M rows of the finished fp32 result by the whole (last) CTA, read back from L2 (ld.cg: other CTAs
// wrote it).  Three passes (sum, squared deviations, normalise), each with every load of every row in flight at once -
// three L2 round trips on the critical path, not one per 8-element chunk.  Same formula as ln_fwd_kernel (layernorm.cu):
// mean = sum / N, rstd = rsqrt(sum((x - mean)^2) / N + eps), y = ((x - mean) * rstd) * gamma + beta.
template <int PASS>
__device__ __forceinline__ void skinny_ln_pass(const SkinnyParams& p, const float* mu, const float* rs, float* red) {
  const int nvec = p.N >> 3, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float acc[SK_MAXM];
#pragma unroll
  for (int m = 0; m < SK_MAXM; ++m) acc[m] = 0.f;
  for (int vi = threadIdx.x; vi < nvec; vi += SK_WARPS * 32) {
    float4 a[SK_MAXM], b[SK_MAXM];
#pragma unroll
    for (int m = 0; m < SK_MAXM; ++m) {
      if (m < p.M) {
        const float4* yr = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.y) + (size_t)m * p.ldy) + 2 * vi;
        a[m] = __ldcg(yr); b[m] = __ldcg(yr + 1);
      }
    }
    uint4 gv, bv;
    if (PASS == 2) { gv = __ldg(reinterpret_cast<const uint4*>(p.ln_gamma) + vi); bv = __ldg(reinterpret_cast<const uint4*>(p.ln_beta) + vi); }
#pragma unroll
    for (int m = 0; m < SK_MAXM; ++m) {
      if (m < p.M) {
        const float v[8] = {a[m].x, a[m].y, a[m].z, a[m].w, b[m].x, b[m].y, b[m].z, b[m].w};
        if (PASS == 0) {
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[m] += v[e];
        } else if (PASS == 1) {
#pragma unroll
          for (int e = 0; e < 8; ++e) { const float d = v[e] - mu[m]; acc[m] += d * d; }
        } else {
          const uint32_t* gp = &gv.x; const uint32_t* bp = &bv.x;
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e)
            o[e] = pack_bf16(fmaf((v[2 * e] - mu[m]) * rs[m], bf16_lo(gp[e]), bf16_lo(bp[e])),
                             fmaf((v[2 * e + 1] - mu[m]) * rs[m], bf16_hi(gp[e]), bf16_hi(bp[e])));
          reinterpret_cast<uint4*>(p.ln_out + (size_t)m * p.ld_ln)[vi] = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
    }
  }
  if (PASS < 2) {
#pragma unroll
    for (int m = 0; m < SK_MAXM; ++m) {
      const float t = warp_sum(acc[m]);
      if (lane == 0) red[warp * SK_MAXM + m] = t;
    }
    __syncthreads();
  }
}
__device__ __forceinline__ void skinny_ln_rows(const SkinnyParams& p, float* red /* [SK_WARPS * SK_MAXM] */) {
  float mu[SK_MAXM], rs[SK_MAXM];
  skinny_ln_pass<0>(p, mu, rs, red);
#pragma unroll
  for (int m = 0; m < SK_MAXM; ++m) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < SK_WARPS; ++w) t += red[w * SK_MAXM + m];
    mu[m] = t / (float)p.N;
  }
  __syncthreads();
  skinny_ln_pass<1>(p, mu, rs, red);
#pragma unroll
  for (int m = 0; m < SK_MAXM; ++m) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < SK_WARPS; ++w) t += red[w * SK_MAXM + m];
    rs[m] = rsqrtf(t / (float)p.N + p.ln_eps);
  }
  skinny_ln_pass<2>(p, mu, rs, red);
}

__device__ __forceinline__ void mma16816_bf16(float (&c)[4], uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  // rows 8..15 of the A operand (a1, a3) are zero: only M <= 8 activation rows exist
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%5}, {%7,%8}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(0u), "r"(a2), "r"(b0), "r"(b1));
}

template <int SK_UNROLL, bool LN>
__global__ void __launch_bounds__(SK_WARPS * 32, (LN ? 2 : 1)) gemm_skinny_kernel(const SkinnyParams p) {
  __shared__ float part[SK_WARPS][64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int ks = p.ksplit, kpart = warp % ks, tile = blockIdx.x * (SK_WARPS / ks) + warp / ks;
  const int n0 = tile * SK_TILE_N;
  const bool live = n0 < p.N;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  griddep_launch();
  if (live) {
    // 16-byte chunks of the K dimension: chunk c = elements [8c, 8c+8); a k-block is 4 chunks (one per t)
    const int nchunk = p.K >> 3, nblk = (nchunk + 3) >> 2;
    const int b_lo = (int)((long)nblk * kpart / ks), b_hi = (int)((long)nblk * (kpart + 1) / ks);
    const uint4* wr = reinterpret_cast<const uint4*>(p.w + (size_t)min(n0 + g, p.N - 1) * p.ldw);
    const uint4* xr = reinterpret_cast<const uint4*>(p.x + (size_t)min(g, p.M - 1) * p.ldx);
    const bool xrow = g < p.M;
    // two register batches of SK_UNROLL k-blocks: the next batch is requested before the current one is consumed, so a
    // warp always has SK_UNROLL..2*SK_UNROLL x 16 bytes of weights in flight
    uint4 wv[SK_UNROLL], xv[SK_UNROLL];
    auto fetch_w = [&](int b, uint4 (&wd)[SK_UNROLL]) {
#pragma unroll
      for (int u = 0; u < SK_UNROLL; ++u) {
        const int c = (b + u) * 4 + t;
        wd[u] = ((b + u) < b_hi && c < nchunk) ? ld_nc_v4(wr + c) : make_uint4(0, 0, 0, 0);
      }
    };
    auto fetch_x = [&](int b, uint4 (&xd)[SK_UNROLL]) {
#pragma unroll
      for (int u = 0; u < SK_UNROLL; ++u) {
        const int c = (b + u) * 4 + t;
        xd[u] = ((b + u) < b_hi && c < nchunk && xrow) ? __ldg(xr + c) : make_uint4(0, 0, 0, 0);
      }
    };
    // the weights do not depend on the previous kernel of the stream: their first batch is already in flight while that
    // kernel drains (programmatic dependent launch); the activations are read only after it has completed
    fetch_w(b_lo, wv);
    griddep_wait();
    fetch_x(b_lo, xv);
    for (int b = b_lo; b < b_hi; b += SK_UNROLL) {
      uint4 wn[SK_UNROLL], xn[SK_UNROLL];
      fetch_w(b + SK_UNROLL, wn);     // (all-zero past the end of the slice)
      fetch_x(b + SK_UNROLL, xn);
#pragma unroll
      for (int u = 0; u < SK_UNROLL; ++u) {
        mma16816_bf16(acc, xv[u].x, xv[u].y, wv[u].x, wv[u].y);
        mma16816_bf16(acc, xv[u].z, xv[u].w, wv[u].z, wv[u].w);
      }
#pragma unroll
      for (int u = 0; u < SK_UNROLL; ++u) { wv[u] = wn[u]; xv[u] = xn[u]; }
    }
  } else {
    griddep_wait();
  }
  // acc[0], acc[1] = (row g, columns n0 + 2t, n0 + 2t + 1) summed over this warp's K slice
  if (ks > 1) {
    part[warp][2 * lane] = acc[0];
    part[warp][2 * lane + 1] = acc[1];
    __syncthreads();
    if (kpart == 0)
      for (int j = 1; j < ks; ++j) { acc[0] += part[warp + j][2 * lane]; acc[1] += part[warp + j][2 * lane + 1]; }
  }
  if (live && kpart == 0 && g < p.M) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int n = n0 + 2 * t + e;
      if (n >= p.N) continue;
      float v = acc[e];
      if (p.bias) v += __bfloat162float(p.bias[n]);
      if (p.act == YMP_ACT_GELU_TANH) v = gelu_tanh(v);
      else if (p.act == YMP_ACT_GELU_ERF) v = gelu_erf(v);
      if (p.residual)
        v += p.res_f32 ? reinterpret_cast<const float*>(p.residual)[(size_t)g * p.ldr + n]
                       : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.residual)[(size_t)g * p.ldr + n]);
      if (p.out_f32) reinterpret_cast<float*>(p.y)[(size_t)g * p.ldy + n] = v;
      else reinterpret_cast<__nv_bfloat16*>(p.y)[(size_t)g * p.ldy + n] = __float2bfloat16(v);
      if (p.y2) p.y2[(long long)g * p.ldy2 + *p.y2_off * p.y2_stride + n] = __float2bfloat16(v);
    }
    if (LN) __threadfence();   // this thread's rows are visible device-wide before its CTA takes a ticket
  }
  if constexpr (LN) {
    // fused LayerNorm: the CTA that takes the last ticket sees every other CTA's rows (writers' fences + atomic) and
    // normalises them
    __shared__ unsigned int ticket;
    __syncthreads();
    if (threadIdx.x == 0) ticket = atomicAdd(p.ln_counter, 1u);
    __syncthreads();
    if (ticket == gridDim.x - 1) {
      __threadfence();
      skinny_ln_rows(p, &part[0][0]);
      if (threadIdx.x == 0) *p.ln_counter = 0u;
    }
  }
}

// 9 <= M <= 64 rows (batched beam search: n_samples x beam rows).  Same CTA / warp / K-slice layout as the kernel above
// (chosen from N and K only), same k permutation, same MMA sequence per k-block and the same cross-warp reduction order,
// so row r of the result depends on row r of x alone, bit for bit, at any M.  The rows are MT m16 tiles of the A
// operand: lane (g, t) feeds rows 16i + g and 16i + 8 + g of tile i, and every tile reuses the weight fragments the lane
// already holds - the weights are still read once.  Only the weights are double-buffered; the activations (L1/L2
// resident) are loaded for the current batch, which keeps the register budget at two CTAs per SM.
__device__ __forceinline__ void mma16816_bf16_full(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                                   uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void skinny_store(const SkinnyParams& p, int m, int n, float v) {
  if (p.bias) v += __bfloat162float(p.bias[n]);
  if (p.act == YMP_ACT_GELU_TANH) v = gelu_tanh(v);
  else if (p.act == YMP_ACT_GELU_ERF) v = gelu_erf(v);
  if (p.residual)
    v += p.res_f32 ? reinterpret_cast<const float*>(p.residual)[(size_t)m * p.ldr + n]
                   : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.residual)[(size_t)m * p.ldr + n]);
  if (p.out_f32) reinterpret_cast<float*>(p.y)[(size_t)m * p.ldy + n] = v;
  else reinterpret_cast<__nv_bfloat16*>(p.y)[(size_t)m * p.ldy + n] = __float2bfloat16(v);
  if (p.y2) p.y2[(long long)m * p.ldy2 + *p.y2_off * p.y2_stride + n] = __float2bfloat16(v);
}

constexpr int SK_WIDE_MAXM = 64, SK_WIDE_UNROLL = 4;

template <int MT>
__global__ void __launch_bounds__(SK_WARPS * 32, 2) gemm_skinny_wide_kernel(const SkinnyParams p) {
  constexpr int U = SK_WIDE_UNROLL;
  __shared__ float part[SK_WARPS][MT * 128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int ks = p.ksplit, kpart = warp % ks, tile = blockIdx.x * (SK_WARPS / ks) + warp / ks;
  const int n0 = tile * SK_TILE_N;
  const bool live = n0 < p.N;
  float acc[MT][4];
#pragma unroll
  for (int i = 0; i < MT; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
  griddep_launch();
  if (live) {
    const int nchunk = p.K >> 3, nblk = (nchunk + 3) >> 2;
    const int b_lo = (int)((long)nblk * kpart / ks), b_hi = (int)((long)nblk * (kpart + 1) / ks);
    const uint4* wr = reinterpret_cast<const uint4*>(p.w + (size_t)min(n0 + g, p.N - 1) * p.ldw);
    const uint4* xr[MT][2];
    bool xrow[MT][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int m = 16 * i + 8 * h + g;
        xrow[i][h] = m < p.M;
        xr[i][h] = reinterpret_cast<const uint4*>(p.x + (size_t)min(m, p.M - 1) * p.ldx);
      }
    uint4 wv[U];
    auto fetch_w = [&](int b, uint4 (&wd)[U]) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = (b + u) * 4 + t;
        wd[u] = ((b + u) < b_hi && c < nchunk) ? ld_nc_v4(wr + c) : make_uint4(0, 0, 0, 0);
      }
    };
    fetch_w(b_lo, wv);
    griddep_wait();
    for (int b = b_lo; b < b_hi; b += U) {
      uint4 wn[U];
      fetch_w(b + U, wn);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = (b + u) * 4 + t;
        const bool in = (b + u) < b_hi && c < nchunk;
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          const uint4 x0 = (in && xrow[i][0]) ? __ldg(xr[i][0] + c) : make_uint4(0, 0, 0, 0);
          const uint4 x1 = (in && xrow[i][1]) ? __ldg(xr[i][1] + c) : make_uint4(0, 0, 0, 0);
          mma16816_bf16_full(acc[i], x0.x, x1.x, x0.y, x1.y, wv[u].x, wv[u].y);
          mma16816_bf16_full(acc[i], x0.z, x1.z, x0.w, x1.w, wv[u].z, wv[u].w);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) wv[u] = wn[u];
    }
  } else {
    griddep_wait();
  }
  // acc[i][2h + e] = (row 16i + 8h + g, column n0 + 2t + e) summed over this warp's K slice
  if (ks > 1) {
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) part[warp][i * 128 + 4 * lane + e] = acc[i][e];
    __syncthreads();
    if (kpart == 0)
      for (int j = 1; j < ks; ++j)
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[i][e] += part[warp + j][i * 128 + 4 * lane + e];
  }
  if (live && kpart == 0) {
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int m = 16 * i + 8 * h + g;
        if (m >= p.M) continue;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int n = n0 + 2 * t + e;
          if (n < p.N) skinny_store(p, m, n, acc[i][2 * h + e]);
        }
      }
  }
}

}  // namespace ymp

using namespace ymp;

// ymp_gemm_skinny (M <= 8) and ymp_gemm_skinny_batch (M <= 64): one implementation, the same kernel for M <= 8
static int gemm_skinny_call(const ymp_gemm_skinny_args* a, void* stream, int max_m) {
  YMP_CHECK_ARG(a && a->x && a->w && a->y, "ymp_gemm_skinny: null pointer");
  YMP_CHECK_ARG(a->M >= 1 && a->M <= max_m && a->N > 0 && a->K > 0 && a->K % 8 == 0, "ymp_gemm_skinny: needs 1 <= M <= %d, K %% 8 == 0 (M=%d K=%d)", max_m, a->M, a->K);
  YMP_CHECK_ARG(!a->ln_out || a->M <= SK_MAXM, "ymp_gemm_skinny: the fused LayerNorm needs M <= 8 (M=%d)", a->M);
  YMP_CHECK_ARG(a->ldx % 8 == 0 && a->ldw % 8 == 0 && a->ldx >= a->K && a->ldw >= a->K && aligned16(a->x) && aligned16(a->w), "ymp_gemm_skinny: x / w rows must be 16-byte aligned");
  YMP_CHECK_ARG(a->act >= 0 && a->act <= 2, "ymp_gemm_skinny: bad act");
  SkinnyParams p;
  p.x = (const __nv_bfloat16*)a->x; p.w = (const __nv_bfloat16*)a->w; p.bias = (const __nv_bfloat16*)a->bias;
  p.residual = a->residual; p.y = a->y;
  YMP_CHECK_ARG(!a->y2 || (a->y2_off_dev && a->out_dtype == YMP_DT_BF16), "ymp_gemm_skinny: y2 needs y2_off_dev and a bf16 result");
  p.y2 = (__nv_bfloat16*)a->y2; p.y2_off = (const long long*)a->y2_off_dev; p.ldy2 = a->ldy2; p.y2_stride = a->y2_off_stride;
  p.M = a->M; p.N = a->N; p.K = a->K; p.ldx = a->ldx; p.ldw = a->ldw; p.ldr = a->ldr; p.ldy = a->ldy;
  const bool ln = a->ln_out != nullptr;
  YMP_CHECK_ARG(!ln || (a->ln_gamma && a->ln_beta && a->ln_counter && a->out_dtype == YMP_DT_F32 && a->N % 8 == 0 && a->ld_ln % 8 == 0 &&
                        a->ldy % 4 == 0 && aligned16(a->y) && aligned16(a->ln_out) && aligned16(a->ln_gamma) && aligned16(a->ln_beta)),
                "ymp_gemm_skinny: fused LayerNorm needs gamma/beta/counter, an fp32 result, N %% 8 == 0 and 16-byte aligned rows");
  p.ln_gamma = (const __nv_bfloat16*)a->ln_gamma; p.ln_beta = (const __nv_bfloat16*)a->ln_beta; p.ln_out = (__nv_bfloat16*)a->ln_out;
  p.ln_counter = a->ln_counter; p.ld_ln = a->ld_ln; p.ln_eps = a->ln_eps;
  p.act = a->act; p.res_f32 = a->residual_dtype == YMP_DT_F32; p.out_f32 = a->out_dtype == YMP_DT_F32;
  // K slices per CTA (the warps of a CTA that share one 8-column tile): as many as leave >= 4 k-blocks of 32 per slice
  int ks = 1;
  static const int force = [] { const char* e = getenv("YMP_SKINNY_KSPLIT"); return e ? atoi(e) : 0; }();
  const int ks_max = a->N <= 4096 ? 8 : 4;   // measured (tools/skinny_probe.py): wide outputs prefer fatter CTAs
  while (ks < ks_max && a->K / (2 * ks) >= 128) ks *= 2;
  if (force == 1 || force == 2 || force == 4 || force == 8) ks = force;
  p.ksplit = ks;
  const int tiles = (a->N + SK_TILE_N - 1) / SK_TILE_N, tiles_per_cta = SK_WARPS / ks;
  const int blocks = (tiles + tiles_per_cta - 1) / tiles_per_cta;
  static const int unroll = [] { const char* e = getenv("YMP_SKINNY_UNROLL"); return e ? atoi(e) : 4; }();
  cudaStream_t st = (cudaStream_t)stream;
  if (a->M > SK_MAXM) {   // same grid, one to four m16 row tiles per warp
    const int mt = (a->M + 15) / 16;
    if (mt == 1) launch_k(gemm_skinny_wide_kernel<1>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
    else if (mt == 2) launch_k(gemm_skinny_wide_kernel<2>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
    else if (mt == 3) launch_k(gemm_skinny_wide_kernel<3>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
    else launch_k(gemm_skinny_wide_kernel<4>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
    YMP_LAUNCH_CHECK();
    return YMP_OK;
  }
  if (ln) launch_k(gemm_skinny_kernel<4, true>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
  else if (unroll == 8) launch_k(gemm_skinny_kernel<8, false>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
  else if (unroll == 2) launch_k(gemm_skinny_kernel<2, false>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
  else launch_k(gemm_skinny_kernel<4, false>, dim3(blocks), dim3(SK_WARPS * 32), 0, st, p);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_gemm_skinny(const ymp_gemm_skinny_args* a, void* stream) { return gemm_skinny_call(a, stream, SK_MAXM); }
extern "C" int ymp_gemm_skinny_batch(const ymp_gemm_skinny_args* a, void* stream) { return gemm_skinny_call(a, stream, SK_WIDE_MAXM); }
