// HBM-bound helper kernels of the path: im2col for the patch embedding, embedding gather,
// fused softmax-cross-entropy forward/backward over the vocabulary, column sums (bias grads),
// small group reductions.  All use 128-bit coalesced accesses where the layout allows.
#include <math_constants.h>

#include "common.h"
#include "philox.cuh"
#include "ptx.cuh"

namespace ymp {

// ------------------------------------------------------------------------------ im2col
// video [B,C,T,H,W] bf16 -> patches [(b, n, t), C*P*P] with n = py*Wp + px, column = (c, iy, ix):
// the row order is the encoder's internal patch-major (n t) order, the column order matches
// conv weight [D, C, P, P].flatten(1).
__global__ void __launch_bounds__(256) im2col_kernel(const __nv_bfloat16* __restrict__ video,
                                                     __nv_bfloat16* __restrict__ out, int B, int C, int T,
                                                     int H, int W, int P, int ldo) {
  const int Hp = H / P, Wp = W / P, N = Hp * Wp;
  const int vec_per_row = C * P * (P / 8);
  const long total = (long)B * N * T * vec_per_row;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int v = (int)(idx % vec_per_row);
    const long row = idx / vec_per_row;
    const int t = (int)(row % T);
    const int n = (int)((row / T) % N);
    const int b = (int)(row / ((long)T * N));
    const int ixv = v % (P / 8);
    const int iy = (v / (P / 8)) % P;
    const int c = v / (P / 8 * P);
    const int py = n / Wp, px = n % Wp;
    const size_t src = ((((size_t)b * C + c) * T + t) * H + (py * P + iy)) * W + px * P + ixv * 8;
    const uint4 val = __ldg(reinterpret_cast<const uint4*>(video + src));
    *reinterpret_cast<uint4*>(out + row * ldo + (size_t)(c * P + iy) * P + ixv * 8) = val;
  }
}

// Any patch size (EVA-g: 14 x 14 patches, row length 588 is not a multiple of 8): one element per thread, columns
// [C*P*P, ldo) of every row are zero-filled so that the GEMM can use a 16-byte aligned, padded K extent.
__global__ void __launch_bounds__(256) im2col_generic_kernel(const __nv_bfloat16* __restrict__ video,
                                                             __nv_bfloat16* __restrict__ out, int B, int C, int T,
                                                             int H, int W, int P, int ldo) {
  const int Hp = H / P, Wp = W / P, N = Hp * Wp, K = C * P * P;
  const long total = (long)B * N * T * ldo;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int col = (int)(idx % ldo);
    const long row = idx / ldo;
    __nv_bfloat16 val = __float2bfloat16(0.f);
    if (col < K) {
      const int t = (int)(row % T), n = (int)((row / T) % N), b = (int)(row / ((long)T * N));
      const int ix = col % P, iy = (col / P) % P, c = col / (P * P);
      const int py = n / Wp, px = n % Wp;
      val = video[((((size_t)b * C + c) * T + t) * H + (py * P + iy)) * W + px * P + ix];
    }
    out[idx] = val;
  }
}

// ------------------------------------------------------------------------------ embedding gather
// out[(b*S + off + l), :] = table[ids[b,l], :] + pos[off + l, :]     (one warp per row)
__global__ void __launch_bounds__(256) embed_gather_kernel(const int64_t* __restrict__ ids,
                                                           const __nv_bfloat16* __restrict__ table,
                                                           const __nv_bfloat16* __restrict__ pos,
                                                           void* __restrict__ out_, int B, int L,
                                                           int S, int off, int Hd, int vocab, int ldo, int out_f32) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nvec = Hd >> 3;
  for (int r = warp; r < B * L; r += nwarps) {
    const int b = r / L, l = r - b * L;
    long id = ids[r];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    const uint4* src = reinterpret_cast<const uint4*>(table + (size_t)id * Hd);
    const uint4* ps = pos ? reinterpret_cast<const uint4*>(pos + (size_t)(off + l) * Hd) : nullptr;
    const size_t orow = (size_t)(b * S + off + l) * ldo;
    for (int v = lane; v < nvec; v += 32) {
      const uint4 a = __ldg(src + v);
      float f[8] = {bf16_lo(a.x), bf16_hi(a.x), bf16_lo(a.y), bf16_hi(a.y), bf16_lo(a.z), bf16_hi(a.z), bf16_lo(a.w), bf16_hi(a.w)};
      if (ps) {
        const uint4 c = __ldg(ps + v);
        f[0] += bf16_lo(c.x); f[1] += bf16_hi(c.x); f[2] += bf16_lo(c.y); f[3] += bf16_hi(c.y);
        f[4] += bf16_lo(c.z); f[5] += bf16_hi(c.z); f[6] += bf16_lo(c.w); f[7] += bf16_hi(c.w);
      }
      if (out_f32) {
        float4* d = reinterpret_cast<float4*>(reinterpret_cast<float*>(out_) + orow) + 2 * v;
        d[0] = make_float4(f[0], f[1], f[2], f[3]);
        d[1] = make_float4(f[4], f[5], f[6], f[7]);
      } else {
        uint4 o;
        o.x = pack_bf16(f[0], f[1]); o.y = pack_bf16(f[2], f[3]); o.z = pack_bf16(f[4], f[5]); o.w = pack_bf16(f[6], f[7]);
        reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(out_) + orow)[v] = o;
      }
    }
  }
}

// ------------------------------------------------------------------------------ softmax CE
constexpr int CE_THREADS = 256;

__device__ __forceinline__ void online_add(float& m, float& s, float x) {
  if (x > m) { s = s * __expf(m - x) + 1.f; m = x; }
  else s += __expf(x - m);
}

// loss[row] = logsumexp(logits[row,:]) - logits[row,label[row]]   (fp32 math over bf16 logits)
__global__ void __launch_bounds__(CE_THREADS) ce_fwd_kernel(const __nv_bfloat16* __restrict__ logits,
                                                            const int64_t* __restrict__ labels,
                                                            float* __restrict__ loss, float* __restrict__ lse,
                                                            int V, int ld) {
  const int row = blockIdx.x;
  const __nv_bfloat16* x = logits + (size_t)row * ld;
  float m = -CUDART_INF_F, s = 0.f;
  const int nvec = V >> 3;
  for (int v = threadIdx.x; v < nvec; v += CE_THREADS) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(x) + v);
    const float f[8] = {bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y),
                        bf16_lo(u.z), bf16_hi(u.z), bf16_lo(u.w), bf16_hi(u.w)};
    float mx = f[0];
#pragma unroll
    for (int e = 1; e < 8; ++e) mx = fmaxf(mx, f[e]);
    if (mx > m) { s *= __expf(m - mx); m = mx; }
#pragma unroll
    for (int e = 0; e < 8; ++e) s += __expf(f[e] - m);
  }
  for (int c = (nvec << 3) + threadIdx.x; c < V; c += CE_THREADS) online_add(m, s, __bfloat162float(x[c]));
  // block reduce of (m, s)
  __shared__ float sm[CE_THREADS / 32], ss[CE_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    const float mn = fmaxf(m, m2);
    s = (mn == -CUDART_INF_F) ? 0.f : s * __expf(m - mn) + s2 * __expf(m2 - mn);
    m = mn;
  }
  if ((threadIdx.x & 31) == 0) { sm[threadIdx.x >> 5] = m; ss[threadIdx.x >> 5] = s; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float M = sm[0], S = ss[0];
    for (int w = 1; w < CE_THREADS / 32; ++w) {
      const float mn = fmaxf(M, sm[w]);
      S = S * __expf(M - mn) + ss[w] * __expf(sm[w] - mn);
      M = mn;
    }
    const float l = M + logf(S);
    long lab = labels[row];
    lab = lab < 0 ? 0 : (lab >= V ? V - 1 : lab);
    loss[row] = l - __bfloat162float(x[lab]);
    if (lse) lse[row] = l;
  }
}

// dlogits[row, v] = g[row] * (softmax(logits[row])[v] - [v == label[row]])   (in place allowed)
__global__ void __launch_bounds__(CE_THREADS) ce_bwd_kernel(const __nv_bfloat16* logits,
                                                            const int64_t* __restrict__ labels,
                                                            const float* __restrict__ lse,
                                                            const float* __restrict__ g,
                                                            __nv_bfloat16* dlogits, int V, int ld) {
  const int row = blockIdx.x;
  const float gr = g[row];
  const __nv_bfloat16* x = logits + (size_t)row * ld;
  __nv_bfloat16* dx = dlogits + (size_t)row * ld;
  const int nvec = V >> 3;
  if (gr == 0.f) {
    for (int v = threadIdx.x; v < nvec; v += CE_THREADS) reinterpret_cast<uint4*>(dx)[v] = make_uint4(0, 0, 0, 0);
    for (int c = (nvec << 3) + threadIdx.x; c < V; c += CE_THREADS) dx[c] = __float2bfloat16(0.f);
    return;
  }
  const float l = lse[row];
  long lab = labels[row];
  lab = lab < 0 ? 0 : (lab >= V ? V - 1 : lab);
  for (int v = threadIdx.x; v < nvec; v += CE_THREADS) {
    const uint4 u = reinterpret_cast<const uint4*>(x)[v];
    float f[8] = {bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y),
                  bf16_lo(u.z), bf16_hi(u.z), bf16_lo(u.w), bf16_hi(u.w)};
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float pr = __expf(f[e] - l);
      if (v * 8 + e == lab) pr -= 1.f;
      f[e] = pr * gr;
    }
    uint4 o;
    o.x = pack_bf16(f[0], f[1]); o.y = pack_bf16(f[2], f[3]);
    o.z = pack_bf16(f[4], f[5]); o.w = pack_bf16(f[6], f[7]);
    reinterpret_cast<uint4*>(dx)[v] = o;
  }
  for (int c = (nvec << 3) + threadIdx.x; c < V; c += CE_THREADS) {
    float pr = __expf(__bfloat162float(x[c]) - l);
    if (c == lab) pr -= 1.f;
    dx[c] = __float2bfloat16(pr * gr);
  }
}

// ------------------------------------------------------------------------------ column sum
// out[c] += sum_r in[r, c]   (fp32; the caller zeroes or carries `out`).
// Block = 8 warps x 32 lanes: a warp reads 512 contiguous bytes of one row (8 columns per lane, 8 rows
// in flight per lane), the 8 warps of a block take interleaved rows and are reduced through shared
// memory; block (x, y) writes its partial column sums to row y of `part` (ldp floats per row), and reduce_partials
// adds the rows in order.
constexpr int CS_WARPS = 8;
__device__ __forceinline__ void acc8(float (&acc)[8], const uint4& u) {
  acc[0] += bf16_lo(u.x); acc[1] += bf16_hi(u.x); acc[2] += bf16_lo(u.y); acc[3] += bf16_hi(u.y);
  acc[4] += bf16_lo(u.z); acc[5] += bf16_hi(u.z); acc[6] += bf16_lo(u.w); acc[7] += bf16_hi(u.w);
}
__global__ void __launch_bounds__(CS_WARPS * 32) colsum_kernel(const __nv_bfloat16* __restrict__ in,
                                                               float* __restrict__ part, int ldp, int R, int C, int ld,
                                                               int rows_per_block) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int v = blockIdx.x * 32 + lane;  // 8-column vector index
  const bool active = v * 8 < C;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(R, r0 + rows_per_block);
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (active) {
    int r = r0 + warp;
    for (; r + 7 * CS_WARPS < r1; r += 8 * CS_WARPS) {
      uint4 u[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) u[j] = __ldg(reinterpret_cast<const uint4*>(in + (size_t)(r + j * CS_WARPS) * ld) + v);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc8(acc, u[j]);
    }
    for (; r < r1; r += CS_WARPS) acc8(acc, __ldg(reinterpret_cast<const uint4*>(in + (size_t)r * ld) + v));
  }
  __shared__ float red[CS_WARPS][32][9];
#pragma unroll
  for (int e = 0; e < 8; ++e) red[warp][lane][e] = acc[e];
  __syncthreads();
  // 256 columns per block: thread t < 64 owns 4 consecutive columns
  if (threadIdx.x < 64) {
    const int l = threadIdx.x >> 1, e0 = (threadIdx.x & 1) * 4;
    float s[4] = {0, 0, 0, 0};
#pragma unroll
    for (int w = 0; w < CS_WARPS; ++w)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[e] += red[w][l][e0 + e];
    const int col = (blockIdx.x * 32 + l) * 8 + e0;
    float* dst = part + (size_t)blockIdx.y * ldp + col;
    if (col + 3 < C) {
      *reinterpret_cast<float4*>(dst) = make_float4(s[0], s[1], s[2], s[3]);
    } else {
      for (int e = 0; e < 4; ++e)
        if (col + e < C) dst[e] = s[e];
    }
  }
}

// ------------------------------------------------------------------------------ group reduce
// out[g, c] = scale * sum_t in[g, t, c]     in: [G, T, C] rows of stride ld_in, out rows ld_out
__global__ void __launch_bounds__(256) group_reduce_kernel(const __nv_bfloat16* __restrict__ in,
                                                           __nv_bfloat16* __restrict__ out, int G, int T,
                                                           int C, int ld_in, int ld_out, float scale) {
  const int nvec = C >> 3;
  const long total = (long)G * nvec;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int gidx = (int)(idx / nvec), v = (int)(idx % nvec);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int t = 0; t < T; ++t) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(in + ((size_t)gidx * T + t) * ld_in) + v);
      acc[0] += bf16_lo(u.x); acc[1] += bf16_hi(u.x); acc[2] += bf16_lo(u.y); acc[3] += bf16_hi(u.y);
      acc[4] += bf16_lo(u.z); acc[5] += bf16_hi(u.z); acc[6] += bf16_lo(u.w); acc[7] += bf16_hi(u.w);
    }
    uint4 o;
    o.x = pack_bf16(acc[0] * scale, acc[1] * scale); o.y = pack_bf16(acc[2] * scale, acc[3] * scale);
    o.z = pack_bf16(acc[4] * scale, acc[5] * scale); o.w = pack_bf16(acc[6] * scale, acc[7] * scale);
    reinterpret_cast<uint4*>(out + (size_t)gidx * ld_out)[v] = o;
  }
}

// out[g, t, c] = scale * in[g, c]   (backward of the mean over frames)
__global__ void __launch_bounds__(256) group_bcast_kernel(const __nv_bfloat16* __restrict__ in,
                                                          __nv_bfloat16* __restrict__ out, int G, int T,
                                                          int C, int ld_in, int ld_out, float scale) {
  const int nvec = C >> 3;
  const long total = (long)G * T * nvec;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int v = (int)(idx % nvec);
    const long gt = idx / nvec;
    const int gidx = (int)(gt / T);
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(in + (size_t)gidx * ld_in) + v);
    uint4 o;
    o.x = pack_bf16(bf16_lo(u.x) * scale, bf16_hi(u.x) * scale); o.y = pack_bf16(bf16_lo(u.y) * scale, bf16_hi(u.y) * scale);
    o.z = pack_bf16(bf16_lo(u.z) * scale, bf16_hi(u.z) * scale); o.w = pack_bf16(bf16_lo(u.w) * scale, bf16_hi(u.w) * scale);
    reinterpret_cast<uint4*>(out + (size_t)gt * ld_out)[v] = o;
  }
}


// ------------------------------------------------------------------------------ clip -> model input
// uint8 [B,T,H,W,C] -> bf16 [B,C,T,H,W] through a per-channel 256-entry table (see include/ymp.h).
// One thread = 8 consecutive pixels of one frame: 8*C contiguous input bytes, one 16-byte store per channel
// plane.  HBM-bound: 1 byte read + 2 bytes written per value.
template <int CH>
__global__ void __launch_bounds__(256) clip_normalize_kernel(const uint8_t* __restrict__ frames, __nv_bfloat16* __restrict__ out,
                                                            const __nv_bfloat16* __restrict__ lut, int B, int T, long HW) {
  __shared__ uint16_t tab[CH * 256];
  for (int i = threadIdx.x; i < CH * 256; i += blockDim.x) tab[i] = reinterpret_cast<const uint16_t*>(lut)[i];
  __syncthreads();
  const long groups_per_frame = HW >> 3;
  const long total = (long)B * T * groups_per_frame;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long)gridDim.x * blockDim.x) {
    const long frame = g / groups_per_frame, pg = g - frame * groups_per_frame;  // frame = b*T + t
    const long b = frame / T, t = frame - b * T;
    const uint8_t* src = frames + (frame * HW + pg * 8) * CH;
    uint8_t px[8 * CH];
    if constexpr ((8 * CH) % 8 == 0) {
#pragma unroll
      for (int i = 0; i < CH; ++i) reinterpret_cast<uint2*>(px)[i] = __ldg(reinterpret_cast<const uint2*>(src) + i);
    } else {
#pragma unroll
      for (int i = 0; i < 8 * CH; ++i) px[i] = __ldg(src + i);
    }
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        w[i] = (uint32_t)tab[c * 256 + px[(2 * i) * CH + c]] | ((uint32_t)tab[c * 256 + px[(2 * i + 1) * CH + c]] << 16);
      __nv_bfloat16* dst = out + ((b * CH + c) * T + t) * HW + pg * 8;
      *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

// ------------------------------------------------------------------------------ elementwise dropout
// y[r, c] = dropout(x[r, c]) with the decoder's Philox convention (logical row = row0 + r): the embedding
// dropout of GPT3Embedding.forward (models/modeling_distributed_gpt3.py:631).  HBM-bound, 4 columns per thread.
template <bool F32>
__global__ void __launch_bounds__(256) dropout_kernel(const void* __restrict__ x, void* __restrict__ y, int rows, int cols,
                                                       int ldx, int ldy, long row0, const DropSpec d) {
  const DropState ds = drop_state(d);
  const int c4n = cols >> 2;
  const long total = (long)rows * c4n;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int r = (int)(idx / c4n), c4 = (int)(idx - (long)r * c4n);
    float a, b, c, e;
    if (F32) {
      const float4 v = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + (size_t)r * ldx + 4 * c4);
      a = v.x; b = v.y; c = v.z; e = v.w;
    } else {
      const uint2 v = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(x) + (size_t)r * ldx + 4 * c4);
      a = bf16_lo(v.x); b = bf16_hi(v.x); c = bf16_lo(v.y); e = bf16_hi(v.y);
    }
    drop4(ds, (uint32_t)(row0 + r), (uint32_t)(4 * c4), a, b, c, e);
    if (F32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + (size_t)r * ldy + 4 * c4) = make_float4(a, b, c, e);
    else *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + (size_t)r * ldy + 4 * c4) = make_uint2(pack_bf16(a, b), pack_bf16(c, e));
  }
}

}  // namespace ymp

using namespace ymp;

extern "C" int ymp_dropout(const ymp_dropout_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->x && a->y && a->rows > 0 && a->cols > 0 && a->cols % 4 == 0, "ymp_dropout: bad args (cols must be a multiple of 4)");
  YMP_CHECK_ARG(a->ldx % 4 == 0 && a->ldy % 4 == 0 && a->ldx >= a->cols && a->ldy >= a->cols, "ymp_dropout: bad ld");
  YMP_CHECK_ARG(aligned16(a->x) && aligned16(a->y), "ymp_dropout: 16-byte alignment required");
  YMP_CHECK_ARG(a->drop.rng && a->drop.p > 0.f && a->drop.p < 1.f, "ymp_dropout: needs rng and 0 < p < 1");
  DropSpec d; d.rng = a->drop.rng; d.site = a->drop.site; d.p = a->drop.p;
  const long total = (long)a->rows * (a->cols / 4);
  const int blocks = (int)min((total + 255) / 256, (long)num_sms() * 8);
  if (a->dtype == YMP_DT_F32)
    dropout_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(a->x, a->y, a->rows, a->cols, a->ldx, a->ldy, (long)a->row0, d);
  else
    dropout_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(a->x, a->y, a->rows, a->cols, a->ldx, a->ldy, (long)a->row0, d);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_im2col(const ymp_im2col_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->video && a->out, "ymp_im2col: null pointer");
  YMP_CHECK_ARG(a->P > 0 && a->H % a->P == 0 && a->W % a->P == 0, "ymp_im2col: need H%%P==0, W%%P==0 (P=%d H=%d W=%d)", a->P, a->H, a->W);
  if (a->P % 8 != 0 || a->W % 8 != 0) {
    YMP_CHECK_ARG(a->ldo >= a->C * a->P * a->P && a->ldo % 8 == 0 && aligned16(a->out), "ymp_im2col: bad ldo / alignment");
    const long tot = (long)a->B * (a->H / a->P) * (a->W / a->P) * a->T * a->ldo;
    const int blk = (int)min((tot + 255) / 256, (long)num_sms() * 16);
    im2col_generic_kernel<<<blk, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a->video, (__nv_bfloat16*)a->out, a->B, a->C,
                                                                 a->T, a->H, a->W, a->P, a->ldo);
    YMP_LAUNCH_CHECK();
    return YMP_OK;
  }
  YMP_CHECK_ARG(a->ldo >= a->C * a->P * a->P && a->ldo % 8 == 0, "ymp_im2col: bad ldo");
  YMP_CHECK_ARG(aligned16(a->video) && aligned16(a->out), "ymp_im2col: alignment");
  const long total = (long)a->B * (a->H / a->P) * (a->W / a->P) * a->T * a->C * a->P * (a->P / 8);
  const int blocks = (int)min((total + 255) / 256, (long)num_sms() * 16);
  im2col_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a->video, (__nv_bfloat16*)a->out,
                                                           a->B, a->C, a->T, a->H, a->W, a->P, a->ldo);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_clip_normalize(const ymp_clip_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->frames && a->out && a->lut, "ymp_clip_normalize: null pointer");
  YMP_CHECK_ARG(a->C == 1 || a->C == 3 || a->C == 4, "ymp_clip_normalize: C must be 1, 3 or 4 (got %d)", a->C);
  const long HW = (long)a->H * a->W;
  YMP_CHECK_ARG(a->B > 0 && a->T > 0 && HW > 0 && HW % 8 == 0, "ymp_clip_normalize: H*W must be a positive multiple of 8");
  YMP_CHECK_ARG((reinterpret_cast<uintptr_t>(a->frames) & 7) == 0 && aligned16(a->out), "ymp_clip_normalize: alignment");
  const long total = (long)a->B * a->T * (HW / 8);
  const int blocks = (int)min((total + 255) / 256, (long)num_sms() * 16);
  cudaStream_t st = (cudaStream_t)stream;
  const uint8_t* f = (const uint8_t*)a->frames;
  __nv_bfloat16* o = (__nv_bfloat16*)a->out;
  const __nv_bfloat16* l = (const __nv_bfloat16*)a->lut;
  if (a->C == 3) clip_normalize_kernel<3><<<blocks, 256, 0, st>>>(f, o, l, a->B, a->T, HW);
  else if (a->C == 4) clip_normalize_kernel<4><<<blocks, 256, 0, st>>>(f, o, l, a->B, a->T, HW);
  else clip_normalize_kernel<1><<<blocks, 256, 0, st>>>(f, o, l, a->B, a->T, HW);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_embed_gather(const ymp_embed_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->ids && a->table && a->out, "ymp_embed_gather: null pointer");
  YMP_CHECK_ARG(a->hidden % 8 == 0 && a->ldo % 8 == 0 && a->ldo >= a->hidden, "ymp_embed_gather: hidden/ldo must be multiples of 8");
  YMP_CHECK_ARG(a->B > 0 && a->L > 0 && a->S >= a->row_offset + a->L, "ymp_embed_gather: bad B/L/S/offset");
  const int rows = a->B * a->L;
  const int blocks = min((rows + 7) / 8, num_sms() * 8);
  embed_gather_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      a->ids, (const __nv_bfloat16*)a->table, (const __nv_bfloat16*)a->pos, a->out, a->B, a->L,
      a->S, a->row_offset, a->hidden, a->vocab, a->ldo, a->out_dtype == YMP_DT_F32 ? 1 : 0);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_ce_fwd(const ymp_ce_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->logits && a->labels && a->loss, "ymp_ce_fwd: null pointer");
  YMP_CHECK_ARG(a->rows > 0 && a->V > 0 && a->ld >= a->V && a->ld % 8 == 0 && aligned16(a->logits), "ymp_ce_fwd: bad shape/alignment");
  ce_fwd_kernel<<<a->rows, CE_THREADS, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a->logits, a->labels, a->loss,
                                                                  a->lse, a->V, a->ld);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_ce_bwd(const ymp_ce_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->logits && a->labels && a->lse && a->grad_rows && a->dlogits, "ymp_ce_bwd: null pointer");
  YMP_CHECK_ARG(a->rows > 0 && a->V > 0 && a->ld >= a->V && a->ld % 8 == 0 && aligned16(a->logits) && aligned16(a->dlogits), "ymp_ce_bwd: bad shape/alignment");
  ce_bwd_kernel<<<a->rows, CE_THREADS, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a->logits, a->labels, a->lse,
                                                                  a->grad_rows, (__nv_bfloat16*)a->dlogits, a->V, a->ld);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

extern "C" int ymp_colsum(const ymp_colsum_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->in && a->out, "ymp_colsum: null pointer");
  // C need not be a multiple of 8: rows are read in 8-column vectors, so the row stride must cover the
  // rounded-up width (the columns beyond C are read and discarded)
  YMP_CHECK_ARG(a->R > 0 && a->C > 0 && a->ld % 8 == 0 && a->ld >= (a->C + 7) / 8 * 8 && aligned16(a->in), "ymp_colsum: bad shape/alignment");
  YMP_CHECK_ARG(aligned16(a->out), "ymp_colsum: out must be 16-byte aligned");
  const int gx = ((a->C + 7) / 8 + 31) / 32;
  int splits = max(1, min((a->R + 63) / 64, (num_sms() * 4 + gx - 1) / gx));
  const int rpb = (a->R + splits - 1) / splits;
  splits = (a->R + rpb - 1) / rpb;
  cudaStream_t st = (cudaStream_t)stream;
  const int ldp = (a->C + 3) / 4 * 4;
  Scratch part;
  int rc = part.alloc(sizeof(float) * (size_t)splits * ldp, st);
  if (rc) return rc;
  colsum_kernel<<<dim3(gx, splits), CS_WARPS * 32, 0, st>>>((const __nv_bfloat16*)a->in, (float*)part.p, ldp, a->R, a->C, a->ld, rpb);
  YMP_LAUNCH_CHECK();
  rc = reduce_partials((const float*)part.p, splits, ldp, a->C, a->out, st);
  if (rc) return rc;
  return part.release();
}

extern "C" int ymp_group_reduce(const ymp_group_args* a, void* stream) {
  YMP_CHECK_ARG(a && a->in && a->out, "ymp_group_reduce: null pointer");
  YMP_CHECK_ARG(a->G > 0 && a->T > 0 && a->C > 0 && a->C % 8 == 0 && a->ld_in % 8 == 0 && a->ld_out % 8 == 0, "ymp_group_reduce: bad shape");
  const long total = (long)a->G * (a->C / 8) * (a->broadcast ? a->T : 1);
  const int blocks = (int)min((total + 255) / 256, (long)num_sms() * 8);
  if (!a->broadcast)
    group_reduce_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a->in, (__nv_bfloat16*)a->out, a->G, a->T, a->C, a->ld_in, a->ld_out, a->scale);
  else
    group_bcast_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a->in, (__nv_bfloat16*)a->out, a->G, a->T, a->C, a->ld_in, a->ld_out, a->scale);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}
