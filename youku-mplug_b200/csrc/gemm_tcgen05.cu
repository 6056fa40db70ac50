// Persistent, warp-specialised bf16 GEMM for sm_100a.
//   warp 0      : TMA producer   (cp.async.bulk.tensor 2D, SWIZZLE_128B, NSTAGE-deep mbarrier ring)
//   warp 1      : MMA issuer     (tcgen05.mma cta_group::1 kind::f16, 128 x BN x 16, fp32 accum in TMEM)
//   warp 2      : TMEM allocator (2 accumulator stages so the epilogue of tile i overlaps tile i+1)
//   warps 4..11 : epilogue       (tcgen05.ld -> bias / GELU / GELU' / residual -> bf16|fp32|fp32 accumulate)
// Operands may be K-major or MN-major (both handled by the UMMA smem descriptors), so the same
// kernel serves forward (x.W^T), dgrad (dy.W) and wgrad (dy^T.x, split-K slices
// reduced in a fixed order, see ymp_gemm).
#include <cuda.h>

#include "common.h"
#include "philox.cuh"
#include "ptx.cuh"

namespace ymp {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int NUM_EPI_WARPS = 8;
constexpr int GEMM_THREADS = (4 + NUM_EPI_WARPS) * 32;
constexpr int A_STAGE_BYTES = BM * BK * 2;

struct GemmKParams {
  void* D;
  const __nv_bfloat16* bias;
  const void* residual;            // bf16 or fp32 (res_f32)
  __nv_bfloat16* aux_out;
  const __nv_bfloat16* aux_in;
  int M, N, K;
  int ldd, ldr;
  int a_mn, b_mn;
  int act, out_f32, accumulate, split_k;
  int kb_per_split;
  int res_row_mod;                 // residual row = row % res_row_mod (0: plain)
  int d_row_block, d_row_stride;   // D row = (row / block) * stride + row % block (0: plain)
  int res_f32;
  int n_fast;                      // tile order: consecutive units walk N first (A streamed once) or M first
  bool v32_d, v32_aux, v32_res, v32_bias;  // 32-byte aligned -> 256-bit accesses
  float alpha;
  int im2col_T, im2col_N, im2col_Wp;  // fused im2col A operand (im2col_T > 0): frames, patches per frame, patches per row
  DropSpec drop;                   // dropout before the residual add (has_drop)
  int has_drop;
  int epi_tma;                     // CTA-pair kernel: outputs staged in swizzled smem and written by TMA (bulk tensor
                                   // store; bulk reduce-add for the fp32 accumulation; one K slice only)
  long long d_split_stride;        // split-K: slice ks of the K range writes D + ks * d_split_stride (0: no split)
};

template <int BN>
struct GemmCfg {
  static constexpr int NSTAGE = (BN == 256) ? 4 : 6;
  static constexpr int B_STAGE_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int TMEM_COLS = 2 * BN;  // 256 or 512 (power of two)
  static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + 256 + 1024;
};

// 256-bit global accesses (sm_100: LDG/STG.E.ENL2.256): one full 32-byte sector per thread per
// instruction, so the row-per-thread epilogue writes whole sectors instead of half sectors.
__device__ __forceinline__ void ld_v8(const void* p, uint32_t (&r)[8]) {
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p));
}
__device__ __forceinline__ void st_v8(void* p, const uint32_t (&r)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// 16 consecutive bf16 (32 bytes) <-> 16 floats
__device__ __forceinline__ void load16(const __nv_bfloat16* p, bool v32, float (&f)[16]) {
  uint32_t r[8];
  if (v32) {
    ld_v8(p, r);
  } else {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) { f[2 * i] = bf16_lo(r[i]); f[2 * i + 1] = bf16_hi(r[i]); }
}
__device__ __forceinline__ void store16(__nv_bfloat16* p, bool v32, const float* f) {
  uint32_t r[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) r[i] = pack_bf16(f[2 * i], f[2 * i + 1]);
  if (v32) {
    st_v8(p, r);
  } else {
    reinterpret_cast<uint4*>(p)[0] = make_uint4(r[0], r[1], r[2], r[3]);
    reinterpret_cast<uint4*>(p)[1] = make_uint4(r[4], r[5], r[6], r[7]);
  }
}

// Global operands of one epilogue chunk (32 columns of one row), fetched BEFORE the tcgen05.wait::ld so
// that their latency overlaps the TMEM read instead of following it (the epilogue warps are only two per
// scheduler: every exposed round trip is paid in full).
struct EpiPrefetch {
  uint32_t bias[16];  // 32 bf16
  uint32_t aux[16];   // 32 bf16 (aux_in)
  uint32_t res[32];   // 32 fp32 or 32 bf16 (first 16 words)
};
__device__ __forceinline__ void load32_raw(const __nv_bfloat16* p, bool v32, uint32_t* r) {
  if (v32) {
    uint32_t a[8], b[8];
    ld_v8(p, a);
    ld_v8(p + 16, b);
#pragma unroll
    for (int i = 0; i < 8; ++i) { r[i] = a[i]; r[8 + i] = b[i]; }
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(p) + j);
      r[4 * j] = a.x; r[4 * j + 1] = a.y; r[4 * j + 2] = a.z; r[4 * j + 3] = a.w;
    }
  }
}
__device__ __forceinline__ void epilogue_prefetch(const GemmKParams& p, int row, int col0, EpiPrefetch& pf) {
  if (row >= p.M || col0 + 32 > p.N) return;
  if (p.bias) load32_raw(p.bias + col0, p.v32_bias, pf.bias);
  if (p.aux_in) load32_raw(p.aux_in + (size_t)row * p.ldd + col0, p.v32_aux, pf.aux);
  if (p.residual) {
    const int rrow = p.res_row_mod ? row % p.res_row_mod : row;
    if (p.res_f32) {
      const float* rf = reinterpret_cast<const float*>(p.residual) + (size_t)rrow * p.ldr + col0;
      if (p.v32_res) {  // one 256-bit load per 32-byte sector (two 128-bit loads would touch every sector twice)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t a[8];
          ld_v8(rf + 8 * j, a);
#pragma unroll
          for (int i = 0; i < 8; ++i) pf.res[8 * j + i] = a[i];
        }
      } else {
        const float4* rp = reinterpret_cast<const float4*>(rf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 a = __ldg(rp + j);
          pf.res[4 * j] = __float_as_uint(a.x); pf.res[4 * j + 1] = __float_as_uint(a.y);
          pf.res[4 * j + 2] = __float_as_uint(a.z); pf.res[4 * j + 3] = __float_as_uint(a.w);
        }
      }
    } else {
      load32_raw(reinterpret_cast<const __nv_bfloat16*>(p.residual) + (size_t)rrow * p.ldr + col0, p.v32_res, pf.res);
    }
  }
}

// Epilogue for one thread: 32 consecutive columns of one output row.
template <bool DROP>
__device__ __forceinline__ void epilogue_chunk(const GemmKParams& p, const uint32_t (&r)[32],
                                               int row, int col0, const EpiPrefetch& pf, const DropState& ds, size_t dsplit) {
  if (row >= p.M || col0 >= p.N) return;
  const bool full = (col0 + 32 <= p.N);
  const int drow = p.d_row_block ? (row / p.d_row_block) * p.d_row_stride + row % p.d_row_block : row;
  const int rrow = p.res_row_mod ? row % p.res_row_mod : row;
  float v[32];
  if (p.alpha == 1.0f) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) * p.alpha;
  }

  if (full) {
    if (p.bias) {
#pragma unroll
      for (int i = 0; i < 16; ++i) { v[2 * i] += bf16_lo(pf.bias[i]); v[2 * i + 1] += bf16_hi(pf.bias[i]); }
    }
    const size_t off = (size_t)row * p.ldd + col0;          // aux tensors: plain rows
    const size_t doff = dsplit + (size_t)drow * p.ldd + col0;   // D: optionally re-blocked rows
    // aux_out: with an activation it receives act'(v) (what the backward epilogue multiplies by),
    // without one the value itself.  aux_in: a plain multiplier.  Switches are warp-uniform.
    if (p.aux_in) {
#pragma unroll
      for (int i = 0; i < 16; ++i) { v[2 * i] *= bf16_lo(pf.aux[i]); v[2 * i + 1] *= bf16_hi(pf.aux[i]); }
    } else if (p.act == YMP_ACT_GELU_ERF) {
      if (p.aux_out) {
        float d[32];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float x8[8], v8[8], d8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) x8[e] = v[8 * j + e];
          gelu_erf_both_x8(x8, v8, d8);
#pragma unroll
          for (int e = 0; e < 8; ++e) { v[8 * j + e] = v8[e]; d[8 * j + e] = d8[e]; }
        }
        store16(p.aux_out + off, p.v32_aux, d);
        store16(p.aux_out + off + 16, p.v32_aux, d + 16);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float x8[8], v8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) x8[e] = v[8 * j + e];
          gelu_erf_x8(x8, v8);
#pragma unroll
          for (int e = 0; e < 8; ++e) v[8 * j + e] = v8[e];
        }
      }
    } else if (p.act == YMP_ACT_GELU_TANH) {
      if (p.aux_out) {
        float d[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = gelu_tanh_both(v[i], d[i]);
        store16(p.aux_out + off, p.v32_aux, d);
        store16(p.aux_out + off + 16, p.v32_aux, d + 16);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = gelu_tanh(v[i]);
      }
    } else if (p.aux_out) {
      store16(p.aux_out + off, p.v32_aux, v);
      store16(p.aux_out + off + 16, p.v32_aux, v + 16);
    }
    if constexpr (DROP) {  // bias-dropout-add: residual + dropout(x + bias)
#pragma unroll
      for (int j = 0; j < 8; ++j) drop4(ds, (uint32_t)row, (uint32_t)(col0 + 4 * j), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
    if (p.residual) {
      if (p.res_f32) {  // fp32 residual stream
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += __uint_as_float(pf.res[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) { v[2 * i] += bf16_lo(pf.res[i]); v[2 * i + 1] += bf16_hi(pf.res[i]); }
      }
    }
    if (!p.out_f32) {
      __nv_bfloat16* dp = reinterpret_cast<__nv_bfloat16*>(p.D) + doff;
      store16(dp, p.v32_d, v);
      store16(dp + 16, p.v32_d, v + 16);
    } else if (!p.accumulate) {
      float* d = reinterpret_cast<float*>(p.D) + doff;
      if (p.v32_d) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t o[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] = __float_as_uint(v[8 * j + i]);
          st_v8(d + 8 * j, o);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          reinterpret_cast<float4*>(d)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
    } else {
      float* d = reinterpret_cast<float*>(p.D) + doff;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(d + 4 * j),
                     "f"(v[4 * j]), "f"(v[4 * j + 1]), "f"(v[4 * j + 2]), "f"(v[4 * j + 3])
                     : "memory");
      }
    }
  } else {
    // ragged N tail: scalar, bounds-checked
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int col = col0 + i;
      if (col < p.N) {
        float x = v[i];
        if (p.bias) x += __bfloat162float(p.bias[col]);
        const size_t off = (size_t)row * p.ldd + col, doff = dsplit + (size_t)drow * p.ldd + col;
        if (p.aux_in) {
          x *= __bfloat162float(p.aux_in[off]);
        } else if (p.act == YMP_ACT_GELU_ERF) {
          float d; x = gelu_erf_both(x, d);
          if (p.aux_out) p.aux_out[off] = __float2bfloat16(d);
        } else if (p.act == YMP_ACT_GELU_TANH) {
          float d; x = gelu_tanh_both(x, d);
          if (p.aux_out) p.aux_out[off] = __float2bfloat16(d);
        } else if (p.aux_out) {
          p.aux_out[off] = __float2bfloat16(x);
        }
        if constexpr (DROP) {
          const uint4 w = drop_words(ds, (uint32_t)row, (uint32_t)col >> 2);
          const uint32_t wc = (col & 3) == 0 ? w.x : (col & 3) == 1 ? w.y : (col & 3) == 2 ? w.z : w.w;
          x = wc >= ds.thresh ? x * ds.scale : 0.f;
        }
        if (p.residual)
          x += p.res_f32 ? reinterpret_cast<const float*>(p.residual)[(size_t)rrow * p.ldr + col]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.residual)[(size_t)rrow * p.ldr + col]);
        if (!p.out_f32) reinterpret_cast<__nv_bfloat16*>(p.D)[doff] = __float2bfloat16(x);
        else if (!p.accumulate) reinterpret_cast<float*>(p.D)[doff] = x;
        else atomicAdd(reinterpret_cast<float*>(p.D) + doff, x);
      }
    }
  }
}

// ---------------------------------------------------------------- fused im2col A operand (patch embedding)
// One 128-row x 64-column tile of the implicit patch matrix (rows m0 .. m0+127 = 128/T consecutive patches x T frames,
// columns kb*64 .. +63 = 4 pixel rows x 16 pixels of one channel) arrives as FOUR 16-column sub-tiles of 4 KB, one per
// pixel row: every patch contributes one 5-D box {16 px, 1 row, T frames} = T rows x 32 bytes, which with
// SWIZZLE_32B is exactly T/8 shared-memory atoms of 8 rows x 32 bytes, dense (a 128-byte-swizzled box would give every
// 32-byte line its own 128-byte row: tools/tma_box_probe.cu).  Each sub-tile is the A operand of one tcgen05.mma K-step
// (K = 16) through a SWIZZLE_32B descriptor; rows past the last sample are out of range and arrive as zeros.
constexpr int IM2COL_SUB_BYTES = BM * 32;  // one 128-row x 16-column sub-tile
template <bool CTA2>
__device__ __forceinline__ void load_a_im2col(uint8_t* sa, const CUtensorMap* tma, uint64_t* bar, int m0, int kb,
                                              const GemmKParams& p) {
  const int T = p.im2col_T, c = kb >> 2, y0 = (kb & 3) * 4;
  const int pt = m0 / T;  // first patch (global index b*N + n) of the tile
  for (int i = 0; i < BM / T; ++i) {
    const int g = pt + i, b = g / p.im2col_N, n = g - b * p.im2col_N;
    const int ny = n / p.im2col_Wp, nx = n - ny * p.im2col_Wp;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint8_t* dst = sa + ks * IM2COL_SUB_BYTES + i * T * 32;
      if (CTA2) tma_load_5d_cta2(dst, tma, bar, nx * 16, ny * 16 + y0 + ks, 0, c, b);
      else tma_load_5d(dst, tma, bar, nx * 16, ny * 16 + y0 + ks, 0, c, b);
    }
  }
}
// SWIZZLE_32B K-major descriptor of sub-tile ks: 8-row atoms of 256 bytes, contiguous along M
__device__ __forceinline__ uint64_t make_smem_desc_sw32(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;                       // LBO: unused (one atom along K)
  d |= (uint64_t)((256 >> 4) & 0x3FFF) << 32;   // SBO: next 8-row group
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;                       // SWIZZLE_32B
  return d;
}

// ---------------------------------------------------------------- TMA epilogue (CTA-pair kernel)
// Every epilogue warp owns two 4 KB staging buffers [32 rows][128 B] in the SWIZZLE_128B layout of the output
// tensor maps.  A lane (= accumulator row) writes its 16-byte chunks at chunk ^ (row & 7): conflict-free for the
// row-per-lane TMEM read-out, and the bulk tensor store turns it into full 128-byte row segments in HBM - instead
// of one 32-byte sector per lane per store instruction (l1tex-bound: profiles/r01_ncu_full_summary.md).
constexpr int EPI_BUF_BYTES = 32 * 128;
constexpr int EPI_SMEM_BYTES = NUM_EPI_WARPS * 2 * EPI_BUF_BYTES;

__device__ __forceinline__ void tma_store_2d(const void* desc, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(desc)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const void* desc, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(desc)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint8_t* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// The arithmetic of epilogue_chunk for one full 32-column chunk, in place on the accumulator registers:
// pre-activation (alpha, bias), then either the whole epilogue (epilogue_post: no aux_out) or, 8 columns at a
// time, the activation together with its derivative (epilogue_act8) - keeping the two results of all 32 columns
// live at once would spill.
__device__ __forceinline__ void epilogue_pre(const GemmKParams& p, uint32_t (&r)[32], const EpiPrefetch& pf) {
  if (p.alpha != 1.0f) {
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * p.alpha);
  }
  if (p.bias) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      r[2 * i] = __float_as_uint(__uint_as_float(r[2 * i]) + bf16_lo(pf.bias[i]));
      r[2 * i + 1] = __float_as_uint(__uint_as_float(r[2 * i + 1]) + bf16_hi(pf.bias[i]));
    }
  }
}
template <bool DROP>
__device__ __forceinline__ void epilogue_post(const GemmKParams& p, uint32_t (&r)[32], const EpiPrefetch& pf, const DropState& ds,
                                              int row, int col0) {
  if (p.aux_in) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      r[2 * i] = __float_as_uint(__uint_as_float(r[2 * i]) * bf16_lo(pf.aux[i]));
      r[2 * i + 1] = __float_as_uint(__uint_as_float(r[2 * i + 1]) * bf16_hi(pf.aux[i]));
    }
  } else if (p.act == YMP_ACT_GELU_ERF) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float x8[8], v8[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x8[e] = __uint_as_float(r[8 * j + e]);
      gelu_erf_x8(x8, v8);
#pragma unroll
      for (int e = 0; e < 8; ++e) r[8 * j + e] = __float_as_uint(v8[e]);
    }
  } else if (p.act == YMP_ACT_GELU_TANH) {
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(gelu_tanh(__uint_as_float(r[i])));
  }
  if constexpr (DROP) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint4 w = drop_words(ds, (uint32_t)row, (uint32_t)(col0 >> 2) + j);
      r[4 * j] = w.x >= ds.thresh ? __float_as_uint(__uint_as_float(r[4 * j]) * ds.scale) : 0u;
      r[4 * j + 1] = w.y >= ds.thresh ? __float_as_uint(__uint_as_float(r[4 * j + 1]) * ds.scale) : 0u;
      r[4 * j + 2] = w.z >= ds.thresh ? __float_as_uint(__uint_as_float(r[4 * j + 2]) * ds.scale) : 0u;
      r[4 * j + 3] = w.w >= ds.thresh ? __float_as_uint(__uint_as_float(r[4 * j + 3]) * ds.scale) : 0u;
    }
  }
  if (p.residual) {
    if (p.res_f32) {
#pragma unroll
      for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(pf.res[i]));
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        r[2 * i] = __float_as_uint(__uint_as_float(r[2 * i]) + bf16_lo(pf.res[i]));
        r[2 * i + 1] = __float_as_uint(__uint_as_float(r[2 * i + 1]) + bf16_hi(pf.res[i]));
      }
    }
  }
}
// columns [8j, 8j+8) of a chunk: value and aux (act' or, without an activation, the value) as packed bf16
__device__ __forceinline__ void epilogue_act8(const GemmKParams& p, const uint32_t (&r)[32], const EpiPrefetch& pf, int j,
                                              uint32_t (&vo)[4], uint32_t (&ao)[4]) {
  float v[8], d[8];
  if (p.act == YMP_ACT_GELU_ERF) {
    float x8[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x8[e] = __uint_as_float(r[8 * j + e]);
    gelu_erf_both_x8(x8, v, d);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float x = __uint_as_float(r[8 * j + e]);
      if (p.act == YMP_ACT_GELU_TANH) v[e] = gelu_tanh_both(x, d[e]);
      else { v[e] = x; d[e] = x; }
    }
  }
  if (p.residual) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int i = 8 * j + e;
      v[e] += p.res_f32 ? __uint_as_float(pf.res[i]) : ((i & 1) ? bf16_hi(pf.res[i >> 1]) : bf16_lo(pf.res[i >> 1]));
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) { vo[e] = pack_bf16(v[2 * e], v[2 * e + 1]); ao[e] = pack_bf16(d[2 * e], d[2 * e + 1]); }
}
// 32 bf16 values of lane-row `lr` into 16-byte chunks [cbase, cbase+4) of its 128-byte row
__device__ __forceinline__ void stage_bf16(uint8_t* buf, int lr, int cbase, const uint32_t (&f)[32]) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    st_shared_v4(buf + lr * 128 + (((cbase + j) ^ (lr & 7)) << 4),
                 pack_bf16(__uint_as_float(f[8 * j]), __uint_as_float(f[8 * j + 1])),
                 pack_bf16(__uint_as_float(f[8 * j + 2]), __uint_as_float(f[8 * j + 3])),
                 pack_bf16(__uint_as_float(f[8 * j + 4]), __uint_as_float(f[8 * j + 5])),
                 pack_bf16(__uint_as_float(f[8 * j + 6]), __uint_as_float(f[8 * j + 7])));
}
__device__ __forceinline__ void stage_f32(uint8_t* buf, int lr, const uint32_t (&f)[32]) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(buf + lr * 128 + ((j ^ (lr & 7)) << 4), f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
}

template <int BN, bool DROP>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a,
                         const __grid_constant__ CUtensorMap tma_b, const GemmKParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int NSTAGE = Cfg::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment in the shared address space
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + NSTAGE * A_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + NSTAGE * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + NSTAGE;
  uint64_t* tfull_bar = empty_bar + NSTAGE;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int num_m = (p.M + BM - 1) / BM;
  const int num_n = (p.N + BN - 1) / BN;
  const int num_units = num_m * num_n * p.split_k;
  const int kb_total = (p.K + BK - 1) / BK;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], NUM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp_idx == 2) {
    tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp_idx == 0) {
    // ===================================================================== TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
        const int ks = u % p.split_k;
        const int t = u / p.split_k;
        const int m_blk = p.n_fast ? t / num_n : t % num_m;
        const int n_blk = p.n_fast ? t % num_n : t / num_m;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
          uint8_t* sa = smem_a + stage * A_STAGE_BYTES;
          uint8_t* sb = smem_b + stage * Cfg::B_STAGE_BYTES;
          if (p.im2col_T) {
            load_a_im2col<false>(sa, &tma_a, &full_bar[stage], m_blk * BM, kb, p);
          } else if (!p.a_mn) {
            tma_load_2d(sa, &tma_a, &full_bar[stage], kb * BK, m_blk * BM);
          } else {
#pragma unroll
            for (int c = 0; c < BM / 64; ++c)
              tma_load_2d(sa + c * (64 * BK * 2), &tma_a, &full_bar[stage], m_blk * BM + c * 64,
                          kb * BK);
          }
          if (!p.b_mn) {
            tma_load_2d(sb, &tma_b, &full_bar[stage], kb * BK, n_blk * BN);
          } else {
#pragma unroll
            for (int c = 0; c < BN / 64; ++c)
              tma_load_2d(sb + c * (64 * BK * 2), &tma_b, &full_bar[stage], n_blk * BN + c * 64,
                          kb * BK);
          }
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================================== MMA issuer
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(BM, BN, p.a_mn, p.b_mn);
      // K-major : rows of 128 B, 8-row swizzle atoms 1024 B apart (SBO); LBO unused.
      // MN-major: 64-element (128 B) MN chunks of 64 k-rows = 8192 B apart (LBO);
      //           8-k-row groups 1024 B apart (SBO).
      const uint32_t a_lbo = p.a_mn ? 64 * BK * 2 : 16, a_kstep = p.a_mn ? UMMA_K * 128 : UMMA_K * 2;
      const uint32_t b_lbo = p.b_mn ? 64 * BK * 2 : 16, b_kstep = p.b_mn ? UMMA_K * 128 : UMMA_K * 2;
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
        const int ks = u % p.split_k;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb_total, kb0 + p.kb_per_split);
        mbar_wait(&tempty_bar[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem_a + stage * A_STAGE_BYTES);
          const uint32_t sb = smem_u32(smem_b + stage * Cfg::B_STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = p.im2col_T ? make_smem_desc_sw32(sa + k * IM2COL_SUB_BYTES) : make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024);
            const uint64_t bdesc = make_smem_desc_sw128(sb + k * b_kstep, b_lbo, 1024);
            umma_bf16(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs retire
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[as]);  // accumulator complete -> epilogue
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp_idx >= 4) {
    // ===================================================================== epilogue
    const int q = warp_idx & 3;              // TMEM lane quarter this warp may access
    const int half = (warp_idx - 4) >> 2;    // which half of the BN columns
    constexpr int CHUNKS = BN / 2 / 32;
    DropState ds;   // only touched by the DROP instantiations
    if constexpr (DROP) ds = drop_state(p.drop);
    int as = 0;
    uint32_t aphase = 0;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      const int t = u / p.split_k;
      const int m_blk = p.n_fast ? t / num_n : t % num_m;
      const int n_blk = p.n_fast ? t % num_n : t / num_m;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const int row = m_blk * BM + q * 32 + lane;
#pragma unroll 1
      for (int c = 0; c < CHUNKS; ++c) {
        const int coff = half * (BN / 2) + c * 32;
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + coff), r);
        EpiPrefetch pf;
        epilogue_prefetch(p, row, n_blk * BN + coff, pf);
        tmem_ld_wait();
        if (c == CHUNKS - 1) {
          // all TMEM reads of this warp are done: hand the accumulator stage back early
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty_bar[as]);
        }
        epilogue_chunk<DROP>(p, r, row, n_blk * BN + coff, pf, ds, (size_t)(u % p.split_k) * p.d_split_stride);
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------ 2-CTA variant
// Tile 256(M) x 256(N) per CTA pair (tcgen05.mma cta_group::2): each CTA stages its own 128 rows of A
// and HALF of the B tile, so per-SM shared-memory traffic (TMA writes + MMA reads) drops from
// 192 to 128 B/clk - the 1-CTA kernel's limiter (B300_MICROARCH: smem crossbar 128 B/clk/SM) - and
// L2->SM traffic per flop drops by a third.  The leader CTA issues all MMAs; completion is multicast
// to both CTAs' mbarriers; both CTAs run their own producer and epilogue warps.
constexpr int BN2 = 256;
constexpr int B2_STAGE_BYTES = (BN2 / 2) * BK * 2;
constexpr int STAGE2_BYTES = A_STAGE_BYTES + B2_STAGE_BYTES;
// operand ring: 6 x 32 KB with the direct (register) epilogue, 5 x 32 KB + 64 KB of staging with the TMA epilogue
// (225 KB of the 227 KB per SM)
template <bool TMA_EPI> struct Pair {
  static constexpr int NSTAGE = TMA_EPI ? 5 : 6;
  static constexpr int SMEM_BYTES = NSTAGE * STAGE2_BYTES + (TMA_EPI ? EPI_SMEM_BYTES : 0) + 256 + 1024;
};

#ifdef YMP_GEMM_DBG
// [0] MMA warp: total cycles, [1] waiting for a free accumulator, [2] waiting for smem stages, [3] tiles
// [4] producer: cycles waiting for empty slots   [5] epilogue warp 4: waiting for tfull, [6] epilogue total
__device__ unsigned long long ymp_gemm_dbg_buf[16];
#define GDBG_T() clock64()
#else
#define GDBG_T() 0ll
#endif

template <bool TMA_EPI, bool DROP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tcgen05_2cta_kernel(const __grid_constant__ CUtensorMap tma_a,
                              const __grid_constant__ CUtensorMap tma_b,
                              const __grid_constant__ CUtensorMap tma_d,
                              const __grid_constant__ CUtensorMap tma_aux, const GemmKParams p) {
  constexpr int NSTAGE2 = Pair<TMA_EPI>::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + NSTAGE2 * A_STAGE_BYTES;
  uint8_t* smem_epi = smem + NSTAGE2 * STAGE2_BYTES;   // 1024-byte aligned: SWIZZLE_128B staging buffers
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_epi + (TMA_EPI ? EPI_SMEM_BYTES : 0));
  uint64_t* empty_bar = full_bar + NSTAGE2;
  uint64_t* tfull_bar = empty_bar + NSTAGE2;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  const int num_m = (p.M + 2 * BM - 1) / (2 * BM);
  const int num_n = (p.N + BN2 - 1) / BN2;
  const int num_units = num_m * num_n * p.split_k;
  const int kb_total = (p.K + BK - 1) / BK;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    if (TMA_EPI) {
      tma_prefetch_desc(&tma_d);
      if (p.aux_out) tma_prefetch_desc(&tma_aux);
    }
  }
  if (warp_idx == 1 && lane == 0) {
    for (int i = 0; i < NSTAGE2; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 2 * NUM_EPI_WARPS);  // epilogue warps of BOTH CTAs (used on the leader)
    }
    fence_mbar_init();
  }
  cluster_sync_all();
  if (warp_idx == 2) tmem_alloc_cta2<2 * BN2>(tmem_ptr);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp_idx == 0) {
    // ===================================================================== TMA producer (both CTAs)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = pair; u < num_units; u += num_pairs) {
        const int ks = u % p.split_k;
        const int t = u / p.split_k;
        const int m0 = (p.n_fast ? t / num_n : t % num_m) * 2 * BM + (int)rank * BM;
        const int n0 = (p.n_fast ? t % num_n : t / num_m) * BN2 + (int)rank * (BN2 / 2);
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
#ifdef YMP_GEMM_DBG
          const long long tw0 = GDBG_T();
#endif
          mbar_wait(&empty_bar[stage], phase ^ 1);
#ifdef YMP_GEMM_DBG
          if (blockIdx.x == 0) ymp_gemm_dbg_buf[4] += GDBG_T() - tw0;
#endif
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * STAGE2_BYTES);  // bytes of both CTAs land here
          uint8_t* sa = smem_a + stage * A_STAGE_BYTES;
          uint8_t* sb = smem_b + stage * B2_STAGE_BYTES;
          if (!p.a_mn) {
            tma_load_2d_cta2(sa, &tma_a, &full_bar[stage], kb * BK, m0);
          } else {
#pragma unroll
            for (int c = 0; c < BM / 64; ++c)
              tma_load_2d_cta2(sa + c * (64 * BK * 2), &tma_a, &full_bar[stage], m0 + c * 64, kb * BK);
          }
          if (!p.b_mn) {
            tma_load_2d_cta2(sb, &tma_b, &full_bar[stage], kb * BK, n0);
          } else {
#pragma unroll
            for (int c = 0; c < BN2 / 2 / 64; ++c)
              tma_load_2d_cta2(sb + c * (64 * BK * 2), &tma_b, &full_bar[stage], n0 + c * 64, kb * BK);
          }
          if (++stage == NSTAGE2) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================================== MMA issuer (leader CTA only)
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc_bf16(2 * BM, BN2, p.a_mn, p.b_mn);
      const uint32_t a_lbo = p.a_mn ? 64 * BK * 2 : 16, a_kstep = p.a_mn ? UMMA_K * 128 : UMMA_K * 2;
      const uint32_t b_lbo = p.b_mn ? 64 * BK * 2 : 16, b_kstep = p.b_mn ? UMMA_K * 128 : UMMA_K * 2;
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int u = pair; u < num_units; u += num_pairs) {
        const int ks = u % p.split_k;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb_total, kb0 + p.kb_per_split);
#ifdef YMP_GEMM_DBG
        const long long ta0 = GDBG_T();
#endif
        mbar_wait(&tempty_bar[as], aphase ^ 1);
        tc_fence_after();
#ifdef YMP_GEMM_DBG
        if (blockIdx.x == 0) { ymp_gemm_dbg_buf[1] += GDBG_T() - ta0; ymp_gemm_dbg_buf[3] += 1; if (ymp_gemm_dbg_buf[7] == 0) ymp_gemm_dbg_buf[7] = ta0; ymp_gemm_dbg_buf[0] = GDBG_T() - ymp_gemm_dbg_buf[7]; }
#endif
        const uint32_t tmem_d = tmem_base + as * BN2;
        for (int kb = kb0; kb < kb1; ++kb) {
#ifdef YMP_GEMM_DBG
          const long long tf0 = GDBG_T();
#endif
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
#ifdef YMP_GEMM_DBG
          if (blockIdx.x == 0) ymp_gemm_dbg_buf[2] += GDBG_T() - tf0;
#endif
          const uint32_t sa = smem_u32(smem_a + stage * A_STAGE_BYTES);
          const uint32_t sb = smem_u32(smem_b + stage * B2_STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024);
            const uint64_t bdesc = make_smem_desc_sw128(sb + k * b_kstep, b_lbo, 1024);
            umma_bf16_cta2(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit_cta2(&empty_bar[stage]);  // frees the slot in both CTAs
          if (++stage == NSTAGE2) { stage = 0; phase ^= 1; }
        }
        umma_commit_cta2(&tfull_bar[as]);  // accumulator halves complete in both CTAs
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp_idx >= 4) {
    // ===================================================================== epilogue (both CTAs)
    const int q = warp_idx & 3;
    const int half = (warp_idx - 4) >> 2;
    constexpr int CHUNKS = BN2 / 2 / 32;
    DropState ds;   // only touched by the DROP instantiations
    if constexpr (DROP) ds = drop_state(p.drop);
    int as = 0;
    uint32_t aphase = 0;
    uint32_t ebox = 0;   // running count of this warp's bulk stores (staging buffer parity)
    for (int u = pair; u < num_units; u += num_pairs) {
      const int t = u / p.split_k;
      const int m0 = (p.n_fast ? t / num_n : t % num_m) * 2 * BM + (int)rank * BM;
      const int n_blk = p.n_fast ? t % num_n : t / num_m;
#ifdef YMP_GEMM_DBG
      const long long te0 = GDBG_T();
#endif
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
#ifdef YMP_GEMM_DBG
      const long long te1 = GDBG_T();
      if (blockIdx.x == 0 && warp_idx == 4 && lane == 0) ymp_gemm_dbg_buf[5] += te1 - te0;
#endif
      const int row = m0 + q * 32 + lane;
      if constexpr (TMA_EPI) {
        // ---- outputs staged in swizzled smem, written by bulk tensor stores (one box = 32 rows x 128 bytes)
        uint8_t* ebuf = smem_epi + (warp_idx - 4) * 2 * EPI_BUF_BYTES;
        const int row0 = m0 + q * 32;
#pragma unroll 1
        for (int c = 0; c < CHUNKS; ++c) {
          const int coff = half * (BN2 / 2) + c * 32;
          const int col0 = n_blk * BN2 + coff;
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN2 + coff), r);
          EpiPrefetch pf;
          epilogue_prefetch(p, row, col0, pf);
          tmem_ld_wait();
          if (c == CHUNKS - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&tempty_bar[as], 0);  // always on the leader's barrier
          }
          epilogue_pre(p, r, pf);
          if (!p.aux_out) epilogue_post<DROP>(p, r, pf, ds, row, col0);
          if (p.out_f32) {
            // one box per chunk (32 fp32 columns = 128 bytes per row); the two buffers alternate
            uint8_t* buf = ebuf + (ebox & 1) * EPI_BUF_BYTES;
            if (lane == 0) bulk_wait_read<1>();   // the store issued two boxes ago has finished reading this buffer
            __syncwarp();
            stage_f32(buf, lane, r);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if (p.accumulate) tma_reduce_add_2d(&tma_d, buf, col0, row0);
              else tma_store_2d(&tma_d, buf, col0, row0);
              bulk_commit();
            }
            ++ebox;
          } else if (p.aux_out) {
            // two bf16 outputs (activation and act'): D through buffer 0, aux_out through buffer 1, one box each per
            // pair of chunks (64 bf16 columns = 128 bytes per row)
            if ((c & 1) == 0) {
              if (lane == 0) bulk_wait_read<0>();
              __syncwarp();
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t vo[4], ao[4];
              epilogue_act8(p, r, pf, j, vo, ao);
              const int off = lane * 128 + ((((c & 1) * 4 + j) ^ (lane & 7)) << 4);
              st_shared_v4(ebuf + off, vo[0], vo[1], vo[2], vo[3]);
              st_shared_v4(ebuf + EPI_BUF_BYTES + off, ao[0], ao[1], ao[2], ao[3]);
            }
            if (c & 1) {
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) {
                tma_store_2d(&tma_d, ebuf, col0 - 32, row0);
                tma_store_2d(&tma_aux, ebuf + EPI_BUF_BYTES, col0 - 32, row0);
                bulk_commit();
              }
            }
          } else {
            uint8_t* buf = ebuf + (ebox & 1) * EPI_BUF_BYTES;
            if ((c & 1) == 0) {
              if (lane == 0) bulk_wait_read<1>();
              __syncwarp();
            }
            stage_bf16(buf, lane, (c & 1) * 4, r);
            if (c & 1) {
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) {
                tma_store_2d(&tma_d, buf, col0 - 32, row0);
                bulk_commit();
              }
              ++ebox;
            }
          }
        }
      } else {
#pragma unroll 1
      for (int c = 0; c < CHUNKS; ++c) {
        const int coff = half * (BN2 / 2) + c * 32;
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN2 + coff), r);
        EpiPrefetch pf;
        epilogue_prefetch(p, row, n_blk * BN2 + coff, pf);
        tmem_ld_wait();
        if (c == CHUNKS - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&tempty_bar[as], 0);  // always on the leader's barrier
        }
        epilogue_chunk<DROP>(p, r, row, n_blk * BN2 + coff, pf, ds, (size_t)(u % p.split_k) * p.d_split_stride);
      }
      }
#ifdef YMP_GEMM_DBG
      if (blockIdx.x == 0 && warp_idx == 4 && lane == 0) ymp_gemm_dbg_buf[6] += GDBG_T() - te1;
#endif
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (TMA_EPI && lane == 0) bulk_wait_all();   // staged rows are read asynchronously: drain before smem goes away
  }

  tc_fence_before();
  cluster_sync_all();  // the peer may still be multicasting into our barriers / reading our smem
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc_cta2<2 * BN2>(tmem_base);
  }
}

// ------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
    else
      cudaGetLastError();
  }
  return fn;
}

// 2D bf16 tensor map: inner (contiguous) extent `inner`, `outer` rows of stride ld elements.
static int make_map(CUtensorMap* m, const void* ptr, uint64_t inner, uint64_t outer, uint64_t ld,
                    uint32_t box_inner, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(YMP_ECUDA, "cuTensorMapEncodeTiled entry point unavailable (no driver?)");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(YMP_ECUDA, "cuTensorMapEncodeTiled failed (%d): inner=%llu outer=%llu ld=%llu",
                     (int)r, (unsigned long long)inner, (unsigned long long)outer,
                     (unsigned long long)ld);
  return YMP_OK;
}

// 5D map over a bf16 video [B, C, T, H, W] for the fused im2col A operand: box {16 px, 1 row, T frames, 1, 1}, SWIZZLE_32B
static int make_video_map(CUtensorMap* m, const ymp_gemm_args* a) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(YMP_ECUDA, "cuTensorMapEncodeTiled entry point unavailable (no driver?)");
  const cuuint64_t W = a->im2col_W, H = a->im2col_H, T = a->im2col_T, C = a->im2col_C, B = a->im2col_B;
  cuuint64_t dims[5] = {W, H, T, C, B};
  cuuint64_t strides[4] = {W * 2, H * W * 2, T * H * W * 2, C * T * H * W * 2};
  cuuint32_t box[5] = {16, 1, (cuuint32_t)T, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(a->A), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(YMP_ECUDA, "cuTensorMapEncodeTiled (video, 5-D) failed (%d)", (int)r);
  return YMP_OK;
}

// 2D output tensor map (bf16 or fp32), box = 128 bytes x 32 rows, SWIZZLE_128B
static int make_out_map(CUtensorMap* m, const void* ptr, bool f32, uint64_t inner, uint64_t outer, uint64_t ld) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(YMP_ECUDA, "cuTensorMapEncodeTiled entry point unavailable (no driver?)");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {f32 ? 32u : 64u, 32u};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(YMP_ECUDA, "cuTensorMapEncodeTiled (output) failed (%d): inner=%llu outer=%llu ld=%llu", (int)r,
                     (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld);
  return YMP_OK;
}

// Split-K: D[r, c] += ws[0][r, c] + ws[1][r, c] + ... + ws[split-1][r, c], slices added in order (deterministic).
// Blocks (x, y) take rows y, y + gridDim.y, ...; 4 consecutive columns per thread (ldw, ldd are multiples of 8 and both
// bases 16-byte aligned).  D rows follow the GEMM's optional re-blocking (d_row_block / d_row_stride).
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ ws, int split, long long slice, int M,
                                                            int N, int ldw, float* __restrict__ D, int ldd, int d_row_block,
                                                            int d_row_stride) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (c >= N) return;
  for (int r = blockIdx.y; r < M; r += gridDim.y) {
    const int drow = d_row_block ? (r / d_row_block) * d_row_stride + r % d_row_block : r;
    const float* w = ws + (size_t)r * ldw + c;
    float* d = D + (size_t)drow * ldd + c;
    if (c + 4 <= N) {
      float4 s = *reinterpret_cast<const float4*>(w);
      for (int k = 1; k < split; ++k) {
        const float4 x = *reinterpret_cast<const float4*>(w + (size_t)k * slice);
        s.x += x.x; s.y += x.y; s.z += x.z; s.w += x.w;
      }
      float4 o = *reinterpret_cast<float4*>(d);
      o.x += s.x; o.y += s.y; o.z += s.z; o.w += s.w;
      *reinterpret_cast<float4*>(d) = o;
    } else {
      for (int e = 0; c + e < N; ++e) {
        float s = w[e];
        for (int k = 1; k < split; ++k) s += w[(size_t)k * slice + e];
        d[e] += s;
      }
    }
  }
}

template <int BN>
static int launch_gemm(const ymp_gemm_args* a, const GemmKParams& kp, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  CUtensorMap ta, tb;
  int rc;
  if (a->im2col_P) rc = make_video_map(&ta, a);
  else if (!a->a_mn_major) rc = make_map(&ta, a->A, a->K, a->M, a->lda, BK, BM);
  else rc = make_map(&ta, a->A, a->M, a->K, a->lda, 64, BK);
  if (rc) return rc;
  if (!a->b_mn_major) rc = make_map(&tb, a->B, a->K, a->N, a->ldb, BK, BN);
  else rc = make_map(&tb, a->B, a->N, a->K, a->ldb, 64, BK);
  if (rc) return rc;

  static DeviceOnce once;
  if (once.first()) {
    YMP_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<BN, false>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    YMP_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<BN, true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  }
  const int num_m = (a->M + BM - 1) / BM, num_n = (a->N + BN - 1) / BN;
  const int units = num_m * num_n * kp.split_k;
  const int grid = units < num_sms() ? units : num_sms();
  if (kp.has_drop) gemm_bf16_tcgen05_kernel<BN, true><<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(ta, tb, kp);
  else gemm_bf16_tcgen05_kernel<BN, false><<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(ta, tb, kp);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

static int launch_gemm_2cta(const ymp_gemm_args* a, GemmKParams kp, cudaStream_t stream) {
  CUtensorMap ta, tb, td, tx;
  int rc;
  // TMA epilogue (5 operand stages + staging) for the short-K, epilogue-bound GEMMs of the ViT (K = 768); the
  // register epilogue with 6 operand stages stays faster when the main loop dominates (measured on one box,
  // profiles/r02c_*: K >= 2048 shapes lose 5-8 % with 5 stages, K = 768 shapes gain 3-10 % from the bulk stores).
  // Conditions: plain row mapping, whole 64-column boxes, 16-byte aligned rows
  static const bool no_tma_epi = [] { const char* e = getenv("YMP_GEMM_LEGACY_EPI"); return e && e[0] == '1'; }();
  static const int tma_epi_max_k = [] { const char* e = getenv("YMP_GEMM_TMA_EPI_MAXK"); return e ? atoi(e) : 1024; }();
  const bool f32 = a->out_dtype == YMP_DT_F32;
  kp.epi_tma = (!no_tma_epi && kp.split_k == 1 && a->K <= tma_epi_max_k && a->N % 64 == 0 && a->d_row_block == 0 && (a->ldd * (f32 ? 4 : 2)) % 16 == 0 &&
                !(f32 && a->aux_out)) ? 1 : 0;
  if (kp.epi_tma) {
    rc = make_out_map(&td, a->D, f32, a->N, a->M, a->ldd);
    if (rc) return rc;
    if (a->aux_out) {
      rc = make_out_map(&tx, a->aux_out, false, a->N, a->M, a->ldd);
      if (rc) return rc;
    }
  }

  if (!a->a_mn_major) rc = make_map(&ta, a->A, a->K, a->M, a->lda, BK, BM);
  else rc = make_map(&ta, a->A, a->M, a->K, a->lda, 64, BK);
  if (rc) return rc;
  if (!a->b_mn_major) rc = make_map(&tb, a->B, a->K, a->N, a->ldb, BK, BN2 / 2);
  else rc = make_map(&tb, a->B, a->N, a->K, a->ldb, 64, BK);
  if (rc) return rc;
  static DeviceOnce once;
  if (once.first()) {
    YMP_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_2cta_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Pair<true>::SMEM_BYTES));
    YMP_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_2cta_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Pair<false>::SMEM_BYTES));
    YMP_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_2cta_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Pair<true>::SMEM_BYTES));
    YMP_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_2cta_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Pair<false>::SMEM_BYTES));
  }
  const int num_m = (a->M + 2 * BM - 1) / (2 * BM), num_n = (a->N + BN2 - 1) / BN2;
  const int units = num_m * num_n * kp.split_k;
  const int pairs = min(units, num_sms() / 2);
  if (!kp.epi_tma) {
    td = tx = ta;        // never dereferenced
    if (kp.has_drop) gemm_bf16_tcgen05_2cta_kernel<false, true><<<2 * pairs, GEMM_THREADS, Pair<false>::SMEM_BYTES, stream>>>(ta, tb, td, tx, kp);
    else gemm_bf16_tcgen05_2cta_kernel<false, false><<<2 * pairs, GEMM_THREADS, Pair<false>::SMEM_BYTES, stream>>>(ta, tb, td, tx, kp);
  } else {
    if (!a->aux_out) tx = td;
    if (kp.has_drop) gemm_bf16_tcgen05_2cta_kernel<true, true><<<2 * pairs, GEMM_THREADS, Pair<true>::SMEM_BYTES, stream>>>(ta, tb, td, tx, kp);
    else gemm_bf16_tcgen05_2cta_kernel<true, false><<<2 * pairs, GEMM_THREADS, Pair<true>::SMEM_BYTES, stream>>>(ta, tb, td, tx, kp);
  }
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

}  // namespace ymp

extern "C" int ymp_gemm(const ymp_gemm_args* a, void* stream) {
  using namespace ymp;
  YMP_CHECK_ARG(a != nullptr, "ymp_gemm: null args");
  YMP_CHECK_ARG(a->A && a->B && a->D, "ymp_gemm: null A/B/D");
  YMP_CHECK_ARG(a->M > 0 && a->N > 0 && a->K > 0, "ymp_gemm: bad shape M=%d N=%d K=%d", a->M, a->N, a->K);
  if (a->im2col_P) {
    const int P = a->im2col_P, T = a->im2col_T;
    YMP_CHECK_ARG(P == 16 && T > 0 && T % 8 == 0 && 128 % T == 0 && a->im2col_H % P == 0 && a->im2col_W % P == 0 && !a->a_mn_major,
                  "ymp_gemm(im2col): needs P = 16, T %% 8 == 0, 128 %% T == 0, H, W multiples of P (P=%d T=%d H=%d W=%d)", P, T,
                  a->im2col_H, a->im2col_W);
    const long rows = (long)a->im2col_B * (a->im2col_H / P) * (a->im2col_W / P) * T;
    YMP_CHECK_ARG(a->M == rows && a->K == a->im2col_C * P * P, "ymp_gemm(im2col): needs M = B*N*T, K = C*P*P (M=%d K=%d)", a->M, a->K);
  }
  const bool ia = a->im2col_P != 0;
  YMP_CHECK_ARG((ia || a->lda % 8 == 0) && a->ldb % 8 == 0, "ymp_gemm: lda/ldb must be multiples of 8 (lda=%d ldb=%d)", a->lda, a->ldb);
  YMP_CHECK_ARG(aligned16(a->A) && aligned16(a->B) && aligned16(a->D), "ymp_gemm: A/B/D must be 16-byte aligned");
  YMP_CHECK_ARG(ia || a->lda >= (a->a_mn_major ? a->M : a->K), "ymp_gemm: lda too small");
  YMP_CHECK_ARG(a->ldb >= (a->b_mn_major ? a->N : a->K), "ymp_gemm: ldb too small");
  YMP_CHECK_ARG(a->ldd >= a->N && a->ldd % 8 == 0, "ymp_gemm: ldd must be >= N and a multiple of 8 (ldd=%d)", a->ldd);
  YMP_CHECK_ARG(a->act >= 0 && a->act <= 2, "ymp_gemm: bad act %d", a->act);
  YMP_CHECK_ARG(!a->residual || (a->ldr >= a->N && a->ldr % 8 == 0 && aligned16(a->residual)), "ymp_gemm: bad residual ld/alignment");
  YMP_CHECK_ARG(a->residual_dtype == YMP_DT_BF16 || a->residual_dtype == YMP_DT_F32, "ymp_gemm: bad residual_dtype");
  YMP_CHECK_ARG(!a->bias || aligned16(a->bias), "ymp_gemm: bias must be 16-byte aligned");
  YMP_CHECK_ARG(!a->aux_out || aligned16(a->aux_out), "ymp_gemm: aux_out alignment");
  YMP_CHECK_ARG(!a->aux_in || aligned16(a->aux_in), "ymp_gemm: aux_in alignment");
  YMP_CHECK_ARG(!(a->accumulate && a->out_dtype != YMP_DT_F32), "ymp_gemm: accumulate needs fp32 output");
  YMP_CHECK_ARG(!(a->accumulate && (a->aux_out || a->aux_in || a->act || a->residual)),
                "ymp_gemm: accumulate mode supports only alpha and bias-free linear epilogue");
  YMP_CHECK_ARG(a->res_row_mod >= 0 && a->d_row_block >= 0 && (a->d_row_block == 0 || a->d_row_stride >= a->d_row_block),
                "ymp_gemm: bad res_row_mod / d_row_block / d_row_stride");
  YMP_CHECK_ARG(!(a->drop.rng && a->drop.p > 0.f) || (a->drop.p < 1.f && !a->aux_out && !a->accumulate),
                "ymp_gemm: dropout needs 0 < p < 1 and is not combined with aux_out / accumulate");
  YMP_CHECK_ARG(a->tile_n == 0 || a->tile_n == 128 || a->tile_n == 256 || a->tile_n == 512,
                "ymp_gemm: tile_n must be 0 (auto), 128, 256 (1-CTA tiles) or 512 (= 256x256 CTA-pair tile)");

  const int kb_total = (a->K + BK - 1) / BK;
  const int sms = num_sms();
  int bn = a->tile_n;
  if (a->im2col_P) bn = (a->N <= 128) ? 128 : 256;   // the fused-im2col producer lives in the 1-CTA kernels (one GEMM per step)
  if (bn == 0) {
    // CTA-pair 256x256 tiles when there are enough of them to fill the machine; otherwise the
    // 128x256 tile, or 128x128 when even that leaves most SMs idle or N is narrow
    const long t2 = (long)((a->M + 2 * BM - 1) / (2 * BM)) * ((a->N + 255) / 256);
    const long t256 = (long)((a->M + BM - 1) / BM) * ((a->N + 255) / 256);
    // a pair tile occupies two SMs: sms / 2 of them already fill the machine
    if (a->N >= 256 && a->M >= 256 && (t2 >= sms / 2 || (a->accumulate && a->split_k != 1))) bn = 512;
    else bn = (a->N <= 128 || (t256 < sms && a->split_k <= 1 && !a->accumulate)) ? 128 : 256;
  }
  int split = a->split_k;
  if (split <= 0) {
    split = 1;
    if (a->accumulate) {
      const long tiles = bn == 512 ? (long)((a->M + 2 * BM - 1) / (2 * BM)) * ((a->N + 255) / 256)
                                   : (long)((a->M + BM - 1) / BM) * ((a->N + bn - 1) / bn);
      // cost model (k-blocks of MMA time): waves x (k-blocks per unit + a fixed pipeline-fill / split-epilogue
      // overhead of ~24 k-blocks).  Tuned on the ViT wgrads when the slices were added with atomics:
      // 768x768x50208 was fastest at 8 splits (72 units = one wave of the 74 CTA pairs, 53 us vs 82 us at 32
      // splits), 3072x768 at 2.  With the ordered reduction through scratch, 768x768x50432 takes 46.3 us (GEMM) + 4.4 us
      // (reduction) against 49.1 us with atomics (torch.profiler, B200 at 1000 W); the split counts were not re-tuned.
      const long workers = bn == 512 ? sms / 2 : sms;
      long best = -1;
      for (int sp = 1; sp <= 64 && sp * 8 <= kb_total; ++sp) {
        const long waves = (tiles * sp + workers - 1) / workers;
        const long cost = waves * ((kb_total + sp - 1) / sp + 24);
        if (best < 0 || cost < best) { best = cost; split = sp; }
      }
    }
  }
  YMP_CHECK_ARG(split == 1 || (a->accumulate && a->out_dtype == YMP_DT_F32), "ymp_gemm: split_k>1 needs accumulate=1 and fp32 output");
  if (split > kb_total) split = kb_total;
  int per = (kb_total + split - 1) / split;
  split = (kb_total + per - 1) / per;  // no empty splits

  GemmKParams kp;
  kp.D = a->D;
  kp.bias = reinterpret_cast<const __nv_bfloat16*>(a->bias);
  kp.residual = a->residual;
  kp.res_f32 = (a->residual_dtype == YMP_DT_F32) ? 1 : 0;
  kp.aux_out = reinterpret_cast<__nv_bfloat16*>(a->aux_out);
  kp.aux_in = reinterpret_cast<const __nv_bfloat16*>(a->aux_in);
  kp.M = a->M; kp.N = a->N; kp.K = a->K;
  kp.ldd = a->ldd; kp.ldr = a->ldr;
  kp.a_mn = a->a_mn_major ? 1 : 0; kp.b_mn = a->b_mn_major ? 1 : 0;
  kp.act = a->act; kp.out_f32 = (a->out_dtype == YMP_DT_F32); kp.accumulate = a->accumulate ? 1 : 0;
  kp.split_k = split; kp.kb_per_split = per;
  kp.alpha = a->alpha;
  // keep the larger operand streaming once from HBM: the smaller one is the re-read (L2-resident) side
  kp.n_fast = ((long)a->M >= (long)a->N) ? 1 : 0;
  kp.res_row_mod = a->res_row_mod; kp.d_row_block = a->d_row_block; kp.d_row_stride = a->d_row_stride;
  kp.epi_tma = 0;
  kp.im2col_T = a->im2col_P ? a->im2col_T : 0;
  kp.im2col_Wp = a->im2col_P ? a->im2col_W / a->im2col_P : 0;
  kp.im2col_N = a->im2col_P ? (a->im2col_H / a->im2col_P) * kp.im2col_Wp : 0;
  kp.has_drop = (a->drop.rng && a->drop.p > 0.f) ? 1 : 0;
  kp.drop.rng = a->drop.rng; kp.drop.site = a->drop.site; kp.drop.p = a->drop.p;
  auto al32 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 31) == 0; };
  const int esz = kp.out_f32 ? 4 : 2;
  kp.v32_d = al32(a->D) && (a->ldd * esz) % 32 == 0;
  kp.v32_aux = (a->ldd * 2) % 32 == 0 && (!a->aux_out || al32(a->aux_out)) && (!a->aux_in || al32(a->aux_in));
  kp.v32_res = a->residual && al32(a->residual) && (a->ldr * 2) % 32 == 0;
  kp.v32_bias = a->bias && al32(a->bias);
  kp.d_split_stride = 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (split == 1) {
    if (bn == 512) return launch_gemm_2cta(a, kp, st);
    if (bn == 256) return launch_gemm<256>(a, kp, st);
    return launch_gemm<128>(a, kp, st);
  }
  // split-K: every slice stores its partial product to its own fp32 scratch matrix (no atomics), then
  // splitk_reduce_kernel adds the slices into D in slice order, so the result does not depend on scheduling
  // (the scratch rows are plain: the reduction applies D's row re-blocking)
  const int ldw = (a->N + 7) / 8 * 8;
  Scratch ws;
  int rc = ws.alloc(sizeof(float) * (size_t)split * a->M * ldw, st);
  if (rc) return rc;
  kp.D = ws.p; kp.ldd = ldw; kp.accumulate = 0;
  kp.d_row_block = 0; kp.d_row_stride = 0;
  kp.d_split_stride = (long long)a->M * ldw;
  kp.v32_d = al32(ws.p) && (ldw * 4) % 32 == 0;
  rc = bn == 512 ? launch_gemm_2cta(a, kp, st) : bn == 256 ? launch_gemm<256>(a, kp, st) : launch_gemm<128>(a, kp, st);
  if (rc) return rc;
  const int vec = (a->N + 3) / 4;
  const int tpb = vec < 256 ? (vec + 31) / 32 * 32 : 256;
  splitk_reduce_kernel<<<dim3((vec + tpb - 1) / tpb, a->M < 65535 ? a->M : 65535), tpb, 0, st>>>(
      (const float*)ws.p, split, kp.d_split_stride, a->M, a->N, ldw, (float*)a->D, a->ldd, a->d_row_block, a->d_row_stride);
  YMP_LAUNCH_CHECK();
  return ws.release();
}

#ifdef YMP_GEMM_DBG
extern "C" int ymp_gemm_dbg_read(unsigned long long* out, int reset) {
  int rc = (int)cudaMemcpyFromSymbol(out, ymp::ymp_gemm_dbg_buf, sizeof(unsigned long long) * 16);
  if (reset) {
    unsigned long long z[16] = {0};
    cudaMemcpyToSymbol(ymp::ymp_gemm_dbg_buf, z, sizeof(z));
  }
  return rc;
}
#endif
