// Fused attention (softmax(scale * Q K^T + mask) V) forward and backward.
//
// This file holds the GENERIC kernels: warp-level mma.sync (m16n8k16 bf16, fp32 accumulate) flash-style
// tiles for any sequence length and head_dim in {64, 80, 96, 128}; the score matrix never touches HBM.
// ymp_attn_fwd / ymp_attn_bwd (bottom of the file) dispatch first to the specialised kernels -
// attention_small.cu (block-diagonal sequences of <= 16 rows: TimeSformer temporal attention) and
// attention_tc.cu (tcgen05, key range <= 256, head_dim 64 / 96: ViT spatial and GPT attention) - and fall
// back to these for everything else (the abstractor's 1570-key cross attention, head_dim 80 / 128, long
// decode contexts) or when YMP_ATTN_LEGACY=1.
//   forward   : CTA = 64 query rows x (seq, head); K/V tiles streamed with cp.async double buffering
//   backward  : two kernels, no atomics, deterministic -
//               dQ   kernel: CTA = 64 query rows, streams K/V   (also emits delta = rowsum(dO*O))
//               dKdV kernel: CTA = 64 key rows,   streams Q/dO
// Sequences are addressed through ymp_seqmap, so Q/K/V are read in place from packed QKV GEMM
// outputs (ViT [3,heads,hd], GPT per-head [q|k|v], TimeSformer per-frame sequences with a shared
// cls row, abstractor cross attention).  Mask modes: none, causal, block-diagonal (packs many
// short TimeSformer temporal sequences into one 64-row tile).
#include <math_constants.h>
#include <stdlib.h>

#include "common.h"
#include "ptx.cuh"

namespace ymp {

struct SeqMap {
  int seq_div, n_prefix, prefix_per_seq;
  long outer_stride, inner_stride, pos_stride, prefix_base, prefix_stride;
};
static SeqMap to_map(const ymp_seqmap& m) {
  SeqMap r;
  r.seq_div = m.seq_div > 0 ? m.seq_div : 1;
  r.n_prefix = m.n_prefix; r.prefix_per_seq = m.prefix_per_seq;
  r.outer_stride = m.outer_stride; r.inner_stride = m.inner_stride; r.pos_stride = m.pos_stride;
  r.prefix_base = m.prefix_base; r.prefix_stride = m.prefix_stride;
  return r;
}
// A seqmap resolved for one sequence (done once per CTA: no divisions on the load path).
struct RSeq {
  long base, pos_stride, prefix0;
  int n_prefix;
};
__device__ __forceinline__ RSeq resolve(const SeqMap& m, int s) {
  const int outer = s / m.seq_div, inner = s - outer * m.seq_div;
  RSeq r;
  r.base = (long)outer * m.outer_stride + (long)inner * m.inner_stride;
  r.pos_stride = m.pos_stride;
  r.prefix0 = m.prefix_base + (long)(m.prefix_per_seq ? s : outer) * m.prefix_stride;
  r.n_prefix = m.n_prefix;
  return r;
}
__device__ __forceinline__ long rrow(const RSeq& r, int i) {
  return i < r.n_prefix ? r.prefix0 + i : r.base + (long)(i - r.n_prefix) * r.pos_stride;
}

// One operand matrix of one (sequence, head): element pointer of position i without any division
// or 64-bit multiply chain on the load path.
struct RMat {
  const __nv_bfloat16* base;    // position n_prefix (first regular row), head/column offset applied
  const __nv_bfloat16* prefix;  // position 0 when n_prefix > 0
  long stride;                  // elements between consecutive regular positions
  int ld, n_prefix;
};
__device__ __forceinline__ RMat rmat(const __nv_bfloat16* p, const RSeq& r, int ld, int col_off) {
  RMat m;
  m.base = p + r.base * ld + col_off;
  m.prefix = p + r.prefix0 * ld + col_off;
  m.stride = r.pos_stride * ld;
  m.ld = ld;
  m.n_prefix = r.n_prefix;
  return m;
}
__device__ __forceinline__ const __nv_bfloat16* mrow(const RMat& m, int i) {
  return i < m.n_prefix ? m.prefix + (long)i * m.ld : m.base + (long)(i - m.n_prefix) * m.stride;
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

constexpr int MASK_NONE = 0, MASK_CAUSAL = 1, MASK_BLOCK = 2;

struct AttnKParams {
  const __nv_bfloat16 *q, *k, *v;
  __nv_bfloat16* o;
  float* lse;
  int ldq, ldk, ldv, ldo, hsq, hsk, hsv, hso;
  SeqMap mq, mkv, mo;
  int n_seq, n_heads, s_q, s_kv, mask, mask_block;
  long total_rows;  // >0: dense packed sequences; the last one may be short
  float scale_log2, scale;
  // backward only
  const __nv_bfloat16* dout;
  __nv_bfloat16 *dq, *dk, *dv;
  float* delta;
  int lddo, hsdo, lddq, lddk, lddv, hsdq, hsdk, hsdv;
  SeqMap mdo, mdq, mdkv;
  const int* skv_dev;  // optional device scalar: number of keys that exist (KV-cache decoding under a CUDA graph)
  const int* kv_rows;  // optional device table: key j of sequence s is K/V row kv_rows[s * ld_kv_rows + j] (decode kernel only)
  int ld_kv_rows;
};

// effective lengths of sequence s (short last sequence when total_rows is set)
__device__ __forceinline__ void eff_len(const AttnKParams& p, int s, int& sq, int& skv) {
  sq = p.s_q; skv = p.s_kv;
  if (p.skv_dev) skv = min(skv, *p.skv_dev);
  if (p.total_rows > 0) {
    const long left = p.total_rows - (long)s * p.s_q;
    if (left < sq) sq = (int)left;
    if (left < skv) skv = (int)left;
  }
}
// Warp-uniform test: does this 16-row x 64-col score tile need any masking at all?
__device__ __forceinline__ bool tile_needs_mask(const AttnKParams& p, int row_lo, int col0, int skv) {
  if (col0 + 64 > skv) return true;
  if (p.mask == MASK_CAUSAL) return col0 + 63 > row_lo;
  return p.mask == MASK_BLOCK;
}
// Set masked entries of a C-fragment tile to `fill`.  rows: row_lo + g (+8), cols: col0 + nb*8 + t4*2 (+1)
__device__ __forceinline__ void apply_mask(const AttnKParams& p, float (&sc)[8][4], int row_lo, int col0, int skv,
                                           int g, int t4, float fill) {
  const int r0 = row_lo + g, r1 = r0 + 8;
  int rb0 = 0, rb1 = 0;
  if (p.mask == MASK_BLOCK) { rb0 = r0 / p.mask_block; rb1 = r1 / p.mask_block; }
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = col0 + nb * 8 + t4 * 2 + e;
      bool m0 = col >= skv, m1 = m0;
      if (p.mask == MASK_CAUSAL) { m0 |= col > r0; m1 |= col > r1; }
      else if (p.mask == MASK_BLOCK) { const int cb = col / p.mask_block; m0 |= cb != rb0; m1 |= cb != rb1; }
      if (m0) sc[nb][e] = fill;
      if (m1) sc[nb][2 + e] = fill;
    }
  }
}

// Asynchronously load a [64 x D] bf16 tile (positions r0..r0+63 of the resolved sequence).
template <int D>
__device__ __forceinline__ void load_tile_async(__nv_bfloat16* dst, const RMat& m, int r0, int n_valid) {
  constexpr int CH = D / 8, LDS = D + 8;
#pragma unroll
  for (int it = 0; it < (64 * CH + 127) / 128; ++it) {
    const int idx = threadIdx.x + it * 128;
    if ((64 * CH) % 128 != 0 && idx >= 64 * CH) break;
    const int r = idx / CH, c = idx - r * CH;
    __nv_bfloat16* d = dst + r * LDS + c * 8;
    if (r0 + r < n_valid) cp_async16(d, mrow(m, r0 + r) + c * 8);
    else *reinterpret_cast<uint4*>(d) = make_uint4(0, 0, 0, 0);
  }
}

// ------------------------------------------------------------------------------ forward
template <int D>
__global__ void __launch_bounds__(128) attn_fwd_kernel(const AttnKParams p) {
  constexpr int LDS = D + 8, KS = D / 16, TILE = 64 * LDS;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* KVs = Qs + TILE;  // [stage][K|V][TILE]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 64, h = blockIdx.y, s = blockIdx.z;
  const int g = lane >> 2, t4 = lane & 3;
  griddep_launch();   // (programmatic dependent launch in the decoding step; no-ops for an ordinary launch)
  griddep_wait();
  int sq, skv;
  eff_len(p, s, sq, skv);
  if (q0 >= sq) return;
  const RSeq mkv = resolve(p.mkv, s), mo = resolve(p.mo, s);
  const RMat Mq = rmat(p.q, resolve(p.mq, s), p.ldq, h * p.hsq);
  const RMat Mk = rmat(p.k, mkv, p.ldk, h * p.hsk), Mv = rmat(p.v, mkv, p.ldv, h * p.hsv);

  int kv_end = skv;
  if (p.mask == MASK_CAUSAL) kv_end = min(skv, q0 + 64);
  int kv_begin = 0;
  if (p.mask == MASK_BLOCK) {  // only key blocks that intersect this tile's query blocks
    kv_begin = (q0 / p.mask_block) * p.mask_block / 64 * 64;
    kv_end = min(skv, ((min(q0 + 64, sq) - 1) / p.mask_block + 1) * p.mask_block);
  }
  const int ntiles = (kv_end - kv_begin + 63) / 64;

  load_tile_async<D>(Qs, Mq, q0, sq);
  load_tile_async<D>(KVs, Mk, kv_begin, skv);
  load_tile_async<D>(KVs + TILE, Mv, kv_begin, skv);
  cp_async_commit();

  uint32_t qf[KS][4];
  float o_acc[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i) { o_acc[i][0] = o_acc[i][1] = o_acc[i][2] = o_acc[i][3] = 0.f; }
  float m_i[2] = {-CUDART_INF_F, -CUDART_INF_F}, l_i[2] = {0.f, 0.f};
  const bool warp_active = (q0 + warp * 16) < sq;

  for (int t = 0; t < ntiles; ++t) {
    const int kv0 = kv_begin + t * 64;
    __nv_bfloat16* Ks = KVs + (t & 1) * 2 * TILE;
    __nv_bfloat16* Vs = Ks + TILE;
    if (t + 1 < ntiles) {
      __nv_bfloat16* Kn = KVs + ((t + 1) & 1) * 2 * TILE;
      load_tile_async<D>(Kn, Mk, kv0 + 64, skv);
      load_tile_async<D>(Kn + TILE, Mv, kv0 + 64, skv);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (t == 0) {
#pragma unroll
      for (int kk = 0; kk < KS; ++kk)
        ldsm_x4(qf[kk], smem_u32(Qs + (warp * 16 + (lane & 15)) * LDS + kk * 16 + (lane >> 4) * 8));
    }
    if (warp_active) {
      // number of key columns of this tile this warp actually needs (warp-uniform)
      int nv = min(64, skv - kv0);
      int nb_lo = 0;  // first 16-column group this warp needs (block mask: only its own diagonal blocks)
      if (p.mask == MASK_CAUSAL) nv = min(nv, q0 + warp * 16 + 16 - kv0);
      if (p.mask == MASK_BLOCK) {
        const int r_lo = q0 + warp * 16;
        const int c_lo = (r_lo / p.mask_block) * p.mask_block, c_hi = ((r_lo + 15) / p.mask_block + 1) * p.mask_block;
        nb_lo = max(0, (c_lo - kv0) / 16);
        nv = min(nv, c_hi - kv0);
      }
      float sc[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { sc[i][0] = sc[i][1] = sc[i][2] = sc[i][3] = 0.f; }
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
#pragma unroll
        for (int nbp = 0; nbp < 4; ++nbp) {
          if (nbp * 16 < nv && nbp >= nb_lo) {
            uint32_t b[4];
            ldsm_x4(b, smem_u32(Ks + (nbp * 16 + (lane & 7) + (lane >> 4) * 8) * LDS + kk * 16 + ((lane >> 3) & 1) * 8));
            mma16816(sc[2 * nbp], qf[kk], b[0], b[1]);
            mma16816(sc[2 * nbp + 1], qf[kk], b[2], b[3]);
          }
        }
      }
      // raw scores; the softmax scale is folded into one FFMA per element below
      if (tile_needs_mask(p, q0 + warp * 16, kv0, skv))
        apply_mask(p, sc, q0 + warp * 16, kv0, skv, g, t4, -CUDART_INF_F);
      float mx[2] = {-CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
        mx[0] = fmaxf(mx[0], fmaxf(sc[nb][0], sc[nb][1]));
        mx[1] = fmaxf(mx[1], fmaxf(sc[nb][2], sc[nb][3]));
      }
      float alpha[2], ms[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        const float mnew = fmaxf(m_i[r], mx[r]);
        ms[r] = (mnew == -CUDART_INF_F) ? 0.f : mnew * p.scale_log2;
        alpha[r] = exp2f(m_i[r] * p.scale_log2 - ms[r]);
        m_i[r] = mnew;
        l_i[r] *= alpha[r];
      }
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float pv = exp2f(fmaf(sc[nb][e], p.scale_log2, -ms[e >> 1]));
          sc[nb][e] = pv;
          l_i[e >> 1] += pv;
        }
      }
#pragma unroll
      for (int i = 0; i < D / 8; ++i) {
        o_acc[i][0] *= alpha[0]; o_acc[i][1] *= alpha[0];
        o_acc[i][2] *= alpha[1]; o_acc[i][3] *= alpha[1];
      }
#pragma unroll
      for (int kk2 = 0; kk2 < 4; ++kk2) {
        if (kk2 * 16 < nv && kk2 >= nb_lo) {
          uint32_t pa[4];
          pa[0] = pack_bf16(sc[2 * kk2][0], sc[2 * kk2][1]);
          pa[1] = pack_bf16(sc[2 * kk2][2], sc[2 * kk2][3]);
          pa[2] = pack_bf16(sc[2 * kk2 + 1][0], sc[2 * kk2 + 1][1]);
          pa[3] = pack_bf16(sc[2 * kk2 + 1][2], sc[2 * kk2 + 1][3]);
#pragma unroll
          for (int dbp = 0; dbp < KS; ++dbp) {
            uint32_t b[4];
            ldsm_x4_t(b, smem_u32(Vs + (kk2 * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LDS + dbp * 16 + (lane >> 4) * 8));
            mma16816(o_acc[2 * dbp], pa, b[0], b[1]);
            mma16816(o_acc[2 * dbp + 1], pa, b[2], b[3]);
          }
        }
      }
    }
    __syncthreads();
  }
  if (!warp_active) return;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_i[r] += __shfl_xor_sync(0xffffffffu, l_i[r], 1);
    l_i[r] += __shfl_xor_sync(0xffffffffu, l_i[r], 2);
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int qi = q0 + warp * 16 + g + r * 8;
    if (qi >= sq) continue;
    const float inv = l_i[r] > 0.f ? 1.f / l_i[r] : 0.f;
    __nv_bfloat16* orow = p.o + rrow(mo, qi) * p.ldo + h * p.hso;
#pragma unroll
    for (int nb = 0; nb < D / 8; ++nb)
      *reinterpret_cast<uint32_t*>(orow + nb * 8 + t4 * 2) =
          pack_bf16(o_acc[nb][2 * r] * inv, o_acc[nb][2 * r + 1] * inv);
    if (p.lse && t4 == 0)
      p.lse[((size_t)s * p.n_heads + h) * p.s_q + qi] = m_i[r] * p.scale + logf(l_i[r]);
  }
}

// ------------------------------------------------------------------------------ backward: dQ
// Also writes delta[s,h,i] = sum_d dO[i,d] * O[i,d] for the dKdV kernel (which runs after this one).
template <int D>
__global__ void __launch_bounds__(128) attn_bwd_dq_kernel(const AttnKParams p) {
  constexpr int LDS = D + 8, KS = D / 16, TILE = 64 * LDS;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* dOs = Qs + TILE;
  __nv_bfloat16* KVs = dOs + TILE;  // [stage][K|V][TILE]
  float* stat = reinterpret_cast<float*>(KVs + 4 * TILE);  // lse(log2)[64], delta[64]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 64, h = blockIdx.y, s = blockIdx.z;
  const int g = lane >> 2, t4 = lane & 3;
  int sq, skv;
  eff_len(p, s, sq, skv);
  if (q0 >= sq) return;
  const RSeq mkv = resolve(p.mkv, s), mo = resolve(p.mo, s), mdo = resolve(p.mdo, s), mdq = resolve(p.mdq, s);
  const RMat Mq = rmat(p.q, resolve(p.mq, s), p.ldq, h * p.hsq), Mdo = rmat(p.dout, mdo, p.lddo, h * p.hsdo);
  const RMat Mk = rmat(p.k, mkv, p.ldk, h * p.hsk), Mv = rmat(p.v, mkv, p.ldv, h * p.hsv);
  int kv_end = skv, kv_begin = 0;
  if (p.mask == MASK_CAUSAL) kv_end = min(skv, q0 + 64);
  if (p.mask == MASK_BLOCK) {
    kv_begin = (q0 / p.mask_block) * p.mask_block / 64 * 64;
    kv_end = min(skv, ((min(q0 + 64, sq) - 1) / p.mask_block + 1) * p.mask_block);
  }
  const int ntiles = (kv_end - kv_begin + 63) / 64;

  load_tile_async<D>(Qs, Mq, q0, sq);
  load_tile_async<D>(dOs, Mdo, q0, sq);
  load_tile_async<D>(KVs, Mk, kv_begin, skv);
  load_tile_async<D>(KVs + TILE, Mv, kv_begin, skv);
  cp_async_commit();
  // delta / lse for this warp's 16 rows, straight from global (O is not needed anywhere else):
  // lane -> (row = lane/2, half of the head dim = lane%2), all 16-byte loads independent
  {
    const int r = lane >> 1, hf = lane & 1;
    const int qi = q0 + warp * 16 + r;
    float acc = 0.f;
    if (qi < sq) {
      const uint4* orow = reinterpret_cast<const uint4*>(p.o + rrow(mo, qi) * p.ldo + h * p.hso + hf * (D / 2));
      const uint4* drow = reinterpret_cast<const uint4*>(p.dout + rrow(mdo, qi) * p.lddo + h * p.hsdo + hf * (D / 2));
#pragma unroll
      for (int c = 0; c < D / 16; ++c) {
        const uint4 a = __ldg(orow + c), b = __ldg(drow + c);
        acc += bf16_lo(a.x) * bf16_lo(b.x) + bf16_hi(a.x) * bf16_hi(b.x) + bf16_lo(a.y) * bf16_lo(b.y) +
               bf16_hi(a.y) * bf16_hi(b.y) + bf16_lo(a.z) * bf16_lo(b.z) + bf16_hi(a.z) * bf16_hi(b.z) +
               bf16_lo(a.w) * bf16_lo(b.w) + bf16_hi(a.w) * bf16_hi(b.w);
      }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    if (hf == 0) {
      const size_t li = ((size_t)s * p.n_heads + h) * p.s_q + qi;
      stat[64 + warp * 16 + r] = acc;
      stat[warp * 16 + r] = (qi < sq) ? p.lse[li] * 1.4426950408889634f : CUDART_INF_F;
      if (qi < sq) p.delta[li] = acc;
    }
  }

  uint32_t qf[KS][4], dof[KS][4];
  float dq_acc[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i) { dq_acc[i][0] = dq_acc[i][1] = dq_acc[i][2] = dq_acc[i][3] = 0.f; }
  const bool warp_active = (q0 + warp * 16) < sq;
  float lse_r[2], del_r[2];

  for (int t = 0; t < ntiles; ++t) {
    const int kv0 = kv_begin + t * 64;
    __nv_bfloat16* Ks = KVs + (t & 1) * 2 * TILE;
    __nv_bfloat16* Vs = Ks + TILE;
    if (t + 1 < ntiles) {
      __nv_bfloat16* Kn = KVs + ((t + 1) & 1) * 2 * TILE;
      load_tile_async<D>(Kn, Mk, kv0 + 64, skv);
      load_tile_async<D>(Kn + TILE, Mv, kv0 + 64, skv);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (t == 0) {
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        const int off = (warp * 16 + (lane & 15)) * LDS + kk * 16 + (lane >> 4) * 8;
        ldsm_x4(qf[kk], smem_u32(Qs + off));
        ldsm_x4(dof[kk], smem_u32(dOs + off));
      }
      lse_r[0] = stat[warp * 16 + g]; lse_r[1] = stat[warp * 16 + g + 8];
      del_r[0] = stat[64 + warp * 16 + g]; del_r[1] = stat[64 + warp * 16 + g + 8];
    }
    if (warp_active) {
      int nv = min(64, skv - kv0);
      int nb_lo = 0;  // first 16-column group this warp needs (block mask: only its own diagonal blocks)
      if (p.mask == MASK_CAUSAL) nv = min(nv, q0 + warp * 16 + 16 - kv0);
      if (p.mask == MASK_BLOCK) {
        const int r_lo = q0 + warp * 16;
        const int c_lo = (r_lo / p.mask_block) * p.mask_block, c_hi = ((r_lo + 15) / p.mask_block + 1) * p.mask_block;
        nb_lo = max(0, (c_lo - kv0) / 16);
        nv = min(nv, c_hi - kv0);
      }
      float sc[8][4], dp[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sc[i][0] = sc[i][1] = sc[i][2] = sc[i][3] = 0.f;
        dp[i][0] = dp[i][1] = dp[i][2] = dp[i][3] = 0.f;
      }
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
#pragma unroll
        for (int nbp = 0; nbp < 4; ++nbp) {
          if (nbp * 16 < nv && nbp >= nb_lo) {
            uint32_t b[4];
            const int off = (nbp * 16 + (lane & 7) + (lane >> 4) * 8) * LDS + kk * 16 + ((lane >> 3) & 1) * 8;
            ldsm_x4(b, smem_u32(Ks + off));
            mma16816(sc[2 * nbp], qf[kk], b[0], b[1]);
            mma16816(sc[2 * nbp + 1], qf[kk], b[2], b[3]);
            ldsm_x4(b, smem_u32(Vs + off));
            mma16816(dp[2 * nbp], dof[kk], b[0], b[1]);
            mma16816(dp[2 * nbp + 1], dof[kk], b[2], b[3]);
          }
        }
      }
      if (tile_needs_mask(p, q0 + warp * 16, kv0, skv))
        apply_mask(p, sc, q0 + warp * 16, kv0, skv, g, t4, -CUDART_INF_F);  // exp2(-inf) = 0
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float pv = exp2f(fmaf(sc[nb][e], p.scale_log2, -lse_r[e >> 1]));
          sc[nb][e] = pv * (dp[nb][e] - del_r[e >> 1]);  // dS
        }
      }
#pragma unroll
      for (int kk2 = 0; kk2 < 4; ++kk2) {
        if (kk2 * 16 < nv && kk2 >= nb_lo) {
          uint32_t da[4];
          da[0] = pack_bf16(sc[2 * kk2][0], sc[2 * kk2][1]);
          da[1] = pack_bf16(sc[2 * kk2][2], sc[2 * kk2][3]);
          da[2] = pack_bf16(sc[2 * kk2 + 1][0], sc[2 * kk2 + 1][1]);
          da[3] = pack_bf16(sc[2 * kk2 + 1][2], sc[2 * kk2 + 1][3]);
#pragma unroll
          for (int dbp = 0; dbp < KS; ++dbp) {
            uint32_t b[4];
            ldsm_x4_t(b, smem_u32(Ks + (kk2 * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LDS + dbp * 16 + (lane >> 4) * 8));
            mma16816(dq_acc[2 * dbp], da, b[0], b[1]);
            mma16816(dq_acc[2 * dbp + 1], da, b[2], b[3]);
          }
        }
      }
    }
    __syncthreads();
  }
  if (!warp_active) return;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int qi = q0 + warp * 16 + g + r * 8;
    if (qi >= sq) continue;
    __nv_bfloat16* dqrow = p.dq + rrow(mdq, qi) * p.lddq + h * p.hsdq;
#pragma unroll
    for (int nb = 0; nb < D / 8; ++nb)
      *reinterpret_cast<uint32_t*>(dqrow + nb * 8 + t4 * 2) =
          pack_bf16(dq_acc[nb][2 * r] * p.scale, dq_acc[nb][2 * r + 1] * p.scale);
  }
}

// ------------------------------------------------------------------------------ backward: dK, dV
template <int D>
__global__ void __launch_bounds__(128) attn_bwd_dkdv_kernel(const AttnKParams p) {
  constexpr int LDS = D + 8, KS = D / 16, TILE = 64 * LDS;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* Vs = Ks + TILE;
  __nv_bfloat16* QDs = Vs + TILE;  // [stage][Q|dO][TILE]
  float* stat = reinterpret_cast<float*>(QDs + 4 * TILE);  // [stage][lse(log2) 64 | delta 64]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kv0 = blockIdx.x * 64, h = blockIdx.y, s = blockIdx.z;
  const int g = lane >> 2, t4 = lane & 3;
  int sq, skv;
  eff_len(p, s, sq, skv);
  if (kv0 >= skv) return;
  const RSeq mkv = resolve(p.mkv, s), mdkv = resolve(p.mdkv, s);
  const RMat Mq = rmat(p.q, resolve(p.mq, s), p.ldq, h * p.hsq), Mdo = rmat(p.dout, resolve(p.mdo, s), p.lddo, h * p.hsdo);
  const RMat Mk = rmat(p.k, mkv, p.ldk, h * p.hsk), Mv = rmat(p.v, mkv, p.ldv, h * p.hsv);
  int q_begin = 0, q_end = sq;
  if (p.mask == MASK_CAUSAL) q_begin = kv0;  // 64-aligned
  if (p.mask == MASK_BLOCK) {
    q_begin = (kv0 / p.mask_block) * p.mask_block / 64 * 64;
    q_end = min(sq, ((min(kv0 + 64, skv) - 1) / p.mask_block + 1) * p.mask_block);
  }
  const int ntiles = (q_end - q_begin + 63) / 64;
  const size_t stat_base = ((size_t)s * p.n_heads + h) * p.s_q;

  auto load_stage = [&](int stage, int qi0) {
    __nv_bfloat16* Qn = QDs + stage * 2 * TILE;
    load_tile_async<D>(Qn, Mq, qi0, sq);
    load_tile_async<D>(Qn + TILE, Mdo, qi0, sq);
    if (threadIdx.x < 64) {
      const int qi = qi0 + threadIdx.x;
      float* st = stat + stage * 128;
      st[threadIdx.x] = (qi < sq) ? p.lse[stat_base + qi] * 1.4426950408889634f : CUDART_INF_F;
      st[64 + threadIdx.x] = (qi < sq) ? p.delta[stat_base + qi] : 0.f;
    }
  };

  load_tile_async<D>(Ks, Mk, kv0, skv);
  load_tile_async<D>(Vs, Mv, kv0, skv);
  load_stage(0, q_begin);
  cp_async_commit();

  float dk_acc[D / 8][4], dv_acc[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i) {
    dk_acc[i][0] = dk_acc[i][1] = dk_acc[i][2] = dk_acc[i][3] = 0.f;
    dv_acc[i][0] = dv_acc[i][1] = dv_acc[i][2] = dv_acc[i][3] = 0.f;
  }
  const bool warp_active = (kv0 + warp * 16) < skv;

  for (int t = 0; t < ntiles; ++t) {
    const int qi0 = q_begin + t * 64;
    __nv_bfloat16* Qs = QDs + (t & 1) * 2 * TILE;
    __nv_bfloat16* dOs = Qs + TILE;
    const float* st = stat + (t & 1) * 128;
    if (t + 1 < ntiles) {
      load_stage((t + 1) & 1, qi0 + 64);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (warp_active) {
      // query columns of this tile this warp needs (warp-uniform)
      int nv = min(64, sq - qi0);
      int nb_lo = 0;  // causal: queries below the first key row of this warp contribute nothing
      if (p.mask == MASK_CAUSAL) nb_lo = max(0, (kv0 + warp * 16 - qi0) / 16);
      if (p.mask == MASK_BLOCK) {  // only the query blocks on this warp's diagonal
        const int k_lo = kv0 + warp * 16;
        const int c_lo = (k_lo / p.mask_block) * p.mask_block, c_hi = ((k_lo + 15) / p.mask_block + 1) * p.mask_block;
        nb_lo = max(0, (c_lo - qi0) / 16);
        nv = min(nv, c_hi - qi0);
      }
      float st_[8][4], dpt[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        st_[i][0] = st_[i][1] = st_[i][2] = st_[i][3] = 0.f;
        dpt[i][0] = dpt[i][1] = dpt[i][2] = dpt[i][3] = 0.f;
      }
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        uint32_t kf[4], vf[4];
        const int aoff = (warp * 16 + (lane & 15)) * LDS + kk * 16 + (lane >> 4) * 8;
        ldsm_x4(kf, smem_u32(Ks + aoff));
        ldsm_x4(vf, smem_u32(Vs + aoff));
#pragma unroll
        for (int nbp = 0; nbp < 4; ++nbp) {
          if (nbp * 16 < nv && nbp >= nb_lo) {
            uint32_t b[4];
            const int off = (nbp * 16 + (lane & 7) + (lane >> 4) * 8) * LDS + kk * 16 + ((lane >> 3) & 1) * 8;
            ldsm_x4(b, smem_u32(Qs + off));
            mma16816(st_[2 * nbp], kf, b[0], b[1]);
            mma16816(st_[2 * nbp + 1], kf, b[2], b[3]);
            ldsm_x4(b, smem_u32(dOs + off));
            mma16816(dpt[2 * nbp], vf, b[0], b[1]);
            mma16816(dpt[2 * nbp + 1], vf, b[2], b[3]);
          }
        }
      }
      {
        // transposed tile: rows are keys, columns are queries
        const int k_lo = kv0 + warp * 16;
        bool need = (k_lo + 16 > skv);
        if (p.mask == MASK_CAUSAL) need |= (k_lo + 15 > qi0);
        if (p.mask == MASK_BLOCK) need = true;
        if (need) {
          const int k0 = k_lo + g, k1 = k0 + 8;
          int kb0 = 0, kb1 = 0;
          if (p.mask == MASK_BLOCK) { kb0 = k0 / p.mask_block; kb1 = k1 / p.mask_block; }
#pragma unroll
          for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int qc = qi0 + nb * 8 + t4 * 2 + e;
              bool m0 = k0 >= skv, m1 = k1 >= skv;
              if (p.mask == MASK_CAUSAL) { m0 |= k0 > qc; m1 |= k1 > qc; }
              else if (p.mask == MASK_BLOCK) { const int qb = qc / p.mask_block; m0 |= qb != kb0; m1 |= qb != kb1; }
              if (m0) st_[nb][e] = -CUDART_INF_F;
              if (m1) st_[nb][2 + e] = -CUDART_INF_F;
            }
          }
        }
      }
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int ql = nb * 8 + t4 * 2 + (e & 1);
          const float pv = exp2f(fmaf(st_[nb][e], p.scale_log2, -st[ql]));  // lse=+inf for absent queries -> 0
          st_[nb][e] = pv;                              // P^T
          dpt[nb][e] = pv * (dpt[nb][e] - st[64 + ql]);  // dS^T
        }
      }
#pragma unroll
      for (int kk2 = 0; kk2 < 4; ++kk2) {
        if (kk2 * 16 < nv && kk2 >= nb_lo) {
          uint32_t pa[4], da[4];
          pa[0] = pack_bf16(st_[2 * kk2][0], st_[2 * kk2][1]);
          pa[1] = pack_bf16(st_[2 * kk2][2], st_[2 * kk2][3]);
          pa[2] = pack_bf16(st_[2 * kk2 + 1][0], st_[2 * kk2 + 1][1]);
          pa[3] = pack_bf16(st_[2 * kk2 + 1][2], st_[2 * kk2 + 1][3]);
          da[0] = pack_bf16(dpt[2 * kk2][0], dpt[2 * kk2][1]);
          da[1] = pack_bf16(dpt[2 * kk2][2], dpt[2 * kk2][3]);
          da[2] = pack_bf16(dpt[2 * kk2 + 1][0], dpt[2 * kk2 + 1][1]);
          da[3] = pack_bf16(dpt[2 * kk2 + 1][2], dpt[2 * kk2 + 1][3]);
#pragma unroll
          for (int dbp = 0; dbp < KS; ++dbp) {
            uint32_t b[4];
            const int off = (kk2 * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LDS + dbp * 16 + (lane >> 4) * 8;
            ldsm_x4_t(b, smem_u32(dOs + off));
            mma16816(dv_acc[2 * dbp], pa, b[0], b[1]);
            mma16816(dv_acc[2 * dbp + 1], pa, b[2], b[3]);
            ldsm_x4_t(b, smem_u32(Qs + off));
            mma16816(dk_acc[2 * dbp], da, b[0], b[1]);
            mma16816(dk_acc[2 * dbp + 1], da, b[2], b[3]);
          }
        }
      }
    }
    __syncthreads();
  }
  if (!warp_active) return;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int kvr = kv0 + warp * 16 + g + r * 8;
    if (kvr >= skv) continue;
    const long row = rrow(mdkv, kvr);
    __nv_bfloat16* dkrow = p.dk + row * p.lddk + h * p.hsdk;
    __nv_bfloat16* dvrow = p.dv + row * p.lddv + h * p.hsdv;
#pragma unroll
    for (int nb = 0; nb < D / 8; ++nb) {
      *reinterpret_cast<uint32_t*>(dkrow + nb * 8 + t4 * 2) =
          pack_bf16(dk_acc[nb][2 * r] * p.scale, dk_acc[nb][2 * r + 1] * p.scale);
      *reinterpret_cast<uint32_t*>(dvrow + nb * 8 + t4 * 2) = pack_bf16(dv_acc[nb][2 * r], dv_acc[nb][2 * r + 1]);
    }
  }
}

// ------------------------------------------------------------------------------ single-query forward (decoding)
// One query row per (sequence, head) over the KV cache: the step of sample() / beam_search()
// (models/modeling_distributed_gpt3.py:874-938).  Pure streaming: every lane owns whole keys (its D-element K and V rows
// arrive as D/8 independent 16-byte loads), keeps a private un-normalised output row in registers under a warp-uniform
// running maximum, and the 128 private rows meet once at the end through shared memory.  Nothing waits on a tile:
// one round trip to the cache per 128 keys instead of a load / mma.sync / softmax pipeline on a 64-row tile with a
// single live row.  Algorithmic bytes: 2 * s_kv * D * 2 per (sequence, head).
// TAB: keys are found through the per-sequence row table kv_rows (batched beam search: a beam reorder rewrites table
// entries, never cached rows); the arithmetic is that of the map_kv variant, key for key.
template <int D, bool TAB>
__global__ void __launch_bounds__(128) attn_decode_kernel(const AttnKParams p) {
  constexpr int CH = D / 8;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  float (*o_part)[D + 1] = reinterpret_cast<float (*)[D + 1]>(smem_attn);   // [128][D + 1]
  float* l_part = reinterpret_cast<float*>(smem_attn) + 128 * (D + 1);      // [128]
  float* m_part = l_part + 128;                                              // [4]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int h = blockIdx.x, s = blockIdx.y;
  griddep_launch();
  griddep_wait();
  const RSeq mkv = resolve(p.mkv, s);
  const RMat Mk = rmat(p.k, mkv, p.ldk, h * p.hsk), Mv = rmat(p.v, mkv, p.ldv, h * p.hsv);
  const __nv_bfloat16* qrow = p.q + rrow(resolve(p.mq, s), 0) * p.ldq + h * p.hsq;
  const int* tab = TAB ? p.kv_rows + (long)s * p.ld_kv_rows : nullptr;
  const __nv_bfloat16* kbase = p.k + h * p.hsk;
  const __nv_bfloat16* vbase = p.v + h * p.hsv;
  constexpr bool TWO_PHASE = D > 80;   // wide heads: V is requested after K has been consumed (register budget)
  uint4 qv[CH], kv[CH], vv[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) qv[c] = __ldg(reinterpret_cast<const uint4*>(qrow) + c);
  auto fetch_k = [&](int key) {
    const uint4* kr = reinterpret_cast<const uint4*>(TAB ? kbase + (long)__ldg(tab + key) * p.ldk : mrow(Mk, key));
#pragma unroll
    for (int c = 0; c < CH; ++c) kv[c] = __ldg(kr + c);
  };
  auto fetch_v = [&](int key) {
    const uint4* vr = reinterpret_cast<const uint4*>(TAB ? vbase + (long)__ldg(tab + key) * p.ldv : mrow(Mv, key));
#pragma unroll
    for (int c = 0; c < CH; ++c) vv[c] = __ldg(vr + c);
  };
  // the first 128 keys are requested before the device-side key count is known (rows < s_kv always exist in the cache
  // buffer; what lies past the count is masked below), so the count's own load is off the critical path
  if (warp * 32 + lane < p.s_kv) {
    fetch_k(warp * 32 + lane);
    if (!TWO_PHASE) fetch_v(warp * 32 + lane);
  }
  int sq, skv;
  eff_len(p, s, sq, skv);
  float o[D];
#pragma unroll
  for (int d = 0; d < D; ++d) o[d] = 0.f;
  float m_run = -CUDART_INF_F, l_run = 0.f;
  for (int k0 = 0; k0 < skv; k0 += 128) {
    const int key = k0 + warp * 32 + lane;
    const bool valid = key < skv;
    if (k0 > 0 && valid) {
      fetch_k(key);
      if (!TWO_PHASE) fetch_v(key);
    }
    float sc = -CUDART_INF_F;
    if (valid) {
      float a0 = 0.f, a1 = 0.f;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const uint32_t* qp = &qv[c].x; const uint32_t* kp = &kv[c].x;
#pragma unroll
        for (int e = 0; e < 4; ++e) { a0 = fmaf(bf16_lo(qp[e]), bf16_lo(kp[e]), a0); a1 = fmaf(bf16_hi(qp[e]), bf16_hi(kp[e]), a1); }
      }
      sc = (a0 + a1) * p.scale_log2;
    }
    if (TWO_PHASE && valid) fetch_v(key);
    const float m_new = fmaxf(m_run, warp_max(sc));   // finite: key k0 + warp*32 is valid whenever this warp has any key
    if (m_new == -CUDART_INF_F) continue;              // (a warp past the end of a short cache)
    const float corr = exp2f(m_run - m_new), pr = valid ? exp2f(sc - m_new) : 0.f;
    l_run = l_run * corr + pr;
    if (valid) {
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const uint32_t* vp = &vv[c].x;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          o[8 * c + 2 * e] = fmaf(pr, bf16_lo(vp[e]), o[8 * c + 2 * e] * corr);
          o[8 * c + 2 * e + 1] = fmaf(pr, bf16_hi(vp[e]), o[8 * c + 2 * e + 1] * corr);
        }
      }
    } else {
#pragma unroll
      for (int d = 0; d < D; ++d) o[d] *= corr;
    }
    m_run = m_new;
  }
#pragma unroll
  for (int d = 0; d < D; ++d) o_part[threadIdx.x][d] = o[d];
  l_part[threadIdx.x] = l_run;
  if (lane == 0) m_part[warp] = m_run;
  __syncthreads();
  const float m_all = fmaxf(fmaxf(m_part[0], m_part[1]), fmaxf(m_part[2], m_part[3]));
  float wgt[4];
#pragma unroll
  for (int w = 0; w < 4; ++w) wgt[w] = m_part[w] == -CUDART_INF_F ? 0.f : exp2f(m_part[w] - m_all);
  float l_all = 0.f;
  for (int r = 0; r < 128; ++r) l_all += l_part[r] * wgt[r >> 5];
  __nv_bfloat16* orow = p.o + rrow(resolve(p.mo, s), 0) * p.ldo + h * p.hso;
  for (int d = threadIdx.x; d < D; d += 128) {
    float acc = 0.f;
    for (int r = 0; r < 128; ++r) acc += o_part[r][d] * wgt[r >> 5];
    orow[d] = __float2bfloat16(acc / l_all);
  }
  if (p.lse && threadIdx.x == 0) p.lse[((long)s * p.n_heads + h) * p.s_q] = (m_all + log2f(l_all)) * 0.6931471805599453f;
}
template <int D, bool TAB>
static int launch_decode_t(const AttnKParams& p, cudaStream_t st) {
  constexpr int smem = (128 * (D + 1) + 128 + 4) * 4;
  static DeviceOnce once;
  if (once.first()) { YMP_CUDA(cudaFuncSetAttribute(attn_decode_kernel<D, TAB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); }
  launch_k(attn_decode_kernel<D, TAB>, dim3(p.n_heads, p.n_seq), dim3(128), smem, st, p);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}
template <int D>
static int launch_decode(const AttnKParams& p, cudaStream_t st) {
  return p.kv_rows ? launch_decode_t<D, true>(p, st) : launch_decode_t<D, false>(p, st);
}

static int fill_params(const ymp_attn_args* a, AttnKParams& p, const char* who) {
  YMP_CHECK_ARG(a && a->q && a->k && a->v, "%s: null q/k/v", who);
  YMP_CHECK_ARG(a->head_dim == 64 || a->head_dim == 80 || a->head_dim == 88 || a->head_dim == 96 || a->head_dim == 128,
                "%s: head_dim %d not in {64,80,88,96,128}", who, a->head_dim);
  YMP_CHECK_ARG(a->n_seq > 0 && a->n_heads > 0 && a->s_q > 0 && a->s_kv > 0, "%s: bad sizes", who);
  YMP_CHECK_ARG(a->ldq % 8 == 0 && a->ldk % 8 == 0 && a->ldv % 8 == 0 && a->ldo % 8 == 0, "%s: row strides must be multiples of 8", who);
  YMP_CHECK_ARG(a->q_head_stride % 8 == 0 && a->k_head_stride % 8 == 0 && a->v_head_stride % 8 == 0 && a->o_head_stride % 8 == 0, "%s: head strides must be multiples of 8", who);
  YMP_CHECK_ARG(aligned16(a->q) && aligned16(a->k) && aligned16(a->v), "%s: q/k/v must be 16-byte aligned", who);
  YMP_CHECK_ARG(a->mask >= 0 && a->mask <= 2, "%s: mask must be 0 (none), 1 (causal) or 2 (block-diagonal)", who);
  YMP_CHECK_ARG(a->mask == YMP_MASK_NONE || a->s_q == a->s_kv, "%s: causal / block masks need s_q == s_kv", who);
  YMP_CHECK_ARG(a->mask != YMP_MASK_BLOCK || a->mask_block > 0, "%s: block mask needs mask_block > 0", who);
  YMP_CHECK_ARG(a->total_rows == 0 || (a->s_q == a->s_kv && a->total_rows > (int64_t)(a->n_seq - 1) * a->s_q),
                "%s: total_rows needs s_q == s_kv and must reach the last sequence", who);
  p.q = (const __nv_bfloat16*)a->q; p.k = (const __nv_bfloat16*)a->k; p.v = (const __nv_bfloat16*)a->v;
  p.o = (__nv_bfloat16*)a->o; p.lse = a->lse;
  p.ldq = a->ldq; p.ldk = a->ldk; p.ldv = a->ldv; p.ldo = a->ldo;
  p.hsq = a->q_head_stride; p.hsk = a->k_head_stride; p.hsv = a->v_head_stride; p.hso = a->o_head_stride;
  p.mq = to_map(a->map_q); p.mkv = to_map(a->map_kv); p.mo = to_map(a->map_o);
  p.n_seq = a->n_seq; p.n_heads = a->n_heads; p.s_q = a->s_q; p.s_kv = a->s_kv;
  p.mask = a->mask; p.mask_block = a->mask_block > 0 ? a->mask_block : 1; p.total_rows = a->total_rows;
  p.scale = a->scale; p.scale_log2 = a->scale * 1.4426950408889634f;
  p.skv_dev = a->s_kv_dev;
  p.kv_rows = a->kv_rows; p.ld_kv_rows = a->ld_kv_rows;
  return YMP_OK;
}

template <int D>
static int launch_fwd(const AttnKParams& p, cudaStream_t st) {
  const int smem = 5 * 64 * (D + 8) * 2;
  static DeviceOnce once;
  if (once.first()) { YMP_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); }
  dim3 grid((p.s_q + 63) / 64, p.n_heads, p.n_seq);
  launch_k(attn_fwd_kernel<D>, grid, dim3(128), smem, st, p);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}
template <int D>
static int launch_bwd(const AttnKParams& p, cudaStream_t st) {
  const int smem = 6 * 64 * (D + 8) * 2 + 1024;
  static DeviceOnce once;
  if (once.first()) {
    YMP_CUDA(cudaFuncSetAttribute(attn_bwd_dq_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    YMP_CUDA(cudaFuncSetAttribute(attn_bwd_dkdv_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  attn_bwd_dq_kernel<D><<<dim3((p.s_q + 63) / 64, p.n_heads, p.n_seq), 128, smem, st>>>(p);
  YMP_LAUNCH_CHECK();
  attn_bwd_dkdv_kernel<D><<<dim3((p.s_kv + 63) / 64, p.n_heads, p.n_seq), 128, smem, st>>>(p);
  YMP_LAUNCH_CHECK();
  return YMP_OK;
}

}  // namespace ymp

namespace ymp {
int attn_tc_fwd_try(const ymp_attn_args* a, cudaStream_t st);
int attn_tc_bwd_try(const ymp_attn_bwd_args* b, cudaStream_t st);
int attn_small_fwd_try(const ymp_attn_args* a, cudaStream_t st);
int attn_small_bwd_try(const ymp_attn_bwd_args* b, cudaStream_t st);
}

static thread_local int g_attn_path = -1;
extern "C" int ymp_attn_last_path(void) { return g_attn_path; }

extern "C" int ymp_attn_fwd(const ymp_attn_args* a, void* stream) {
  using namespace ymp;
  AttnKParams p = {};
  int rc = fill_params(a, p, "ymp_attn_fwd");
  if (rc) return rc;
  YMP_CHECK_ARG(a->o && aligned16(a->o), "ymp_attn_fwd: bad o");
  cudaStream_t st = (cudaStream_t)stream;
  // short key ranges run on the tcgen05 kernel (attention_tc.cu); YMP_ATTN_LEGACY=1 forces mma.sync
  static const bool legacy = [] { const char* e = getenv("YMP_ATTN_LEGACY"); return e && e[0] == '1'; }();
  const bool dropped = a->drop.rng && a->drop.p > 0.f;
  YMP_CHECK_ARG(!dropped || a->drop.p < 1.f, "ymp_attn_fwd: dropout p must be < 1");
  const bool decode = a->s_q == 1 && a->mask == YMP_MASK_NONE && a->total_rows == 0 && !dropped && a->head_dim != 88 && a->head_dim != 128;
  YMP_CHECK_ARG(!a->kv_rows || (decode && a->ld_kv_rows >= a->s_kv),
                "ymp_attn_fwd: kv_rows needs the single-query decoding kernel (s_q == 1, mask none, no dropout, no total_rows, "
                "head_dim 64 / 80 / 96) and ld_kv_rows >= s_kv");
  if (decode && (!legacy || a->kv_rows)) {
    g_attn_path = YMP_ATTN_PATH_DECODE;   // one query row per sequence: the streaming kernel (also follows s_kv_dev)
    switch (a->head_dim) {
      case 64: return launch_decode<64>(p, st);
      case 80: return launch_decode<80>(p, st);
      default: return launch_decode<96>(p, st);
    }
  }
  const bool dev_len = a->s_kv_dev != nullptr;  // key count read on the device: the mma.sync kernels bound their KV loop by it
  YMP_CHECK_ARG(!dev_len || (!dropped && a->mask == YMP_MASK_NONE && a->total_rows == 0 && a->head_dim != 88),
                "ymp_attn_fwd: s_kv_dev needs mask none, no dropout, no total_rows, head_dim in {64,80,96,128}");
  if ((!legacy || dropped) && !dev_len) {
    if (!dropped) {
      rc = attn_small_fwd_try(a, st);  // short dense block-diagonal sequences (attention_small.cu)
      if (rc != YMP_ENOSUP) { g_attn_path = YMP_ATTN_PATH_SMALL; return rc; }
    }
    rc = attn_tc_fwd_try(a, st);
    if (rc != YMP_ENOSUP) { g_attn_path = YMP_ATTN_PATH_TCGEN05; return rc; }
  }
  if (dropped) return set_error(YMP_ENOSUP, "ymp_attn_fwd: dropout of the probabilities is implemented by the tcgen05 kernels only");
  g_attn_path = YMP_ATTN_PATH_MMA_SYNC;
  if (a->head_dim == 88) return set_error(YMP_ENOSUP, "ymp_attn_fwd: head_dim 88 is served by the tcgen05 kernels only (dense or cross attention, s_q >= 16)");
  switch (a->head_dim) {
    case 64: return launch_fwd<64>(p, st);
    case 80: return launch_fwd<80>(p, st);
    case 96: return launch_fwd<96>(p, st);
    default: return launch_fwd<128>(p, st);
  }
}

extern "C" int ymp_attn_bwd(const ymp_attn_bwd_args* b, void* stream) {
  using namespace ymp;
  YMP_CHECK_ARG(b != nullptr, "ymp_attn_bwd: null args");
  const ymp_attn_args* a = &b->fwd;
  AttnKParams p = {};
  int rc = fill_params(a, p, "ymp_attn_bwd");
  if (rc) return rc;
  YMP_CHECK_ARG(a->o && a->lse && b->dout && b->dq && b->dk && b->dv && b->delta_ws, "ymp_attn_bwd: null o/lse/dout/dq/dk/dv/delta_ws");
  YMP_CHECK_ARG(b->lddo % 8 == 0 && b->lddq % 8 == 0 && b->lddk % 8 == 0 && b->lddv % 8 == 0, "ymp_attn_bwd: grad row strides must be multiples of 8");
  YMP_CHECK_ARG(!a->s_kv_dev, "ymp_attn_bwd: s_kv_dev is forward only");
  YMP_CHECK_ARG(!a->kv_rows, "ymp_attn_bwd: kv_rows is served by the single-query decoding kernel only");
  p.dout = (const __nv_bfloat16*)b->dout; p.dq = (__nv_bfloat16*)b->dq; p.dk = (__nv_bfloat16*)b->dk; p.dv = (__nv_bfloat16*)b->dv;
  p.delta = b->delta_ws;
  p.lddo = b->lddo; p.hsdo = b->do_head_stride;
  p.lddq = b->lddq; p.lddk = b->lddk; p.lddv = b->lddv;
  p.hsdq = b->dq_head_stride; p.hsdk = b->dk_head_stride; p.hsdv = b->dv_head_stride;
  p.mdo = to_map(b->map_do); p.mdq = to_map(b->map_dq); p.mdkv = to_map(b->map_dkv);
  cudaStream_t st = (cudaStream_t)stream;
  static const bool legacy = [] { const char* e = getenv("YMP_ATTN_LEGACY"); return e && e[0] == '1'; }();
  const bool dropped = a->drop.rng && a->drop.p > 0.f;
  if (!legacy || dropped) {
    if (!dropped) {
      rc = attn_small_bwd_try(b, st);
      if (rc != YMP_ENOSUP) { g_attn_path = YMP_ATTN_PATH_SMALL; return rc; }
    }
    rc = attn_tc_bwd_try(b, st);
    if (rc != YMP_ENOSUP) { g_attn_path = YMP_ATTN_PATH_TCGEN05; return rc; }
  }
  if (dropped) return set_error(YMP_ENOSUP, "ymp_attn_bwd: dropout of the probabilities is implemented by the tcgen05 kernels only");
  g_attn_path = YMP_ATTN_PATH_MMA_SYNC;
  if (a->head_dim == 88) return set_error(YMP_ENOSUP, "ymp_attn_bwd: head_dim 88 is served by the tcgen05 kernels only");
  switch (a->head_dim) {
    case 64: return launch_bwd<64>(p, st);
    case 80: return launch_bwd<80>(p, st);
    case 96: return launch_bwd<96>(p, st);
    default: return launch_bwd<128>(p, st);
  }
}
