"""Tensor-level wrappers over the C ABI (one function per entry point of include/ymp.h).

Inputs are torch CUDA tensors used purely as device buffers; every function enqueues exactly the
kernels of one ABI call on the current stream and returns the output tensor(s).
"""
import torch

from . import lib as L
from .lib import (ACT_NONE, ACT_GELU_ERF, ACT_GELU_TANH, DT_BF16, DT_F32,  # noqa: F401
                  MASK_NONE, MASK_CAUSAL, MASK_BLOCK)

bf16 = torch.bfloat16


class Drop:
    """One dropout call site: (rng tensor {seed, offset} int64[2] on the device, site id, probability)."""
    __slots__ = ("rng", "site", "p")

    def __init__(self, rng, site, p):
        assert rng.dtype == torch.int64 and rng.numel() == 2 and rng.is_cuda
        self.rng, self.site, self.p = rng, int(site), float(p)


def _set_drop(spec, drop):
    if drop is not None and drop.p > 0.0:
        spec.rng, spec.site, spec.p = drop.rng.data_ptr(), drop.site, drop.p


def site_embed():
    return 0


def site_attn(layer):
    return 4 * layer + 1


def site_bda_attn(layer):
    return 4 * layer + 2


def site_bda_mlp(layer):
    return 4 * layer + 3


def dropout(x, drop, out=None, row0=0):
    """y = dropout(x) for a 2-D bf16 / fp32 tensor with the decoder's Philox convention (in place by default)."""
    _chk2d(x, "x")
    out = x if out is None else out
    assert out.dtype == x.dtype and out.shape == x.shape and x.dtype in (bf16, torch.float32)
    a = L.DropoutArgs()
    a.x, a.y, a.rows, a.cols, a.ldx, a.ldy = x.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1], x.stride(0), out.stride(0)
    a.dtype, a.row0 = (DT_F32 if x.dtype == torch.float32 else DT_BF16), row0
    _set_drop(a.drop, drop)
    L.call(L._dropout, a, "ymp_dropout")
    return out


def _chk2d(t, name):
    assert t.is_cuda and t.dim() == 2 and t.stride(1) == 1, f"{name}: need 2-D row-major CUDA tensor"


def gemm(a, b, *, a_t=False, b_t=False, bias=None, residual=None, act=ACT_NONE, aux_out=None,
         aux_in=None, out=None, out_dtype=bf16, accumulate=False, split_k=0, alpha=1.0, tile_n=0,
         res_row_mod=0, d_row_block=0, d_row_stride=0, drop=None, _im2col=None):
    """D[M,N] = epilogue(alpha * op(A) @ op(B)^T).

    a: [M,K] (or [K,M] when a_t)      b: [N,K] like nn.Linear.weight (or [K,N] when b_t)
    """
    _chk2d(a, "a"); _chk2d(b, "b")
    assert a.dtype == bf16 and b.dtype == bf16
    if _im2col is not None:
        P, vB, vC, vT, vH, vW = _im2col
        M, K = vB * (vH // P) * (vW // P) * vT, vC * P * P
    else:
        M, K = (a.shape[1], a.shape[0]) if a_t else (a.shape[0], a.shape[1])
    N, Kb = (b.shape[1], b.shape[0]) if b_t else (b.shape[0], b.shape[1])
    assert K == Kb, f"gemm: K mismatch {K} vs {Kb}"
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=out_dtype)
        assert not accumulate, "accumulate needs an explicit (zeroed or running) output"
    _chk2d(out, "out")
    if d_row_block:
        assert out.shape[1] == N and M % d_row_block == 0
        assert out.shape[0] >= (M // d_row_block - 1) * d_row_stride + d_row_block  # last row written
    else:
        assert out.shape == (M, N), f"gemm: out shape {tuple(out.shape)} != {(M, N)}"
    g = L.GemmArgs()
    g.A, g.B, g.D = a.data_ptr(), b.data_ptr(), out.data_ptr()
    g.M, g.N, g.K = M, N, K
    g.lda, g.ldb, g.ldd = a.stride(0), b.stride(0), out.stride(0)
    g.a_mn_major, g.b_mn_major = int(a_t), int(b_t)
    g.bias = L.ptr(bias)
    g.residual = L.ptr(residual)
    g.ldr = residual.stride(0) if residual is not None else 0
    if residual is not None:
        assert residual.dtype in (bf16, torch.float32) and residual.stride(1) == 1
        g.residual_dtype = DT_F32 if residual.dtype == torch.float32 else DT_BF16
    g.act = act
    if aux_out is not None:
        assert aux_out.dtype == bf16 and aux_out.shape == (M, N) and aux_out.stride(0) == out.stride(0)
    if aux_in is not None:
        assert aux_in.dtype == bf16 and aux_in.shape == (M, N) and aux_in.stride(0) == out.stride(0)
    g.aux_out, g.aux_in = L.ptr(aux_out), L.ptr(aux_in)
    g.out_dtype = DT_F32 if out.dtype == torch.float32 else DT_BF16
    g.accumulate = int(accumulate)
    g.split_k = split_k
    g.alpha = alpha
    g.tile_n = tile_n
    g.res_row_mod, g.d_row_block, g.d_row_stride = res_row_mod, d_row_block, d_row_stride
    _set_drop(g.drop, drop)
    if _im2col is not None:
        g.im2col_P, g.im2col_B, g.im2col_C, g.im2col_T, g.im2col_H, g.im2col_W = _im2col
    L.call(L._gemm, g, "ymp_gemm")
    return out


SKINNY_MAX_ROWS = 8        # one beam search (the captured per-sample decoding step); the fused LayerNorm stops here
SKINNY_WIDE_MAX_ROWS = 64  # a batch of beam searches


def gemm_skinny(x, w, **kw):
    """y[M, N] = act(x[M, K] @ w[N, K]^T + bias) + residual for M <= 8 rows (single-token decoding): one pass over
    the weights on the HBM-bound kernel of csrc/gemv.cu instead of a mostly empty 128-row tensor-core tile.  Row m of y
    depends on row m of x only, bit for bit, whatever M is.  Keywords:
    bias, residual, act, out, out_dtype: the epilogue and the result buffer / dtype.
    out2 [R, N] bf16 with out2_off (int64 device scalar): result row m is also written to out2 row
    m * out2_row_stride + out2_off (the KV-cache row at the device-side cache length).
    ln = (gamma, beta, eps, counter): also returns LN(y) [M, N] bf16, computed inside the same kernel by the CTA that
    finishes last (counter: uint32/int32 device scalar, zero at launch, reset by the kernel); result is then (y, ln_y)."""
    return _skinny(L._gemm_skinny, "ymp_gemm_skinny", SKINNY_MAX_ROWS, x, w, **kw)


def gemm_skinny_batch(x, w, **kw):
    """gemm_skinny for up to 64 rows (ymp_gemm_skinny_batch): the step of a batch of beam searches.  Same keywords;
    the fused LayerNorm `ln` still needs M <= 8.  Row m of the result has the bits gemm_skinny gives it."""
    return _skinny(L._gemm_skinny_batch, "ymp_gemm_skinny_batch", SKINNY_WIDE_MAX_ROWS, x, w, **kw)


def _skinny(entry, name, max_rows, x, w, *, bias=None, residual=None, act=ACT_NONE, out=None, out_dtype=bf16, out2=None,
            out2_row_stride=0, out2_off=None, ln=None):
    _chk2d(x, "x"); _chk2d(w, "w")
    assert x.dtype == bf16 and w.dtype == bf16 and x.shape[1] == w.shape[1] and x.shape[0] <= max_rows
    M, K, N = x.shape[0], x.shape[1], w.shape[0]
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=out_dtype)
    _chk2d(out, "out")
    assert out.shape == (M, N)
    a = L.GemmSkinnyArgs()
    a.x, a.w, a.bias, a.residual, a.y = x.data_ptr(), w.data_ptr(), L.ptr(bias), L.ptr(residual), out.data_ptr()
    a.M, a.N, a.K, a.ldx, a.ldw, a.ldy = M, N, K, x.stride(0), w.stride(0), out.stride(0)
    if residual is not None:
        assert residual.dtype in (bf16, torch.float32) and residual.stride(1) == 1 and residual.shape == (M, N)
        a.ldr = residual.stride(0)
        a.residual_dtype = DT_F32 if residual.dtype == torch.float32 else DT_BF16
    a.act = act
    a.out_dtype = DT_F32 if out.dtype == torch.float32 else DT_BF16
    if out2 is not None:
        _chk2d(out2, "out2")
        assert out2.dtype == bf16 and out2.shape[1] == N and out2_off.dtype == torch.int64 and out2_off.numel() == 1
        assert out2.shape[0] >= (M - 1) * out2_row_stride + 1
        a.y2, a.y2_off_dev = out2.data_ptr(), out2_off.data_ptr()
        a.ldy2, a.y2_off_stride = out2_row_stride * out2.stride(0), out2.stride(0)
    ln_out = None
    if ln is not None:
        gamma, beta, eps, counter = ln
        assert out.dtype == torch.float32 and gamma.dtype == bf16 and beta.dtype == bf16 and counter.numel() == 1
        assert counter.dtype in (torch.int32, torch.uint32) and gamma.numel() == N and beta.numel() == N
        ln_out = torch.empty((M, N), device=x.device, dtype=bf16)
        a.ln_gamma, a.ln_beta, a.ln_out, a.ln_counter = gamma.data_ptr(), beta.data_ptr(), ln_out.data_ptr(), counter.data_ptr()
        a.ld_ln, a.ln_eps = ln_out.stride(0), eps
    L.call(entry, a, name)
    return out if ln is None else (out, ln_out)


# ---------------------------------------------------------------------------------- LayerNorm
def layernorm_fwd(x, gamma, beta, eps, out=None, in_rows=None, rows=None, stats=True, out_dtype=bf16):
    """y = LN(x) row-wise (fp32 statistics); x and y may each be bf16 or fp32.  Returns (y, mean, rstd)."""
    _chk2d(x, "x")
    D = x.shape[1]
    rows = rows if rows is not None else (in_rows.numel() if in_rows is not None else x.shape[0])
    if out is None:
        out = torch.empty((rows, D), device=x.device, dtype=out_dtype)
    mean = torch.empty(rows, device=x.device, dtype=torch.float32) if stats else None
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32) if stats else None
    a = L.LayerNormArgs()
    a.x, a.gamma, a.beta, a.y = x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr()
    a.mean, a.rstd, a.in_rows = L.ptr(mean), L.ptr(rstd), L.ptr(in_rows)
    a.rows, a.D, a.ldx, a.ldy, a.eps = rows, D, x.stride(0), out.stride(0), eps
    a.x_dtype = DT_F32 if x.dtype == torch.float32 else DT_BF16
    a.y_dtype = DT_F32 if out.dtype == torch.float32 else DT_BF16
    L.call(L._ln_fwd, a, "ymp_layernorm_fwd")
    return out, mean, rstd


def layernorm_bwd(dy, x, gamma, mean, rstd, add=None, dgamma=None, dbeta=None, in_rows=None, dx=None, drop=None,
                  dx_drop=None):
    """dx (+ add) and, when dgamma/dbeta (fp32, accumulated) are given, the affine grads.  With `drop` the
    kernel also writes dx_drop = dx * mask / (1 - p) for that dropout site (returned as the second value)."""
    _chk2d(dy, "dy"); _chk2d(x, "x")
    rows, D = dy.shape
    if dx is None:
        dx = torch.empty((x.shape[0], D), device=x.device, dtype=bf16)
    assert dx.stride(0) == x.stride(0)
    a = L.LayerNormBwdArgs()
    a.dy, a.x, a.gamma, a.mean, a.rstd = dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr()
    a.add, a.dx, a.dgamma, a.dbeta, a.in_rows = L.ptr(add), dx.data_ptr(), L.ptr(dgamma), L.ptr(dbeta), L.ptr(in_rows)
    a.rows, a.D, a.ldx, a.lddy = rows, D, x.stride(0), dy.stride(0)
    a.ldadd = add.stride(0) if add is not None else 0
    a.x_dtype = DT_F32 if x.dtype == torch.float32 else DT_BF16
    assert dx.dtype == bf16 and dy.dtype == bf16
    if drop is not None and drop.p > 0.0:
        if dx_drop is None:
            dx_drop = torch.empty_like(dx) if in_rows is None else torch.zeros_like(dx)
        assert dx_drop.dtype == bf16 and dx_drop.stride(0) == dx.stride(0)
        a.dx_drop = dx_drop.data_ptr()
        _set_drop(a.drop, drop)
        L.call(L._ln_bwd, a, "ymp_layernorm_bwd")
        return dx, dx_drop
    L.call(L._ln_bwd, a, "ymp_layernorm_bwd")
    return dx


# ---------------------------------------------------------------------------------- attention
def seqmap(seq_div=1, outer_stride=0, inner_stride=0, pos_stride=1, n_prefix=0, prefix_base=0,
           prefix_stride=0, prefix_per_seq=0):
    m = L.SeqMap()
    m.seq_div, m.n_prefix, m.prefix_per_seq = seq_div, n_prefix, prefix_per_seq
    m.outer_stride, m.inner_stride, m.pos_stride = outer_stride, inner_stride, pos_stride
    m.prefix_base, m.prefix_stride = prefix_base, prefix_stride
    return m


def dense_map(S):
    return seqmap(seq_div=1, outer_stride=S, pos_stride=1)


class TView:
    """A (tensor, column offset, head stride, seqmap) view: where one of q/k/v/o lives."""
    __slots__ = ("t", "col", "hs", "m")

    def __init__(self, t, col, hs, m):
        assert t.dtype == bf16 and t.dim() == 2 and t.stride(1) == 1
        self.t, self.col, self.hs, self.m = t, col, hs, m

    @property
    def p(self):
        return self.t.data_ptr() + 2 * self.col

    @property
    def ld(self):
        return self.t.stride(0)


def _attn_args(q, k, v, o, lse, n_seq, n_heads, head_dim, s_q, s_kv, causal, scale, mask_block=0, total_rows=0, drop=None,
               s_kv_dev=None, kv_rows=None):
    a = L.AttnArgs()
    a.q, a.k, a.v, a.o, a.lse = q.p, k.p, v.p, o.p, L.ptr(lse)
    a.ldq, a.ldk, a.ldv, a.ldo = q.ld, k.ld, v.ld, o.ld
    a.q_head_stride, a.k_head_stride, a.v_head_stride, a.o_head_stride = q.hs, k.hs, v.hs, o.hs
    a.map_q, a.map_kv, a.map_o = q.m, k.m, o.m
    a.n_seq, a.n_heads, a.head_dim, a.s_q, a.s_kv = n_seq, n_heads, head_dim, s_q, s_kv
    # `causal` may be a bool or one of MASK_NONE / MASK_CAUSAL / MASK_BLOCK
    a.mask, a.mask_block, a.total_rows, a.scale = int(causal), mask_block, total_rows, scale
    _set_drop(a.drop, drop)
    if s_kv_dev is not None:
        assert s_kv_dev.dtype == torch.int32 and s_kv_dev.is_cuda and s_kv_dev.numel() == 1
        a.s_kv_dev = s_kv_dev.data_ptr()
    if kv_rows is not None:
        assert kv_rows.dtype == torch.int32 and kv_rows.is_cuda and kv_rows.dim() == 2 and kv_rows.stride(1) == 1
        assert kv_rows.shape[0] >= n_seq
        a.kv_rows, a.ld_kv_rows = kv_rows.data_ptr(), kv_rows.stride(0)
    return a


def attn_fwd(q, k, v, o, *, n_seq, n_heads, head_dim, s_q, s_kv, causal, scale, lse=None, mask_block=0,
             total_rows=0, drop=None, s_kv_dev=None, kv_rows=None):
    """q,k,v,o: TView.  Returns lse [n_seq, n_heads, s_q] fp32.  s_kv_dev: int32 device scalar, only the first
    min(s_kv, s_kv_dev) keys exist (the captured decoding step).  kv_rows: int32 device table [n_seq, >= s_kv]: key j
    of sequence s is row kv_rows[s, j] of k's and v's tensors (k.m is then unused; single-query decoding only)."""
    if lse is None:
        lse = torch.empty((n_seq, n_heads, s_q), device=q.t.device, dtype=torch.float32)
    a = _attn_args(q, k, v, o, lse, n_seq, n_heads, head_dim, s_q, s_kv, causal, scale, mask_block, total_rows, drop, s_kv_dev,
                   kv_rows)
    L.call(L._attn_fwd, a, "ymp_attn_fwd")
    return lse


def attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, *, n_seq, n_heads, head_dim, s_q, s_kv, causal, scale,
             mask_block=0, total_rows=0, drop=None):
    """dout,dq,dk,dv: TView (dk and dv share dk's seqmap)."""
    b = L.AttnBwdArgs()
    b.fwd = _attn_args(q, k, v, o, lse, n_seq, n_heads, head_dim, s_q, s_kv, causal, scale, mask_block, total_rows, drop)
    delta = torch.empty_like(lse)
    b.delta_ws = delta.data_ptr()
    b.dout, b.dq, b.dk, b.dv = dout.p, dq.p, dk.p, dv.p
    b.lddo, b.lddq, b.lddk, b.lddv = dout.ld, dq.ld, dk.ld, dv.ld
    b.do_head_stride, b.dq_head_stride, b.dk_head_stride, b.dv_head_stride = dout.hs, dq.hs, dk.hs, dv.hs
    b.map_do, b.map_dq, b.map_dkv = dout.m, dq.m, dk.m
    L.call(L._attn_bwd, b, "ymp_attn_bwd")


def temporal_pack(R, T):
    """Pack consecutive length-T sequences into <=64-row tiles: (n_seq, P) with P = (64 // T) * T."""
    P = max(1, 64 // T) * T
    return (R + P - 1) // P, P


def attn_temporal_fwd(qkv, out, *, R, n_heads, T, D, scale):
    """TimeSformer temporal attention: rows are [.., T] consecutive frames of one patch; qkv [R, 3C] in ViT
    layout [3, heads, D]; out [R, C].  Block-diagonal mask inside packed tiles.  Returns lse."""
    C = n_heads * D
    n_seq, P = temporal_pack(R, T)
    m = dense_map(P)
    q, k, v = (TView(qkv, i * C, D, m) for i in range(3))
    return attn_fwd(q, k, v, TView(out, 0, D, m), n_seq=n_seq, n_heads=n_heads, head_dim=D, s_q=P, s_kv=P,
                    causal=MASK_BLOCK, scale=scale, mask_block=T, total_rows=R)


def attn_temporal_bwd(qkv, out, lse, dout, dqkv, *, R, n_heads, T, D, scale):
    C = n_heads * D
    n_seq, P = temporal_pack(R, T)
    m = dense_map(P)
    q, k, v = (TView(qkv, i * C, D, m) for i in range(3))
    dq, dk, dv = (TView(dqkv, i * C, D, m) for i in range(3))
    attn_bwd(q, k, v, TView(out, 0, D, m), lse, TView(dout, 0, D, m), dq, dk, dv, n_seq=n_seq, n_heads=n_heads,
             head_dim=D, s_q=P, s_kv=P, causal=MASK_BLOCK, scale=scale, mask_block=T, total_rows=R)
    return dqkv


# ---------------------------------------------------------------------------------- misc
def patch_embed_gemm(video, weight2d, P, **kw):
    """Conv2d(k = stride = P, no padding) over every frame as ONE GEMM whose A operand is gathered from the video
    [B,C,T,H,W] by the TMA producer (fused im2col): rows (b, n, t), weight2d = conv_weight.flatten(1) [D, C*P*P].
    Remaining keyword arguments are those of `gemm` (bias, residual table with res_row_mod, out, ...)."""
    assert video.is_contiguous() and video.dtype == bf16 and video.dim() == 5
    B, Cc, T, H, W = video.shape
    return gemm(video.view(B * Cc * T * H, W), weight2d, _im2col=(P, B, Cc, T, H, W), **kw)


def fused_im2col_ok(T, P):
    import os
    return os.environ.get("YMP_FUSED_IM2COL", "1") != "0" and P == 16 and T % 8 == 0 and 128 % T == 0


def im2col(video, P, out=None):
    """video [B,C,T,H,W] bf16 contiguous -> [(b n t), C*P*P] (row length rounded up to 8 and zero-padded when
    C*P*P is not a multiple of 8, e.g. the 14 x 14 patches of EVA-g: returns the padded [rows, ld] tensor)."""
    assert video.is_contiguous() and video.dtype == bf16
    B, Cc, T, H, W = video.shape
    rows = B * (H // P) * (W // P) * T
    if out is None:
        out = torch.empty((rows, (Cc * P * P + 7) // 8 * 8), device=video.device, dtype=bf16)
    a = L.Im2colArgs()
    a.video, a.out = video.data_ptr(), out.data_ptr()
    a.B, a.C, a.T, a.H, a.W, a.P, a.ldo = B, Cc, T, H, W, P, out.stride(0)
    L.call(L._im2col, a, "ymp_im2col")
    return out


_CLIP_LUT = {}


def clip_lut(mean, std, device):
    """bf16 table [C*256]: lut[c*256+v] = bf16(((v / 255.) - mean[c]) / std[c]) evaluated with the reference's own
    fp32 torch ops (ClipToTensor: `clip / 255.`; normalize: `sub_(mean).div_(std)`), hence bit-exact."""
    key = (tuple(float(m) for m in mean), tuple(float(x) for x in std), str(device))
    if key not in _CLIP_LUT:
        v = torch.arange(256, dtype=torch.uint8)[None, :].repeat(len(mean), 1)      # [C, 256] uint8
        x = v / 255.
        x.sub_(torch.as_tensor(mean, dtype=x.dtype)[:, None]).div_(torch.as_tensor(std, dtype=x.dtype)[:, None])
        _CLIP_LUT[key] = x.to(bf16).reshape(-1).contiguous().to(device)
    return _CLIP_LUT[key]


def clip_normalize(frames, mean, std, out=None):
    """frames uint8 [B,T,H,W,C] (CUDA, contiguous) -> bf16 [B,C,T,H,W] = Normalize(ClipToTensor(frames))."""
    assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 5 and frames.is_contiguous()
    B, T, H, W, Cc = frames.shape
    assert len(mean) == Cc and len(std) == Cc
    if out is None:
        out = torch.empty((B, Cc, T, H, W), device=frames.device, dtype=bf16)
    a = L.ClipArgs()
    a.frames, a.out, a.lut = frames.data_ptr(), out.data_ptr(), clip_lut(mean, std, frames.device).data_ptr()
    a.B, a.T, a.H, a.W, a.C = B, T, H, W, Cc
    L.call(L._clip, a, "ymp_clip_normalize")
    return out


def embed_gather(ids, table, pos, out, S, row_offset):
    """out[(b*S + row_offset + l)] = table[ids[b,l]] + pos[row_offset + l]."""
    assert ids.dtype == torch.int64 and ids.is_contiguous()
    B, Ln = ids.shape
    a = L.EmbedArgs()
    a.ids, a.table, a.pos, a.out = ids.data_ptr(), table.data_ptr(), L.ptr(pos), out.data_ptr()
    a.B, a.L, a.S, a.row_offset = B, Ln, S, row_offset
    a.hidden, a.vocab, a.ldo = table.shape[1], table.shape[0], out.stride(0)
    a.out_dtype = DT_F32 if out.dtype == torch.float32 else DT_BF16
    L.call(L._embed, a, "ymp_embed_gather")
    return out


def ce_fwd(logits, labels):
    """Per-row losses and logsumexp (fp32) of bf16 logits [rows, V]."""
    _chk2d(logits, "logits")
    rows, V = logits.shape
    labels = labels.reshape(-1)
    assert labels.dtype == torch.int64 and labels.numel() == rows and labels.is_contiguous()
    loss = torch.empty(rows, device=logits.device, dtype=torch.float32)
    lse = torch.empty(rows, device=logits.device, dtype=torch.float32)
    a = L.CeArgs()
    a.logits, a.labels, a.loss, a.lse = logits.data_ptr(), labels.data_ptr(), loss.data_ptr(), lse.data_ptr()
    a.rows, a.V, a.ld = rows, V, logits.stride(0)
    L.call(L._ce_fwd, a, "ymp_ce_fwd")
    return loss, lse


def ce_bwd(logits, labels, lse, grad_rows, dlogits=None):
    """dlogits = grad_rows[:,None] * (softmax(logits) - onehot); in place when dlogits is None."""
    rows, V = logits.shape
    if dlogits is None:
        dlogits = logits
    labels = labels.reshape(-1)
    a = L.CeArgs()
    a.logits, a.labels, a.lse = logits.data_ptr(), labels.data_ptr(), lse.data_ptr()
    a.grad_rows, a.dlogits = grad_rows.data_ptr(), dlogits.data_ptr()
    assert grad_rows.dtype == torch.float32 and grad_rows.is_contiguous()
    a.rows, a.V, a.ld = rows, V, logits.stride(0)
    L.call(L._ce_bwd, a, "ymp_ce_bwd")
    return dlogits


def colsum(x, out):
    """out[c] (fp32, accumulated) += sum_r x[r,c]."""
    _chk2d(x, "x")
    assert out.dtype == torch.float32 and out.numel() == x.shape[1]
    a = L.ColsumArgs()
    a.in_, a.out, a.R, a.C, a.ld = x.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1], x.stride(0)
    L.call(L._colsum, a, "ymp_colsum")
    return out


def group_reduce(x, G, T, out, scale=1.0, broadcast=False):
    """broadcast=False: out[g] = scale*sum_t x[g,t];  True: out[g,t] = scale*x[g]."""
    a = L.GroupArgs()
    a.in_, a.out, a.G, a.T, a.C = x.data_ptr(), out.data_ptr(), G, T, x.shape[1]
    a.ld_in, a.ld_out, a.broadcast, a.scale = x.stride(0), out.stride(0), int(broadcast), scale
    L.call(L._group, a, "ymp_group_reduce")
    return out


# ---------------------------------------------------------------------------------- optimizer
def sumsq(g, out):
    """out (fp32 scalar tensor, accumulated) += sum(g^2)."""
    assert g.dtype == torch.float32 and g.is_contiguous()
    L.check(L._sumsq(g.data_ptr(), g.numel(), out.data_ptr(), L.cur_stream()), "ymp_sumsq")
    return out


def adamw(master, param, grad, m, v, *, step, lr, beta1, beta2, eps, weight_decay, grad_scale=1.0,
          max_grad_norm=0.0, sumsq_t=None, hyper=None, zero_grad=False):
    a = L.AdamwArgs()
    a.hyper = L.ptr(hyper)
    a.master, a.param, a.grad, a.m, a.v = master.data_ptr(), param.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr()
    a.sumsq = L.ptr(sumsq_t)
    a.n, a.step = master.numel(), step
    a.lr, a.beta1, a.beta2, a.eps, a.weight_decay = lr, beta1, beta2, eps, weight_decay
    a.grad_scale, a.max_grad_norm = grad_scale, max_grad_norm
    a.zero_grad = int(zero_grad)
    L.call(L._adamw, a, "ymp_adamw")
