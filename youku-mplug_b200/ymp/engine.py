"""Hand-scheduled forward/backward of the mPLUG-Video pre-training hot path on the C-ABI kernels.

No autograd inside: every stage saves exactly what its backward needs, weight gradients are
accumulated in fp32 (split-K slices added in a fixed order after the GEMM), and the frozen GPT-3 decoder runs
dgrad only (SURVEY.md section 2.2: no wgrad GEMMs, no saved GEMM inputs).

Weights are addressed by the reference's own state_dict keys.  `W` maps key -> bf16 CUDA tensor,
`G` maps key -> fp32 gradient accumulator for the *trainable* keys (absent key == frozen).

The residual streams (ViT x / xt / y, decoder x / x1) are kept in fp32: they are only ever read by
LayerNorm and by the GEMM epilogue's residual add, never by a tensor-core operand, and rounding them
to bf16 84 times along the depth is the dominant error term against the fp32 reference (measured on
the 1.3B config: 1.3 % -> 0.66 % relative L2 error of the logits).  Everything a GEMM consumes is bf16.

Row layouts (all activations are 2-D [rows, features]; bf16 unless noted):
  ViT tokens : row = (b*N + n)*T + t  (patch-major, as inside the reference Block,
               models/vision_transformer.py:247-274), followed by B cls rows  -> RB = B*N*T + B rows
  decoder    : row = b*S + s  (the reference uses [s,b,h]; per-(b,head) arithmetic is identical)
"""
import math

import torch

from . import lib as L
from . import ops
from .ops import ACT_GELU_ERF, ACT_GELU_TANH, TView, bf16

GPT = "text_decoder.dist_model.language_model."
VE = "visual_encoder."
AP = "attn_pool."


def _zeros_f32(n, dev):
    return torch.zeros(n, device=dev, dtype=torch.float32)


class Ctx(dict):
    """Saved activations of one forward (attribute access for brevity)."""
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


# ------------------------------------------------------------------------------------------
# linear helpers
# ------------------------------------------------------------------------------------------
def linear_wgrad(dy, x, wkey, bkey, G):
    """G[wkey] += dy^T x ; G[bkey] += colsum(dy)   (both optional / skipped when frozen)."""
    if wkey in G:
        g = G[wkey]
        ops.gemm(dy, x, a_t=True, b_t=True, out=g.view(dy.shape[1], x.shape[1]), accumulate=True)
    if bkey is not None and bkey in G:
        ops.colsum(dy, G[bkey])


def linear_dgrad(dy, w, **kw):
    """dx = dy @ w   (w is the forward [out, in] weight, consumed MN-major: no transpose copy)."""
    return ops.gemm(dy, w, b_t=True, **kw)


# ------------------------------------------------------------------------------------------
# TimeSformer encoder
# ------------------------------------------------------------------------------------------
class VitDims:
    def __init__(self, vcfg, B):
        self.P, self.D, self.depth = vcfg["patch_size"], vcfg["embed_dim"], vcfg["depth"]
        self.heads, self.T = vcfg["num_heads"], vcfg["num_frames"]
        self.hd = self.D // self.heads
        self.N = (vcfg["img_size"] // self.P) ** 2
        self.hid = int(self.D * vcfg["mlp_ratio"])
        self.B = B
        self.R = B * self.N * self.T
        self.RB = self.R + B
        self.eps = 1e-6
        self.scale = self.hd ** -0.5


_gather_cache = {}


def _final_gather_rows(d, dev):
    """Output row (b, 0)=cls, (b, 1 + t*N + n) <- internal token row (b*N + n)*T + t
    (models/vision_transformer.py:582-585 emits (t n) order after the cls token)."""
    key = (d.B, d.N, d.T, str(dev))
    if key not in _gather_cache:
        b = torch.arange(d.B).view(d.B, 1, 1)
        t = torch.arange(d.T).view(1, d.T, 1)
        n = torch.arange(d.N).view(1, 1, d.N)
        tok = ((b * d.N + n) * d.T + t).reshape(d.B, d.T * d.N)
        cls = (d.R + torch.arange(d.B)).view(d.B, 1)
        _gather_cache[key] = torch.cat([cls, tok], 1).reshape(-1).int().to(dev)
    return _gather_cache[key]


def _qkv_bias(W, pre):
    """cat(q_bias, 0, v_bias) - models/vision_transformer.py:171-175 (K has no bias)."""
    qb, vb = W[pre + "q_bias"], W[pre + "v_bias"]
    return torch.cat([qb, torch.zeros_like(vb), vb])


def _spatial_maps(d, prefix_base_in, prefix_base_out):
    m_in = ops.seqmap(seq_div=d.T, outer_stride=d.N * d.T, inner_stride=1, pos_stride=d.T, n_prefix=1,
                      prefix_base=prefix_base_in, prefix_stride=1, prefix_per_seq=0)
    m_out = ops.seqmap(seq_div=d.T, outer_stride=d.N * d.T, inner_stride=1, pos_stride=d.T, n_prefix=1,
                       prefix_base=prefix_base_out, prefix_stride=1, prefix_per_seq=1)
    return m_in, m_out


def vit_block_fwd(W, pre, x, d, save=True):
    """Block.forward - models/vision_transformer.py:243-275.  x [RB, D] -> [RB, D]."""
    R, RB, D, B, T = d.R, d.RB, d.D, d.B, d.T
    c = Ctx()
    # ---- temporal attention over the T frames of each patch
    ln_t, c.m_t, c.r_t = ops.layernorm_fwd(x[:R], W[pre + "temporal_ln.weight"], W[pre + "temporal_ln.bias"], d.eps)
    qkv_t = ops.gemm(ln_t, W[pre + "temporal_attn.qkv.weight"], bias=_qkv_bias(W, pre + "temporal_attn."))
    att_t = torch.empty((R, D), device=x.device, dtype=bf16)
    c.lse_t = ops.attn_temporal_fwd(qkv_t, att_t, R=R, n_heads=d.heads, T=T, D=d.hd, scale=d.scale)
    proj_t = ops.gemm(att_t, W[pre + "temporal_attn.proj.weight"], bias=W[pre + "temporal_attn.proj.bias"])
    xt = torch.empty((RB, D), device=x.device, dtype=torch.float32)
    ops.gemm(proj_t, W[pre + "temporal_fc.weight"], bias=W[pre + "temporal_fc.bias"], residual=x[:R], out=xt[:R])
    xt[R:].copy_(x[R:])
    # ---- spatial attention per frame, cls token shared by the T frames of a sample
    ln_s, c.m_s, c.r_s = ops.layernorm_fwd(xt, W[pre + "norm1.weight"], W[pre + "norm1.bias"], d.eps)
    qkv_s = ops.gemm(ln_s, W[pre + "attn.qkv.weight"], bias=_qkv_bias(W, pre + "attn."))
    att_s = torch.empty((RB + B * T, D), device=x.device, dtype=bf16)  # tokens | cls mean | per-frame cls
    m_in, m_out = _spatial_maps(d, R, RB)
    q, k, v = (TView(qkv_s, i * D, d.hd, m_in) for i in range(3))
    c.lse_s = ops.attn_fwd(q, k, v, TView(att_s, 0, d.hd, m_out), n_seq=B * T, n_heads=d.heads, head_dim=d.hd,
                           s_q=d.N + 1, s_kv=d.N + 1, causal=False, scale=d.scale)
    ops.group_reduce(att_s[RB:], B, T, att_s[R:RB], scale=1.0 / T)  # cls averaged over frames (:262)
    y = ops.gemm(att_s[:RB], W[pre + "attn.proj.weight"], bias=W[pre + "attn.proj.bias"], residual=xt,
                 out_dtype=torch.float32)
    # ---- MLP
    ln_m, c.m_m, c.r_m = ops.layernorm_fwd(y, W[pre + "norm2.weight"], W[pre + "norm2.bias"], d.eps)
    dact = torch.empty((RB, d.hid), device=x.device, dtype=bf16)
    h = ops.gemm(ln_m, W[pre + "mlp.fc1.weight"], bias=W[pre + "mlp.fc1.bias"], act=ACT_GELU_ERF, aux_out=dact)
    out = ops.gemm(h, W[pre + "mlp.fc2.weight"], bias=W[pre + "mlp.fc2.bias"], residual=y, out_dtype=torch.float32)
    if save:
        c.update(x=x, ln_t=ln_t, qkv_t=qkv_t, att_t=att_t, proj_t=proj_t, xt=xt, ln_s=ln_s, qkv_s=qkv_s,
                 att_s=att_s, y=y, ln_m=ln_m, dact=dact, h=h)
    return out, c


def vit_block_bwd(W, G, pre, c, dout, d):
    """Backward of vit_block_fwd: dout [RB, D] -> dx [RB, D]; accumulates the block's weight grads."""
    R, RB, D, B, T = d.R, d.RB, d.D, d.B, d.T
    dev = dout.device
    # ---- MLP
    linear_wgrad(dout, c.h, pre + "mlp.fc2.weight", pre + "mlp.fc2.bias", G)
    dpre = linear_dgrad(dout, W[pre + "mlp.fc2.weight"], act=ACT_GELU_ERF, aux_in=c.dact)
    linear_wgrad(dpre, c.ln_m, pre + "mlp.fc1.weight", pre + "mlp.fc1.bias", G)
    dln_m = linear_dgrad(dpre, W[pre + "mlp.fc1.weight"])
    dy = ops.layernorm_bwd(dln_m, c.y, W[pre + "norm2.weight"], c.m_m, c.r_m, add=dout,
                           dgamma=G.get(pre + "norm2.weight"), dbeta=G.get(pre + "norm2.bias"))
    # ---- spatial attention
    linear_wgrad(dy, c.att_s[:RB], pre + "attn.proj.weight", pre + "attn.proj.bias", G)
    datt = torch.empty((RB + B * T, D), device=dev, dtype=bf16)
    linear_dgrad(dy, W[pre + "attn.proj.weight"], out=datt[:RB])
    ops.group_reduce(datt[R:RB], B, T, datt[RB:], scale=1.0 / T, broadcast=True)
    dqkv = torch.empty((RB + B * T, 3 * D), device=dev, dtype=bf16)
    m_in, m_out = _spatial_maps(d, R, RB)
    q, k, v = (TView(c.qkv_s, i * D, d.hd, m_in) for i in range(3))
    dq, dk, dv = (TView(dqkv, i * D, d.hd, m_out) for i in range(3))
    ops.attn_bwd(q, k, v, TView(c.att_s, 0, d.hd, m_out), c.lse_s, TView(datt, 0, d.hd, m_out), dq, dk, dv,
                 n_seq=B * T, n_heads=d.heads, head_dim=d.hd, s_q=d.N + 1, s_kv=d.N + 1, causal=False, scale=d.scale)
    ops.group_reduce(dqkv[RB:], B, T, dqkv[R:RB], scale=1.0)  # the shared cls row collects all T frames
    _qkv_wgrad(G, pre + "attn.", dqkv[:RB], c.ln_s, D, dev)
    dln_s = linear_dgrad(dqkv[:RB], W[pre + "attn.qkv.weight"])
    dxt = ops.layernorm_bwd(dln_s, c.xt, W[pre + "norm1.weight"], c.m_s, c.r_s, add=dy,
                            dgamma=G.get(pre + "norm1.weight"), dbeta=G.get(pre + "norm1.bias"))
    # ---- temporal attention
    linear_wgrad(dxt[:R], c.proj_t, pre + "temporal_fc.weight", pre + "temporal_fc.bias", G)
    dproj = linear_dgrad(dxt[:R], W[pre + "temporal_fc.weight"])
    linear_wgrad(dproj, c.att_t, pre + "temporal_attn.proj.weight", pre + "temporal_attn.proj.bias", G)
    datt_t = linear_dgrad(dproj, W[pre + "temporal_attn.proj.weight"])
    dqkv_t = torch.empty((R, 3 * D), device=dev, dtype=bf16)
    ops.attn_temporal_bwd(c.qkv_t, c.att_t, c.lse_t, datt_t, dqkv_t, R=R, n_heads=d.heads, T=T, D=d.hd, scale=d.scale)
    _qkv_wgrad(G, pre + "temporal_attn.", dqkv_t, c.ln_t, D, dev)
    dln_t = linear_dgrad(dqkv_t, W[pre + "temporal_attn.qkv.weight"])
    dx = torch.empty((RB, D), device=dev, dtype=bf16)
    ops.layernorm_bwd(dln_t, c.x[:R], W[pre + "temporal_ln.weight"], c.m_t, c.r_t, add=dxt[:R],
                      dgamma=G.get(pre + "temporal_ln.weight"), dbeta=G.get(pre + "temporal_ln.bias"), dx=dx[:R])
    dx[R:].copy_(dxt[R:])
    return dx


def _qkv_wgrad(G, apre, dqkv, x, D, dev):
    linear_wgrad(dqkv, x, apre + "qkv.weight", None, G)
    # the qkv bias is cat(q_bias, 0, v_bias) (models/vision_transformer.py:171-175): only the q and the v column blocks
    # have a bias gradient, and their column sums accumulate straight into the flat gradient buffer
    if apre + "q_bias" in G:
        ops.colsum(dqkv[:, :D], G[apre + "q_bias"].view(-1))
    if apre + "v_bias" in G:
        ops.colsum(dqkv[:, 2 * D:], G[apre + "v_bias"].view(-1))


def vit_fwd(W, video, vcfg, save=True):
    """TimeSformer.forward_features - models/vision_transformer.py:544-587.
    video [B,3,T,H,W] bf16 -> image_embeds [B*(1+T*N), D] in the reference's (t n) order."""
    B = video.shape[0]
    d = VitDims(vcfg, B)
    assert video.shape[2] == d.T, f"video has {video.shape[2]} frames, model expects {d.T}"
    dev = video.device
    c = Ctx(d=d, blocks=[])
    video = video.contiguous()
    pos, temb = W[VE + "pos_embed"], W[VE + "temporal_embed"]
    table = (pos[0, 1:, None, :] + temb[0, None, :, :]).reshape(d.N * d.T, d.D).contiguous()
    x0 = torch.empty((d.RB, d.D), device=dev, dtype=torch.float32)
    wp = W[VE + "patch_embed.proj.weight"].reshape(d.D, -1)
    # PatchEmbed (:392-398) + position / temporal embedding add (:552-566) in ONE GEMM: the TMA producer gathers the
    # 16x16 patches straight from the video (fused im2col), the epilogue adds bias and the (pos + temporal) table
    fused = ops.fused_im2col_ok(d.T, d.P) and video.shape[1] * d.P * d.P % 64 == 0
    patches = None
    if fused:
        ops.patch_embed_gemm(video, wp, d.P, bias=W.get(VE + "patch_embed.proj.bias"), residual=table, res_row_mod=d.N * d.T,
                             out=x0[:d.R])
    else:   # frame counts below 8 (tiny test configs): explicit patch matrix
        patches = ops.im2col(video, d.P)
        ops.gemm(patches, wp, bias=W.get(VE + "patch_embed.proj.bias"), residual=table, res_row_mod=d.N * d.T, out=x0[:d.R])
    x0[d.R:] = (W[VE + "cls_token"][0, 0].float() + pos[0, 0].float())
    if VE + "norm_pre.weight" in W:
        x, c.m0, c.r0 = ops.layernorm_fwd(x0, W[VE + "norm_pre.weight"], W[VE + "norm_pre.bias"], d.eps,
                                          out_dtype=torch.float32)
    else:
        x = x0
    for i in range(d.depth):
        x, bc = vit_block_fwd(W, f"{VE}blocks.{i}.", x, d, save)
        c.blocks.append(bc)
    rows = _final_gather_rows(d, dev)
    out, c.mf, c.rf = ops.layernorm_fwd(x, W[VE + "norm.weight"], W[VE + "norm.bias"], d.eps, in_rows=rows)
    if save:
        c.update(patches=patches, video=video if fused else None, x0=x0, xL=x, rows=rows)
    return out, c


def vit_bwd(W, G, c, d_out):
    """d_out [B*(1+T*N), D] (grad of image_embeds) -> accumulates all encoder weight grads."""
    d = c.d
    dev = d_out.device
    dx = ops.layernorm_bwd(d_out, c.xL, W[VE + "norm.weight"], c.mf, c.rf, in_rows=c.rows,
                           dgamma=G.get(VE + "norm.weight"), dbeta=G.get(VE + "norm.bias"))
    for i in reversed(range(d.depth)):
        dx = vit_block_bwd(W, G, f"{VE}blocks.{i}.", c.blocks[i], dx, d)
        c.blocks[i] = None  # release activations as we go
        if hasattr(G, "ready"):
            G.ready(f"{VE}blocks.{i}.")  # this block's weight gradients are final: their all-reduce may start
    if VE + "norm_pre.weight" in W:
        dx0 = ops.layernorm_bwd(dx, c.x0, W[VE + "norm_pre.weight"], c.m0, c.r0,
                                dgamma=G.get(VE + "norm_pre.weight"), dbeta=G.get(VE + "norm_pre.bias"))
    else:
        dx0 = dx
    # cls_token + pos[0]
    if VE + "cls_token" in G or VE + "pos_embed" in G:
        dcls = _zeros_f32(d.D, dev)
        ops.colsum(dx0[d.R:], dcls)
        if VE + "cls_token" in G:
            G[VE + "cls_token"].view(-1).add_(dcls)
        if VE + "pos_embed" in G:
            G[VE + "pos_embed"].view(d.N + 1, d.D)[0].add_(dcls)
    # pos[1+n] + temporal[t] table: sum over the batch, then over t / n
    if VE + "pos_embed" in G or VE + "temporal_embed" in G:
        dtab = _zeros_f32(d.N * d.T * d.D, dev)
        ops.colsum(dx0[:d.R].view(d.B, d.N * d.T * d.D), dtab)
        dtab = dtab.view(d.N, d.T, d.D)
        if VE + "pos_embed" in G:
            G[VE + "pos_embed"].view(d.N + 1, d.D)[1:].add_(dtab.sum(1))
        if VE + "temporal_embed" in G:
            G[VE + "temporal_embed"].view(d.T, d.D).add_(dtab.sum(0))
    patches = c.patches
    if patches is None and VE + "patch_embed.proj.weight" in G:
        # the forward gathered its operand tiles from the video; the weight gradient (an MN-major B operand: four pixel
        # rows per 128-byte shared-memory row, which TMA boxes cannot produce from [B,C,T,H,W]) materialises the patch
        # matrix here, in the backward only
        patches = ops.im2col(c.video, d.P)
    if patches is not None:
        linear_wgrad(dx0[:d.R], patches, VE + "patch_embed.proj.weight", VE + "patch_embed.proj.bias", G)
    elif VE + "patch_embed.proj.bias" in G:
        ops.colsum(dx0[:d.R], G[VE + "patch_embed.proj.bias"])


# ------------------------------------------------------------------------------------------
# EVA image encoder (SURVEY 8f N3): plain pre-LN ViT over [cls | 16 x 16 patches of 14 x 14 pixels]
# ------------------------------------------------------------------------------------------
class EvaDims:
    def __init__(self, ecfg, B):
        self.P, self.D, self.depth, self.heads = ecfg["patch_size"], ecfg["embed_dim"], ecfg["depth"], ecfg["num_heads"]
        self.hd = self.D // self.heads
        self.N = (ecfg["img_size"] // self.P) ** 2
        self.S = self.N + 1
        self.hid = int(self.D * ecfg["mlp_ratio"])
        self.B, self.R = B, B * (self.N + 1)
        self.eps = ecfg.get("eps", 1e-6)
        self.scale = self.hd ** -0.5


def eva_fwd(W, image, ecfg, save=True):
    """EVA VisionTransformer.forward_features - models/eva_vit.py:334-350 (Block :174-181, Attention :117-145, PatchEmbed
    :200-207 with bias, final norm).  image [B,3,H,W] bf16 -> tokens [B*(1+N), D], row b*(N+1) + i, cls first."""
    B = image.shape[0]
    d = EvaDims(ecfg, B)
    dev = image.device
    c = Ctx(d=d, blocks=[])
    patches = ops.im2col(image.contiguous().unsqueeze(2), d.P)               # [B*N, Kp] (588 -> 592 zero-padded)
    Kp = patches.shape[1]
    wp = W[VE + "patch_embed.proj.weight"].reshape(d.D, -1)
    if wp.shape[1] != Kp:
        wpad = torch.zeros((d.D, Kp), device=dev, dtype=bf16)
        wpad[:, :wp.shape[1]] = wp
        wp = wpad
    pos = W[VE + "pos_embed"][0]
    x = torch.empty((d.R, d.D), device=dev, dtype=torch.float32)
    # patch rows land at b*(N+1) + 1 + n (row re-blocking), position embeddings added by the epilogue
    ops.gemm(patches, wp, bias=W[VE + "patch_embed.proj.bias"], residual=pos[1:], res_row_mod=d.N, out=x[1:], d_row_block=d.N,
             d_row_stride=d.S)
    x.view(B, d.S, d.D)[:, 0] = W[VE + "cls_token"][0, 0].float() + pos[0].float()
    m = ops.dense_map(d.S)
    for i in range(d.depth):
        pre = f"{VE}blocks.{i}."
        bc = Ctx()
        ln1, bc.m1, bc.r1 = ops.layernorm_fwd(x, W[pre + "norm1.weight"], W[pre + "norm1.bias"], d.eps)
        qkv = ops.gemm(ln1, W[pre + "attn.qkv.weight"], bias=_qkv_bias(W, pre + "attn."))
        att = torch.empty((d.R, d.D), device=dev, dtype=bf16)
        q, k, v = (TView(qkv, j * d.D, d.hd, m) for j in range(3))
        bc.lse = ops.attn_fwd(q, k, v, TView(att, 0, d.hd, m), n_seq=B, n_heads=d.heads, head_dim=d.hd, s_q=d.S, s_kv=d.S,
                              causal=False, scale=d.scale)
        x1 = ops.gemm(att, W[pre + "attn.proj.weight"], bias=W[pre + "attn.proj.bias"], residual=x, out_dtype=torch.float32)
        ln2, bc.m2, bc.r2 = ops.layernorm_fwd(x1, W[pre + "norm2.weight"], W[pre + "norm2.bias"], d.eps)
        dact = torch.empty((d.R, d.hid), device=dev, dtype=bf16)
        h = ops.gemm(ln2, W[pre + "mlp.fc1.weight"], bias=W[pre + "mlp.fc1.bias"], act=ACT_GELU_ERF, aux_out=dact)
        xn = ops.gemm(h, W[pre + "mlp.fc2.weight"], bias=W[pre + "mlp.fc2.bias"], residual=x1, out_dtype=torch.float32)
        if save:
            bc.update(x=x, ln1=ln1, qkv=qkv, att=att, x1=x1, ln2=ln2, dact=dact, h=h)
        c.blocks.append(bc)
        x = xn
    out, c.mf, c.rf = ops.layernorm_fwd(x, W[VE + "norm.weight"], W[VE + "norm.bias"], d.eps)
    if save:
        c.update(patches=patches, xL=x, Kp=Kp)
    return out, c


def eva_bwd(W, G, c, d_out):
    """d_out [B*(1+N), D] -> accumulates every encoder weight gradient."""
    d = c.d
    dev = d_out.device
    B = d.B
    m = ops.dense_map(d.S)
    dx = ops.layernorm_bwd(d_out, c.xL, W[VE + "norm.weight"], c.mf, c.rf, dgamma=G.get(VE + "norm.weight"), dbeta=G.get(VE + "norm.bias"))
    for i in reversed(range(d.depth)):
        pre, bc = f"{VE}blocks.{i}.", c.blocks[i]
        linear_wgrad(dx, bc.h, pre + "mlp.fc2.weight", pre + "mlp.fc2.bias", G)
        dpre = linear_dgrad(dx, W[pre + "mlp.fc2.weight"], act=ACT_GELU_ERF, aux_in=bc.dact)
        linear_wgrad(dpre, bc.ln2, pre + "mlp.fc1.weight", pre + "mlp.fc1.bias", G)
        dln2 = linear_dgrad(dpre, W[pre + "mlp.fc1.weight"])
        dx1 = ops.layernorm_bwd(dln2, bc.x1, W[pre + "norm2.weight"], bc.m2, bc.r2, add=dx,
                                dgamma=G.get(pre + "norm2.weight"), dbeta=G.get(pre + "norm2.bias"))
        linear_wgrad(dx1, bc.att, pre + "attn.proj.weight", pre + "attn.proj.bias", G)
        datt = linear_dgrad(dx1, W[pre + "attn.proj.weight"])
        dqkv = torch.empty_like(bc.qkv)
        q, k, v = (TView(bc.qkv, j * d.D, d.hd, m) for j in range(3))
        dq, dk, dv = (TView(dqkv, j * d.D, d.hd, m) for j in range(3))
        ops.attn_bwd(q, k, v, TView(bc.att, 0, d.hd, m), bc.lse, TView(datt, 0, d.hd, m), dq, dk, dv, n_seq=B, n_heads=d.heads,
                     head_dim=d.hd, s_q=d.S, s_kv=d.S, causal=False, scale=d.scale)
        _qkv_wgrad(G, pre + "attn.", dqkv, bc.ln1, d.D, dev)
        dln1 = linear_dgrad(dqkv, W[pre + "attn.qkv.weight"])
        dx = ops.layernorm_bwd(dln1, bc.x, W[pre + "norm1.weight"], bc.m1, bc.r1, add=dx1,
                               dgamma=G.get(pre + "norm1.weight"), dbeta=G.get(pre + "norm1.bias"))
        c.blocks[i] = None
    dx3 = dx.view(B, d.S, d.D)
    if VE + "cls_token" in G:
        G[VE + "cls_token"].view(-1).add_(dx3[:, 0].float().sum(0))
    if VE + "pos_embed" in G:
        G[VE + "pos_embed"].view(d.S, d.D).add_(dx3.float().sum(0))
    dpatch = dx3[:, 1:].reshape(B * d.N, d.D).contiguous()
    pk = VE + "patch_embed.proj.weight"
    if pk in G:
        K = G[pk].numel() // d.D
        if c.Kp == K:
            ops.gemm(dpatch, c.patches, a_t=True, b_t=True, out=G[pk].view(d.D, K), accumulate=True)
        else:   # padded patch rows: accumulate into a padded buffer, fold the real columns back
            tmp = torch.zeros((d.D, c.Kp), device=dev, dtype=torch.float32)
            ops.gemm(dpatch, c.patches, a_t=True, b_t=True, out=tmp, accumulate=True)
            G[pk].view(d.D, K).add_(tmp[:, :K])
    if VE + "patch_embed.proj.bias" in G:
        ops.colsum(dpatch, G[VE + "patch_embed.proj.bias"])


# ------------------------------------------------------------------------------------------
# visual abstractor (AttentionPool) + visual_fc
# ------------------------------------------------------------------------------------------
_pad_cache = {}


def _kv_pad_rows(B, K1, dev):
    """in_rows for the key LayerNorm: each sample gets K1 real rows plus one slot (-1) that the
    learned bias_k / bias_v row (nn.MultiheadAttention add_bias_kv) is written into."""
    key = (B, K1, str(dev))
    if key not in _pad_cache:
        r = torch.arange(B * K1).view(B, K1)
        _pad_cache[key] = torch.cat([r, torch.full((B, 1), -1)], 1).reshape(-1).int().to(dev)
    return _pad_cache[key]


def attn_pool_fwd(W, image_embeds, B, heads, save=True):
    """AttentionPool.forward - models/vision_transformer.py:368-374 on
    learnable_queries.repeat(B) (models/distributed_gpt3.py:134).  image_embeds [B*K1, D] -> [B*Q, D]."""
    dev = image_embeds.device
    D = image_embeds.shape[1]
    K1 = image_embeds.shape[0] // B
    KP = K1 + 1
    hd = D // heads
    lq = W["learnable_queries"][0]
    Q = lq.shape[0]
    c = Ctx(B=B, Q=Q, K1=K1, D=D, heads=heads, hd=hd)
    eps = 1e-6
    # the query block is identical for every sample: normalise / project it once
    xq, c.mq, c.rq = ops.layernorm_fwd(lq, W[AP + "norm1.weight"], W[AP + "norm1.bias"], eps)
    rows = _kv_pad_rows(B, K1, dev)
    kvn, c.mk, c.rk = ops.layernorm_fwd(image_embeds, W[AP + "normk.weight"], W[AP + "normk.bias"], eps, in_rows=rows)
    w_in, b_in = W[AP + "attn.in_proj_weight"], W[AP + "attn.in_proj_bias"]
    qp = ops.gemm(xq, w_in[:D], bias=b_in[:D])
    kvp = ops.gemm(kvn, w_in[D:], bias=b_in[D:])                      # [B*KP, 2D]: k | v
    kvp.view(B, KP, 2 * D)[:, K1] = torch.cat([W[AP + "attn.bias_k"].view(-1), W[AP + "attn.bias_v"].view(-1)])
    att = torch.empty((B * Q, D), device=dev, dtype=bf16)
    mq = ops.seqmap(seq_div=1, outer_stride=0, pos_stride=1)
    mkv, mo = ops.dense_map(KP), ops.dense_map(Q)
    c.lse = ops.attn_fwd(TView(qp, 0, hd, mq), TView(kvp, 0, hd, mkv), TView(kvp, D, hd, mkv), TView(att, 0, hd, mo),
                         n_seq=B, n_heads=heads, head_dim=hd, s_q=Q, s_kv=KP, causal=False, scale=hd ** -0.5)
    # residual from the *normalised* queries (:369-371)
    x1 = ops.gemm(att, W[AP + "attn.out_proj.weight"], bias=W[AP + "attn.out_proj.bias"], residual=xq, res_row_mod=Q,
                  out_dtype=torch.float32)
    ln2, c.m2, c.r2 = ops.layernorm_fwd(x1, W[AP + "norm2.weight"], W[AP + "norm2.bias"], eps)
    dact = torch.empty((B * Q, W[AP + "mlp.fc1.weight"].shape[0]), device=dev, dtype=bf16)
    h = ops.gemm(ln2, W[AP + "mlp.fc1.weight"], bias=W[AP + "mlp.fc1.bias"], act=ACT_GELU_ERF, aux_out=dact)
    out = ops.gemm(h, W[AP + "mlp.fc2.weight"], bias=W[AP + "mlp.fc2.bias"], residual=x1)
    if save:
        c.update(lq=lq, xq=xq, kvn=kvn, qp=qp, kvp=kvp, att=att, x1=x1, ln2=ln2, dact=dact, h=h,
                 image_embeds=image_embeds, rows=rows)
    return out, c


def attn_pool_bwd(W, G, c, dout):
    """dout [B*Q, D] -> d_image_embeds [B*K1, D]; accumulates abstractor + learnable_queries grads."""
    B, Q, K1, D, hd, heads = c.B, c.Q, c.K1, c.D, c.hd, c.heads
    KP = K1 + 1
    dev = dout.device
    linear_wgrad(dout, c.h, AP + "mlp.fc2.weight", AP + "mlp.fc2.bias", G)
    dpre = linear_dgrad(dout, W[AP + "mlp.fc2.weight"], act=ACT_GELU_ERF, aux_in=c.dact)
    linear_wgrad(dpre, c.ln2, AP + "mlp.fc1.weight", AP + "mlp.fc1.bias", G)
    dln2 = linear_dgrad(dpre, W[AP + "mlp.fc1.weight"])
    dx1 = ops.layernorm_bwd(dln2, c.x1, W[AP + "norm2.weight"], c.m2, c.r2, add=dout,
                            dgamma=G.get(AP + "norm2.weight"), dbeta=G.get(AP + "norm2.bias"))
    linear_wgrad(dx1, c.att, AP + "attn.out_proj.weight", AP + "attn.out_proj.bias", G)
    datt = linear_dgrad(dx1, W[AP + "attn.out_proj.weight"])
    dqp_b = torch.empty((B * Q, D), device=dev, dtype=bf16)
    dkvp = torch.empty((B * KP, 2 * D), device=dev, dtype=bf16)
    mq = ops.seqmap(seq_div=1, outer_stride=0, pos_stride=1)
    mkv, mo = ops.dense_map(KP), ops.dense_map(Q)
    ops.attn_bwd(TView(c.qp, 0, hd, mq), TView(c.kvp, 0, hd, mkv), TView(c.kvp, D, hd, mkv), TView(c.att, 0, hd, mo),
                 c.lse, TView(datt, 0, hd, mo), TView(dqp_b, 0, hd, mo), TView(dkvp, 0, hd, mkv), TView(dkvp, D, hd, mkv),
                 n_seq=B, n_heads=heads, head_dim=hd, s_q=Q, s_kv=KP, causal=False, scale=hd ** -0.5)
    # learned bias_k / bias_v row, then zero it so it does not leak into the projection grads
    dkv3 = dkvp.view(B, KP, 2 * D)
    dbias = dkv3[:, K1].float().sum(0)
    if AP + "attn.bias_k" in G:
        G[AP + "attn.bias_k"].view(-1).add_(dbias[:D])
    if AP + "attn.bias_v" in G:
        G[AP + "attn.bias_v"].view(-1).add_(dbias[D:])
    dkv3[:, K1].zero_()
    # shared query block: sum the per-sample grads (query path + residual path)
    dq_sum = _zeros_f32(Q * D, dev)
    ops.colsum(dqp_b.view(B, Q * D), dq_sum)
    dqp = dq_sum.view(Q, D).to(bf16)
    dres = _zeros_f32(Q * D, dev)
    ops.colsum(dx1.view(B, Q * D), dres)
    w_in = W[AP + "attn.in_proj_weight"]
    if AP + "attn.in_proj_weight" in G:
        gw = G[AP + "attn.in_proj_weight"].view(3 * D, D)
        ops.gemm(dqp, c.xq, a_t=True, b_t=True, out=gw[:D], accumulate=True)
        ops.gemm(dkvp, c.kvn, a_t=True, b_t=True, out=gw[D:], accumulate=True)
    if AP + "attn.in_proj_bias" in G:
        gb = G[AP + "attn.in_proj_bias"]
        ops.colsum(dqp, gb[:D])
        ops.colsum(dkvp, gb[D:])
    dxq = linear_dgrad(dqp, w_in[:D], out_dtype=torch.float32)
    dxq = (dxq + dres.view(Q, D)).to(bf16)
    dlq = ops.layernorm_bwd(dxq, c.lq, W[AP + "norm1.weight"], c.mq, c.rq,
                            dgamma=G.get(AP + "norm1.weight"), dbeta=G.get(AP + "norm1.bias"))
    if "learnable_queries" in G:
        G["learnable_queries"].view(Q, D).add_(dlq.float())
    dkvn = linear_dgrad(dkvp, w_in[D:])
    d_img = torch.empty_like(c.image_embeds)
    ops.layernorm_bwd(dkvn, c.image_embeds, W[AP + "normk.weight"], c.mk, c.rk, in_rows=c.rows,
                      dgamma=G.get(AP + "normk.weight"), dbeta=G.get(AP + "normk.bias"), dx=d_img)
    return d_img


# ------------------------------------------------------------------------------------------
# GPT-3 decoder
# ------------------------------------------------------------------------------------------
class GptDrop:
    """Dropout of one decoder pass (the reference runs the frozen decoder in train() mode: hidden_dropout on the
    embeddings and the two bias-dropout-adds, attention_dropout on the probabilities - modeling_distributed_gpt3.py:
    631,732,1056-1078).  `rng` is the pass's {seed, offset} device tensor; the backward regenerates the same masks."""

    def __init__(self, rng, p_hidden, p_attn):
        self.rng, self.p_hidden, self.p_attn = rng, float(p_hidden), float(p_attn)

    def embed(self):
        return ops.Drop(self.rng, ops.site_embed(), self.p_hidden) if self.p_hidden > 0 else None

    def attn(self, i):
        return ops.Drop(self.rng, ops.site_attn(i), self.p_attn) if self.p_attn > 0 else None

    def bda_attn(self, i):
        return ops.Drop(self.rng, ops.site_bda_attn(i), self.p_hidden) if self.p_hidden > 0 else None

    def bda_mlp(self, i):
        return ops.Drop(self.rng, ops.site_bda_mlp(i), self.p_hidden) if self.p_hidden > 0 else None


class GptDims:
    def __init__(self, gcfg):
        self.H = gcfg["hidden_size"]
        self.heads = gcfg["num_attention_heads"]
        self.hd = self.H // self.heads
        self.layers = gcfg["num_hidden_layers"]
        self.F = gcfg.get("ffn_hidden_size") or 4 * self.H
        self.V = gcfg["vocab_size"]
        self.eps = gcfg.get("layernorm_epsilon", 1e-12)
        # q.k / (sqrt(hn)*layer) * layer == q.k / sqrt(hn)  (modeling_distributed_gpt3.py:718-762)
        self.scale = 1.0 / math.sqrt(self.hd)


def gpt_layer_fwd(W, pre, x, g, B, S, train_w=False, drop=None, li=0):
    """GPT3ParallelTransformerLayer.forward - models/modeling_distributed_gpt3.py:1034-1089
    (causal mask over the whole [prefix|text] sequence, :1329-1332; `drop`: GptDrop or None, li: layer index)."""
    H, hd = g.H, g.hd
    c = Ctx()
    d_at = drop.attn(li) if drop else None
    d_b1 = drop.bda_attn(li) if drop else None
    d_b2 = drop.bda_mlp(li) if drop else None
    ln1, c.m1, c.r1 = ops.layernorm_fwd(x, W[pre + "input_layernorm.weight"], W[pre + "input_layernorm.bias"], g.eps)
    qkv = ops.gemm(ln1, W[pre + "self_attention.query_key_value.weight"], bias=W[pre + "self_attention.query_key_value.bias"])
    att = torch.empty((B * S, H), device=x.device, dtype=bf16)
    m = ops.dense_map(S)
    q, k, v = (TView(qkv, i * hd, 3 * hd, m) for i in range(3))  # rows grouped per head as [q|k|v] (:894-902)
    c.lse = ops.attn_fwd(q, k, v, TView(att, 0, hd, m), n_seq=B, n_heads=g.heads, head_dim=hd, s_q=S, s_kv=S,
                         causal=True, scale=g.scale, drop=d_at)
    x1 = ops.gemm(att, W[pre + "self_attention.dense.weight"], bias=W[pre + "self_attention.dense.bias"], residual=x,
                  out_dtype=torch.float32, drop=d_b1)
    ln2, c.m2, c.r2 = ops.layernorm_fwd(x1, W[pre + "post_attention_layernorm.weight"], W[pre + "post_attention_layernorm.bias"], g.eps)
    dact = torch.empty((B * S, g.F), device=x.device, dtype=bf16)
    h = ops.gemm(ln2, W[pre + "mlp.dense_h_to_4h.weight"], bias=W[pre + "mlp.dense_h_to_4h.bias"], act=ACT_GELU_TANH, aux_out=dact)
    out = ops.gemm(h, W[pre + "mlp.dense_4h_to_h.weight"], bias=W[pre + "mlp.dense_4h_to_h.bias"], residual=x1,
                   out_dtype=torch.float32, drop=d_b2)
    c.update(x=x, qkv=qkv, att=att, x1=x1, dact=dact)
    if train_w:
        c.update(ln1=ln1, ln2=ln2, h=h)
    return out, c


def gpt_layer_bwd(W, G, pre, c, dout, g, B, S, drop=None, li=0, dout_d=None):
    """dout: gradient of the layer output (residual stream).  With dropout, dout_d = dropout_backward(dout) for this
    layer's MLP bias-dropout-add (the gradient of the branch output); returns (dx, dx_d) where dx_d is masked for the
    dropout site that produced this layer's input (previous layer's MLP bias-dropout-add, or the embedding)."""
    hd = g.hd
    dev = dout.device
    if dout_d is None:
        dout_d = dout
    if "h" in c:
        linear_wgrad(dout_d, c.h, pre + "mlp.dense_4h_to_h.weight", pre + "mlp.dense_4h_to_h.bias", G)
    dpre = linear_dgrad(dout_d, W[pre + "mlp.dense_4h_to_h.weight"], act=ACT_GELU_TANH, aux_in=c.dact)
    if "ln2" in c:
        linear_wgrad(dpre, c.ln2, pre + "mlp.dense_h_to_4h.weight", pre + "mlp.dense_h_to_4h.bias", G)
    dln2 = linear_dgrad(dpre, W[pre + "mlp.dense_h_to_4h.weight"])
    d_b1 = drop.bda_attn(li) if drop else None
    r = ops.layernorm_bwd(dln2, c.x1, W[pre + "post_attention_layernorm.weight"], c.m2, c.r2, add=dout,
                          dgamma=G.get(pre + "post_attention_layernorm.weight"), dbeta=G.get(pre + "post_attention_layernorm.bias"),
                          drop=d_b1)
    dx1, dx1_d = r if d_b1 is not None else (r, r)
    linear_wgrad(dx1_d, c.att, pre + "self_attention.dense.weight", pre + "self_attention.dense.bias", G)
    datt = linear_dgrad(dx1_d, W[pre + "self_attention.dense.weight"])
    dqkv = torch.empty_like(c.qkv)
    m = ops.dense_map(S)
    q, k, v = (TView(c.qkv, i * hd, 3 * hd, m) for i in range(3))
    dq, dk, dv = (TView(dqkv, i * hd, 3 * hd, m) for i in range(3))
    ops.attn_bwd(q, k, v, TView(c.att, 0, hd, m), c.lse, TView(datt, 0, hd, m), dq, dk, dv, n_seq=B, n_heads=g.heads,
                 head_dim=hd, s_q=S, s_kv=S, causal=True, scale=g.scale, drop=drop.attn(li) if drop else None)
    if "ln1" in c:
        linear_wgrad(dqkv, c.ln1, pre + "self_attention.query_key_value.weight", pre + "self_attention.query_key_value.bias", G)
    dln1 = linear_dgrad(dqkv, W[pre + "self_attention.query_key_value.weight"])
    d_in = (drop.bda_mlp(li - 1) if li > 0 else drop.embed()) if drop else None
    r = ops.layernorm_bwd(dln1, c.x, W[pre + "input_layernorm.weight"], c.m1, c.r1, add=dx1,
                          dgamma=G.get(pre + "input_layernorm.weight"), dbeta=G.get(pre + "input_layernorm.bias"), drop=d_in)
    return r if d_in is not None else (r, r)


def gpt_fwd(W, x, gcfg, B, S, train_w=False, save=True, out_rows=None, drop=None):
    """x [B*S, H] fp32: input embeddings with the learned position embeddings already added
    (GPT3Embedding.forward, :640-666); with `drop` (GptDrop) the embedding dropout (:631) is applied to x IN PLACE
    first.  Returns final-LN hidden states [B*S, H], or only the rows listed in out_rows (int32 row indices,
    compact [len(out_rows), H]) when the caller needs no others."""
    g = GptDims(gcfg)
    if drop is not None and drop.p_hidden <= 0 and drop.p_attn <= 0:
        drop = None
    c = Ctx(g=g, B=B, S=S, layers=[], out_rows=out_rows, drop=drop)
    if drop is not None and drop.embed() is not None:
        ops.dropout(x, drop.embed())
    for i in range(g.layers):
        x, lc = gpt_layer_fwd(W, f"{GPT}encoder.layers.{i}.", x, g, B, S, train_w, drop, i)
        c.layers.append(lc if save else None)
    hid, c.mf, c.rf = ops.layernorm_fwd(x, W[GPT + "encoder.final_layernorm.weight"], W[GPT + "encoder.final_layernorm.bias"], g.eps,
                                        in_rows=out_rows)
    if save:
        c.xL = x
    return hid, c


def gpt_bwd(W, G, c, dhid):
    """Returns the gradient w.r.t. the decoder input embeddings (before the embedding dropout when active)."""
    g, B, S, drop = c.g, c.B, c.S, c.drop
    dx = dx_d = None
    if c.out_rows is not None:  # rows without a consumer get no gradient from the final LayerNorm
        dx = torch.zeros((c.xL.shape[0], c.xL.shape[1]), device=dhid.device, dtype=torch.bfloat16)
    d_last = drop.bda_mlp(g.layers - 1) if drop else None
    r = ops.layernorm_bwd(dhid, c.xL, W[GPT + "encoder.final_layernorm.weight"], c.mf, c.rf,
                          dgamma=G.get(GPT + "encoder.final_layernorm.weight"), dbeta=G.get(GPT + "encoder.final_layernorm.bias"),
                          in_rows=c.out_rows, dx=dx, drop=d_last)
    dx, dx_d = r if d_last is not None else (r, r)
    for i in reversed(range(g.layers)):
        dx, dx_d = gpt_layer_bwd(W, G, f"{GPT}encoder.layers.{i}.", c.layers[i], dx, g, B, S, drop, i, dx_d)
        c.layers[i] = None
    return dx_d


class KVCache:
    """Incremental-decoding state (SURVEY.md 8f N2; the reference's InferenceParams.key_value_memory_dict,
    models/modeling_distributed_gpt3.py:874-923).  One packed QKV buffer [B*max_len, 3H] per layer in the
    per-head [q|k|v] column layout of the QKV GEMM, so new rows are written by the GEMM epilogue itself
    (row re-blocking) and the attention kernels read K/V of all cached positions in place.  All layers live in
    one allocation that never moves (the captured single-token step holds its pointers), and the number of
    cached positions is mirrored on the device (`len_idx`, `len1`) for that graph."""

    def __init__(self, gcfg, batch, max_len, device):
        g = GptDims(gcfg)
        self.g, self.B, self.max_len, self.len = g, batch, max_len, 0
        self.store = torch.zeros((g.layers, batch * max_len, 3 * g.H), device=device, dtype=bf16)
        self.qkv = [self.store[i] for i in range(g.layers)]
        self.len_idx = torch.zeros(1, device=device, dtype=torch.int64)   # = len: position / cache row of the next token
        self.len1 = torch.ones(1, device=device, dtype=torch.int32)       # = len + 1: keys the next token attends to
        self.token = None   # TokenStep of the single-token steps (built by the caller that owns the weights)

    def reset(self):
        """Forget the cached positions (the rows are overwritten by the next prefill; stale rows past `len` are never read)."""
        self.len = 0
        self.len_idx.zero_()
        self.len1.fill_(1)

    def _set_len(self, n):
        self.len = n
        self.len_idx.fill_(n)
        self.len1.fill_(n + 1)

    def reorder(self, idx):
        """Row b of the cache becomes old row idx[b] (beam search, swap_key_value_dict :1460-1473), in place and for
        the cached positions only: two launches for all layers."""
        assert idx.numel() == self.B
        if self.len == 0:
            return
        v = self.store.view(self.g.layers, self.B, self.max_len, -1)[:, :, :self.len]
        v.copy_(v.index_select(1, idx))


class _RowBlock:
    """Rows [r0, r0 + rows) of a KVCache, seen as a cache of their own by gpt_decode (the per-sample prefill of a batched
    beam search writes one sample's beams into its block with exactly the call a single beam search makes)."""

    def __init__(self, cache, r0, rows):
        ML = cache.max_len
        self.g, self.B, self.max_len, self.len = cache.g, rows, ML, 0
        self.qkv = [t[r0 * ML:(r0 + rows) * ML] for t in cache.qkv]

    def _set_len(self, n):
        self.len = n


class BeamBatchCache(KVCache):
    """KV cache of a batch of beam searches: R = n_samples x beam rows, sample i owning rows [i*beam, (i+1)*beam).
    Attention finds key j of row r through the int32 device table `table[r, j]` (a cache row index), so a beam reorder
    moves table entries - `table[:, :len] = table[parent, :len]`, a few kilobytes - instead of every cached position of
    every layer.  The new token of row r is still written to slot r * max_len + len: no table entry refers to it before
    that step (entries at and past `len` are the identity), so cached K/V is never rewritten.  After the prefill every
    beam of a sample reads its prefix positions from the sample's beam-0 rows (`start_table`), which keeps one copy of
    each prefix in L2 instead of `beam`."""

    def __init__(self, gcfg, n_samples, beam, max_len, device):
        super().__init__(gcfg, n_samples * beam, max_len, device)
        self.n_samples, self.beam = n_samples, beam
        self.table = torch.empty((self.B, max_len), device=device, dtype=torch.int32)
        self.start_table(0)

    def block(self, i):
        """Sample i's rows as a cache of `beam` sequences (for its prefill)."""
        return _RowBlock(self, i * self.beam, self.beam)

    def start_table(self, prefix_len):
        """Identity table, except that positions < prefix_len of every row read the rows of its sample's beam 0."""
        R, ML = self.B, self.max_len
        rows = torch.arange(R, dtype=torch.int64)
        src = rows.clone()
        src_prefix = (rows // self.beam) * self.beam
        tab = src[:, None] * ML + torch.arange(ML, dtype=torch.int64)[None, :]
        tab[:, :prefix_len] = src_prefix[:, None] * ML + torch.arange(prefix_len, dtype=torch.int64)[None, :]
        self.table.copy_(tab.to(torch.int32))

    def reorder_table(self, idx):
        """Row r continues the history of row idx[r] (idx: int64 device tensor [R])."""
        assert idx.numel() == self.B
        if self.len == 0:
            return
        t = self.table[:, :self.len]
        t.copy_(t.index_select(0, idx))


class TokenStep:
    """The single-token decoding step (n == 1, cache not empty) for at most ops.SKINNY_MAX_ROWS sequences, as ONE CUDA
    graph: every linear is a skinny GEMM (one pass over its weights, csrc/gemv.cu), the new K/V row goes into the cache
    at the device-side position `len_idx`, attention reads `len1` keys (ymp_attn_args.s_kv_dev), and the graph ends by
    advancing both counters - so one captured graph serves every position of every generate() call that reuses this
    cache.  ~8 kernels per layer; the latency floor is the weight stream (2.6 GB at 1.3B).
    Over a BeamBatchCache the same step serves up to ops.SKINNY_WIDE_MAX_ROWS rows (a batch of beam searches), the
    decode attention reading its keys through the cache's row table."""

    def __init__(self, cache, W, emb_dtype, sig=None, static=True):
        """sig: anything that changes when the weight tensors behind W move; static: W may be captured (raw pointers)."""
        g, dev = cache.g, cache.store.device
        self.cache, self.W, self.sig, self.static = cache, W, sig, static
        self.emb_in = torch.zeros((cache.B, g.H), device=dev, dtype=emb_dtype)
        self.stage = torch.zeros((cache.B, 3 * g.H), device=dev, dtype=bf16)   # the new token's [q|k|v] row per sequence
        self.ticket = torch.zeros(1, device=dev, dtype=torch.int32)            # last-CTA ticket of the fused LayerNorms
        self.graph = None
        self.out = None
        self.warm = False

    def body(self):
        """Enqueue the step on the current stream (eagerly or under capture): reads emb_in, returns (hid, logits).
        YMP_DECODE_PDL=1 chains the kernels by programmatic dependent launch (each may start - and the GEMMs already
        stream their first weights - while the previous one drains).  Off by default: measured SLOWER inside the
        captured graph on B200 (1.63 vs 1.47 ms per token at 1.3B / beam 5, profiles/r02l_pdl.log)."""
        import os
        prev = L.set_pdl(os.environ.get("YMP_DECODE_PDL", "0") == "1")
        try:
            return self._body()
        finally:
            L.set_pdl(prev)

    def _body(self):
        c, W = self.cache, self.W
        g, B, ML = c.g, c.B, c.max_len
        H, hd = g.H, g.hd
        pos = W[GPT + "embedding.position_embeddings.weight"]
        x = self.emb_in.float() + pos.index_select(0, c.len_idx).float()
        mkv = ops.dense_map(ML)

        import os
        # YMP_DECODE_FUSED_LN=1: every LayerNorm but the first is computed by the last CTA of the GEMM that completes its
        # input (one kernel boundary less per sub-layer).  Off by default: measured neutral on B200 (captured step 1.466
        # vs 1.438 ms, profiles/r02p_decode_ab.log) - the ticket + three L2 round trips of the tail cost what the
        # stand-alone kernel and its launch gap cost.
        fused_ln = os.environ.get("YMP_DECODE_FUSED_LN", "0") == "1" and B <= ops.SKINNY_MAX_ROWS
        kv_rows = getattr(c, "table", None)   # BeamBatchCache: keys through the per-row table
        skinny = ops.gemm_skinny if B <= ops.SKINNY_MAX_ROWS else ops.gemm_skinny_batch

        def ln_of(prefix):
            return (W[prefix + ".weight"], W[prefix + ".bias"], g.eps, self.ticket)

        def gemm_ln(a, wname, residual, ln_prefix):
            """fp32 residual-stream GEMM followed by the LayerNorm of its complete result: (y, LN(y))."""
            if fused_ln:  # the LayerNorm is computed by the GEMM's last CTA
                return skinny(a, W[wname + ".weight"], bias=W[wname + ".bias"], residual=residual, out_dtype=torch.float32,
                                       ln=ln_of(ln_prefix))
            y = skinny(a, W[wname + ".weight"], bias=W[wname + ".bias"], residual=residual, out_dtype=torch.float32)
            return y, ops.layernorm_fwd(y, W[ln_prefix + ".weight"], W[ln_prefix + ".bias"], g.eps, stats=False)[0]

        ln1, _, _ = ops.layernorm_fwd(x, W[f"{GPT}encoder.layers.0.input_layernorm.weight"], W[f"{GPT}encoder.layers.0.input_layernorm.bias"],
                                      g.eps, stats=False)
        for i in range(g.layers):
            pre = f"{GPT}encoder.layers.{i}."
            st = self.stage
            buf = c.qkv[i]
            # [q|k|v] of the new token: into the staging rows (q for this step) and into cache row b*ML + len (k, v)
            skinny(ln1, W[pre + "self_attention.query_key_value.weight"], bias=W[pre + "self_attention.query_key_value.bias"],
                            out=st, out2=buf, out2_row_stride=ML, out2_off=c.len_idx)
            att = torch.empty((B, H), device=x.device, dtype=bf16)
            q = TView(st, 0, 3 * hd, ops.dense_map(1))
            k, v = TView(buf, hd, 3 * hd, mkv), TView(buf, 2 * hd, 3 * hd, mkv)
            ops.attn_fwd(q, k, v, TView(att, 0, hd, ops.dense_map(1)), n_seq=B, n_heads=g.heads, head_dim=hd, s_q=1, s_kv=ML,
                         causal=False, scale=g.scale, s_kv_dev=c.len1, kv_rows=kv_rows)
            x1, ln2 = gemm_ln(att, pre + "self_attention.dense", x, pre + "post_attention_layernorm")
            h = skinny(ln2, W[pre + "mlp.dense_h_to_4h.weight"], bias=W[pre + "mlp.dense_h_to_4h.bias"], act=ACT_GELU_TANH)
            nxt = f"{GPT}encoder.layers.{i + 1}.input_layernorm" if i + 1 < g.layers else GPT + "encoder.final_layernorm"
            x, ln1 = gemm_ln(h, pre + "mlp.dense_4h_to_h", x1, nxt)
        hid = ln1
        logits = skinny(hid, W[GPT + "embedding.word_embeddings.weight"], out_dtype=torch.float32)
        c.len_idx += 1
        c.len1 += 1
        return hid, logits

    def run(self, emb):
        c = self.cache
        use_graph = self.static and decode_graph_enabled()
        if c.len + 1 > c.max_len:
            raise ValueError(f"KV cache overflow: {c.len} + 1 > {c.max_len}")
        self.emb_in.copy_(emb)
        if not use_graph or not self.warm:
            # the first step runs eagerly: it is also the warm-up the capture needs (lazy kernel attributes)
            hid, logits = self.body()
            self.warm = True
        else:
            if self.graph is None:
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    self.out = self.body()
                self.graph = graph
            self.graph.replay()
            hid, logits = self.out[0].clone(), self.out[1].clone()
        c.len += 1
        return hid, logits


def decode_graph_enabled():
    import os
    return os.environ.get("YMP_DECODE_GRAPH", "1") != "0"


def gpt_decode(W, x, cache, n):
    """n new positions per sequence through all layers with the KV cache.  x [B*n, H] fp32 = embeddings +
    learned positions of positions cache.len .. cache.len+n-1 (rows b*n + i).  Either the first call
    (cache empty: causal attention inside the block) or single-token steps (n == 1: the query sees every
    cached key).  Returns the final-LayerNorm hidden state of the LAST new position of every sequence [B, H]."""
    g, B, ML, off = cache.g, cache.B, cache.max_len, cache.len
    H, hd = g.H, g.hd
    if off + n > ML:
        raise ValueError(f"KV cache overflow: {off} + {n} > {ML}")
    if off > 0 and n != 1:
        raise NotImplementedError("multi-token continuation after the first block is not supported")
    for i in range(g.layers):
        pre = f"{GPT}encoder.layers.{i}."
        ln1, _, _ = ops.layernorm_fwd(x, W[pre + "input_layernorm.weight"], W[pre + "input_layernorm.bias"], g.eps, stats=False)
        buf = cache.qkv[i]
        new_rows = buf[off:]  # GEMM row (b, i) -> buffer row b*max_len + off + i
        ops.gemm(ln1, W[pre + "self_attention.query_key_value.weight"], bias=W[pre + "self_attention.query_key_value.bias"],
                 out=new_rows, d_row_block=n, d_row_stride=ML)
        att = torch.empty((B * n, H), device=x.device, dtype=bf16)
        mq = ops.seqmap(seq_div=1, outer_stride=ML, pos_stride=1)
        mkv = ops.dense_map(ML)
        q = TView(new_rows, 0, 3 * hd, mq)
        k, v = TView(buf, hd, 3 * hd, mkv), TView(buf, 2 * hd, 3 * hd, mkv)
        ops.attn_fwd(q, k, v, TView(att, 0, hd, ops.dense_map(n)), n_seq=B, n_heads=g.heads, head_dim=hd, s_q=n, s_kv=off + n,
                     causal=(off == 0 and n > 1), scale=g.scale)
        x1 = ops.gemm(att, W[pre + "self_attention.dense.weight"], bias=W[pre + "self_attention.dense.bias"], residual=x,
                      out_dtype=torch.float32)
        ln2, _, _ = ops.layernorm_fwd(x1, W[pre + "post_attention_layernorm.weight"], W[pre + "post_attention_layernorm.bias"], g.eps,
                                      stats=False)
        h = ops.gemm(ln2, W[pre + "mlp.dense_h_to_4h.weight"], bias=W[pre + "mlp.dense_h_to_4h.bias"], act=ACT_GELU_TANH)
        x = ops.gemm(h, W[pre + "mlp.dense_4h_to_h.weight"], bias=W[pre + "mlp.dense_4h_to_h.bias"], residual=x1,
                     out_dtype=torch.float32)
    cache._set_len(off + n)
    last = torch.arange(B, device=x.device, dtype=torch.int32) * n + (n - 1)
    hid, _, _ = ops.layernorm_fwd(x, W[GPT + "encoder.final_layernorm.weight"], W[GPT + "encoder.final_layernorm.bias"], g.eps,
                                  in_rows=last, stats=False)
    return hid


def lm_head_fwd(W, hid, labels):
    """Tied LM head + per-token CE on fp32 math (modeling_distributed_gpt3.py:1348-1359).
    Returns (logits [B*S, V] bf16, losses [B*S] fp32, lse)."""
    logits = ops.gemm(hid, W[GPT + "embedding.word_embeddings.weight"])
    losses, lse = ops.ce_fwd(logits, labels.reshape(-1).contiguous())
    return logits, losses, lse


def lm_head_bwd(W, G, hid, logits, labels, lse, grad_rows, keep_logits=False):
    """grad_rows [B*S] fp32 = d loss / d losses.  Overwrites `logits` with dlogits unless keep_logits."""
    dlogits = ops.ce_bwd(logits, labels.reshape(-1).contiguous(), lse, grad_rows.contiguous(),
                         dlogits=torch.empty_like(logits) if keep_logits else None)
    emb = GPT + "embedding.word_embeddings.weight"
    if emb in G:
        ops.gemm(dlogits, hid, a_t=True, b_t=True, out=G[emb].view(dlogits.shape[1], hid.shape[1]), accumulate=True)
    return linear_dgrad(dlogits, W[emb])
