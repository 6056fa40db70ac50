"""mPLUG-Video task models on the B200 kernels - drop-in for the reference `models/distributed_gpt3.py`.

DistributedGPT3_Pretrain (:31-226) is the hot path: TimeSformer -> AttentionPool abstractor ->
visual_fc -> frozen GPT-3 causal decoder over [visual prefix | text] -> masked token CE.  Same
constructor (config dict, tokenizer), same forward(image, text) -> (loss_caption, loss_contrastive),
same parameter names.  Integer work (targets / loss_mask, :142-159) is done with the same torch
index ops as the reference and is bit-exact.
"""
import json
from functools import partial

import torch
import torch.nn.functional as F
from torch import nn

from ymp import functional as YF

from ._params import add_param, linear_default, named_param_list, trunc_normal
from .distributed_utils import all_gather_cat, concat_all_gather  # noqa: F401
from .modeling_distributed_gpt3 import DistributedGPT3, GPT3Config
from .vision_transformer import AttentionPool, LayerNormWithForceFP32, TimeSformer, _convert_pretrained_vit


class _Linear(nn.Linear):
    """nn.Linear whose forward runs on the tcgen05 GEMM (same parameters / state_dict keys)."""

    def forward(self, x):
        return YF.LinearFn.apply(x, self.weight, self.bias)


class _VisualNorm(nn.LayerNorm):
    """visual_norm of `connect_ln` configs (reference :112-116): LayerNormWithForceFP32(text_width)."""

    def forward(self, x):
        return YF.LayerNormFn.apply(x, self.weight, self.bias, self.eps)


def _build_visual_encoder(visual_cfg, num_frames):
    return TimeSformer(
        img_size=visual_cfg['img_size'], num_frames=num_frames, patch_size=visual_cfg['patch_size'],
        embed_dim=visual_cfg['embed_dim'], depth=visual_cfg['depth'], num_heads=visual_cfg['num_heads'],
        mlp_ratio=visual_cfg['mlp_ratio'], qkv_bias=True, norm_layer=partial(LayerNormWithForceFP32, eps=1e-6),
        init_std=0.015, grad_ckpt=visual_cfg.get('grad_ckpt', True), drop_path_rate=visual_cfg.get('drop_path', False),
        stop_grad_conv1=visual_cfg.get('stop_grad_conv1', False),
        use_shared_rel_pos_bias=visual_cfg.get('use_shared_rel_pos_bias', False),
        use_abs_pos_emb=visual_cfg.get('use_abs_pos_emb', True),
        init_values=visual_cfg.get('layer_scale_init_value', 0), postnorm=visual_cfg.get('postnorm', False),
        clip_model=visual_cfg.get('clip_model', False))


def _load_pretrained_vit(encoder, visual_cfg):
    ckpt = visual_cfg.get("pretrained_ckpt", None)
    if ckpt is None:
        return
    if ckpt.startswith("clip"):
        path = "/".join(ckpt.split("/")[1:])
        weights = _convert_pretrained_vit(torch.load(path, map_location='cpu'))
        msg = encoder.load_state_dict(weights, strict=False)
        print("Initialize Vision Encoder from CKPT {}".format(path))
        print(msg)
    else:
        raise NotImplementedError(f"pretrained_ckpt={ckpt!r}: timm hub checkpoints need network access")


class _PrefixModelBase(nn.Module):
    """Shared construction: visual encoder + frozen decoder + learnable queries + abstractor + visual_fc
    (reference :31-116 / :431-520 / :662-750)."""

    def _build(self, config, tokenizer, num_frames):
        self.tokenizer = tokenizer
        with open(config['visual_cfg'], 'r') as f:
            visual_cfg = json.load(f)
        text_cfg = GPT3Config.from_json_file(config['text_cfg'])
        self.visual_cfg = visual_cfg
        self.visual_encoder = _build_visual_encoder(visual_cfg, num_frames if num_frames is not None else visual_cfg['num_frames'])
        _load_pretrained_vit(self.visual_encoder, visual_cfg)
        rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
        self.text_decoder = DistributedGPT3(
            model_dir=config['text_decoder'], rank=rank, path_load_tag='model', megatron_cfg=config['megatron_cfg'],
            checkpoint_model_parallel_size=1 if text_cfg.num_hidden_layers < 40 else 8)
        if config.get('freeze_vit', False):
            for name, param in self.visual_encoder.named_parameters():
                if not any(x in name for x in ['time', 'temporal']):
                    param.requires_grad = False
        if config.get('freeze_text_decoder', True):
            for param in self.text_decoder.parameters():
                param.requires_grad = False
        self.vision_width = visual_cfg['embed_dim']
        self.text_width = self.text_decoder.config.hidden_size
        self.learnable_token = True
        self.num_learnable_token = config.get('num_learnable_token', 256)
        self.learnable_queries = nn.Parameter(trunc_normal((1, self.num_learnable_token, self.vision_width), 0.015))
        self.attn_pool = AttentionPool(self.vision_width, num_heads=visual_cfg['num_heads'],
                                       mlp_ratio=visual_cfg['mlp_ratio'],
                                       norm_layer=partial(LayerNormWithForceFP32, eps=1e-6))
        self.visual_fc = _Linear(self.vision_width, self.text_width)
        with torch.no_grad():
            self.visual_fc.weight.copy_(trunc_normal((self.text_width, self.vision_width), 0.015))
        self.connect_ln = bool(visual_cfg.get('connect_ln', False))
        self.visual_norm = _VisualNorm(self.text_width, eps=1e-6) if self.connect_ln else nn.Identity()
        self.prompt = config.get('prompt', "")

    def _word_embedding(self):
        return self.text_decoder.dist_model.language_model.embedding.word_embeddings

    def visual_prefix(self, image):
        """image -> (image_embeds [B,1+TN,D], image_query [B,Q,D], query_features [B,Q,H])."""
        pooled, image_embeds = self.visual_encoder(image)
        image_query = self.attn_pool(None, image_embeds, queries_param=self.learnable_queries)
        query_features = self.visual_norm(self.visual_fc(image_query))
        return pooled, image_embeds, image_query, query_features

    @torch.jit.ignore
    def no_weight_decay(self):
        return {'visual_encoder.pos_embed', 'visual_encoder.cls_token', 'visual_encoder.temporal_embed'}


def mask_prompt(text_loss_atts, prompt_lengths):
    """text_loss_atts[i, :prompt_lengths[i]] = 0 for every sample (the reference loops over `.cpu().tolist()`,
    models/distributed_gpt3.py:760-766) as one device-side comparison: same integers, no host synchronisation, so
    the step stays CUDA-graph capturable."""
    pos = torch.arange(text_loss_atts.shape[1], device=text_loss_atts.device)[None, :]
    return text_loss_atts * (pos >= prompt_lengths.to(text_loss_atts.device).view(-1, 1)).to(text_loss_atts.dtype)


def build_targets(input_ids, text_loss_atts, num_query):
    """targets = [100]*Q ++ ids[:,1:] ++ ids[:,1] ; loss_mask = [0]*Q ++ mask[:,1:]  (:142-159)."""
    B = input_ids.shape[0]
    targets = input_ids[:, 1:].clone()
    targets = torch.cat([targets, targets[:, 0:1]], dim=1)  # last column is not used
    empty_targets = torch.ones((B, num_query), dtype=torch.long, device=input_ids.device).fill_(100)
    targets = torch.cat([empty_targets, targets], dim=1)
    query_atts = torch.ones((B, num_query), dtype=torch.long, device=input_ids.device)
    loss_mask = torch.cat([1 - query_atts, text_loss_atts], dim=1)
    return targets, loss_mask


class DistributedGPT3_Pretrain(_PrefixModelBase):
    def __init__(self, config=None, tokenizer=None):
        super().__init__()
        self._build(config, tokenizer, None)
        self.use_contrastive = config.get('use_contrastive', False)
        if self.use_contrastive:
            embed_dim = config.get('contrastive_embed_dim', 256)
            self.vision_proj = _Linear(self.vision_width, embed_dim)
            self.text_proj = _Linear(self.text_width, embed_dim)
            self.temp = nn.Parameter(torch.ones([]) * config.get('temp', 0.07))
        self.last_losses = None

    def _fused_params(self):
        keys, params = named_param_list(self)
        drop = ("vision_proj.", "text_proj.", "temp")
        kp = [(k, p) for k, p in zip(keys, params) if not k.startswith(drop)]
        return [k for k, _ in kp], [p for _, p in kp]

    def forward(self, image, text):
        if self.prompt != "":
            raise NotImplementedError("a non-empty prompt crashes in the reference too (prompt_length is "
                                      "never set, models/distributed_gpt3.py:118-120,146-148)")
        text_loss_atts = text.attention_mask[:, 1:]
        targets, loss_mask = build_targets(text.input_ids, text_loss_atts, self.num_learnable_token)
        if not self.use_contrastive and not self.connect_ln:
            keys, params = self._fused_params()
            loss_caption, losses = YF.PretrainFn.apply(image, text.input_ids, targets, loss_mask,
                                                       self.visual_encoder.vcfg, self.text_decoder.config.engine_cfg(self.text_decoder.training),
                                                       keys, *params)
            self.last_losses = losses
            return loss_caption, loss_caption.new_zeros(())   # device-side (CUDA-graph capturable)

        # ---- contrastive variant (:168-217) / connect_ln: component path so that image_query is exposed
        _, image_embeds, image_query, query_features = self.visual_prefix(image)
        input_embeds = torch.cat([query_features, self._word_embedding()(text.input_ids).to(query_features.dtype)], dim=1)
        outputs = self.text_decoder(input_embeds=input_embeds, loss_mask=loss_mask, labels=targets)
        loss_caption = outputs.loss
        self.last_losses = None
        if not self.use_contrastive:
            return loss_caption, loss_caption.new_zeros(())
        targets_dep = torch.cat([text.input_ids[:, 1:], text.input_ids[:, 1:2]], dim=1)
        outputs_text = self.text_decoder(tokens=text.input_ids, loss_mask=text.attention_mask[:, 1:].clone(),
                                         labels=targets_dep)
        vision_feats = F.normalize(self.vision_proj(image_query).float(), dim=-1)
        pooled = outputs_text.last_hidden_state
        pooled = pooled[torch.arange(pooled.shape[0], device=pooled.device), text.attention_mask.sum(dim=-1) - 1]
        text_feat = F.normalize(self.text_proj(pooled).float(), dim=-1)
        dist_on = torch.distributed.is_initialized()
        vision_feats_all = all_gather_cat(vision_feats) if dist_on else vision_feats   # [B*W, Q, E]
        text_feat_all = all_gather_cat(text_feat) if dist_on else text_feat            # [B*W, E]
        # sim_q2t[b, j, q] = <vision_feats[b,q], text_all[j]> ; max over queries (:186-202).  Both contractions
        # run on the tcgen05 GEMM (bf16 operands like the reference's bf16 module, fp32 accumulation / output).
        Bv, Qv, E = vision_feats.shape
        J = text_feat_all.shape[0]
        sim_i2t = YF.matmul_nt(vision_feats.reshape(Bv * Qv, E), text_feat_all).view(Bv, Qv, J).max(1)[0] / self.temp
        sim_t2i = YF.matmul_nt(text_feat, vision_feats_all.reshape(J * Qv, E)).view(Bv, J, Qv).max(-1)[0] / self.temp
        rank = torch.distributed.get_rank() if dist_on else 0
        bs = image.size(0)
        tgt = torch.arange(rank * bs, rank * bs + bs, device=image.device)
        loss_contrastive = (F.cross_entropy(sim_i2t, tgt, label_smoothing=0.1)
                            + F.cross_entropy(sim_t2i, tgt, label_smoothing=0.1)) / 2
        return loss_caption, loss_contrastive


class DistributedGPT3_Pretrain_Image(_PrefixModelBase):
    """Image pre-training variant (reference :230-427; SURVEY 8f N3) with the EVA-g encoder (`use_eva_g: true`): image
    [B,3,H,W] -> EVA tokens [B,257,1408] -> abstractor -> visual_fc -> frozen decoder -> masked token CE.  The
    reference's other branch (a plain image ViT from models/vision_transformer.py) is not part of this package."""

    def __init__(self, config=None, tokenizer=None):
        super().__init__()
        from . import eva_vit
        if not config.get('use_eva_g', False):
            raise NotImplementedError("DistributedGPT3_Pretrain_Image on the B200 path implements the EVA-g encoder (use_eva_g: true)")
        self.tokenizer = tokenizer
        with open(config['visual_cfg'], 'r') as f:
            visual_cfg = json.load(f)
        text_cfg = GPT3Config.from_json_file(config['text_cfg'])
        self.visual_cfg = visual_cfg
        self.visual_encoder = eva_vit.create_eva_vit_g(img_size=visual_cfg['img_size'], norm_layer=partial(LayerNormWithForceFP32, eps=1e-6),
                                                       drop_path_rate=visual_cfg.get('drop_path', False), use_checkpoint=True)
        ckpt = visual_cfg.get("pretrained_ckpt", None)
        if ckpt is not None:
            if not ckpt.startswith("eva"):
                raise NotImplementedError(f"pretrained_ckpt={ckpt!r}: only eva/<path> checkpoints load into the EVA-g encoder")
            weights = torch.load("/".join(ckpt.split("/")[1:]), map_location='cpu')
            eva_vit.interpolate_pos_embed(self.visual_encoder, weights)
            print(self.visual_encoder.load_state_dict(weights, strict=False))
        rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
        self.text_decoder = DistributedGPT3(model_dir=config['text_decoder'], rank=rank, path_load_tag='model',
                                            megatron_cfg=config['megatron_cfg'],
                                            checkpoint_model_parallel_size=1 if text_cfg.num_hidden_layers < 40 else 8)
        if config.get('freeze_vit', False):
            for param in self.visual_encoder.parameters():
                param.requires_grad = False
        if config.get('freeze_text_decoder', True):
            for param in self.text_decoder.parameters():
                param.requires_grad = False
        self.vision_width = visual_cfg['embed_dim']
        self.text_width = self.text_decoder.config.hidden_size
        self.learnable_token = True
        self.num_learnable_token = config.get('num_learnable_token', 256)
        self.learnable_queries = nn.Parameter(trunc_normal((1, self.num_learnable_token, self.vision_width), 0.015))
        self.attn_pool = AttentionPool(self.vision_width, num_heads=visual_cfg['num_heads'], mlp_ratio=visual_cfg['mlp_ratio'],
                                       norm_layer=partial(LayerNormWithForceFP32, eps=1e-6))
        self.visual_fc = _Linear(self.vision_width, self.text_width)
        with torch.no_grad():
            self.visual_fc.weight.copy_(trunc_normal((self.text_width, self.vision_width), 0.015))
        self.connect_ln = bool(visual_cfg.get('connect_ln', False))
        self.visual_norm = _VisualNorm(self.text_width, eps=1e-6) if self.connect_ln else nn.Identity()
        self.prompt = config.get('prompt', "")
        self.use_contrastive = config.get('use_contrastive', False)
        if self.use_contrastive:
            raise NotImplementedError("DistributedGPT3_Pretrain_Image: the contrastive branch is implemented for the video model "
                                      "(DistributedGPT3_Pretrain) only")

    def forward(self, image, text):
        _, _, _, query_features = self.visual_prefix(image)
        Q = query_features.shape[1]
        text_loss_atts = text.attention_mask[:, 1:].clone()
        prompt_lengths = getattr(text, "prompt_lengths", None)
        if prompt_lengths is not None:
            text_loss_atts = mask_prompt(text_loss_atts, prompt_lengths)
        targets, loss_mask = build_targets(text.input_ids, text_loss_atts, Q)
        input_embeds = torch.cat([query_features, self._word_embedding()(text.input_ids).to(query_features.dtype)], dim=1)
        loss_caption = self.text_decoder(input_embeds=input_embeds, loss_mask=loss_mask, labels=targets).loss
        return loss_caption, loss_caption.new_zeros(())

    @torch.jit.ignore
    def no_weight_decay(self):
        return {'visual_encoder.pos_embed', 'visual_encoder.cls_token'}


class DistributedGPT3_Caption(_PrefixModelBase):
    """Caption fine-tuning forward (:751-788) and generate() (:790-809, beam search over the KV cache)."""

    def __init__(self, config=None, tokenizer=None):
        super().__init__()
        self._build(config, tokenizer, config.get('num_frames', None))

    def forward(self, image, text=None):
        """Caption loss over [prefix | prompt+caption]; prompt tokens (text.prompt_lengths, :760-766) carry
        no loss."""
        _, _, _, query_features = self.visual_prefix(image)
        Q = query_features.shape[1]
        text_loss_atts = text.attention_mask[:, 1:].clone()
        prompt_lengths = getattr(text, "prompt_lengths", None)
        if prompt_lengths is not None:
            text_loss_atts = mask_prompt(text_loss_atts, prompt_lengths)
        targets, loss_mask = build_targets(text.input_ids, text_loss_atts, Q)
        input_embeds = torch.cat([query_features, self._word_embedding()(text.input_ids).to(query_features.dtype)], dim=1)
        return self.text_decoder(input_embeds=input_embeds, loss_mask=loss_mask, labels=targets).loss

    @torch.no_grad()
    def generate(self, image, text):
        """Per-sample beam search (beam 5) over the visual prefix (:790-809): list of [1, len] LongTensors on
        the CPU.  prompt_length = attention_mask.sum(-1) - 1, stop token = the tokenizer's <|endoftext|>."""
        _, _, _, query_features = self.visual_prefix(image)
        eos = self.tokenizer.tokenizer.eos if self.tokenizer is not None else self.text_decoder.config.eod_id
        res = []
        for i in range(len(text.input_ids)):
            out = self.text_decoder.generate(text.input_ids[i:i + 1], query_embeds=query_features[i:i + 1], termination_id=eos,
                                             do_sample=False, prompt_length=text.attention_mask.sum(-1)[i] - 1)
            res.append(out.sequences.cpu())
        return res

    @torch.no_grad()
    def generate_batch(self, image, text):
        """What generate(image, text) returns - the same list of [1, len] CPU LongTensors, same stop token and prompt
        lengths - with the visual prefix computed once and the clips decoded together (DistributedGPT3.beam_search_batch:
        the beams of up to 64 // beam clips of equal prompt length share every decoding step)."""
        _, _, _, query_features = self.visual_prefix(image)
        eos = self.tokenizer.tokenizer.eos if self.tokenizer is not None else self.text_decoder.config.eod_id
        out = self.text_decoder.beam_search_batch(text.input_ids, query_embeds=query_features,
                                                  prompt_length=text.attention_mask.sum(-1) - 1, stop_token=eos)
        return [o.sequences.cpu() for o in out]


class _PromptClsBase(_PrefixModelBase):
    """Shared forward pieces of DistributedGPT3_Cls (:431-657) and DistributedGPT3_Retrieval_Cls (:988-1218):
    a caption-style generation loss over `text` ([prompt+answer] pairs, prompt tokens masked out of the
    loss via text.prompt_lengths) and an optional cls_head on the decoder state at the last valid token of
    `prompt_text`."""

    def _gen_pass(self, query_features, text):
        """Decoder pass over [visual prefix | text]; returns (outputs, loss_mask [B, S-1])."""
        Q = query_features.shape[1]
        text_loss_atts = mask_prompt(text.attention_mask[:, 1:].clone(), text.prompt_lengths)
        targets, loss_mask = build_targets(text.input_ids, text_loss_atts, Q)
        emb = self._word_embedding()(text.input_ids).to(query_features.dtype)
        out = self.text_decoder(input_embeds=torch.cat([query_features, emb], dim=1), loss_mask=loss_mask, labels=targets)
        return out, loss_mask

    def _cls_pass(self, query_features, prompt_text, train):
        """cls_head(last_hidden_state at the last valid position of [prefix | prompt])."""
        Q = query_features.shape[1]
        att = prompt_text.attention_mask
        # the reference's (unused) loss of this pass masks with 1-att in training and att in eval
        text_loss_atts = (1 - att[:, 1:]) if train else att[:, 1:].clone()
        targets, loss_mask = build_targets(prompt_text.input_ids, text_loss_atts, Q)
        emb = self._word_embedding()(prompt_text.input_ids).to(query_features.dtype)
        out = self.text_decoder(input_embeds=torch.cat([query_features, emb], dim=1), loss_mask=loss_mask, labels=targets)
        hid = out.last_hidden_state
        pooled = hid[torch.arange(hid.shape[0], device=hid.device), Q + att.sum(dim=-1) - 1]
        return self.cls_head(pooled)


class DistributedGPT3_Cls(_PromptClsBase):
    """Video category prediction (:431-657).  Training: generation loss on [prompt+label] (+ optional
    cls_head CE); eval: every class prompt of every video scored by softmax(-sum(losses * mask))."""

    def __init__(self, config=None, tokenizer=None):
        super().__init__()
        self._build(config, tokenizer, config.get('num_frames', None))
        self.use_cls = config.get('use_cls', False)
        self.num_classes = config.get('num_classes', 45)
        if self.use_cls:
            self.cls_head = nn.Sequential(_Linear(self.text_width, self.text_width), nn.ReLU(),
                                          _Linear(self.text_width, self.num_classes))

    def forward(self, image, text=None, prompt_text=None, labels=None, train=True):
        _, _, _, query_features = self.visual_prefix(image)
        B, Q, _ = query_features.shape
        if train:
            out, _ = self._gen_pass(query_features, text)
            if self.use_cls:
                loss_cls = F.cross_entropy(self._cls_pass(query_features, prompt_text, True).float(), labels)
            else:
                loss_cls = out.loss.new_zeros(())
            return out.loss, loss_cls
        num_cls = text.input_ids.shape[0] // B
        qf = query_features.unsqueeze(1).repeat(1, num_cls, 1, 1).reshape(B * num_cls, Q, -1)
        out, loss_mask = self._gen_pass(qf, text)
        generation_logits = (-(out.losses * loss_mask).sum(dim=-1)).view(B, num_cls).softmax(dim=-1)
        cls_logits = self._cls_pass(query_features, prompt_text, False) if self.use_cls else None
        return generation_logits, cls_logits


class DistributedGPT3_Retrieval_Cls(_PromptClsBase):
    """Video-text matching used by downstream/run_retrieval_distributed_gpt3_itm.py (:988-1218): the B
    prefixes are extended with `negative_indices` (hard negatives), a generation loss plus a 2-way
    match/no-match cls_head; eval scores every (video, text) pair."""

    def __init__(self, config=None, tokenizer=None):
        super().__init__()
        self._build(config, tokenizer, config.get('num_frames', None))
        self.use_cls = config.get('use_cls', False)
        if self.use_cls:
            self.cls_head = nn.Sequential(_Linear(self.text_width, self.text_width), nn.ReLU(),
                                          _Linear(self.text_width, 2))

    def forward(self, image, text=None, prompt_text=None, negative_indices=None, labels=None, train=True):
        _, _, _, query_features = self.visual_prefix(image)
        if train:
            qf = torch.cat([query_features, query_features[negative_indices]], dim=0)
            out, _ = self._gen_pass(qf, text)
            if self.use_cls:
                loss_cls = F.cross_entropy(self._cls_pass(qf, prompt_text, True).float(), labels)
            else:
                loss_cls = out.loss.new_zeros(())
            return out.loss, loss_cls
        V = query_features.shape[0]
        t = text.input_ids.shape[0] // V
        qf = query_features.repeat_interleave(t, dim=0)
        out, loss_mask = self._gen_pass(qf, text)
        generation_logits = (-(out.losses * loss_mask).sum(dim=-1)).view(V, t)
        cls_logits = None
        if self.use_cls:
            cls_logits = self._cls_pass(qf, prompt_text, False).float().softmax(dim=-1)[:, 1].view(V, t)
        return generation_logits, cls_logits


class DistributedGPT3_Retrieval(_PrefixModelBase):
    """Contrastive video-text retrieval (:817-985): CLS-pooled ViT feature vs last-valid-token GPT
    hidden state, all-gathered across ranks (C2/C3 of SURVEY.md section 2.3)."""

    def __init__(self, config=None, tokenizer=None):
        super().__init__()
        self._build(config, tokenizer, config.get('num_frames', None))
        embed_dim = config.get('contrastive_embed_dim', 256)
        self.vision_proj = _Linear(self.vision_width, embed_dim)
        self.text_proj = _Linear(self.text_width, embed_dim)
        self.temp = nn.Parameter(torch.ones([]) * config.get('temp', 0.07))

    def extract_vision_feature(self, image):
        pooled, _ = self.visual_encoder(image)
        return F.normalize(self.vision_proj(pooled).float(), dim=-1)

    def extract_text_feature(self, text):
        targets = torch.cat([text.input_ids[:, 1:], text.input_ids[:, 1:2]], dim=1)
        out = self.text_decoder(tokens=text.input_ids, loss_mask=text.attention_mask[:, 1:].clone(), labels=targets)
        hid = out.last_hidden_state
        pooled = hid[torch.arange(hid.shape[0], device=hid.device), text.attention_mask.sum(dim=-1) - 1]
        return F.normalize(self.text_proj(pooled).float(), dim=-1)

    def forward(self, image, text, idx):
        image_feat = self.extract_vision_feature(image)
        text_feat = self.extract_text_feature(text)
        if torch.distributed.is_initialized():
            image_feat_all = all_gather_cat(image_feat)
            text_feat_all = all_gather_cat(text_feat)
            idx_all = concat_all_gather(idx.view(-1))
        else:
            image_feat_all, text_feat_all, idx_all = image_feat, text_feat, idx.view(-1)
        sim_i2t = YF.matmul_nt(image_feat, text_feat_all) / self.temp
        sim_t2i = YF.matmul_nt(text_feat, image_feat_all) / self.temp
        pos = torch.eq(idx.view(-1, 1), idx_all.view(1, -1)).float()
        sim_targets = pos / pos.sum(1, keepdim=True)
        loss_i2t = -torch.sum(F.log_softmax(sim_i2t, dim=1) * sim_targets, dim=1).mean()
        loss_t2i = -torch.sum(F.log_softmax(sim_t2i, dim=1) * sim_targets, dim=1).mean()
        return (loss_i2t + loss_t2i) / 2
