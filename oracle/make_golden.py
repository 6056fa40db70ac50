"""TEST INFRASTRUCTURE - generates tests/golden/*.pt from the UNMODIFIED reference.

Run in the dev container (needs /root/reference):   python oracle/make_golden.py [--full]

For each config it (1) builds weights with oracle.port.init_state_dict (seeded, reproducible
anywhere), (2) loads them into the reference's DistributedGPT3_Pretrain (via oracle/ref_shims.py),
(3) runs the reference forward+backward on seeded inputs, (4) runs oracle/port.py on the same
inputs and ASSERTS agreement to fp32 round-off - this is what pins the oracle - and (5) stores the
REFERENCE's outputs as the fixture.  Fixtures hold outputs + the recipe (seeds/configs), not weights.
"""
import argparse
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import port, ref_shims  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def make_inputs(B, vcfg, L, vocab, seed):
    g = torch.Generator().manual_seed(seed)
    video = torch.randn(B, 3, vcfg["num_frames"], vcfg["img_size"], vcfg["img_size"], generator=g)
    ids = torch.randint(0, vocab, (B, L), generator=g)
    lens = torch.randint(max(2, L // 4), L + 1, (B,), generator=g)
    att = (torch.arange(L)[None, :] < lens[:, None]).long()
    return video, ids, att


GRAD_KEYS = ["learnable_queries", "visual_fc.weight", "visual_fc.bias", "visual_encoder.cls_token",
             "visual_encoder.pos_embed", "visual_encoder.temporal_embed",
             "visual_encoder.patch_embed.proj.weight", "visual_encoder.norm_pre.weight",
             "visual_encoder.blocks.0.temporal_fc.weight", "visual_encoder.blocks.0.temporal_attn.qkv.weight",
             "visual_encoder.blocks.0.temporal_attn.q_bias", "visual_encoder.blocks.0.attn.qkv.weight",
             "visual_encoder.blocks.0.attn.v_bias", "visual_encoder.blocks.0.attn.proj.bias",
             "visual_encoder.blocks.0.norm1.weight", "visual_encoder.blocks.0.mlp.fc1.weight",
             "visual_encoder.blocks.1.mlp.fc2.bias", "visual_encoder.blocks.1.temporal_ln.bias",
             "visual_encoder.norm.bias", "attn_pool.attn.in_proj_weight", "attn_pool.attn.bias_k",
             "attn_pool.attn.bias_v", "attn_pool.attn.out_proj.weight", "attn_pool.normk.weight",
             "attn_pool.mlp.fc2.weight"]


def sample_grad(g, n=4096):
    """(stride, flattened[::stride]) - keeps fixtures small; tests apply the same stride."""
    flat = g.flatten()
    stride = max(1, flat.numel() // n)
    return stride, flat[::stride].clone()


def run(name, vcfg, gcfg, Q, B, L, wseed, iseed, randomize, sample_logits=None, grads=True):
    t0 = time.time()
    sd = port.init_state_dict(vcfg, gcfg, Q, seed=wseed, randomize=randomize)
    ref_vcfg = dict(vcfg, drop_path=0, use_abs_pos_emb=True)
    model, G = ref_shims.build_reference_pretrain(ref_vcfg, gcfg, Q)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert not missing, missing
    video, ids, att = make_inputs(B, vcfg, L, gcfg["vocab_size"], iseed)
    text = G.BatchEncoding(dict(input_ids=ids, attention_mask=att))
    print(f"[{name}] built in {time.time() - t0:.1f}s; running reference ...", flush=True)

    # ---- reference forward (+ hooks for intermediates) and backward
    inter = {}
    h1 = model.visual_encoder.register_forward_hook(lambda m, i, o: inter.__setitem__("image_embeds", o[1].detach()))
    h2 = model.visual_fc.register_forward_hook(lambda m, i, o: inter.__setitem__("query_features", o.detach()))
    h3 = model.text_decoder.register_forward_hook(lambda m, i, o: inter.__setitem__("gpt", o))
    t0 = time.time()
    loss_ref, _ = model(video, text)
    t_fwd = time.time() - t0
    t0 = time.time()
    if grads:
        loss_ref.backward()
    t_bwd = time.time() - t0
    for h in (h1, h2, h3):
        h.remove()
    out = inter["gpt"]
    ref_grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()
                 if p.grad is not None} if grads else {}
    print(f"[{name}] reference loss {loss_ref.item():.6f} fwd {t_fwd:.1f}s bwd {t_bwd:.1f}s", flush=True)
    del model

    # ---- the port on the same weights/inputs: this comparison is what pins the oracle
    psd = {k: v.clone().requires_grad_(k in port.trainable_keys(sd) and grads) for k, v in sd.items()}
    res = port.pretrain_forward(video, ids, att, psd, vcfg, gcfg, return_all=True)
    if grads:
        res["loss"].backward()

    def chk(a, b, what, tol=2e-4):
        err = (a.float() - b.float()).abs().max().item()
        scale = b.float().abs().max().item() + 1e-12
        assert err <= tol * scale + 1e-6, f"{name}: port != reference for {what}: {err} (scale {scale})"
        return err / scale

    worst = 0.0
    worst = max(worst, chk(res["loss"], loss_ref, "loss", 1e-5))
    worst = max(worst, chk(res["image_embeds"], inter["image_embeds"], "image_embeds"))
    worst = max(worst, chk(res["query_features"], inter["query_features"], "query_features"))
    worst = max(worst, chk(res["logits"], out.logits, "logits"))
    worst = max(worst, chk(res["losses"][:, :-1], out.losses, "losses"))
    worst = max(worst, chk(res["hidden"], out.last_hidden_state, "hidden"))
    ref_targets, ref_mask = port.build_targets(ids, att, Q)
    assert torch.equal(res["targets"], ref_targets)
    for k, gref in ref_grads.items():
        worst = max(worst, chk(psd[k].grad, gref, "grad " + k, 5e-4))
    assert set(ref_grads) == {k for k in psd if psd[k].grad is not None}, "trainable set differs"
    print(f"[{name}] port == reference (worst rel err {worst:.2e}); {len(ref_grads)} grads", flush=True)

    fix = dict(name=name, vcfg=vcfg, gcfg=gcfg, Q=Q, B=B, L=L, wseed=wseed, iseed=iseed,
               randomize=randomize, torch_version=torch.__version__,
               sd_checksum=float(sum(v.double().abs().sum() for v in sd.values())),
               input_checksum=float(video.double().abs().sum() + ids.double().sum() + att.double().sum()),
               loss=loss_ref.detach(), losses=out.losses.detach(), targets=ref_targets, loss_mask=ref_mask,
               ref_fwd_s=t_fwd, ref_bwd_s=t_bwd, port_vs_ref_worst_rel=worst)
    if sample_logits is None:
        fix.update(logits=out.logits.detach(), hidden=out.last_hidden_state.detach(),
                   image_embeds=inter["image_embeds"], query_features=inter["query_features"],
                   grad_norms={k: v.norm() for k, v in ref_grads.items()},
                   grads={k: sample_grad(ref_grads[k]) for k in GRAD_KEYS if k in ref_grads})
    else:
        g = torch.Generator().manual_seed(7)
        lg = out.logits.detach()
        idx = torch.stack([torch.randint(0, n, (sample_logits,), generator=g) for n in lg.shape], dim=1)
        fix.update(logit_idx=idx, logit_vals=lg[idx[:, 0], idx[:, 1], idx[:, 2]],
                   logits_abs_mean=lg.abs().mean(), logits_absmax=lg.abs().max(),
                   image_embeds_norm=inter["image_embeds"].norm(dim=-1),
                   query_features_norm=inter["query_features"].norm(dim=-1),
                   hidden_norm=out.last_hidden_state.detach().norm(dim=-1),
                   grad_norms={k: v.norm() for k, v in ref_grads.items()},
                   grads={k: sample_grad(ref_grads[k]) for k in GRAD_KEYS if k in ref_grads})
    os.makedirs(GOLD, exist_ok=True)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_dropout(name, vcfg, gcfg, Q, B, L, wseed, iseed, p_hidden=0.1, p_attn=0.1, seed=20240924, offset=0):
    """Decoder dropout (the ★ row of the coverage table): the UNMODIFIED reference's DistributedGPT3_Pretrain in
    train() mode with hidden_dropout / attention_dropout live (as in real training: the frozen decoder stays in
    train mode), its F.dropout masks drawn from the B200 kernels' Philox convention (ref_shims.philox_dropout).
    The oracle's restatement with the same masks must agree (pins port.gpt3_layer(drop=...)); the reference's
    outputs and gradients become the fixture the GPU kernels are checked against WITH dropout active."""
    sd = port.init_state_dict(vcfg, gcfg, Q, seed=wseed, randomize=True)
    ref_vcfg = dict(vcfg, drop_path=0, use_abs_pos_emb=True)
    # bias_dropout_fusion=False: the same bias_dropout_add arithmetic (:953-957) through the plain Python function
    # instead of its torch.jit.script twin (:968-979), whose dropout a Python-level patch cannot reach
    model, G = ref_shims.build_reference_model("DistributedGPT3_Pretrain", ref_vcfg, dict(gcfg, bias_dropout_fusion=False), Q,
                                               dropout=(p_hidden, p_attn))
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    model.train()
    video, ids, att = make_inputs(B, vcfg, L, gcfg["vocab_size"], iseed)
    text = G.BatchEncoding(dict(input_ids=ids, attention_mask=att))
    inter = {}
    h3 = model.text_decoder.register_forward_hook(lambda m, i, o: inter.__setitem__("gpt", o))
    with ref_shims.philox_dropout(seed, offset) as pd:
        loss_ref, _ = model(video, text)
        loss_ref.backward()
    h3.remove()
    n_layers = gcfg["num_hidden_layers"]
    assert pd.calls == 1 + 3 * n_layers, pd.calls
    out = inter["gpt"]
    ref_grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    # the same forward without dropout differs (the masks really were applied)
    model.eval()
    with torch.no_grad():
        loss_eval, _ = model(video, text)
    assert abs(loss_eval.item() - loss_ref.item()) > 1e-4 * abs(loss_eval.item())
    del model
    drop = dict(seed=seed, offset=offset, p_hidden=p_hidden, p_attn=p_attn)
    psd = {k: v.clone().requires_grad_(k in port.trainable_keys(sd)) for k, v in sd.items()}
    res = port.pretrain_forward(video, ids, att, psd, vcfg, gcfg, return_all=True, drop=drop)
    res["loss"].backward()

    def chk(a, b, what, tol=2e-4):
        err = (a.float() - b.float()).abs().max().item()
        scale = b.float().abs().max().item() + 1e-12
        assert err <= tol * scale + 1e-6, f"{name}: port != reference for {what}: {err} (scale {scale})"
        return err / scale

    worst = max(chk(res["loss"], loss_ref, "loss", 1e-5), chk(res["logits"], out.logits, "logits"),
                chk(res["losses"][:, :-1], out.losses, "losses"), chk(res["hidden"], out.last_hidden_state, "hidden"))
    for k, gref in ref_grads.items():
        worst = max(worst, chk(psd[k].grad, gref, "grad " + k, 5e-4))
    print(f"[{name}] reference (train mode, Philox masks) loss {loss_ref.item():.6f} vs eval {loss_eval.item():.6f}; "
          f"port == reference (worst rel err {worst:.2e}); {len(ref_grads)} grads", flush=True)
    fix = dict(name=name, vcfg=vcfg, gcfg=gcfg, Q=Q, B=B, L=L, wseed=wseed, iseed=iseed, drop=drop, loss=loss_ref.detach(),
               loss_eval=loss_eval.detach(), losses=out.losses.detach(), logits=out.logits.detach(),
               hidden=out.last_hidden_state.detach(), grad_norms={k: v.norm() for k, v in ref_grads.items()},
               grads={k: sample_grad(ref_grads[k]) for k in GRAD_KEYS if k in ref_grads},
               port_vs_ref_worst_rel=worst, torch_version=torch.__version__)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_image(name, ecfg, gcfg, Q, B, L, wseed, iseed):
    """SURVEY 8f N3: the UNMODIFIED reference's DistributedGPT3_Pretrain_Image with the EVA encoder class
    (models/eva_vit.py VisionTransformer - the class create_eva_vit_g instantiates at 1408 x 40) at tiny dims
    (head_dim 88 kept).  create_eva_vit_g hard-codes the EVA-g dims (:413-424), so the module-level name the model
    constructor looks up is pointed at a small instance of the same class - no reference code is changed."""
    import tempfile, json
    V, G, D = ref_shims.import_reference()
    import models.eva_vit as E
    from functools import partial
    sd = port.eva_state_dict(ecfg, gcfg, Q, seed=wseed)
    td = tempfile.mkdtemp(prefix="ymp_ref_img_")
    json.dump(dict(gcfg, hidden_dropout=0.0, attention_dropout=0.0), open(os.path.join(td, "config.json"), "w"))
    json.dump(dict(img_size=ecfg["img_size"], embed_dim=ecfg["embed_dim"], num_heads=ecfg["num_heads"], mlp_ratio=ecfg["mlp_ratio"],
                   pretrained_ckpt=None, drop_path=0), open(os.path.join(td, "vis.json"), "w"))
    orig = D.create_eva_vit_g
    D.create_eva_vit_g = lambda img_size, norm_layer, drop_path_rate, use_checkpoint: E.VisionTransformer(
        img_size=img_size, patch_size=ecfg["patch_size"], use_mean_pooling=False, embed_dim=ecfg["embed_dim"], depth=ecfg["depth"],
        num_heads=ecfg["num_heads"], mlp_ratio=ecfg["mlp_ratio"], qkv_bias=True, drop_path_rate=drop_path_rate or 0.0,
        norm_layer=norm_layer, use_checkpoint=False)
    try:
        config = dict(visual_cfg=os.path.join(td, "vis.json"), text_cfg=os.path.join(td, "config.json"), text_decoder=td,
                      megatron_cfg={}, num_learnable_token=Q, use_contrastive=False, freeze_text_decoder=True, use_eva_g=True)
        torch.manual_seed(0)
        model = D.DistributedGPT3_Pretrain_Image(config=config, tokenizer=None).eval()
    finally:
        D.create_eva_vit_g = orig
    ref_keys = sorted(k for k in model.state_dict() if not k.endswith("relative_position_index"))
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    g = torch.Generator().manual_seed(iseed)
    image = torch.randn(B, 3, ecfg["img_size"], ecfg["img_size"], generator=g)
    ids = torch.randint(0, gcfg["vocab_size"], (B, L), generator=g)
    lens = torch.randint(max(2, L // 4), L + 1, (B,), generator=g)
    att = (torch.arange(L)[None, :] < lens[:, None]).long()
    inter = {}
    h1 = model.visual_encoder.register_forward_hook(lambda m, i, o: inter.__setitem__("image_embeds", o[1].detach()))
    h3 = model.text_decoder.register_forward_hook(lambda m, i, o: inter.__setitem__("gpt", o))
    loss_ref, _ = model(image, G.BatchEncoding(dict(input_ids=ids, attention_mask=att)))
    loss_ref.backward()
    h1.remove(); h3.remove()
    out = inter["gpt"]
    ref_grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    del model
    train = [k for k in sd if not k.startswith("text_decoder.")]
    psd = {k: v.clone().requires_grad_(k in train) for k, v in sd.items()}
    res = port.pretrain_image_forward(image, ids, att, psd, ecfg, gcfg, return_all=True)
    res["loss"].backward()

    def chk(a, b, what, tol=2e-4):
        err = (a.float() - b.float()).abs().max().item()
        scale = b.float().abs().max().item() + 1e-12
        assert err <= tol * scale + 1e-6, f"{name}: port != reference for {what}: {err} (scale {scale})"
        return err / scale

    worst = max(chk(res["loss"], loss_ref, "loss", 1e-5), chk(res["image_embeds"], inter["image_embeds"], "image_embeds"),
                chk(res["logits"], out.logits, "logits"), chk(res["losses"][:, :-1], out.losses, "losses"))
    assert set(ref_grads) == {k for k in psd if psd[k].grad is not None}
    for k, gref in ref_grads.items():
        worst = max(worst, chk(psd[k].grad, gref, "grad " + k, 5e-4))
    print(f"[{name}] reference loss {loss_ref.item():.6f}; port == reference (worst rel err {worst:.2e}); {len(ref_grads)} grads", flush=True)
    fix = dict(name=name, ecfg=ecfg, gcfg=gcfg, Q=Q, B=B, L=L, wseed=wseed, iseed=iseed, keys=ref_keys, image=image, ids=ids, att=att,
               loss=loss_ref.detach(), losses=out.losses.detach(), logits=out.logits.detach(), image_embeds=inter["image_embeds"],
               grad_norms={k: v.norm() for k, v in ref_grads.items()},
               grads={k: sample_grad(v) for k, v in ref_grads.items() if k.startswith(("visual_encoder.blocks.0.", "visual_encoder.patch_embed",
                                                                                        "visual_encoder.cls_token", "visual_encoder.pos_embed",
                                                                                        "visual_encoder.norm.", "visual_fc", "learnable_queries"))},
               port_vs_ref_worst_rel=worst, torch_version=torch.__version__)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_hostside(name):
    """Pins the two host-side restatements that round 1 only checked against themselves:
    (1) port.clip_to_model_input against the reference's own ClipToTensor + Normalize transform objects
        (dataset/video_utils/volume_transforms.py:15-37, video_transforms.py:1405-1428 -> functional.normalize) -
        the two modules are loaded from their files (the `dataset` package __init__ pulls in decord);
    (2) the product's DistributedGPT3Tokenizer wrapper against the reference's (models/modeling_distributed_gpt3.py:
        42-137,180-319: padding / truncation / [prompt, text] pairs / decode) on a tiny tokenizer.json, with a
        whitespace `jieba.cut` stand-in on both sides (jieba is not in this image; the product falls back to the same
        whitespace segmentation).  The reference's outputs are stored; tests/test_host_cpu.py replays them."""
    import importlib.util
    import tempfile
    import types
    import numpy as np

    def load(modname, path):
        spec = importlib.util.spec_from_file_location(modname, path)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m

    vu = os.path.join(ref_shims.REFERENCE_ROOT, "dataset", "video_utils")
    vol = load("ymp_ref_volume_transforms", os.path.join(vu, "volume_transforms.py"))
    fn = load("ymp_ref_functional", os.path.join(vu, "functional.py"))
    g = torch.Generator().manual_seed(5)
    frames = torch.randint(0, 256, (2, 3, 8, 16, 3), generator=g, dtype=torch.uint8)      # [B,T,H,W,C]
    to_tensor = vol.ClipToTensor(channel_nb=3)
    ref_t = torch.stack([fn.normalize(to_tensor(f), port.CLIP_MEAN, port.CLIP_STD) for f in frames])           # torch uint8 input
    ref_n = torch.stack([fn.normalize(to_tensor(f.numpy()), port.CLIP_MEAN, port.CLIP_STD) for f in frames])   # numpy input (decord off)
    assert torch.equal(ref_t, ref_n)
    got = port.clip_to_model_input(frames)
    assert torch.equal(got.view(torch.int16), ref_t.bfloat16().view(torch.int16)), "port.clip_to_model_input != reference transforms"
    # ---- tokenizer wrapper
    from tokenizers import Tokenizer, models as tk_models, pre_tokenizers
    td = tempfile.mkdtemp(prefix="ymp_tok_")
    vocab = {"<|endoftext|>": 0, "<sep>": 1, "[UNK]": 2, "\n": 3}
    for i, w in enumerate("a b c d e f g hello world video cat dog".split()):
        vocab[w] = 4 + i
    tok = Tokenizer(tk_models.WordLevel(vocab, unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    tok.save(os.path.join(td, "tokenizer.json"))
    jb = types.ModuleType("jieba")
    jb.cut = lambda s: s.split()
    jb.setLogLevel = lambda *_: None
    sys.modules.setdefault("jieba", jb)
    V, G, D = ref_shims.import_reference()
    rt = G.DistributedGPT3Tokenizer(td)
    cases = [dict(data=["hello world", "a b c d e f g"], padding="max_length", truncation=True, max_length=6),
             dict(data=["hello world", "a b c"], padding="longest", truncation=True, max_length=64),
             dict(data=[["video cat", "dog"], ["a b c d e f g", "hello world"]], padding="max_length", max_length=8),
             dict(data=["cat dog video", "hello", "world world world world"], padding="max_length", truncation=True, max_length=4),
             dict(data=[["hello", "a b c d e f g a b c"], ["a b", "c"]], padding="longest", truncation=True, max_length=7)]
    outs = []
    for c in cases:
        kw = {k: v for k, v in c.items() if k != "data"}
        o = rt(c["data"], return_tensors="pt", add_special_tokens=True, **kw)
        outs.append({k: v.clone() for k, v in o.data.items() if torch.is_tensor(v)})
    dec = rt.decode(torch.tensor([11, 12]))
    fix = dict(name=name, clip_frames=frames, clip_out=ref_t, vocab=vocab, cases=cases, outputs=outs, decode_11_12=dec,
               eos=rt.tokenizer.eos, torch_version=torch.__version__)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] reference clip transform == port (bit-exact); {len(cases)} tokenizer cases stored; wrote {path} "
          f"({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_task_configs(name):
    """Stores what the reference ships as data for its task scripts: every configs/**/*.yaml parsed with the YAML loader
    the scripts use (the package's ruamel.yaml stand-in: 1e-6 is a float), keyed by its path under configs/, and the
    class-name table of the classification task (classname.json).  tests/test_host_cpu.py compares the package's yamls
    with the first; the downstream workspace of tests/plumbing.py takes its labels from the second."""
    import glob
    import importlib
    import json
    compat = os.path.join(ROOT, "youku-mplug_b200", "compat")
    sys.path.append(compat)
    try:
        ryaml = importlib.import_module("ruamel.yaml")
    finally:
        sys.path.remove(compat)
    cfg_root = os.path.join(ref_shims.REFERENCE_ROOT, "configs")
    paths = sorted(glob.glob(os.path.join(cfg_root, "**", "*.yaml"), recursive=True))
    configs = {os.path.relpath(p, cfg_root): ryaml.load(open(p), Loader=ryaml.Loader) for p in paths}
    with open(os.path.join(ref_shims.REFERENCE_ROOT, "classname.json")) as f:
        classnames = json.load(f)
    path = os.path.join(GOLD, name + ".json")
    with open(path, "w") as f:
        json.dump(dict(configs=configs, classnames=classnames), f, indent=1)
        f.write("\n")
    print(f"[{name}] {len(configs)} task configs, {len(classnames)} class names; wrote {path} "
          f"({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_generate(name, vcfg, gcfg, Q, B, L, wseed, iseed, beam_size=3, n_new=6, pos_gain=30.0, ln_gain=16.0, stop_after=3):
    """Golden vectors for the generation path (SURVEY 8f N2): the UNMODIFIED reference's per-sample beam
    search and batched greedy sampling over its KV cache, with the visual prefix, next to the oracle's
    full-recompute restatement.  A random tiny decoder with tied embeddings just repeats its last input
    token, so the position embeddings (x pos_gain) and the final LayerNorm affine (x ln_gain) are scaled up:
    the continuations then vary from step to step.  The stop token is chosen as the token greedy decoding
    of sample 0 emits at step `stop_after`, so early termination and finished beams are exercised."""
    def build(eod):
        g = dict(gcfg, tokens_to_generate=n_new, top_k=1, top_p=0.0, eod_id=eod)
        return g, port.generation_state_dict(vcfg, g, Q, wseed, pos_gain, ln_gain)

    video, ids, att = make_inputs(B, vcfg, L, gcfg["vocab_size"], iseed)
    plen = att.sum(-1) - 1               # DistributedGPT3_Caption.generate: prompt_length = mask.sum(-1) - 1
    g0, sd = build(eod=gcfg["vocab_size"] - 1)
    with torch.no_grad():
        qf_port = port.visual_prefix(video, sd, vcfg)[3]
        probe = port.sample_generate(ids.clone(), sd, g0, query_features=qf_port, prompt_length=plen.clone(), tokens_to_generate=n_new,
                                     eod_id=g0["eod_id"], top_k=1, top_p=0.0)
    eod = int(probe[0, int(plen[0]) + stop_after])
    ids[ids == eod] = (eod + 1) % gcfg["vocab_size"]   # no accidental stop tokens inside the prompts
    gcfg, sd = build(eod)
    ref_vcfg = dict(vcfg, drop_path=0, use_abs_pos_emb=True)
    model, G = ref_shims.build_reference_pretrain(ref_vcfg, gcfg, Q)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    with torch.no_grad():
        _, image_embeds = model.visual_encoder(video)
        image_query = model.attn_pool(model.learnable_queries.repeat(B, 1, 1), image_embeds)
        qf = model.visual_norm(model.visual_fc(image_query))
        ref_beam = [model.text_decoder.generate(ids[i:i + 1], query_embeds=qf[i:i + 1], termination_id=eod, do_sample=False,
                                                prompt_length=plen[i], beam_size=beam_size) for i in range(B)]
        ref_greedy = model.text_decoder.generate(ids.clone(), query_embeds=qf, termination_id=eod, do_sample=True,
                                                 prompt_length=plen.clone())
    del model
    # the reference's sampling filters on seeded logits (pure torch functions of the reference module)
    fl = torch.randn(4, 50, generator=torch.Generator().manual_seed(0))
    a, b = fl.clone(), fl.clone()
    G.modify_logits_for_top_k_filtering(a, 5)
    G.modify_logits_for_top_p_filtering(b, 0.7)
    torch.manual_seed(3)
    drawn = G.sample(fl, top_k=0, top_p=0.9, temperature=0.7, vocab_size=40)
    filters = dict(logits=fl, top_k5=a, top_p07=b, sample_seed3_p09_t07_v40=drawn, greedy=G.sample(fl, top_k=1))
    assert torch.equal(a, port.filter_top_k(fl, 5)) and torch.equal(b, port.filter_top_p(fl, 0.7))
    torch.manual_seed(3)
    assert torch.equal(drawn, port.pick_token(fl, top_k=0, top_p=0.9, temperature=0.7, vocab_size=40))
    with torch.no_grad():
        qf_port = port.visual_prefix(video, sd, vcfg)[3]
        assert (qf_port - qf).abs().max() <= 2e-4 * qf.abs().max()
        beams = []
        for i in range(B):
            seq, sc = port.beam_search_generate(ids[i:i + 1], sd, gcfg, query_features=qf_port[i:i + 1], prompt_length=plen[i],
                                                beam_size=beam_size, stop_token=eod, tokens_to_generate=n_new, eod_id=eod)
            assert torch.equal(seq, ref_beam[i].sequences), (name, i, seq, ref_beam[i].sequences)
            assert (sc - ref_beam[i].scores.reshape(-1)).abs().max() < 1e-4, (sc, ref_beam[i].scores)
            beams.append((ref_beam[i].sequences.clone(), ref_beam[i].scores.reshape(-1).clone()))
        greedy = port.sample_generate(ids.clone(), sd, gcfg, query_features=qf_port, prompt_length=plen.clone(), tokens_to_generate=n_new,
                                      eod_id=eod, top_k=1, top_p=0.0, termination_id=eod)
        assert torch.equal(greedy, ref_greedy), (greedy, ref_greedy)
        # teacher-forced next-token log-probs along the greedy sequences (what a bf16 run is compared with)
        steps = []
        for i in range(B):
            for t in range(int(plen[i]), ref_greedy.shape[1]):
                lp = torch.log_softmax(port.next_token_logits(qf_port[i:i + 1], ref_greedy[i:i + 1, :t], sd, gcfg)[0], -1)
                top = torch.topk(lp, 2)
                steps.append(dict(sample=i, pos=t, logprobs=lp.clone(), margin=float(top[0][0] - top[0][1])))
    print(f"[{name}] stop token {eod}; port == reference: beam {[b[0].tolist() for b in beams]} scores {[b[1].tolist() for b in beams]}\n"
          f"[{name}] greedy {ref_greedy.tolist()} min margin {min(s['margin'] for s in steps):.3f}", flush=True)
    fix = dict(name=name, vcfg=vcfg, gcfg=gcfg, Q=Q, B=B, L=L, wseed=wseed, iseed=iseed, beam_size=beam_size, n_new=n_new,
               pos_gain=pos_gain, ln_gain=ln_gain, eod=eod, ids=ids, att=att, prompt_length=plen, video_checksum=float(video.double().abs().sum()),
               query_features=qf.detach(), beam_sequences=[b[0] for b in beams], beam_scores=[b[1] for b in beams], greedy=ref_greedy,
               steps=steps, filters=filters, torch_version=torch.__version__)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_downstream(name, vcfg, gcfg, Q, wseed):
    """Golden vectors for the downstream task models (SURVEY 8a rows a20-a23): the UNMODIFIED reference's
    DistributedGPT3_Cls (train + eval, use_cls), _Caption (forward), _Retrieval (features + loss) and
    _Retrieval_Cls (train + eval) on CPU next to the oracle's compositions (oracle/port.py)."""
    import torch.distributed as dist
    if not dist.is_initialized():  # the retrieval model all-gathers its features (world size 1 here)
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:29533", rank=0, world_size=1)
    ref_vcfg = dict(vcfg, drop_path=0, use_abs_pos_emb=True)
    H, D = gcfg["hidden_size"], vcfg["embed_dim"]
    g = torch.Generator().manual_seed(wseed + 1)

    def sd_with(extra):
        sd = port.init_state_dict(vcfg, gcfg, Q, seed=wseed, randomize=True)
        for k, shape in extra.items():
            sd[k] = 0.05 * torch.randn(shape, generator=g)
        return sd

    def load(cls_name, sd, **cfg):
        model, G = ref_shims.build_reference_model(cls_name, ref_vcfg, gcfg, Q, **cfg)
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected and not missing, (cls_name, missing, unexpected)
        return model, G

    def chk(a, b, what, tol=2e-4):
        err = (a.float() - b.float()).abs().max().item()
        scale = b.float().abs().max().item() + 1e-12
        assert err <= tol * scale + 1e-6, f"{name}: port != reference for {what}: {err} (scale {scale})"

    fix = dict(name=name, vcfg=vcfg, gcfg=gcfg, Q=Q, wseed=wseed, torch_version=torch.__version__)
    B, L, ncls = 2, 8, 3
    head = {"cls_head.0.weight": (H, H), "cls_head.0.bias": (H,), "cls_head.2.weight": (5, H), "cls_head.2.bias": (5,)}
    with torch.no_grad():
        # ---------------- DistributedGPT3_Cls
        sd = sd_with(head)
        model, G = load("DistributedGPT3_Cls", sd, use_cls=True, num_classes=5)
        video, ids, att = make_inputs(B, vcfg, L, gcfg["vocab_size"], 31)
        _, pids, patt = make_inputs(B, vcfg, L, gcfg["vocab_size"], 32)
        pl, labels = torch.tensor([2, 3]), torch.tensor([1, 4])
        enc = lambda **kw: G.BatchEncoding(dict(kw))  # noqa: E731
        lc, lk = model(video, enc(input_ids=ids, attention_mask=att, prompt_lengths=pl), enc(input_ids=pids, attention_mask=patt),
                       labels, train=True)
        qf = port.visual_prefix(video, sd, vcfg)[3]
        plc, plk = port.cls_train_losses(qf, ids, att, pl, pids, patt, labels, sd, gcfg)
        chk(plc, lc, "cls train loss_caption", 1e-5)
        chk(plk, lk, "cls train loss_cls", 1e-5)
        _, cids, catt = make_inputs(B * ncls, vcfg, L, gcfg["vocab_size"], 33)
        cpl = torch.randint(1, 4, (B * ncls,), generator=torch.Generator().manual_seed(5))
        gen, clsl = model(video, enc(input_ids=cids, attention_mask=catt, prompt_lengths=cpl), enc(input_ids=pids, attention_mask=patt),
                          train=False)
        chk(port.cls_eval_scores(qf, cids, catt, cpl, sd, gcfg, ncls), gen, "cls eval generation_logits")
        chk(port.cls_head(port.prompt_pooled_hidden(qf, pids, patt, sd, gcfg), sd), clsl, "cls eval cls_logits")
        fix["cls"] = dict(seeds=(31, 32, 33), prompt_lengths=pl, labels=labels, eval_prompt_lengths=cpl, ncls=ncls,
                          head={k: sd[k] for k in head}, loss_caption=lc, loss_cls=lk, eval_generation=gen, eval_cls_logits=clsl)
        del model
        # ---------------- DistributedGPT3_Caption
        sd = sd_with({})
        model, G = load("DistributedGPT3_Caption", sd)
        loss = model(video, G.BatchEncoding(dict(input_ids=ids, attention_mask=att, prompt_lengths=pl)))
        chk(port.prefix_decoder_pass(qf, ids, att, pl, sd, gcfg)["loss"], loss, "caption loss", 1e-5)
        fix["caption"] = dict(seed=31, prompt_lengths=pl, loss=loss)
        del model
        # ---------------- DistributedGPT3_Retrieval
        proj = {"vision_proj.weight": (32, D), "vision_proj.bias": (32,), "text_proj.weight": (32, H), "text_proj.bias": (32,)}
        sd = sd_with(proj)
        sd["temp"] = torch.tensor(0.07)
        model, G = load("DistributedGPT3_Retrieval", sd, contrastive_embed_dim=32)
        video3, ids3, att3 = make_inputs(3, vcfg, L, gcfg["vocab_size"], 41)
        idx = torch.tensor([7, 9, 7])
        text3 = G.BatchEncoding(dict(input_ids=ids3, attention_mask=att3))
        rv, rt = model.extract_vision_feature(video3), model.extract_text_feature(text3)
        rloss = model(video3, text3, idx)
        pv, pt = port.retrieval_features(video3, ids3, att3, sd, vcfg, gcfg)
        chk(pv, rv, "retrieval vision feature")
        chk(pt, rt, "retrieval text feature")
        chk(port.retrieval_loss(pv, pt, idx, 0.07), rloss, "retrieval loss", 1e-5)
        fix["retrieval"] = dict(seed=41, idx=idx, proj={k: sd[k] for k in proj}, vision_feats=rv, text_feats=rt, loss=rloss)
        del model
        # ---------------- DistributedGPT3_Retrieval_Cls
        head2 = {"cls_head.0.weight": (H, H), "cls_head.0.bias": (H,), "cls_head.2.weight": (2, H), "cls_head.2.bias": (2,)}
        sd = sd_with(head2)
        model, G = load("DistributedGPT3_Retrieval_Cls", sd, use_cls=True, num_classes=2)
        videoB, _, _ = make_inputs(B, vcfg, L, gcfg["vocab_size"], 51)
        _, ids4, att4 = make_inputs(2 * B, vcfg, L, gcfg["vocab_size"], 52)       # positives then negatives
        pl4, neg, lab4 = torch.tensor([2, 2, 3, 1]), torch.tensor([1, 0]), torch.tensor([1, 1, 0, 0])
        text4 = G.BatchEncoding(dict(input_ids=ids4, attention_mask=att4, prompt_lengths=pl4))
        prompt4 = G.BatchEncoding(dict(input_ids=ids4, attention_mask=att4))
        lc4, lk4 = model(videoB, text4, prompt4, neg, lab4, train=True)
        qfB = port.visual_prefix(videoB, sd, vcfg)[3]
        p_lc4, p_lk4 = port.retrieval_cls_train_losses(qfB, neg, ids4, att4, pl4, ids4, att4, lab4, sd, gcfg)
        chk(p_lc4, lc4, "retrieval_cls train loss_caption", 1e-5)
        chk(p_lk4, lk4, "retrieval_cls train loss_cls", 1e-5)
        gen4, cls4 = model(videoB, text4, prompt4, train=False)
        p_gen4, p_cls4 = port.retrieval_cls_eval(qfB, ids4, att4, pl4, ids4, att4, sd, gcfg)
        chk(p_gen4, gen4, "retrieval_cls eval generation_logits")
        chk(p_cls4, cls4, "retrieval_cls eval cls_logits")
        fix["retrieval_cls"] = dict(seeds=(51, 52), prompt_lengths=pl4, negative_indices=neg, labels=lab4, head={k: sd[k] for k in head2},
                                    loss_caption=lc4, loss_cls=lk4, eval_generation=gen4, eval_cls=cls4)
        del model
        # ---------------- DistributedGPT3_Pretrain with the contrastive branch (SURVEY 8a row a17)
        sd = sd_with(proj)
        sd["temp"] = torch.tensor(0.07)
        model, G = load("DistributedGPT3_Pretrain", sd, use_contrastive=True, contrastive_embed_dim=32)
        lcap, lcon = model(video3, G.BatchEncoding(dict(input_ids=ids3, attention_mask=att3)))
        chk(port.pretrain_forward(video3, ids3, att3, sd, vcfg, gcfg), lcap, "pretrain(contrastive) loss_caption", 1e-5)
        chk(port.pretrain_contrastive_loss(video3, ids3, att3, sd, vcfg, gcfg, 0.07), lcon, "pretrain loss_contrastive", 1e-5)
        fix["pretrain_contrastive"] = dict(seed=41, proj={k: sd[k] for k in proj}, loss_caption=lcap, loss_contrastive=lcon)
        del model
    print(f"[{name}] port == reference for Cls (train/eval), Caption, Retrieval (features/loss), Retrieval_Cls (train/eval), "
          f"Pretrain + contrastive", flush=True)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def run_caption_full(name, vcfg, gcfg, Q, B, L, wseed, iseed, sample_logits=2048):
    """BASELINE config-4 at its real dims (configs/caption/caption_gpt3_2.7B_youku_v0.yaml:19,30 + BASELINE.json:
    GPT-3 2.7B = 32 layers x 2560, 32 heads x 80; 16 frames; text 256 -> S = 128 + 256 = 384): the UNMODIFIED
    reference's DistributedGPT3_Caption.forward + backward (models/distributed_gpt3.py:751-788) on CPU in fp32, the
    oracle's restatement beside it (asserted equal), and the reference's loss / sampled logits / norms / sampled
    gradients stored as the fixture."""
    t0 = time.time()
    sd = port.init_state_dict(vcfg, gcfg, Q, seed=wseed, randomize=False)
    ref_vcfg = dict(vcfg, drop_path=0, use_abs_pos_emb=True)
    model, G = ref_shims.build_reference_model("DistributedGPT3_Caption", ref_vcfg, gcfg, Q)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    video, ids, att = make_inputs(B, vcfg, L, gcfg["vocab_size"], iseed)
    pl = torch.tensor([5] * B)
    text = G.BatchEncoding(dict(input_ids=ids, attention_mask=att, prompt_lengths=pl))
    print(f"[{name}] built in {time.time() - t0:.1f}s; running reference ...", flush=True)
    inter = {}
    h1 = model.visual_encoder.register_forward_hook(lambda m, i, o: inter.__setitem__("image_embeds", o[1].detach()))
    h2 = model.visual_fc.register_forward_hook(lambda m, i, o: inter.__setitem__("query_features", o.detach()))
    h3 = model.text_decoder.register_forward_hook(lambda m, i, o: inter.__setitem__("gpt", o))
    t0 = time.time()
    loss_ref = model(video, text)
    t_fwd = time.time() - t0
    t0 = time.time()
    loss_ref.backward()
    t_bwd = time.time() - t0
    for h in (h1, h2, h3):
        h.remove()
    out = inter["gpt"]
    ref_grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    print(f"[{name}] reference loss {loss_ref.item():.6f} fwd {t_fwd:.1f}s bwd {t_bwd:.1f}s", flush=True)
    lg = out.logits.detach()
    g = torch.Generator().manual_seed(7)
    idx = torch.stack([torch.randint(0, n, (sample_logits,), generator=g) for n in lg.shape], dim=1)
    fix = dict(name=name, vcfg=vcfg, gcfg=gcfg, Q=Q, B=B, L=L, wseed=wseed, iseed=iseed, prompt_lengths=pl,
               torch_version=torch.__version__,
               sd_checksum=float(sum(v.double().abs().sum() for v in sd.values())),
               loss=loss_ref.detach(), losses=out.losses.detach(),
               logit_idx=idx, logit_vals=lg[idx[:, 0], idx[:, 1], idx[:, 2]].clone(),
               logits_abs_mean=lg.abs().mean(), logits_absmax=lg.abs().max(),
               image_embeds_norm=inter["image_embeds"].norm(dim=-1),
               query_features_norm=inter["query_features"].norm(dim=-1),
               hidden_norm=out.last_hidden_state.detach().norm(dim=-1),
               grad_norms={k: v.norm() for k, v in ref_grads.items()},
               grads={k: sample_grad(ref_grads[k]) for k in GRAD_KEYS if k in ref_grads},
               ref_fwd_s=t_fwd, ref_bwd_s=t_bwd)
    del model, lg, inter["gpt"]
    # ---- the oracle on the same weights / inputs (pins the 2.7B-shape restatement: hd 80, S 384, T 16)
    train = set(port.trainable_keys(sd))
    psd = {k: v.clone().requires_grad_(k in train) for k, v in sd.items()}
    qf = port.visual_prefix(video, psd, vcfg)[3]
    res = port.prefix_decoder_pass(qf, ids, att, pl, psd, gcfg)
    res["loss"].backward()
    worst = 0.0

    def chk(a, b, what, tol=2e-4):
        err = (a.float() - b.float()).abs().max().item()
        scale = b.float().abs().max().item() + 1e-12
        assert err <= tol * scale + 1e-6, f"{name}: port != reference for {what}: {err} (scale {scale})"
        return err / scale

    worst = max(worst, chk(res["loss"], loss_ref, "loss", 1e-5))
    worst = max(worst, chk(res["losses"], out.losses, "losses"))
    worst = max(worst, chk(res["logits"][idx[:, 0], idx[:, 1], idx[:, 2]], fix["logit_vals"], "sampled logits"))
    for k, gref in ref_grads.items():
        worst = max(worst, chk(psd[k].grad, gref, "grad " + k, 5e-4))
    fix["port_vs_ref_worst_rel"] = worst
    print(f"[{name}] port == reference (worst rel err {worst:.2e}); {len(ref_grads)} grads", flush=True)
    path = os.path.join(GOLD, name + ".pt")
    torch.save(fix, path)
    print(f"[{name}] wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also the real 1.3B / T=8 / B=1 config (~6 GB RAM, minutes)")
    ap.add_argument("--caption27b", action="store_true", help="only the 2.7B caption config at its real dims (~35 GB RAM, minutes)")
    ap.add_argument("--only-image", action="store_true", help="only the EVA / Pretrain_Image fixture (N3)")
    ap.add_argument("--only-hostside", action="store_true", help="only the clip-transform / tokenizer fixture")
    ap.add_argument("--only-dropout", action="store_true", help="only (re)write the decoder-dropout fixture")
    ap.add_argument("--only-generate", action="store_true", help="only (re)write the generation fixture")
    ap.add_argument("--only-downstream", action="store_true", help="only (re)write the downstream-model fixture")
    ap.add_argument("--only-task-configs", action="store_true", help="only (re)write the task-config / class-name fixture")
    a = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    if a.caption27b:
        run_caption_full("full_2p7b_caption_T16_B1", dict(port.VCFG_CLIP_B16, num_frames=16), port.GCFG_2_7B, Q=128, B=1, L=256,
                         wseed=0, iseed=4321)
        sys.exit(0)
    if a.only_image:
        run_image("tiny_pretrain_image", port.ECFG_TINY, port.GCFG_TINY, Q=8, B=2, L=8, wseed=71, iseed=72)
        sys.exit(0)
    if a.only_hostside:
        run_hostside("tiny_hostside")
        sys.exit(0)
    if a.only_dropout:
        run_dropout("tiny_pretrain_dropout", port.VCFG_TINY, port.GCFG_TINY, Q=8, B=2, L=8, wseed=61, iseed=62)
        sys.exit(0)
    if a.only_downstream:
        run_downstream("tiny_downstream", port.VCFG_TINY, port.GCFG_TINY, Q=8, wseed=21)
        sys.exit(0)
    if a.only_task_configs:
        run_task_configs("reference_task_configs")
        sys.exit(0)
    run_task_configs("reference_task_configs")
    run_hostside("tiny_hostside")
    run_image("tiny_pretrain_image", port.ECFG_TINY, port.GCFG_TINY, Q=8, B=2, L=8, wseed=71, iseed=72)
    run_generate("tiny_generate", port.VCFG_TINY, port.GCFG_TINY, Q=8, B=2, L=8, wseed=51, iseed=52)
    if a.only_generate:
        sys.exit(0)
    run_downstream("tiny_downstream", port.VCFG_TINY, port.GCFG_TINY, Q=8, wseed=21)
    run_dropout("tiny_pretrain_dropout", port.VCFG_TINY, port.GCFG_TINY, Q=8, B=2, L=8, wseed=61, iseed=62)
    run("tiny_pretrain", port.VCFG_TINY, port.GCFG_TINY, Q=8, B=2, L=8, wseed=11, iseed=12, randomize=True)
    run("tiny_pretrain_refinit", port.VCFG_TINY, port.GCFG_TINY, Q=8, B=1, L=6, wseed=13, iseed=14, randomize=False)
    if a.full:
        run("full_1p3b_T8_B1", port.VCFG_CLIP_B16, port.GCFG_1_3B, Q=128, B=1, L=128, wseed=0, iseed=1234,
            randomize=False, sample_logits=2048)
