"""CPU: host-side logic of the drop-in package - state_dict surface, config checks, tokenizer
padding rules, C-ABI exports.  No kernel is launched here."""
import ctypes
import json
import os
import re

import pytest
import torch

from oracle import port
from helpers import build_pretrain, make_model_dir, pretrain_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "ymp.h")).read()
    names = set(re.findall(r"\b(ymp_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 15
    lib = ctypes.CDLL(os.path.join(ROOT, "youku-mplug_b200", "ymp", "libymp_b200.so"))
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/ymp.h but not exported"
    lib.ymp_abi_version.restype = ctypes.c_int
    assert lib.ymp_abi_version() == 3


def test_ctypes_structs_match_header_field_order():
    """Every struct in include/ymp.h has a ctypes mirror with the same field names in order."""
    from ymp import lib as L
    hdr = open(os.path.join(ROOT, "include", "ymp.h")).read()
    mirrors = {"ymp_gemm_args": L.GemmArgs, "ymp_layernorm_args": L.LayerNormArgs, "ymp_layernorm_bwd_args": L.LayerNormBwdArgs,
               "ymp_seqmap": L.SeqMap, "ymp_attn_args": L.AttnArgs, "ymp_attn_bwd_args": L.AttnBwdArgs,
               "ymp_adamw_args": L.AdamwArgs, "ymp_im2col_args": L.Im2colArgs, "ymp_clip_args": L.ClipArgs, "ymp_embed_args": L.EmbedArgs,
               "ymp_ce_args": L.CeArgs, "ymp_colsum_args": L.ColsumArgs, "ymp_group_args": L.GroupArgs,
               "ymp_dropout_spec": L.DropoutSpec, "ymp_dropout_args": L.DropoutArgs, "ymp_gemm_skinny_args": L.GemmSkinnyArgs}
    for name, cls in mirrors.items():
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), hdr, re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        fields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(","):
                fields.append(re.findall(r"([A-Za-z_][A-Za-z0-9_]*)\s*$", part.strip())[0])
        py = [f[0].rstrip("_") for f in cls._fields_]
        assert [f.rstrip("_") for f in fields] == py, (name, fields, py)


def test_gemm_rejects_bad_arguments_without_gpu():
    from ymp import lib as L
    g = L.GemmArgs()
    rc = L._gemm(ctypes.byref(g), None)
    assert rc == -1 and b"null" in L.lib.ymp_last_error()


def test_state_dict_keys_match_reference_surface():
    m = build_pretrain(port.VCFG_TINY, port.GCFG_TINY, 8)
    ref = port.init_state_dict(port.VCFG_TINY, port.GCFG_TINY, 8)  # == reference keys (pinned by make_golden)
    sd = m.state_dict()
    assert set(sd) == set(ref)
    for k in ref:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k
    # frozen decoder, trainable rest (models/distributed_gpt3.py:86-93)
    train = {k for k, p in m.named_parameters() if p.requires_grad}
    assert train == set(port.trainable_keys(ref))
    assert m.no_weight_decay() == {'visual_encoder.pos_embed', 'visual_encoder.cls_token', 'visual_encoder.temporal_embed'}


def test_freeze_vit_keeps_only_temporal_parameters():
    m = build_pretrain(port.VCFG_TINY, port.GCFG_TINY, 8, freeze_vit=True)
    train = {k for k, p in m.named_parameters() if p.requires_grad}
    ref = port.init_state_dict(port.VCFG_TINY, port.GCFG_TINY, 8)
    assert train == set(port.trainable_keys(ref, freeze_vit=True))


def test_tensor_parallel_config_is_rejected():
    td = make_model_dir(port.VCFG_TINY, port.GCFG_TINY)
    cfg = pretrain_config(td, 8)
    cfg["megatron_cfg"] = {"world_size": 1, "model_parallel_size": 8, "tensor_model_parallel_size": 8}
    os.environ["YMP_ALLOW_RANDOM_INIT"] = "1"
    import models.distributed_gpt3 as D
    with pytest.raises(ValueError):
        D.DistributedGPT3_Pretrain(config=cfg, tokenizer=None)


def test_cpu_forward_fails_loudly():
    """No CPU fallback: the product path must refuse to run without the CUDA kernels."""
    m = build_pretrain(port.VCFG_TINY, port.GCFG_TINY, 8)
    import models.modeling_distributed_gpt3 as G
    text = G.BatchEncoding(dict(input_ids=torch.randint(0, 512, (1, 6)), attention_mask=torch.ones(1, 6, dtype=torch.long)))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 3, 2, 32, 32), text)


def test_build_targets_bit_exact_vs_oracle():
    import models.distributed_gpt3 as D
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(0, 51200, (4, 16), generator=g)
    att = (torch.arange(16)[None] < torch.tensor([[16], [9], [2], [5]])).long()
    t, m = D.build_targets(ids, att[:, 1:], 7)
    t2, m2 = port.build_targets(ids, att, 7)
    assert torch.equal(t, t2) and torch.equal(m, m2)


def _tiny_tokenizer_dir():
    from tokenizers import Tokenizer, models, pre_tokenizers
    td = make_model_dir(port.VCFG_TINY, port.GCFG_TINY)
    vocab = {"<|endoftext|>": 0, "<sep>": 1, "[UNK]": 2, "\n": 3}
    for i, w in enumerate("a b c d e f g hello world video cat dog".split()):
        vocab[w] = 4 + i
    tok = Tokenizer(models.WordLevel(vocab, unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    tok.save(os.path.join(td, "tokenizer.json"))
    return td


def test_tokenizer_padding_and_truncation_rules():
    import models.modeling_distributed_gpt3 as G
    tk = G.DistributedGPT3Tokenizer(_tiny_tokenizer_dir())
    out = tk(["hello world", "a b c d e f g"], padding='max_length', truncation=True, max_length=6, return_tensors='pt')
    assert out.input_ids.shape == (2, 6) and out.input_ids.dtype == torch.long
    assert out.input_ids[0].tolist() == [1, 11, 12, 0, 0, 0]          # <sep> hello world <eot> pad pad
    assert out.attention_mask[0].tolist() == [1, 1, 1, 1, 0, 0]
    assert out.input_ids[1].tolist() == [1, 4, 5, 6, 7, 8]             # truncated, no eos left
    assert out.attention_mask[1].tolist() == [1] * 6
    out = tk(["hello world", "a b c"], padding='longest', truncation=True, max_length=64)
    assert out.input_ids.shape == (2, 5)
    pair = tk([["video cat", "dog"], ["a b c d e f g", "hello world"]], padding='max_length', max_length=8)
    assert pair.input_ids.shape == (2, 8)
    assert pair.prompt_lengths.tolist() == [2, 4]                      # second prompt cut to make room
    assert pair.input_ids[1].tolist() == [1, 4, 5, 6, 7, 11, 12, 0]
    assert pair.to("cpu").attention_mask[0].tolist() == [1, 1, 1, 1, 1, 0, 0, 0]
    assert tk.decode(torch.tensor([11, 12])) == "hello world"
    assert tk.tokenizer.eos == 0


def test_resize_embeddings():
    import models.vision_transformer as V
    pe = torch.randn(1, 1 + 4, 8)
    out = V.resize_pos_embed(pe, torch.zeros(1, 1 + 16, 8))
    assert out.shape == (1, 17, 8) and torch.equal(out[:, 0], pe[:, 0])
    te = torch.randn(1, 4, 8)
    assert V.resize_temporal_embed(te, torch.zeros(1, 8, 8)).shape == (1, 8, 8)
    assert torch.equal(V.resize_temporal_embed(te, torch.zeros(1, 4, 8)), te)


def test_clip_lut_equals_reference_ops():
    """The table the GPU kernel gathers from reproduces ClipToTensor + Normalize + bf16 cast bit for bit."""
    from ymp import ops
    g = torch.Generator().manual_seed(5)
    frames = torch.randint(0, 256, (2, 3, 8, 16, 3), generator=g, dtype=torch.uint8)
    ref = port.clip_to_model_input(frames)
    lut = ops.clip_lut(port.CLIP_MEAN, port.CLIP_STD, "cpu").view(3, 256)
    got = torch.stack([lut[c][frames[..., c].long()] for c in range(3)], dim=1)  # [B,C,T,H,W]
    assert torch.equal(got.view(torch.int16), ref.view(torch.int16))


def test_hostside_fixture_from_the_reference():
    """tests/golden/tiny_hostside.pt (oracle/make_golden.py run_hostside): the reference's own ClipToTensor + Normalize
    output and the reference's own DistributedGPT3Tokenizer outputs; the oracle's clip restatement and the product's
    tokenizer wrapper must reproduce them exactly (token ids, masks, prompt lengths are integer work)."""
    import models.modeling_distributed_gpt3 as G
    from tokenizers import Tokenizer, models, pre_tokenizers
    fx = torch.load(os.path.join(ROOT, "tests", "golden", "tiny_hostside.pt"), weights_only=False)
    got = port.clip_to_model_input(fx["clip_frames"])
    assert torch.equal(got.view(torch.int16), fx["clip_out"].bfloat16().view(torch.int16))
    td = make_model_dir(port.VCFG_TINY, port.GCFG_TINY)
    tok = Tokenizer(models.WordLevel(fx["vocab"], unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    tok.save(os.path.join(td, "tokenizer.json"))
    tk = G.DistributedGPT3Tokenizer(td)
    for case, want in zip(fx["cases"], fx["outputs"]):
        kw = {k: v for k, v in case.items() if k != "data"}
        out = tk(case["data"], return_tensors="pt", add_special_tokens=True, **kw)
        for k, v in want.items():
            assert torch.equal(getattr(out, k), v), (case, k, getattr(out, k), v)
    assert tk.decode(torch.tensor([11, 12])) == fx["decode_11_12"]
    assert tk.tokenizer.eos == fx["eos"]


def test_pretrain_image_state_dict_surface_and_oracle():
    """SURVEY 8f N3: DistributedGPT3_Pretrain_Image (EVA encoder) exposes the reference's state-dict keys (from the
    unmodified reference, tests/golden/tiny_pretrain_image.pt) and the oracle's eva restatement reproduces the
    reference's loss / logits / encoder output on the fixture's inputs."""
    from helpers import build_pretrain_image
    fx = torch.load(os.path.join(ROOT, "tests", "golden", "tiny_pretrain_image.pt"), weights_only=False)
    m = build_pretrain_image(fx["ecfg"], fx["gcfg"], fx["Q"])
    assert sorted(m.state_dict().keys()) == fx["keys"]
    frozen = {k for k, p in m.named_parameters() if not p.requires_grad}
    assert frozen and all(k.startswith("text_decoder.") for k in frozen)
    sd = port.eva_state_dict(fx["ecfg"], fx["gcfg"], fx["Q"], seed=fx["wseed"])
    with torch.no_grad():
        res = port.pretrain_image_forward(fx["image"], fx["ids"], fx["att"], sd, fx["ecfg"], fx["gcfg"], return_all=True)
    assert abs(res["loss"].item() - fx["loss"].item()) < 1e-5 * abs(fx["loss"].item())
    assert (res["image_embeds"] - fx["image_embeds"]).abs().max() < 2e-4 * fx["image_embeds"].abs().max()
    assert (res["logits"] - fx["logits"]).abs().max() < 2e-4 * fx["logits"].abs().max()
    import models.eva_vit as E
    g = E.create_eva_vit_g(img_size=224, drop_path_rate=0, norm_layer=None)
    assert g.ecfg["embed_dim"] == 1408 and g.ecfg["depth"] == 40 and g.ecfg["num_heads"] == 16 and g.pos_embed.shape == (1, 257, 1408)
    assert g.get_parameter("blocks.39.mlp.fc1.weight").shape == (6144, 1408)


def test_task_configs_mirror_the_reference_yamls():
    """configs/{pretrain,caption,cls,retrieval}/*.yaml: every file the reference ships for the GPT-3 models exists here
    under the same name, parses with the YAML loader the scripts use (ruamel.yaml semantics: 1e-6 is a float), and
    carries the same keys and values as the reference's file except for megatron_cfg (tensor parallel size 1 here)."""
    import importlib
    import sys
    compat = os.path.join(ROOT, "youku-mplug_b200", "compat")
    sys.path.append(compat)
    try:
        ryaml = importlib.import_module("ruamel.yaml")
    finally:
        sys.path.remove(compat)
        for k in [k for k in sys.modules if k == "ruamel" or k.startswith("ruamel.")]:
            del sys.modules[k]
    cfg_root = os.path.join(ROOT, "youku-mplug_b200", "configs")
    names = ["caption/caption_gpt3_1.3B_youku_v0.yaml", "caption/caption_gpt3_2.7B_youku_v0.yaml",
             "cls/cls_gpt3_1.3B_youku_v0_sharp_2.yaml", "cls/cls_gpt3_2.7B_youku_v0_sharp_2.yaml",
             "retrieval/retrieval_gpt3_1.3B_youku_v0.yaml", "retrieval/retrieval_gpt3_2.7B_youku_v0.yaml",
             "retrieval/retrieval_itm_gpt3_1.3B_youku_v0.yaml", "retrieval/retrieval_itm_gpt3_2.7B_youku_v0.yaml",
             "pretrain/gpt3_1.3B/pretrain_gpt3_freezeGPT_youku_v0.yaml", "pretrain/gpt3_2.7B/pretrain_gpt3_freezeGPT_youku_v0.yaml"]
    # the reference's own yamls, parsed with the same loader (oracle/make_golden.py run_task_configs)
    with open(os.path.join(ROOT, "tests", "golden", "reference_task_configs.json")) as f:
        ref_configs = json.load(f)["configs"]
    for n in names:
        cfg = ryaml.load(open(os.path.join(cfg_root, n)), Loader=ryaml.Loader)
        assert cfg["megatron_cfg"]["tensor_model_parallel_size"] == 1 and cfg["megatron_cfg"]["model_parallel_size"] == 1
        assert isinstance(cfg["optimizer"]["lr"], float) and isinstance(cfg["optimizer"]["opt_eps"], float)
        assert isinstance(cfg["schedular"]["min_lr"], float) and cfg["freeze_text_decoder"] is True and cfg["num_learnable_token"] == 128
        assert os.path.exists(os.path.join(ROOT, "youku-mplug_b200", cfg["text_cfg"])) and os.path.exists(os.path.join(ROOT, "youku-mplug_b200", cfg["visual_cfg"]))
        ref = ref_configs[n]
        assert set(ref) == set(cfg), (n, set(ref) ^ set(cfg))
        for k in ref:
            if k != "megatron_cfg":
                assert ref[k] == cfg[k], (n, k, ref[k], cfg[k])
    shipped = set(ref_configs)
    assert shipped <= set(names) | {n for n in shipped if "b200" in n}, shipped - set(names)
