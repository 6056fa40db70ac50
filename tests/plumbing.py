"""Test helper: a synthetic workspace the reference's run_pretrain_distributed_gpt3.py can run on - tiny model
directory (config.json / visual json / tokenizer.json), the task yaml with the reference's own keys
(configs/pretrain/gpt3_1.3B/pretrain_gpt3_freezeGPT_youku_v0.yaml), a csv in the loader's format
(dataset/video_pretrain_dataset.py:22-24) and .npy clips for the decord stand-in."""
import json
import os

import numpy as np

from oracle import port


def make_workspace(td, num_videos=8, batch_size=2, max_length=8, num_workers=0):
    from tokenizers import Tokenizer, models, pre_tokenizers
    md = os.path.join(td, "text_decoder")
    os.makedirs(md, exist_ok=True)
    vcfg = dict(port.VCFG_TINY, pretrained_ckpt=None, grad_ckpt=False, drop_path=0, stop_grad_conv1=False,
                use_shared_rel_pos_bias=False, use_abs_pos_emb=True)
    with open(os.path.join(td, "vis.json"), "w") as f:
        json.dump(vcfg, f)
    with open(os.path.join(md, "config.json"), "w") as f:
        json.dump(dict(port.GCFG_TINY, hidden_dropout=0.0, attention_dropout=0.0), f)
    vocab = {"<|endoftext|>": 0, "<sep>": 1, "[UNK]": 2, "\n": 3}
    words = "a b c d e f g hello world video cat dog runs on the grass".split()
    for i, w in enumerate(words):
        vocab[w] = 4 + i
    tok = Tokenizer(models.WordLevel(vocab, unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    tok.save(os.path.join(md, "tokenizer.json"))
    vids = os.path.join(td, "videos")
    os.makedirs(vids, exist_ok=True)
    rng = np.random.default_rng(0)
    rows = ["video_id:FILE,title"]
    for i in range(num_videos):
        np.save(os.path.join(vids, f"clip{i}.npy"), rng.integers(0, 256, (6, 40, 48, 3), dtype=np.uint8))
        rows.append(f"clip{i}.npy,{' '.join(rng.choice(words, 4))}")
    with open(os.path.join(td, "pretrain.csv"), "w") as f:
        f.write("\n".join(rows) + "\n")
    cfg = f"""train_file: [
  {os.path.join(td, 'pretrain.csv')}
]
read_local_data: true

train_video_root: "{vids}/"

text_decoder: '{md}/'
text_cfg: {os.path.join(md, 'config.json')}
visual_cfg: '{os.path.join(td, 'vis.json')}'

megatron_cfg: {{
  "world_size": 1,
  "model_parallel_size": 1,
  "tensor_model_parallel_size": 1,
}}

batch_size: {batch_size}
num_workers: {num_workers}
max_length: {max_length}

freeze_vit: false
freeze_text_decoder: true

num_learnable_token: 8
use_contrastive: false

temp: 0.07
embed_dim: 256

optimizer: {{
  lr: 1e-4,
  opt: "AdamW",
  weight_decay: 0.05,
  clip_grad: 3.0,
  opt_betas: [0.9, 0.999],
  opt_eps: 1e-6
}}

schedular: {{
  epochs: 1,
  min_lr: 1e-6,
  warmup_epochs: -1,
  warmup_steps: 1,
  lr_sched_type: "cosine"
}}
"""
    path = os.path.join(td, "pretrain_tiny.yaml")
    with open(path, "w") as f:
        f.write(cfg)
    return dict(config=path, model_dir=md, output_dir=os.path.join(td, "out"), videos=vids)


def make_downstream_workspace(td, task, num_videos=8, batch_size=2, max_length=8, num_frames=2):
    """Workspace for the reference's downstream scripts (downstream/run_{cls,caption,retrieval,retrieval_itm}...py): the
    tiny model directory of make_workspace plus train / val / test csv files in the format the task's dataset class reads
    (dataset/video_downstream_datasets.py:34-41,118-125,335-347,413-423) and a task yaml with the reference's keys."""
    ws = make_workspace(td, num_videos=num_videos, batch_size=batch_size, max_length=max_length)
    rng = np.random.default_rng(1)
    words = "a b c d e f g hello world video cat dog runs on the grass".split()
    clips = [f"clip{i}.npy" for i in range(num_videos)]
    if task == "cls":
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_task_configs.json")) as f:
            classes = list(json.load(f)["classnames"])       # the reference's classname.json
        header, rows = "video_id:FILE,title,label", [f"{c},{' '.join(rng.choice(words, 3))},{classes[i % len(classes)]}" for i, c in enumerate(clips)]
        prefix, extra = "classification", "use_cls: true\nnum_frames: %d\nnum_classes: %d\n" % (num_frames, len(classes))
    elif task == "caption":
        header, rows = "video_id:FILE,golden_caption", [f"{c},\"['{' '.join(rng.choice(words, 3))}']\"" for c in clips]
        prefix, extra = "captioning", "use_cls: true\nnum_frames: %d\nprompt: \"\"\n" % num_frames
    else:
        header, rows = "clip_name:FILE,caption", [f"{c},{' '.join(rng.choice(words, 3))}" for c in clips]
        prefix = "retrieval"
        extra = ("use_cls: true\n" if task == "retrieval_itm" else "") + "num_frames: %d\ntemp: 0.07\nembed_dim: 32\n" % num_frames
    files = {}
    for split in ("train", "val", "test"):
        files[split] = os.path.join(td, f"{prefix}_{split}.csv")
        with open(files[split], "w") as f:
            f.write(header + "\n" + "\n".join(rows) + "\n")
    cfg = f"""train_file: '{files['train']}'
val_file: '{files['val']}'
test_file: '{files['test']}'
read_local_data: true
video_root: "{ws['videos']}/"
text_decoder: '{ws['model_dir']}/'
text_cfg: {os.path.join(ws['model_dir'], 'config.json')}
visual_cfg: '{os.path.join(td, 'vis.json')}'
megatron_cfg: {{
  "world_size": 1,
  "model_parallel_size": 1,
  "tensor_model_parallel_size": 1,
}}
batch_size: {batch_size}
num_workers: 0
max_length: {max_length}
freeze_vit: false
freeze_text_decoder: true
num_learnable_token: 8
{extra}optimizer: {{
  lr: 2e-5,
  opt: "AdamW",
  weight_decay: 0.05,
  clip_grad: 3.0,
  opt_betas: [0.9, 0.999],
  opt_eps: 1e-6
}}
schedular: {{
  epochs: 1,
  min_lr: 1e-6,
  warmup_epochs: -1,
  warmup_steps: 1,
  lr_sched_type: "cosine"
}}
"""
    path = os.path.join(td, f"{task}_tiny.yaml")
    with open(path, "w") as f:
        f.write(cfg)
    return dict(ws, config=path)
