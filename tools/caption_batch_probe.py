"""GPU probe: caption decoding throughput of the batched beam search against the per-clip one, at the 1.3B configuration
with random weights (YMP_ALLOW_RANDOM_INIT=1), a CLIP-B/16 encoder over 8 frames of 224^2, a 128-query visual prefix,
equal 16-token prompts and beam 5, all timed with CUDA events.  Prints one JSON line per measurement, the card's name
and power limit first:
  CAPTION   DistributedGPT3_Caption.generate (visual prefix once, then one beam search per clip) against
            generate_batch (visual prefix once, then all clips' beams in each decoding step), end to end, stop token
            = the config's eod id (both arms decode the same tokens);
  DECODE    the decoder alone, DistributedGPT3.beam_search per clip against beam_search_batch, with a stop token outside
            the vocabulary so that every clip decodes exactly STEPS tokens;
  STEP      the captured decoding step alone at 5 rows (one beam search) and at 60 rows (12 clips);
  PART      per-launch device time of the step's non-GEMM kernels at 5 and 60 rows: the decode attention (32 heads,
            head_dim 64, mid-decode key count; through the key-row table at 60 rows) and the LayerNorm of a [rows, 2048]
            fp32 residual row block (two per layer plus the first one: 49 per step at 24 layers).
Per-GEMM times at 5 / 60 rows come from `ROWS=5|60 tools/skinny_probe.py`.
Env: CLIPS (default "12,24"), STEPS (default 16)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "youku-mplug_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
os.environ["YMP_ALLOW_RANDOM_INIT"] = "1"
import torch  # noqa: E402
from helpers import make_model_dir, pretrain_config  # noqa: E402
from bench import GCFG, VCFG_CLIP_B16  # noqa: E402  (model-shape constants)
import models.distributed_gpt3 as D  # noqa: E402
import models.modeling_distributed_gpt3 as M  # noqa: E402
from ymp import ops  # noqa: E402
from ymp.ops import TView  # noqa: E402

dev, bf16 = torch.device("cuda"), torch.bfloat16
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("CARD " + json.dumps(dict(nvidia_smi=smi[0] if smi else None, torch_name=torch.cuda.get_device_name(0))), flush=True)

STEPS = int(os.environ.get("STEPS", "16"))
CLIPS = [int(c) for c in os.environ.get("CLIPS", "12,24").split(",")]
beam, Q, P, T = 5, 128, 16, 8
gcfg = dict(GCFG["1.3B"], tokens_to_generate=STEPS)
H, V = gcfg["hidden_size"], gcfg["vocab_size"]
td = make_model_dir(dict(VCFG_CLIP_B16, num_frames=T), gcfg)
torch.manual_seed(0)
with torch.device(dev):
    model = D.DistributedGPT3_Caption(config=pretrain_config(td, Q, num_frames=T), tokenizer=None)
model = model.to(bf16).eval()
dec = model.text_decoder
n_max = max(CLIPS)
g = torch.Generator().manual_seed(1)
video = torch.randn(n_max, 3, T, 224, 224, generator=g).to(bf16).to(dev)
prompt = torch.randint(0, V, (1, P), generator=g).repeat(n_max, 1)
# [prompt | one more token]: generate() takes prompt_length = attention_mask.sum(-1) - 1 = P
ids = torch.cat([prompt, torch.full((n_max, 1), 5)], 1).to(dev)
qf = (torch.randn(n_max, Q, H, generator=g) * 0.1).to(bf16).to(dev)
prompt = prompt.to(dev)
STOP = V        # outside the vocabulary: never ranked


def timed(fn, n, reps=2):
    fn(n)                                   # warm-up: caches, graph capture
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn(n)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def same_lists(a, b):
    return len(a) == len(b) and all(x.shape == y.shape and torch.equal(x, y) for x, y in zip(a, b))


with torch.no_grad():
    for n in CLIPS:
        sub = M.BatchEncoding(dict(input_ids=ids[:n], attention_mask=torch.ones_like(ids[:n])))
        ms_ref, ref = timed(lambda k: model.generate(video[:k], sub), n)
        ms_bat, got = timed(lambda k: model.generate_batch(video[:k], sub), n)
        print("CAPTION " + json.dumps(dict(clips=n, beam=beam, tokens_to_generate=STEPS, frames=T, prefix=Q, prompt=P,
                                           generate_ms=round(ms_ref, 2), generate_batch_ms=round(ms_bat, 2),
                                           generate_clips_per_s=round(n / ms_ref * 1e3, 2),
                                           generate_batch_clips_per_s=round(n / ms_bat * 1e3, 2),
                                           speedup=round(ms_ref / ms_bat, 2), identical=same_lists(ref, got))), flush=True)

    def per_clip(n):
        return [dec.beam_search(prompt[i:i + 1], query_embeds=qf[i:i + 1], prompt_length=P, beam_size=beam, stop_token=STOP)
                for i in range(n)]

    def batched(n):
        return dec.beam_search_batch(prompt[:n], query_embeds=qf[:n], prompt_length=torch.full((n,), P), beam_size=beam,
                                     stop_token=STOP)

    for n in CLIPS:
        ms_ref, ref = timed(per_clip, n)
        ms_bat, got = timed(batched, n)
        same = all(torch.equal(a.sequences, b.sequences) and torch.equal(a.scores, b.scores) for a, b in zip(ref, got))
        print("DECODE " + json.dumps(dict(clips=n, beam=beam, steps=STEPS, prefix=Q, prompt=P,
                                          beam_search_ms=round(ms_ref, 2), beam_search_batch_ms=round(ms_bat, 2),
                                          beam_search_clips_per_s=round(n / ms_ref * 1e3, 2),
                                          beam_search_batch_clips_per_s=round(n / ms_bat * 1e3, 2),
                                          speedup=round(ms_ref / ms_bat, 2), identical=same)), flush=True)


def replay_ms(ts):
    """The captured step alone: device time of back-to-back replays from the prefix length on (each replay advances the
    device-side cache length, so at most max_len - prefix - 1 of them fit)."""
    c = ts.cache
    c._set_len(Q + P)
    reps = c.max_len - (Q + P) - 1
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ts.graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


with torch.no_grad():
    dec.beam_search(prompt[:1], query_embeds=qf[:1], prompt_length=P, beam_size=beam, stop_token=STOP)
    ts5 = next(iter(dec._decode_pool.values())).token
    batched(12)
    ts60 = next(iter(dec._beam_batch_pool.values())).token
for rows, ts in ((5, ts5), (60, ts60)):
    if ts is not None and ts.graph is not None:
        print("STEP " + json.dumps(dict(rows=rows, captured_step_ms=round(replay_ms(ts), 3), layers=gcfg["num_hidden_layers"])),
              flush=True)


def graph_us(call, per_graph=24, reps=20):
    """Per-launch device time of `call`, captured per_graph times into one CUDA graph and replayed."""
    call()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(per_graph):
            call()
    gr.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        gr.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (reps * per_graph) * 1e3


heads, hd = gcfg["num_attention_heads"], H // gcfg["num_attention_heads"]
keys = Q + P + STEPS // 2                      # mid-decode key count
ML = Q + P + STEPS
for rows in (5, 60):
    buf = torch.randn(rows * ML, 3 * H, device=dev).to(bf16)
    q = torch.randn(rows, 3 * H, device=dev).to(bf16)
    o = torch.empty(rows, H, device=dev, dtype=bf16)
    lse = torch.empty(rows, heads, 1, device=dev)
    len1 = torch.tensor([keys], device=dev, dtype=torch.int32)
    # at 60 rows the batched step's layout: beams of a clip share the prefix rows of their clip's beam 0
    tab = None
    if rows > 8:
        r = torch.arange(rows)
        tab = r[:, None] * ML + torch.arange(ML)[None]
        tab[:, :Q + P] = ((r // beam) * beam)[:, None] * ML + torch.arange(Q + P)[None]
        tab = tab.int().to(dev)
    m1, mkv = ops.dense_map(1), ops.dense_map(ML)

    def attn():
        ops.attn_fwd(TView(q, 0, 3 * hd, m1), TView(buf, hd, 3 * hd, mkv), TView(buf, 2 * hd, 3 * hd, mkv), TView(o, 0, hd, m1),
                     n_seq=rows, n_heads=heads, head_dim=hd, s_q=1, s_kv=ML, causal=False, scale=hd ** -0.5, lse=lse,
                     s_kv_dev=len1, kv_rows=tab)
    x = torch.randn(rows, H, device=dev)
    gamma, beta, y = torch.ones(H, device=dev, dtype=bf16), torch.zeros(H, device=dev, dtype=bf16), torch.empty(rows, H, device=dev, dtype=bf16)

    def ln():
        ops.layernorm_fwd(x, gamma, beta, 1e-5, out=y, stats=False)
    print("PART " + json.dumps(dict(rows=rows, keys=keys, decode_attention_us=round(graph_us(attn), 2),
                                    layernorm_us=round(graph_us(ln), 2), table=tab is not None)), flush=True)
