#!/usr/bin/env python
"""Benchmark of the mPLUG-Video pre-training hot path (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            # this repo's B200 path
  python bench.py --impl reference --gpus N --steps K ...   # the reference's algorithm on host cores
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's results as DIR/*.npy

A step = one pre-training iteration through the public model API: forward (TimeSformer ->
abstractor -> frozen GPT-3 1.3B -> masked CE), backward (dgrad everywhere, wgrad for the 130 M
trainable parameters), gradient all-reduce (N>1), global-norm clip + AdamW.  Workload: 32
samples/GPU of (3, 8, 224, 224) video + 128 text tokens, 128 learnable queries, bf16, random-init
weights, synthetic data (weak scaling).  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "youku-mplug_b200")
for _p in (ROOT, PKG, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "video-text samples/sec (pretrain 1.3B, 8f x 224^2)"
GF_PER_SAMPLE = 2563.8  # algorithmic fwd+bwd GFLOP per sample, SURVEY.md section 8(d) config 2

# model dims of the BASELINE configs (configs/models/{clip-b16,config_gpt3_1.3B,config_gpt3_2.7B}.json of the
# reference; the package's own copies live in youku-mplug_b200/configs/models/)
VCFG_CLIP_B16 = dict(img_size=224, patch_size=16, embed_dim=768, depth=12, num_heads=8, mlp_ratio=4, num_frames=8, clip_model=True)
GCFG = {"1.3B": dict(vocab_size=51200, hidden_size=2048, ffn_hidden_size=8192, num_hidden_layers=24, num_attention_heads=32,
                     max_position_embeddings=2048, layernorm_epsilon=1e-5, init_method_std=0.02),
        "2.7B": dict(vocab_size=51200, hidden_size=2560, ffn_hidden_size=10240, num_hidden_layers=32, num_attention_heads=32,
                     max_position_embeddings=2048, layernorm_epsilon=1e-5, init_method_std=0.02)}
# --config: (model class, decoder, frames, text length, batch/GPU, metric)
CONFIGS = {
    "pretrain": dict(cls="DistributedGPT3_Pretrain", gpt="1.3B", frames=8, text_len=128, batch=32, metric=METRIC,
                     workload="mPLUG-Video GPT-3 1.3B pretrain step (BASELINE configs[1])"),
    "caption27b": dict(cls="DistributedGPT3_Caption", gpt="2.7B", frames=16, text_len=256, batch=32,
                       metric="video-text samples/sec (caption fine-tuning 2.7B, 16f x 224^2, text 256)",
                       workload="mPLUG-Video GPT-3 2.7B caption fine-tuning step (BASELINE configs[3])"),
    "retrieval": dict(cls="DistributedGPT3_Retrieval", gpt="1.3B", frames=8, text_len=80, batch=96,
                      metric="video-text samples/sec (contrastive retrieval 1.3B, 8f x 224^2, text 80)",
                      workload="mPLUG-Video GPT-3 1.3B contrastive retrieval step, feature all-gather across ranks (BASELINE configs[2])"),
}


def algorithmic_gflop(kind, vcfg, gcfg, T, L, Q):
    """fwd+bwd GFLOP per sample as the reference computes the work (SURVEY.md section 8d formulas: multiply-add = 2,
    full S x S attention, no recompute, frozen decoder = dgrad only, trainable encoder = dgrad + wgrad)."""
    D, N, depth, V = vcfg["embed_dim"], (vcfg["img_size"] // vcfg["patch_size"]) ** 2, vcfg["depth"], gcfg["vocab_size"]
    h, layers = gcfg["hidden_size"], gcfg["num_hidden_layers"]
    TN = T * N
    block = (2 * TN * D * 3 * D + 4 * N * T * T * D + 2 * (2 * TN * D * D) + 2 * T * (N + 1) * D * 3 * D + 4 * T * (N + 1) ** 2 * D
             + 2 * T * (N + 1) * D * D + 4 * (TN + 1) * D * 4 * D)
    vit = depth * block + 2 * TN * 768 * D
    K = TN + 1
    abstractor = 4 * Q * D * D + 4 * K * D * D + 4 * Q * (K + 1) * D + 16 * Q * D * D + 2 * Q * D * h
    if kind == "retrieval":      # CLS-pooled ViT feature + text-only decoder pass (its LM head / CE is computed and unused)
        S = L
        fwd = vit + layers * (S * 24 * h * h + 4 * S * S * h) + 2 * S * h * V
        return (fwd + 2 * vit) / 1e9          # nothing trainable sits below the decoder: no decoder backward
    S = Q + L
    gpt = layers * (S * 24 * h * h + 4 * S * S * h)
    lm = 2 * S * h * V
    return (vit + abstractor + gpt + lm + 2 * (vit + abstractor) + gpt + lm) / 1e9


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if mx and x > 0.5 * mx] or sm
        return dict(sm_mhz=statistics.median(busy) if busy else None, sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm))


def make_text(G, B, L, vocab, seed, bos=1, pad=0):
    import torch
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, vocab, (B, L), generator=g)
    ids[:, 0] = bos
    lens = torch.randint(16, L + 1, (B,), generator=g)
    att = (torch.arange(L)[None, :] < lens[:, None]).long()
    ids = torch.where(att.bool(), ids, torch.full_like(ids, pad))
    return ids, att


def cpu_baseline(port, torch, T, L, Q, iters=1, warmup=1, cold_cutoff_s=None):
    """The oracle port (fp32, host threads) on a bounded sample: fwd+bwd of ONE sample of the same
    workload, `warmup` untimed + `iters` timed iterations (the first call pays page faults for ~10 GB of
    weights / saved activations).  With cold_cutoff_s, a last warm-up iteration slower than that is taken as the
    only timed one, which keeps an informational baseline within minutes on slow hosts.
    Returns (samples/s, threads, description)."""
    vcfg = dict(port.VCFG_CLIP_B16, num_frames=T)
    threads = min(os.cpu_count() or 1, 32)   # beyond ~32 threads the small-GEMM torch CPU path slows down
    torch.set_num_threads(threads)
    sd = port.init_state_dict(vcfg, port.GCFG_1_3B, Q, seed=0, fast=True)
    train = set(port.trainable_keys(sd))
    psd = {k: v.requires_grad_(k in train) for k, v in sd.items()}
    g = torch.Generator().manual_seed(1234)
    video2 = torch.randn(2, 3, T, 224, 224, generator=g)
    ids2 = torch.randint(0, 51200, (2, L), generator=g)
    att2 = torch.ones(2, L, dtype=torch.long)
    video, ids, att = video2[:1], ids2[:1], att2[:1]

    def one(video=video, ids=ids, att=att):
        t0 = time.time()
        loss = port.pretrain_forward(video, ids, att, psd, vcfg, port.GCFG_1_3B)
        loss.backward()
        for v in psd.values():
            v.grad = None
        return time.time() - t0

    cold = [one() for _ in range(warmup)]
    note = ""
    if cold_cutoff_s is not None and cold and cold[-1] > cold_cutoff_s:
        times, note = cold[-1:], " (cold first iteration: the host was too slow for a warm-up + timed pass)"
    else:
        times = [one() for _ in range(iters)]
    dt = statistics.median(times)
    b2 = ""
    if not note and dt < 20.0:     # batch 2 for the CPU path's own batch scaling (SURVEY 8d), when the host is fast enough
        t2 = statistics.median([one(video2, ids2, att2) for _ in range(2)])
        b2 = f"; batch 2: {2.0 / t2:.3f} samples/s ({t2:.1f}s per step)"
    return 1.0 / dt, threads, (f"median of {len(times)} x (fwd+bwd of 1 sample, T={T}, L={L}, Q={Q}, fp32 torch CPU, {threads} threads, "
                               f"{dt:.1f}s each, {warmup} warm-up){note}{b2}")


def run_reference(args, rank):
    """--impl reference: the reference's algorithm (oracle/port.py, pinned against the unmodified
    reference) on the box's host cores; the Python reference itself cannot travel to the GPU box."""
    if rank != 0:
        return
    import torch
    from oracle import port
    val, cores, sample = cpu_baseline(port, torch, args.frames, args.text_len, args.queries, iters=args.steps,
                                      warmup=1 if args.warmup > 0 else 0)
    line = dict(metric=METRIC, value=val, unit="samples/s", n_gpus=args.gpus, steps=args.steps, warmup=1 if args.warmup > 0 else 0,
                ms_per_step=1000.0 / val, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload="mPLUG-Video GPT-3 1.3B pretrain step, 8f x 224^2, text 128, 128 queries",
                            per_step="1 sample fwd+bwd (bounded sample of the 32/GPU workload)"),
                cpu_baseline=dict(value=val, unit="samples/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=val, unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


DUMP_SAMPLE = 1 << 21     # values drawn from each flat training-state vector by --dump-outputs (8 MB each in fp32)


def dump_outputs(out_dir, eng, loss):
    """--dump-outputs: what the last timed step handed back, as float32 / float64 .npy files - its loss, the global
    gradient norm AdamW clipped with, and, at a fixed seeded sample of DUMP_SAMPLE flat positions (sample_index.npy),
    the trainable parameters it wrote (fp32 master copy) and AdamW's first moment.  With the same arguments the
    inputs and initial weights are the same from run to run and every reduction of the step adds in a fixed order,
    so one build writes the same bits every run and two builds can be compared file by file."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = eng.master.numel()
    idx = torch.randint(0, n, (min(DUMP_SAMPLE, n),), generator=torch.Generator().manual_seed(0)).sort().values
    arrays = dict(loss=np.asarray([float(loss.float().item())], dtype=np.float32),
                  grad_norm=np.asarray([float(eng.optimizer._global_grad_norm)], dtype=np.float64),
                  sample_index=idx.numpy().astype(np.float64),
                  trainable_params=eng.master[idx.to(eng.master.device)].cpu().numpy(),
                  adam_exp_avg=eng.exp_avg[idx.to(eng.exp_avg.device)].cpu().numpy())
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ymp(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    os.environ["YMP_ALLOW_RANDOM_INIT"] = "1"
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from helpers import make_model_dir, pretrain_config
    import models.distributed_gpt3 as D
    import models.modeling_distributed_gpt3 as G
    from ymp import lib, ops, train

    cfg = CONFIGS[args.config]
    B, T, L, Q = args.batch, args.frames, args.text_len, args.queries
    gcfg = GCFG[cfg["gpt"]]
    vcfg = dict(VCFG_CLIP_B16, num_frames=T)
    td = make_model_dir(vcfg, gcfg, dropout=(args.dropout, args.dropout))
    torch.manual_seed(0)
    with torch.device(dev):
        model = getattr(D, cfg["cls"])(config=pretrain_config(td, Q, num_frames=T), tokenizer=None)
    model = model.to(torch.bfloat16)
    model.train()
    n_train = sum(p.numel() for p in model.parameters() if p.requires_grad)
    eng = train.TrainEngine(model, lr=1e-4, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.05, clip_grad=3.0)

    g = torch.Generator().manual_seed(1234 + rank)
    video_h = torch.randn(B, 3, T, 224, 224, generator=g).pin_memory()      # fp32 host frames (the loader's dtype)
    ids_h, att_h = make_text(G, B, L, 51200, 4321 + rank)
    ids_h, att_h = ids_h.pin_memory(), att_h.pin_memory()
    video_d = video_h.to(dev).bfloat16()
    extra_h = {}
    if args.config == "caption27b":     # [prompt + caption] pairs: prompt tokens carry no loss (distributed_gpt3.py:760-766)
        extra_h["prompt_lengths"] = torch.full((B,), 4, dtype=torch.long).pin_memory()
    tail_h = ()
    if args.config == "retrieval":      # video ids: equal ids are positives of each other (:944-958)
        tail_h = (torch.arange(rank * B, (rank + 1) * B, dtype=torch.long).pin_memory(),)

    def enc(ids, att, extra):
        return G.BatchEncoding(dict(input_ids=ids, attention_mask=att, **extra))

    text_d = enc(ids_h.to(dev), att_h.to(dev), {k: v.to(dev) for k, v in extra_h.items()})
    tail_d = tuple(t.to(dev) for t in tail_h)

    use_graph = not args.no_graph

    def step_resident():
        return eng.train_step(video_d, text_d, *tail_d, use_graph=use_graph)

    from ymp.data import DevicePrefetcher
    pf = DevicePrefetcher(dev)

    def step_e2e():
        # every step copies one batch of pinned fp32 host frames (+ token ids, mask) to the device: the NEXT step's
        # batch is staged on a side stream while this step computes, as a prefetching loader does
        host = (video_h, ids_h, att_h) + tuple(extra_h.values()) + tail_h
        if not len(pf):
            pf.submit(*host)
        got = pf.take()
        pf.submit(*host)
        v, ids_d, att_d = got[:3]
        extra_d = dict(zip(extra_h.keys(), got[3:3 + len(extra_h)]))
        loss = eng.train_step(v, enc(ids_d, att_d, extra_d), *got[3 + len(extra_h):], use_graph=use_graph)
        return loss.item()     # D2H read of the step's result, as the reference loop does (run_pretrain...py:115)

    def step_eager():
        out = eng(video_d, text_d, *tail_d)
        loss = sum(out[1:], out[0]) if isinstance(out, tuple) else out
        eng.backward(loss)
        eng.step()
        return loss

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for _ in range(steps):
            last = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), last

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, last_loss = timed(step_resident, args.steps)
    if args.dump_outputs and rank == 0:     # before any further step changes the weights
        dump_outputs(args.dump_outputs, eng, last_loss)
    # kernels of ours enqueued per timed step: counted on one eager step (a graph replay re-launches the
    # same kernels without going through the library's host entry points)
    n0 = lib.launch_count()
    step_eager()
    torch.cuda.synchronize()
    launches = (lib.launch_count() - n0) * args.steps
    clocks = sampler.stop() if rank == 0 else None
    final_loss = float(last_loss.item())
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)

    # informational: the same end-to-end step fed with uint8 clips [B,T,H,W,3] (SURVEY 8f N4): normalisation, layout
    # change and bf16 cast run on the device (ymp_clip_normalize), the host sends 1 byte per value
    frames_h = torch.randint(0, 256, (B, T, 224, 224, 3), generator=g, dtype=torch.uint8).pin_memory()
    CLIP_MEAN = [0.48145466, 0.4578275, 0.40821073]   # dataset/__init__.py:69-72
    CLIP_STD = [0.26862954, 0.26130258, 0.27577711]

    pf8 = DevicePrefetcher(dev)

    def step_e2e_u8():
        host = (frames_h, ids_h, att_h) + tuple(extra_h.values()) + tail_h
        if not len(pf8):
            pf8.submit(*host)
        got = pf8.take()
        pf8.submit(*host)
        v = ops.clip_normalize(got[0], CLIP_MEAN, CLIP_STD)
        extra_d = dict(zip(extra_h.keys(), got[3:3 + len(extra_h)]))
        return eng.train_step(v, enc(got[1], got[2], extra_d), *got[3 + len(extra_h):], use_graph=use_graph).item()

    for _ in range(2):
        step_e2e_u8()
    ms_e2e_u8, _ = timed(step_e2e_u8, args.steps)

    # ---- roofline of the dominant kernel (tcgen05 GEMM): CUDA events around every launch of one
    # extra, untimed step on the launching stream; achieved = sum(2MNK) / sum(duration)
    rec = []
    orig = ops.gemm

    def gemm_rec(a, b, **kw):
        M, K = (a.shape[1], a.shape[0]) if kw.get("a_t") else (a.shape[0], a.shape[1])
        if kw.get("_im2col") is not None:       # fused patch embedding: A is the video, rows (b, n, t) x columns C*P*P
            P_, B_, C_, T_, H_, W_ = kw["_im2col"]
            M, K = B_ * (H_ // P_) * (W_ // P_) * T_, C_ * P_ * P_
        N = b.shape[1] if kw.get("b_t") else b.shape[0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = orig(a, b, **kw)
        e1.record()
        rec.append((2.0 * M * N * K, e0, e1, (M, N, K, int(bool(kw.get("a_t"))), int(bool(kw.get("b_t"))),
                                              int(bool(kw.get("accumulate"))), int(kw.get("act", 0)),
                                              int(kw.get("aux_out") is not None), int(kw.get("aux_in") is not None),
                                              int(kw.get("residual") is not None), int(out.dtype == torch.float32),
                                              int(kw.get("residual") is not None and kw["residual"].dtype == torch.float32))))
        return out

    ops.gemm = gemm_rec
    step_eager()
    torch.cuda.synchronize()
    ops.gemm = orig
    gemm_ms = sum(e0.elapsed_time(e1) for _, e0, e1, _ in rec)
    gemm_flop = sum(f for f, _, _, _ in rec)
    if args.gemm_report and rank == 0:
        shapes = {}
        for f, e0, e1, key in rec:
            ent = shapes.setdefault(key, [0, 0.0, 0.0])
            ent[0] += 1; ent[1] += e0.elapsed_time(e1); ent[2] += f
        rows = sorted(([dict(M=k[0], N=k[1], K=k[2], a_t=k[3], b_t=k[4], acc=k[5], act=k[6], aux_out=k[7], aux_in=k[8],
                             res=k[9], out_f32=k[10], res_f32=k[11], n=v[0], ms=v[1], tflops=v[2] / v[1] / 1e9)
                        for k, v in shapes.items()]),
                      key=lambda r: -r["ms"])
        with open(args.gemm_report, "w") as fh:
            json.dump(rows, fh, indent=1)
    pk = peaks()
    tf = gemm_flop / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    ms_step = ms / args.steps
    gf_sample = algorithmic_gflop(args.config, vcfg, gcfg, T, L, Q)
    if args.config == "pretrain" and (T, L, Q) == (8, 128, 128):
        assert abs(gf_sample - GF_PER_SAMPLE) < 0.5, gf_sample       # SURVEY.md section 8(d), config 2
    step_tf = gf_sample * B / ms_step  # GFLOP/ms == TFLOP/s
    traffic, traffic_note = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_gemm_traffic.json")
    if os.path.exists(tpath) and args.config == "pretrain" and (B, T, L, Q) == (32, 8, 128, 128):
        with open(tpath) as fh:
            tj = json.load(fh)
        traffic = tj["bytes_per_launch"]
        traffic_note = (f"dram__bytes_read+write per GEMM launch, ncu capture committed in profiles/{os.path.basename(tpath)} "
                        f"(= {tj['measured_over_algorithmic']:.2f} x the algorithmic operand bytes)")
    roofline = dict(bound="tensor", kernel="gemm_bf16_tcgen05_2cta_kernel", achieved=tf, peak=pk["tf_sustained"], unit="TFLOP/s",
                    frac=tf / pk["tf_sustained"], traffic=traffic, traffic_note=traffic_note,
                    peak_source=pk["source"] + ", sustained figure",
                    launches_per_step=len(rec), gemm_ms_per_step=gemm_ms, gemm_share_of_step=gemm_ms / ms_step,
                    note="events around each GEMM launch of one extra untimed step; algorithmic 2MNK per launch")
    value = B * world * args.steps / (ms * 1e-3)
    e2e_val = B * world * args.steps / (ms_e2e * 1e-3)
    h2d = video_h.numel() * 4 + ids_h.numel() * 8 + att_h.numel() * 8
    if rank != 0:
        _teardown(eng, world)
        return
    line = dict(metric=cfg["metric"], value=value, unit="samples/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
                data="synthetic", impl="ymp_b200",
                config=dict(workload=cfg["workload"], model=cfg["cls"], decoder="GPT-3 " + cfg["gpt"], batch_per_gpu=B,
                            global_batch=B * world, frames=T, image=224, text_len=L, queries=Q, parallelism=f"dp{world}",
                            trainable_params=n_train,
                            step=f"fwd+bwd+allreduce+clip+AdamW, decoder dropout {args.dropout:g}"
                                 + (" (parity mode; the reference default 0.1: --dropout 0.1)" if args.dropout == 0 else
                                    " (hidden + attention, Philox masks regenerated in the backward)"),
                            cuda_graph=use_graph,
                            lm_head_rows="B*L text rows: the B*Q visual-prefix rows have loss_mask 0 in the reference "
                                         "(distributed_gpt3.py:142-159) and get no final-LN / LM-head / CE work; loss and all "
                                         "gradients are unchanged, algorithmic FLOPs still count them",
                            l2="per-step working set (~30 GB of activations) >> 126 MB L2; no explicit flush"),
                clocks=clocks, gpu_launches=int(launches),
                e2e=dict(value=e2e_val, unit="samples/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=4,
                         ms_per_step=ms_e2e / args.steps,
                         note="pinned fp32 frames; one batch copied per step on a side stream (ymp.data.DevicePrefetcher) "
                              "while the previous step computes; loss.item() read back every step"),
                e2e_uint8_input=dict(value=B * world * args.steps / (ms_e2e_u8 * 1e-3), unit="samples/s",
                                     h2d_bytes_per_step=int(frames_h.numel() + ids_h.numel() * 8 + att_h.numel() * 8),
                                     ms_per_step=ms_e2e_u8 / args.steps,
                                     note="uint8 clips normalised on the device (N4); not the headline e2e"),
                roofline=roofline,
                step_model=dict(algorithmic_gflop_per_sample=gf_sample, achieved_tflops=step_tf,
                                frac_of_sustained_peak=step_tf / pk["tf_sustained"],
                                executed_gflop_per_sample=gf_sample - (2 * 2 * Q * gcfg["hidden_size"] * gcfg["vocab_size"] / 1e9
                                                                       if args.config == "pretrain" else 0.0),
                                note="executed = algorithmic minus the LM-head rows of the visual prefix (fwd + dgrad), which "
                                     "carry loss_mask 0 and are skipped"),
                final_loss=final_loss)
    if world == 1 and not args.no_cpu_baseline and args.config == "pretrain":
        del eng, model
        torch.cuda.empty_cache()
        from oracle import port          # the CPU restatement, timed as the baseline only (never on the product path)
        val, cores, sample = cpu_baseline(port, torch, T, L, Q, iters=3, warmup=1, cold_cutoff_s=90.0)
        line["cpu_baseline"] = dict(value=val, unit="samples/s", cores=cores, kind="port", sample=sample)
    print(json.dumps(line), flush=True)
    if world > 1:
        _teardown(eng, world)


def _teardown(eng, world):
    """Leave a multi-rank run without hanging: the captured step graphs hold NCCL kernels and the engine holds async
    work handles, so they are released before the communicator on EVERY rank (a rank that simply returned used to
    block in interpreter shutdown while its peer sat in destroy_process_group); a watchdog guarantees the exit."""
    if world <= 1:
        return
    import gc
    import threading
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    t = threading.Timer(30.0, lambda: os._exit(0))
    t.daemon = True
    t.start()
    torch.cuda.synchronize()
    eng._graphs.clear()
    eng._pending.clear()
    gc.collect()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    sys.stdout.flush()
    os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ymp", choices=["ymp", "reference"])
    ap.add_argument("--config", default="pretrain", choices=sorted(CONFIGS),
                    help="pretrain = BASELINE configs[1] (the headline); caption27b = configs[3]; retrieval = configs[2]")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--frames", type=int, default=None)
    ap.add_argument("--text-len", type=int, default=None)
    ap.add_argument("--queries", type=int, default=128)
    ap.add_argument("--dropout", type=float, default=0.0,
                    help="hidden + attention dropout of the (frozen, train-mode) decoder; the reference default is 0.1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gemm-report", default=None, help="write per-shape GEMM timings of one step to this json file")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly (no CUDA graph replay)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the last one's loss, grad norm and a seeded sample of the updated "
                         "trainable parameters and AdamW first moment to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ymp":
        ap.error("--dump-outputs writes the results of the B200 path (--impl ymp)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    c = CONFIGS[args.config]
    args.batch = args.batch or c["batch"]
    args.frames = args.frames or c["frames"]
    args.text_len = args.text_len or c["text_len"]
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)
    run_ymp(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
