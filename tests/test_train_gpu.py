"""GPU parity of everything the timed training step runs after the model's backward (SURVEY 8f N1):
fused grad-norm + clip + AdamW against torch.optim.AdamW + clip_grad_norm_ (the arithmetic of DeepSpeed
FusedAdam(adam_w_mode) + gradient_clipping the reference configures, utils.py:490-526), the CUDA-graph
`train_step` against the eager `engine(); backward(); step()` loop of run_pretrain_distributed_gpt3.py:
109,134-137, gradient accumulation, checkpoint round trip, parameters whose gradient comes from plain
autograd, and (2 GPUs, NCCL) the data-parallel gradient and the differentiable all-gather."""
import os
import socket
import tempfile

import pytest
import torch

from oracle import port
from oracle.make_golden import make_inputs
from helpers import build_pretrain

pytestmark = pytest.mark.gpu


def _text(ids, att, dev, **extra):
    import models.modeling_distributed_gpt3 as G
    d = dict(input_ids=ids.to(dev), attention_mask=att.to(dev))
    d.update({k: v.to(dev) for k, v in extra.items()})
    return G.BatchEncoding(d)


def test_fused_adamw_and_clip_match_torch(cuda):
    from ymp import ops
    torch.manual_seed(0)
    n1, n2 = 1_000_003 // 8 * 8, 4096       # a decay group and a no-decay group sharing one global norm
    n = n1 + n2
    lr, betas, eps, wd, clip, gscale = 3e-4, (0.9, 0.999), 1e-6, 0.05, 3.0, 1.0 / 8
    w0 = torch.randn(n, device=cuda) * 0.02
    ref_a = torch.nn.Parameter(w0[:n1].clone())
    ref_b = torch.nn.Parameter(w0[n1:].clone())
    opt = torch.optim.AdamW([dict(params=[ref_a], weight_decay=wd), dict(params=[ref_b], weight_decay=0.0, lr=0.1 * lr)],
                            lr=lr, betas=betas, eps=eps)
    master = w0.clone()
    param = w0.bfloat16()
    m, v = torch.zeros_like(master), torch.zeros_like(master)
    sumsq = torch.zeros(1, device=cuda)
    for step in range(1, 4):
        # the second step's gradient is large (clipping active), the third small (clipping inactive)
        g = torch.randn(n, device=cuda) * (40.0 if step == 2 else 1e-3) * 8
        ref_a.grad, ref_b.grad = g[:n1] * gscale, g[n1:] * gscale
        tn = torch.nn.utils.clip_grad_norm_([ref_a, ref_b], clip)
        opt.step()
        sumsq.zero_()
        ops.sumsq(g, sumsq)
        assert abs(sumsq.sqrt().item() * gscale - tn.item()) <= 1e-4 * tn.item()
        for (a, b, w_d, l) in ((0, n1, wd, lr), (n1, n, 0.0, 0.1 * lr)):
            ops.adamw(master[a:b], param[a:b], g[a:b], m[a:b], v[a:b], step=step, lr=l, beta1=betas[0], beta2=betas[1],
                      eps=eps, weight_decay=w_d, grad_scale=gscale, max_grad_norm=clip, sumsq_t=sumsq)
        ref = torch.cat([ref_a.detach(), ref_b.detach()])
        st = [opt.state[ref_a], opt.state[ref_b]]
        ref_m = torch.cat([s["exp_avg"] for s in st])
        ref_v = torch.cat([s["exp_avg_sq"] for s in st])
        assert (master - ref).abs().max().item() <= 1e-6, step
        assert (m - ref_m).abs().max().item() <= 1e-6 * max(1.0, ref_m.abs().max().item()), step
        assert (v - ref_v).abs().max().item() <= 1e-6 * max(1.0, ref_v.abs().max().item()), step
        assert torch.equal(param, master.bfloat16()), step      # bf16 weights refreshed bit-exactly from the master


def _tiny(cuda, seed=3, **extra):
    sd = port.init_state_dict(port.VCFG_TINY, port.GCFG_TINY, 8, seed=seed, randomize=True)
    return build_pretrain(port.VCFG_TINY, port.GCFG_TINY, 8, sd=sd, device=cuda, dtype=torch.bfloat16, **extra)


def _batches(n, cuda, B=2, L=8):
    out = []
    for i in range(n):
        video, ids, att = make_inputs(B, port.VCFG_TINY, L, port.GCFG_TINY["vocab_size"], 100 + i)
        out.append((video.to(cuda).bfloat16(), _text(ids, att, cuda)))
    return out


def test_graph_train_step_equals_eager_loop(cuda):
    """4 consecutive iterations: CUDA-graph replay (captured at the 2nd call) vs the reference loop's
    model(); model.backward(loss); model.step().  The weight-gradient accumulators are zeroed between
    replays by step(); the comparisons keep a tolerance for fp32 rounding."""
    from ymp.train import TrainEngine
    lr = 1e-3
    eng_g = TrainEngine(_tiny(cuda), lr=lr)
    eng_e = TrainEngine(_tiny(cuda), lr=lr)
    losses_g, losses_e = [], []
    for video, text in _batches(4, cuda):
        losses_g.append(eng_g.train_step(video, text, use_graph=True, graph_warmup=1).item())
        loss, zero = eng_e(video, text)
        eng_e.backward(loss + zero)
        eng_e.step()
        losses_e.append(loss.item())
    assert any("graph" in st for st in eng_g._graphs.values())       # the graph path really ran
    for a, b in zip(losses_g, losses_e):
        assert abs(a - b) <= 1e-3 * abs(b), (losses_g, losses_e)
    assert losses_e[0] != losses_e[1]
    d = (eng_g.master - eng_e.master).abs()
    # Adam's update is +-lr per step wherever |g| is far above its rounding noise
    assert (d > 0.05 * lr).float().mean().item() < 2e-3
    assert d.max().item() <= 2.0 * lr * 4
    assert eng_g.global_steps == eng_e.global_steps == 4
    assert float(eng_g.flat_grad.abs().max()) == 0.0                   # zeroed for the next replay
    gn_g, gn_e = float(eng_g.optimizer._global_grad_norm), float(eng_e.optimizer._global_grad_norm)
    assert abs(gn_g - gn_e) <= 2e-2 * gn_e


def test_gradient_accumulation_boundary(cuda):
    """gradient_accumulation_steps=2: no optimizer step on the first micro-batch, and the update equals one
    step on the mean gradient (DeepSpeed scales the loss by 1/gas)."""
    from ymp.train import TrainEngine
    (v1, t1), (v2, t2) = _batches(2, cuda)
    eng = TrainEngine(_tiny(cuda), lr=1e-3, gradient_accumulation_steps=2)
    m0 = eng.master.clone()
    loss, _ = eng(v1, t1)
    eng.backward(loss)
    eng.step()
    assert torch.equal(eng.master, m0) and eng.global_steps == 0 and float(eng.flat_grad.abs().max()) > 0
    g1 = eng.flat_grad.clone()
    loss, _ = eng(v2, t2)
    eng.backward(loss)
    acc = eng.flat_grad.clone()
    eng.step()
    assert eng.global_steps == 1 and not torch.equal(eng.master, m0)
    # reference: two separate engines' gradients averaged
    ref = TrainEngine(_tiny(cuda), lr=1e-3)
    l1, _ = ref(v1, t1)
    ref.backward(l1)
    ga = ref.flat_grad.clone()
    ref.flat_grad.zero_()
    l2, _ = ref(v2, t2)
    ref.backward(l2)
    gb = ref.flat_grad.clone()
    scale = max(ga.abs().max().item(), 1e-12)
    assert (g1 - 0.5 * ga).abs().max().item() <= 2e-2 * scale
    assert (acc - 0.5 * (ga + gb)).abs().max().item() <= 2e-2 * scale


def test_checkpoint_round_trip(cuda):
    from ymp.train import TrainEngine
    batches = _batches(3, cuda)
    eng = TrainEngine(_tiny(cuda), lr=1e-3)
    for video, text in batches[:2]:
        eng.train_step(video, text, use_graph=False)
    td = tempfile.mkdtemp(prefix="ymp_ckpt_")
    eng.save_checkpoint(td, tag="checkpoint-0", client_state={"epoch": 0})
    saved = dict(master=eng.master.clone(), m=eng.exp_avg.clone(), v=eng.exp_avg_sq.clone(), p=eng.flat_param.clone())
    loss_next = eng.train_step(*batches[2], use_graph=False).item()
    after = eng.master.clone()
    # perturb everything, then restore (utils.auto_load_model: model.load_checkpoint(dir, tag=...))
    eng.master.add_(1.0); eng.exp_avg.fill_(7.0); eng.exp_avg_sq.fill_(7.0); eng.flat_param.zero_()
    _, client = eng.load_checkpoint(td, tag="checkpoint-0")
    assert client == {"epoch": 0} and eng.global_steps == 2
    assert torch.equal(eng.master, saved["master"]) and torch.equal(eng.exp_avg, saved["m"])
    assert torch.equal(eng.exp_avg_sq, saved["v"]) and torch.equal(eng.flat_param, saved["p"])
    # the module's parameters are views of flat_param: the model sees the restored weights
    p0 = next(p for p in eng.module.parameters() if p.requires_grad)
    assert p0.data_ptr() >= eng.flat_param.data_ptr() and p0.data_ptr() < eng.flat_param.data_ptr() + eng.flat_param.numel() * 2
    # a fresh engine loading `latest` continues identically (up to fp32 rounding)
    eng2 = TrainEngine(_tiny(cuda, seed=99), lr=1e-3)
    eng2.load_checkpoint(td)
    loss2 = eng2.train_step(*batches[2], use_graph=False).item()
    assert abs(loss2 - loss_next) <= 1e-3 * abs(loss_next)
    assert ((eng2.master - after).abs() > 0.05e-3).float().mean().item() < 2e-3


def test_engine_trains_autograd_side_parameters(cuda):
    """`temp` of the contrastive pre-training model and the narrow cls_head output layer get their gradients
    outside PretrainFn; the engine must still update them, and train_step must optimise
    loss_caption + loss_ita (run_pretrain_distributed_gpt3.py:113)."""
    from ymp.train import TrainEngine
    model = _tiny(cuda, use_contrastive=True, contrastive_embed_dim=32)
    with torch.no_grad():
        model.vision_proj.weight.normal_(0, 0.05); model.text_proj.weight.normal_(0, 0.05)
    eng = TrainEngine(model, lr=1e-3)
    video, text = _batches(1, cuda, B=3)[0]
    before = {k: p.detach().float().clone() for k, p in model.named_parameters() if p.requires_grad}
    lc, li = eng(video, text)
    assert li.item() != 0.0
    loss = eng.train_step(video, text, use_graph=False)
    assert abs(loss.item() - (lc + li).item()) <= 2e-3 * abs((lc + li).item())
    changed = {k for k, p in model.named_parameters() if p.requires_grad and not torch.equal(p.detach().float(), before[k])}
    for k in ("temp", "vision_proj.weight", "text_proj.weight", "visual_fc.weight", "visual_encoder.blocks.0.attn.qkv.weight"):
        assert k in changed, k
    assert all(p.grad is None for p in model.parameters())

    sd = port.init_state_dict(port.VCFG_TINY, port.GCFG_TINY, 8, seed=4, randomize=True)
    cls = build_pretrain(port.VCFG_TINY, port.GCFG_TINY, 8, sd=sd, device=cuda, dtype=torch.bfloat16,
                         cls_name="DistributedGPT3_Cls", use_cls=True, num_classes=5, num_frames=port.VCFG_TINY["num_frames"])
    eng = TrainEngine(cls, lr=1e-3)
    videoc, ids, att = make_inputs(2, port.VCFG_TINY, 8, port.GCFG_TINY["vocab_size"], 31)
    _, pids, patt = make_inputs(2, port.VCFG_TINY, 8, port.GCFG_TINY["vocab_size"], 32)
    before = {k: p.detach().float().clone() for k, p in cls.named_parameters() if p.requires_grad}
    lcap, lcls = eng(videoc.to(cuda).bfloat16(), _text(ids, att, cuda, prompt_lengths=torch.tensor([2, 3])),
                     _text(pids, patt, cuda), torch.tensor([1, 4], device=cuda), train=True)
    eng.backward(lcap + lcls)
    eng.step()
    for k in ("cls_head.0.weight", "cls_head.2.weight", "cls_head.2.bias"):
        assert not torch.equal(dict(cls.named_parameters())[k].detach().float(), before[k]), k


def test_narrow_linear_and_matmul_nt_against_torch(cuda):
    """LinearFn with out_features not a multiple of 8 (2 / 5 / 45-way heads) and the similarity GEMM, fwd + bwd."""
    from ymp import functional as YF
    torch.manual_seed(1)
    for (M, K, N) in ((6, 128, 5), (37, 128, 45), (4, 64, 2)):
        x = torch.randn(M, K, device=cuda).bfloat16().requires_grad_(True)
        w = (torch.randn(N, K, device=cuda) * 0.1).bfloat16().requires_grad_(True)
        b = torch.randn(N, device=cuda).bfloat16().requires_grad_(True)
        y = YF.LinearFn.apply(x, w, b)
        assert y.shape == (M, N)
        gy = torch.randn(M, N, device=cuda)
        y.float().backward(gy)
        xr, wr, br = (t.detach().float().requires_grad_(True) for t in (x, w, b))
        yr = torch.nn.functional.linear(xr, wr, br)
        yr.backward(gy.bfloat16().float())
        assert (y.float() - yr).abs().max() <= 2e-2 * yr.abs().max()
        for got, ref in ((x.grad, xr.grad), (w.grad, wr.grad), (b.grad, br.grad)):
            assert (got.float() - ref).abs().max() <= 2e-2 * ref.abs().max() + 1e-3, (M, K, N)
    for (M, K, N) in ((24, 32, 3), (6, 256, 96), (3, 32, 24)):
        x = torch.randn(M, K, device=cuda).requires_grad_(True)
        y = torch.randn(N, K, device=cuda).requires_grad_(True)
        s = YF.matmul_nt(x, y)
        gs = torch.randn(M, N, device=cuda)
        s.backward(gs)
        xr, yr = (t.detach().bfloat16().float().requires_grad_(True) for t in (x, y))
        sr = xr @ yr.t()
        sr.backward(gs.bfloat16().float())
        assert s.dtype == torch.float32 and (s - sr).abs().max() <= 1e-3 * sr.abs().max() + 1e-4
        assert (x.grad - xr.grad).abs().max() <= 2e-2 * xr.grad.abs().max()
        assert (y.grad - yr.grad).abs().max() <= 2e-2 * yr.grad.abs().max()


# ------------------------------------------------------------------------------------------ 2 GPUs / NCCL
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port_no, q):
    import sys
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port_no), RANK=str(rank), WORLD_SIZE=str(world),
                      YMP_ALLOW_RANDOM_INIT="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "youku-mplug_b200"), os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from models.distributed_utils import all_gather_cat, concat_all_gather
        from ymp.train import TrainEngine
        res = {}
        # ---- differentiable all-gather on NCCL (reference models/distributed_utils.py:285-311)
        torch.manual_seed(100 + rank)
        x = torch.randn(3, 4, device=dev, requires_grad=True)
        full = all_gather_cat(x)
        base = torch.arange(world * 3 * 4, dtype=torch.float32, device=dev).view(world * 3, 4)
        (full * base * (rank + 1)).sum().backward()
        expect = sum(base[rank * 3:(rank + 1) * 3] * (r + 1) for r in range(world))
        torch.manual_seed(100)
        r0 = torch.randn(3, 4, device=dev)
        res["gather_bwd"] = bool(torch.allclose(x.grad, expect))
        res["gather_fwd"] = bool(torch.equal(full[:3].detach(), r0)) and full.shape == (world * 3, 4)
        idx = torch.tensor([rank * 10 + 1, rank * 10 + 2], dtype=torch.int64, device=dev)
        res["gather_idx"] = concat_all_gather(idx).tolist() == [1, 2, 11, 12]
        # ---- data-parallel gradient: all-reduced flat_grad / world == mean of the per-shard gradients
        video, ids, att = make_inputs(2 * world, port.VCFG_TINY, 8, port.GCFG_TINY["vocab_size"], 77)
        video = video.to(dev).bfloat16()
        shard = lambda r: (video[2 * r:2 * r + 2], _text(ids[2 * r:2 * r + 2], att[2 * r:2 * r + 2], dev))  # noqa: E731
        for overlap in (False, True):
            eng = TrainEngine(_tiny(dev), lr=1e-3, overlap_comm=overlap)
            loss, _ = eng(*shard(rank))
            eng.backward(loss)
            eng.allreduce_gradients()
            got = eng.flat_grad.clone() / world
            ref = torch.zeros_like(got)
            single = TrainEngine(_tiny(dev), lr=1e-3, overlap_comm=False)
            single.world = 1
            for r in range(world):
                l, _ = single(*shard(r))
                single.backward(l)
            ref = single.flat_grad / world
            scale = ref.abs().max().item()
            res[f"dp_grad_overlap{int(overlap)}"] = (got - ref).abs().max().item() / scale
            res[f"buckets{int(overlap)}"] = len(eng._buckets)
        # ---- whole steps stay in lock-step across ranks: graph replay with the bucket all-reduces captured
        eng = TrainEngine(_tiny(dev), lr=1e-3, overlap_comm=True)
        for i in range(4):
            v, i2, a2 = make_inputs(2, port.VCFG_TINY, 8, port.GCFG_TINY["vocab_size"], 500 + 10 * i + rank)
            eng.train_step(v.to(dev).bfloat16(), _text(i2, a2, dev), use_graph=True, graph_warmup=1)
        flat = eng.master.clone()
        other = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(other, flat)
        res["replicas_identical"] = bool(all(torch.equal(o, other[0]) for o in other))
        res["graph_used"] = any("graph" in st for st in eng._graphs.values())
        # ---- contrastive pre-training across ranks (SURVEY 8a row a17): runs, finite, in-batch targets offset by rank
        model = _tiny(dev, use_contrastive=True, contrastive_embed_dim=32)
        v, i2, a2 = make_inputs(3, port.VCFG_TINY, 8, port.GCFG_TINY["vocab_size"], 900 + rank)
        lc, li = model(v.to(dev).bfloat16(), _text(i2, a2, dev))
        (lc + li).backward()
        res["contrastive_finite"] = bool(torch.isfinite(li)) and model.temp.grad is not None
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_two_gpu_data_parallel_gradient_and_allgather(cuda):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (run with gpurun --gpus 2)")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port_no = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port_no, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
    for rank, r in res:
        print("rank", rank, r)
        assert r["gather_fwd"] and r["gather_bwd"] and r["gather_idx"], r
        assert r["dp_grad_overlap0"] < 2e-2 and r["dp_grad_overlap1"] < 2e-2, r
        assert r["buckets1"] > 0 or True
        assert r["replicas_identical"] and r["graph_used"], r
        assert r["contrastive_finite"], r
