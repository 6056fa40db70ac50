"""GPU: batched beam search (DistributedGPT3.beam_search_batch, DistributedGPT3_Caption.generate_batch) and the kernels
under it - the skinny GEMM at up to 64 rows and the decode attention that finds its keys through a per-row table -
against the per-sample path, bit for bit."""
import os

import pytest
import torch

from oracle import port
from oracle.make_golden import make_inputs
from helpers import build_pretrain, make_model_dir

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
bf16 = torch.bfloat16

# (name, N, K) of the decoding step's linears: QKV, attention dense, fc1, fc2, tied LM head
SHAPES = {"1.3B": [("qkv", 6144, 2048), ("dense", 2048, 2048), ("fc1", 8192, 2048), ("fc2", 2048, 8192), ("lm_head", 51200, 2048)],
          "2.7B": [("qkv", 7680, 2560), ("dense", 2560, 2560), ("fc1", 10240, 2560), ("fc2", 2560, 10240), ("lm_head", 51200, 2560)]}
ROWS = [1, 5, 8, 9, 16, 17, 40, 60, 64]
# (act, bias, residual dtype, out dtype, KV-cache copy)
EPILOGUES = [(0, False, None, bf16, False), (2, True, None, bf16, True), (1, True, bf16, torch.float32, False),
             (0, True, torch.float32, torch.float32, False), (2, False, torch.float32, bf16, True)]


@pytest.mark.parametrize("model", ["1.3B", "2.7B"])
@pytest.mark.parametrize("epi", range(len(EPILOGUES)))
def test_skinny_gemm_wide_rows(cuda, model, epi):
    """ops.gemm_skinny_batch (ymp_gemm_skinny_batch) at every M in ROWS: against fp32 torch within bf16 tolerance, and
    every row bit-identical to the same row computed alone (M = 1) - the kernel layout depends on N and K only; the
    8-row entry point gives the same bits."""
    from ymp import ops
    act, has_bias, res_dt, out_dt, copy = EPILOGUES[epi]
    g = torch.Generator(device=cuda).manual_seed(7 + epi)
    for name, N, K in SHAPES[model]:
        w = (torch.randn(N, K, device=cuda, generator=g) * 0.02).to(bf16)
        x = torch.randn(64, K, device=cuda, generator=g).to(bf16)
        bias = (torch.randn(N, device=cuda, generator=g) * 0.1).to(bf16) if has_bias else None
        res = torch.randn(64, N, device=cuda, generator=g).to(res_dt) if res_dt is not None else None
        ref = x.float() @ w.float().t()
        if bias is not None:
            ref = ref + bias.float()
        if act == 2:
            ref = torch.nn.functional.gelu(ref, approximate="tanh")
        elif act == 1:
            ref = torch.nn.functional.gelu(ref)
        if res is not None:
            ref = ref + res.float()

        def run(rows):
            M = rows.stop - rows.start
            kw = dict(bias=bias, act=act, out_dtype=out_dt, residual=None if res is None else res[rows])
            if not copy:
                return ops.gemm_skinny_batch(x[rows], w, **kw), None
            ML, off = 4, torch.tensor([2], device=cuda, dtype=torch.int64)
            cache = torch.zeros(M * ML, N, device=cuda, dtype=bf16)
            y = ops.gemm_skinny_batch(x[rows], w, out2=cache, out2_row_stride=ML, out2_off=off, **kw)
            return y, cache.view(M, ML, N)[:, 2]

        alone = [run(slice(r, r + 1)) for r in range(64)]
        for M in ROWS:
            y, y2 = run(slice(0, M))
            err = (y.float() - ref[:M]).abs().max().item()
            assert err <= 2e-2 * ref[:M].abs().max().item() + 1e-2, (name, M, err)
            same = torch.cat([a[0] for a in alone[:M]])
            assert torch.equal(y, same), (name, M, (y.float() - same.float()).abs().max().item())
            if copy:
                assert torch.equal(y2, y), (name, M)
            if M <= 8 and not copy:
                assert torch.equal(ops.gemm_skinny(x[:M], w, bias=bias, act=act, out_dtype=out_dt,
                                                   residual=None if res is None else res[:M]), y), (name, M)


def test_skinny_gemm_rejects_65_rows_and_wide_layernorm(cuda):
    import ctypes
    from ymp import lib, ops
    w = torch.randn(256, 128, device=cuda).to(bf16)
    x = torch.randn(65, 128, device=cuda).to(bf16)
    a = lib.GemmSkinnyArgs()
    a.x, a.w, a.y = x.data_ptr(), w.data_ptr(), torch.empty(65, 256, device=cuda, dtype=bf16).data_ptr()
    a.M, a.N, a.K, a.ldx, a.ldw, a.ldy = 65, 256, 128, 128, 128, 256
    assert lib._gemm_skinny_batch(ctypes.byref(a), lib.cur_stream()) == -1 and b"M <= 64" in lib.lib.ymp_last_error()
    with pytest.raises(AssertionError):
        ops.gemm_skinny_batch(x, w)
    ln = (torch.ones(256, device=cuda, dtype=bf16), torch.zeros(256, device=cuda, dtype=bf16), 1e-5,
          torch.zeros(1, device=cuda, dtype=torch.int32))
    ops.gemm_skinny(torch.randn(8, 128, device=cuda).to(bf16), w, out_dtype=torch.float32, ln=ln)   # 8 rows: accepted
    with pytest.raises(Exception, match="LayerNorm needs M <= 8"):
        ops.gemm_skinny_batch(torch.randn(9, 128, device=cuda).to(bf16), w, out_dtype=torch.float32, ln=ln)


@pytest.mark.parametrize("hd", [64, 80, 96])
@pytest.mark.parametrize("dev_len", [False, True])
def test_table_attention_equals_gathered_cache(cuda, hd, dev_len):
    """Decode attention through a random key-row table (rows shared between sequences) against the plain kernel over a
    cache physically gathered into the table's order, bit for bit; other paths reject the table."""
    from ymp import lib as L
    from ymp import ops
    from ymp.ops import TView
    R, heads, ML, s_kv = 24, 4, 300, 257
    g = torch.Generator(device=cuda).manual_seed(hd)
    buf = torch.randn(R * ML, 3 * heads * hd, device=cuda, generator=g).to(bf16)
    q = torch.randn(R, 3 * heads * hd, device=cuda, generator=g).to(bf16)
    table = torch.randint(0, R * ML, (R, ML), device=cuda, generator=g)
    table[1::2, :100] = table[0::2, :100]                                       # pairs of rows share their first slots
    table[:, 200:230] = table[:1, 200:230]                                      # and every row shares a few more
    table = table.int().contiguous()
    gathered = buf[table.long().reshape(-1)].contiguous()                       # [R * ML, 3 * heads * hd]
    len1 = torch.tensor([131], device=cuda, dtype=torch.int32) if dev_len else None
    m1, mkv = ops.dense_map(1), ops.dense_map(ML)

    def attn(kvbuf, tab):
        o = torch.empty(R, heads * hd, device=cuda, dtype=bf16)
        ops.attn_fwd(TView(q, 0, 3 * hd, m1), TView(kvbuf, hd, 3 * hd, mkv), TView(kvbuf, 2 * hd, 3 * hd, mkv), TView(o, 0, hd, m1),
                     n_seq=R, n_heads=heads, head_dim=hd, s_q=1, s_kv=s_kv, causal=False, scale=hd ** -0.5, s_kv_dev=len1,
                     kv_rows=tab)
        return o

    plain = attn(gathered, None)
    via_table = attn(buf, table)
    assert torch.equal(via_table, plain)
    # the rows the table does not reach make no difference
    buf2 = buf.clone()
    used = torch.zeros(R * ML, dtype=torch.bool, device=cuda)
    used[table[:, :s_kv].long().reshape(-1)] = True
    buf2[~used] = 0
    assert torch.equal(attn(buf2, table), plain)
    # s_q > 1 (mma.sync / tcgen05 paths) rejects the table
    o = torch.empty(R * 2, heads * hd, device=cuda, dtype=bf16)
    m2 = ops.dense_map(2)
    with pytest.raises(Exception, match="kv_rows"):
        ops.attn_fwd(TView(buf, 0, 3 * hd, m2), TView(buf, hd, 3 * hd, mkv), TView(buf, 2 * hd, 3 * hd, mkv), TView(o, 0, hd, m2),
                     n_seq=R, n_heads=heads, head_dim=hd, s_q=2, s_kv=s_kv, causal=False, scale=0.1, kv_rows=table)
    b = L.AttnBwdArgs()
    lse = torch.empty(R, heads, 2, device=cuda)
    b.fwd = ops._attn_args(TView(buf, 0, 3 * hd, m2), TView(buf, hd, 3 * hd, mkv), TView(buf, 2 * hd, 3 * hd, mkv), TView(o, 0, hd, m2),
                           lse, R, heads, hd, 2, s_kv, False, 0.1, kv_rows=table)
    b.dout = b.dq = b.dk = b.dv = o.data_ptr()      # never written: the call is rejected first
    b.delta_ws = lse.data_ptr()
    b.lddo = b.lddq = b.lddk = b.lddv = o.stride(0)
    with pytest.raises(Exception, match="kv_rows"):
        L.call(L._attn_bwd, b, "ymp_attn_bwd")


# ---------------------------------------------------------------------------------------------- decoder level
def _tiny(dev):
    fx = torch.load(os.path.join(GOLD, "tiny_generate.pt"), weights_only=False)
    sd = port.generation_state_dict(fx["vcfg"], fx["gcfg"], fx["Q"], fx["wseed"], fx["pos_gain"], fx["ln_gain"])
    model = build_pretrain(fx["vcfg"], fx["gcfg"], fx["Q"], sd=sd, device=dev, dtype=bf16,
                           cls_name="DistributedGPT3_Caption", num_frames=fx["vcfg"]["num_frames"]).eval()
    return fx, model


def _decoder_13b(dev, layers):
    import bench
    import models.modeling_distributed_gpt3 as M
    os.environ["YMP_ALLOW_RANDOM_INIT"] = "1"
    td = make_model_dir(bench.VCFG_CLIP_B16, dict(bench.GCFG["1.3B"], num_hidden_layers=layers, tokens_to_generate=16))
    torch.manual_seed(0)
    with torch.device(dev):
        return M.DistributedGPT3(td, 0, megatron_cfg={}).to(bf16).eval()


def _teacher_forced(dec, qf, prompt, beam, n_steps, seed):
    """Per-sample path (dec(tokens=...) + swap_key_value_dict) and the batched step over all samples, fed the same tokens
    and the same beam reorders; returns both logits stacks [n_steps + 1, n * beam, V]."""
    import models.modeling_distributed_gpt3 as M
    n, P = prompt.shape
    dev, V = prompt.device, dec.config.vocab_size
    g = torch.Generator().manual_seed(seed)
    toks = torch.randint(0, V, (n_steps, n * beam, 1), generator=g)
    perms = torch.randint(0, beam, (n_steps, n, beam), generator=g)
    ML = qf.size(1) + P + n_steps + 1
    ref = []
    with torch.no_grad():
        for i in range(n):
            dec.inference_params = M.InferenceParams(beam, ML)
            out = dec(tokens=prompt[i:i + 1].repeat(beam, 1), query_embeds=qf[i:i + 1].repeat(beam, 1, 1))
            rows = [out.logits[:, -1].clone()]
            for t in range(n_steps):
                dec.inference_params.swap_key_value_dict(perms[t, i].tolist())
                out = dec(tokens=toks[t, i * beam:(i + 1) * beam].to(dev))
                rows.append(out.logits[:, -1].clone())
            ref.append(torch.stack(rows))
        bd = M._BeamBatchDecoder(dec, qf, beam, n, ML, dev)
        got = [bd.step(list(range(n)), prompt.repeat_interleave(beam, 0), True).clone()]
        for t in range(n_steps):
            idx = (perms[t] + torch.arange(n)[:, None] * beam).reshape(-1)
            bd.reorder(idx.to(dev))
            got.append(bd.step(list(range(n)), toks[t].to(dev), False).clone())
    return torch.cat(ref, dim=1), torch.stack(got), bd


def test_batched_step_logits_equal_per_sample_tiny(cuda):
    fx, model = _tiny(cuda)
    dec, Q, H = model.text_decoder, fx["Q"], fx["gcfg"]["hidden_size"]
    n, beam = 7, 3
    g = torch.Generator().manual_seed(3)
    qf = (torch.randn(n, Q, H, generator=g) * 0.5).to(bf16).to(cuda)
    prompt = torch.randint(0, fx["gcfg"]["vocab_size"], (n, 5), generator=g).to(cuda)
    ref, got, _ = _teacher_forced(dec, qf, prompt, beam, 10, seed=4)
    for t in range(ref.size(0)):
        assert torch.equal(got[t], ref[t]), (t, (got[t] - ref[t]).abs().max().item())


def test_batched_step_logits_equal_per_sample_1p3b(cuda):
    dec = _decoder_13b(cuda, layers=6)
    n, beam, Q = 12, 5, 128
    g = torch.Generator().manual_seed(5)
    qf = (torch.randn(n, Q, 2048, generator=g) * 0.1).to(bf16).to(cuda)
    prompt = torch.randint(0, 51200, (n, 9), generator=g).to(cuda)
    ref, got, _ = _teacher_forced(dec, qf, prompt, beam, 6, seed=6)
    for t in range(ref.size(0)):
        assert torch.equal(got[t], ref[t]), (t, (got[t] - ref[t]).abs().max().item())


def test_batched_graph_equals_eager_and_is_reused(cuda, monkeypatch):
    fx, model = _tiny(cuda)
    dec, Q, H = model.text_decoder, fx["Q"], fx["gcfg"]["hidden_size"]
    n, beam = 6, 3
    g = torch.Generator().manual_seed(8)
    qf = (torch.randn(n, Q, H, generator=g) * 0.5).to(bf16).to(cuda)
    prompt = torch.randint(0, fx["gcfg"]["vocab_size"], (n, 4), generator=g).to(cuda)
    monkeypatch.setenv("YMP_DECODE_GRAPH", "0")
    dec.__dict__.pop("_beam_batch_pool", None)
    _, eager, _ = _teacher_forced(dec, qf, prompt, beam, 6, seed=9)
    monkeypatch.setenv("YMP_DECODE_GRAPH", "1")
    dec.__dict__.pop("_beam_batch_pool", None)
    _, graphed, bd = _teacher_forced(dec, qf, prompt, beam, 6, seed=9)
    assert torch.equal(eager, graphed)
    cache, ts = bd.cache, bd.cache.token
    assert ts is not None and ts.graph is not None
    _, again, bd2 = _teacher_forced(dec, qf, prompt, beam, 6, seed=9)     # the per-sample calls in between recapture nothing
    assert bd2.cache is cache and cache.token is ts and torch.equal(again, eager)


# ---------------------------------------------------------------------------------------------- end to end
def _caption_setup(model, fx, beam):
    import models.modeling_distributed_gpt3 as M
    model.text_decoder.config.tokens_to_generate = fx["n_new"]

    class _Tok:
        class tokenizer:
            eos = fx["eod"]
    model.tokenizer = _Tok()
    dec = model.text_decoder
    orig, orig_b = dec.beam_search, dec.beam_search_batch
    dec.beam_search = lambda *a, **k: orig(*a, **dict(k, beam_size=beam))
    dec.beam_search_batch = lambda *a, **k: orig_b(*a, **dict(k, beam_size=beam))
    return M


def _assert_same(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and torch.equal(x, y), (i, x.tolist(), y.tolist())


def test_generate_batch_equals_generate_golden(cuda):
    fx, model = _tiny(cuda)
    M = _caption_setup(model, fx, fx["beam_size"])
    video, _, _ = make_inputs(fx["B"], fx["vcfg"], fx["L"], fx["gcfg"]["vocab_size"], fx["iseed"])
    text = M.BatchEncoding(dict(input_ids=fx["ids"].to(cuda), attention_mask=fx["att"].to(cuda)))
    v = video.to(cuda).bfloat16()
    _assert_same(model.generate_batch(v, text), model.generate(v, text))


def test_generate_batch_equals_generate_many_clips(cuda):
    """27 clips with the fixture's first prompt (two chunks of 64 // 3 = 21 clips at beam 3, the second one padded),
    then a batch of three prompt lengths."""
    fx, model = _tiny(cuda)
    M = _caption_setup(model, fx, fx["beam_size"])
    B = 27
    video, _, _ = make_inputs(B, fx["vcfg"], fx["L"], fx["gcfg"]["vocab_size"], 77)
    v = video.to(cuda).bfloat16()
    ids, att = fx["ids"][:1].repeat(B, 1), fx["att"][:1].repeat(B, 1)
    text = M.BatchEncoding(dict(input_ids=ids.to(cuda), attention_mask=att.to(cuda)))
    _assert_same(model.generate_batch(v, text), model.generate(v, text))
    # mixed prompt lengths: the fixture's two prompts plus shortened copies
    B2 = 9
    ids2, att2 = fx["ids"][torch.arange(B2) % 2].clone(), fx["att"][torch.arange(B2) % 2].clone()
    for i in range(B2):
        n = int(att2[i].sum()) - i % 3
        att2[i, n:] = 0
    text2 = M.BatchEncoding(dict(input_ids=ids2.to(cuda), attention_mask=att2.to(cuda)))
    assert len(set((att2.sum(-1) - 1).tolist())) >= 3
    _assert_same(model.generate_batch(v[:B2], text2), model.generate(v[:B2], text2))


def test_beam_search_batch_equals_beam_search_1p3b(cuda):
    dec = _decoder_13b(cuda, layers=6)
    n, beam, Q = 12, 5, 128
    g = torch.Generator().manual_seed(12)
    qf = (torch.randn(n, Q, 2048, generator=g) * 0.1).to(bf16).to(cuda)
    tokens = torch.randint(0, 51200, (n, 10), generator=g).to(cuda)
    plen = torch.full((n,), 7, dtype=torch.long)
    got = dec.beam_search_batch(tokens, query_embeds=qf, prompt_length=plen, beam_size=beam, stop_token=7)
    for i in range(n):
        ref = dec.beam_search(tokens[i:i + 1], query_embeds=qf[i:i + 1], prompt_length=7, beam_size=beam, stop_token=7)
        assert torch.equal(got[i].sequences, ref.sequences), i
        assert torch.equal(got[i].scores, ref.scores), i
