"""CPU: the batched beam-search host loop (models.modeling_distributed_gpt3.run_beam_search_batch) against the
per-sample loop (run_beam_search) with the same deterministic fake decoder: every sample's sequences and scores must be
equal, whatever chunk, group or padding the sample lands in."""
import pytest
import torch

V, STOP = 16, 2


def _logits(row, boost):
    """Next-token logits of one row: a seeded function of the row's token history.  The stop token gains `boost` per
    generated token past a history-dependent delay, so samples finish at different steps; boost None: never stop."""
    h = 0
    for t in row.tolist():
        h = (h * 1000003 + int(t) + 1) % (2 ** 31 - 1)
    g = torch.Generator().manual_seed(h)
    z = torch.randn(V, generator=g) * 2.0
    if boost is None:
        z[STOP] -= 50.0
        return z
    delay = 2 + int(row[0]) % 4
    z[STOP] += boost * max(0, row.numel() - 6 - delay)
    return z


class _PerSample:
    def __init__(self, boost):
        self.boost, self.hist, self.calls = boost, None, 0

    def step(self, new_tokens, first):
        self.calls += 1
        self.hist = new_tokens.clone() if first else torch.cat([self.hist, new_tokens], 1)
        return torch.stack([_logits(r, self.boost) for r in self.hist])

    def reorder(self, idx):
        self.hist = self.hist[idx]


class _Batch:
    def __init__(self, boost):
        self.boost, self.hist, self.chunks = boost, None, []

    def step(self, samples, new_tokens, first):
        if first:
            self.chunks.append(list(samples))
        self.hist = new_tokens.clone() if first else torch.cat([self.hist, new_tokens], 1)
        return torch.stack([_logits(r, self.boost) for r in self.hist])

    def reorder(self, idx):
        assert idx.dtype == torch.long and idx.numel() == self.hist.size(0)
        self.hist = self.hist[idx]


def _prompts(B, L, plens, seed):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(3, V, (B, L), generator=g)
    for i, p in enumerate(plens):
        tok[i, p:] = STOP     # padding past the prompt, as a tokenizer's pad id would be
    return tok


@pytest.mark.parametrize("boost,num_return_gen", [(None, 1), (None, 2), (0.6, 1), (1.5, 2), (4.0, 3)])
def test_batch_loop_equals_per_sample_loop(boost, num_return_gen):
    import models.modeling_distributed_gpt3 as M
    beam, L, ttg = 3, 6, 9
    plens = [3, 3, 4, 3, 4, 5, 3, 3, 4]
    tokens = _prompts(len(plens), L, plens, seed=11)
    kw = dict(beam_size=beam, num_return_gen=num_return_gen, stop_token=STOP, tokens_to_generate=ttg,
              max_position_embeddings=64)
    bat = _Batch(boost)
    got = M.run_beam_search_batch(bat.step, bat.reorder, tokens, torch.tensor(plens), 4, max_rows=9, **kw)   # 3 per chunk
    calls = []
    for i, p in enumerate(plens):
        ref_dec = _PerSample(boost)
        ref = M.run_beam_search(ref_dec.step, ref_dec.reorder, tokens[i:i + 1], p, 4, **kw)
        calls.append(ref_dec.calls)
        assert torch.equal(got[i].sequences, ref.sequences), (i, got[i].sequences, ref.sequences)
        assert got[i].scores.dtype == ref.scores.dtype and torch.equal(got[i].scores, ref.scores), (i, got[i].scores, ref.scores)
        assert ref.sequences.size(0) == min(num_return_gen, beam)
    # groups by prompt length, chunks of 3 samples, short chunks padded with their first sample
    assert bat.chunks == [[0, 1, 3], [6, 7, 6], [2, 4, 8], [5, 5, 5]]
    full = [L + ttg - p for p in plens]
    if boost is None:
        assert calls == full                                      # every sample reaches the final length
    if boost is not None and boost >= 1.5:
        assert all(c < f for c, f in zip(calls, full))            # early stop through is_done
        assert len(set(calls)) > 1                                # at different steps


def test_batch_loop_more_samples_than_one_chunk_default_rows():
    """The default 64-row chunks at beam 5 hold 12 samples: 25 equal-length samples take three chunks, the last one
    padded."""
    import models.modeling_distributed_gpt3 as M
    beam, B, plen = 5, 25, 4
    tokens = _prompts(B, 5, [plen] * B, seed=5)
    kw = dict(beam_size=beam, num_return_gen=1, stop_token=STOP, tokens_to_generate=6, max_position_embeddings=64)
    bat = _Batch(1.0)
    got = M.run_beam_search_batch(bat.step, bat.reorder, tokens, [plen] * B, 2, **kw)
    assert [len(c) for c in bat.chunks] == [12, 12, 12] and bat.chunks[2] == [24] * 12
    for i in range(B):
        ref_dec = _PerSample(1.0)
        ref = M.run_beam_search(ref_dec.step, ref_dec.reorder, tokens[i:i + 1], plen, 2, **kw)
        assert torch.equal(got[i].sequences, ref.sequences) and torch.equal(got[i].scores, ref.scores), i


def test_beam_chunks_and_bad_arguments():
    import models.modeling_distributed_gpt3 as M
    assert list(M.beam_chunks([5, 3, 5, 5, 3], 2)) == [(5, [0, 2]), (5, [3]), (3, [1, 4])]
    tokens = _prompts(2, 4, [4, 4], seed=1)
    kw = dict(num_return_gen=1, stop_token=STOP, tokens_to_generate=0, max_position_embeddings=64)
    with pytest.raises(ValueError, match="too large"):
        M.run_beam_search_batch(None, None, tokens, [4, 4], 0, beam_size=2, **kw)
    with pytest.raises(ValueError, match="max_rows"):
        M.run_beam_search_batch(None, None, tokens, [4, 4], 0, beam_size=65, **kw)


def test_beam_batch_cache_table_start_and_reorder():
    """ymp.engine.BeamBatchCache host logic: the table starts as the identity with every beam's prefix read from its
    sample's beam 0; a reorder copies table rows over the cached positions only and never touches the K/V store."""
    from oracle import port
    from ymp import engine
    gcfg = dict(port.GCFG_TINY)
    n, beam, ML = 2, 3, 7
    c = engine.BeamBatchCache(gcfg, n, beam, ML, torch.device("cpu"))
    assert c.B == 6 and c.table.shape == (6, ML) and c.table.dtype == torch.int32
    ident = (torch.arange(6)[:, None] * ML + torch.arange(ML)[None]).int()
    assert torch.equal(c.table, ident)
    blk = c.block(1)
    assert blk.B == beam and all(t.data_ptr() == s[beam * ML:].data_ptr() and t.shape[0] == beam * ML for t, s in zip(blk.qkv, c.qkv))
    c._set_len(3)
    c.start_table(3)
    for r in range(6):
        base = (r // beam) * beam
        assert c.table[r, :3].tolist() == [base * ML + j for j in range(3)]
        assert torch.equal(c.table[r, 3:], ident[r, 3:])
    c._set_len(5)
    store = c.store.clone()
    before = c.table.clone()
    idx = torch.tensor([2, 2, 0, 3, 5, 4])
    c.reorder_table(idx)
    assert torch.equal(c.table[:, :5], before[idx, :5]) and torch.equal(c.table[:, 5:], before[:, 5:])
    assert torch.equal(c.store, store)
