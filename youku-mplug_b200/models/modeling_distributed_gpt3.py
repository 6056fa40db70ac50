"""GPT-3 (1.3B / 2.7B Megatron-style) decoder of mPLUG-Video on the B200 kernels.

Mirrors the reference module `models/modeling_distributed_gpt3.py`: GPT3Config (:459-547),
BatchEncoding (:139-178), DistributedGPT3Tokenizer (:180-319), DistributedGPT3 (:1522-1618).
No megatron_util: tensor-model-parallel size must be 1 (SURVEY.md D6) - the path is pure data
parallel.  Parameter names equal the reference's (`dist_model.language_model....`), including the
per-head [q|k|v] row grouping of query_key_value, so `model/mp_rank_00_model_states.pt` loads as is.

Host-side API helpers whose behaviour has to match the reference token for token - BatchEncoding (:139-176), the
top-k / top-p logit filters and `sample` (:1369-1443), BeamHypotheses (:1908-1961) - keep the reference's control flow
and messages on purpose (they are thin re-statements of upstream Megatron / HF utilities and are pinned against the
reference's own outputs in tests/golden/tiny_generate.pt); everything that touches the device - parameter containers,
the KV cache, the decoding loops run_sample / run_beam_search, the captured single-token step - is this package's own.
"""
import json
import math
import os
import os.path as osp

import numpy as np
import torch
import torch.nn as nn

from ymp import functional as YF

from ._params import EmbedHolder, Holder, add_param, named_param_list


class AttrDict(dict):
    """addict.Dict-like result container (attribute access; missing keys -> None)."""
    __getattr__ = dict.get
    __setattr__ = dict.__setitem__


class GPT3Config:
    model_type = 'gpt3'

    def __init__(self, vocab_size=25600, hidden_size=768, ffn_hidden_size=None, num_hidden_layers=12,
                 num_attention_heads=12, intermediate_size=3072, hidden_act='gelu', hidden_dropout_prob=0.1,
                 attention_probs_dropout_prob=0.1, max_position_embeddings=2048, type_vocab_size=2,
                 layernorm_epsilon=1e-12, bias_gelu_fusion=True, fp32_residual_connection=False,
                 sequence_parallel=False, fp16=False, bf16=False, apply_query_key_layer_scaling=True,
                 attention_softmax_in_fp32=False, kv_channels=None, masked_softmax_fusion=True,
                 attention_dropout=0.1, bias_dropout_fusion=True,
                 apply_residual_connection_post_layernorm=False, hidden_dropout=0.1, init_method_std=0.02,
                 eod_id=7, tokens_to_generate=100, top_k=0, top_p=0.9, **kwargs):
        self.vocab_size = vocab_size
        self.hidden_size = hidden_size
        self.ffn_hidden_size = 4 * hidden_size if ffn_hidden_size is None else ffn_hidden_size
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.intermediate_size = intermediate_size
        self.hidden_act = hidden_act
        self.hidden_dropout_prob = hidden_dropout_prob
        self.attention_probs_dropout_prob = attention_probs_dropout_prob
        self.max_position_embeddings = max_position_embeddings
        self.type_vocab_size = type_vocab_size
        self.layernorm_epsilon = layernorm_epsilon
        self.layer_norm_eps = layernorm_epsilon
        self.fp16, self.bf16 = fp16, bf16
        assert not (fp16 and bf16)
        assert hidden_size % num_attention_heads == 0
        self.kv_channels = hidden_size // num_attention_heads if kv_channels is None else kv_channels
        self.attention_dropout = attention_dropout
        self.hidden_dropout = hidden_dropout
        self.init_method_std = init_method_std
        self.apply_query_key_layer_scaling = apply_query_key_layer_scaling
        self.apply_residual_connection_post_layernorm = apply_residual_connection_post_layernorm
        self.sequence_parallel = sequence_parallel
        self.eod_id, self.tokens_to_generate, self.top_k, self.top_p = eod_id, tokens_to_generate, top_k, top_p
        for k, v in kwargs.items():
            setattr(self, k, v)
        if apply_residual_connection_post_layernorm or sequence_parallel or fp32_residual_connection:
            raise NotImplementedError("unsupported GPT3Config option for the B200 path")

    @classmethod
    def from_json_file(cls, path):
        with open(path, 'r') as f:
            return cls(**json.load(f))

    @classmethod
    def from_pretrained(cls, model_dir):
        return cls.from_json_file(osp.join(model_dir, 'config.json'))

    def to_dict(self):
        return dict(self.__dict__)

    def engine_cfg(self, training=False):
        """Dims + the dropout setting of one decoder pass: hidden_dropout / attention_dropout are live only in
        train() mode (the reference keeps the frozen decoder in train mode during training)."""
        return dict(vocab_size=self.vocab_size, hidden_size=self.hidden_size, ffn_hidden_size=self.ffn_hidden_size,
                    num_hidden_layers=self.num_hidden_layers, num_attention_heads=self.num_attention_heads,
                    max_position_embeddings=self.max_position_embeddings, layernorm_epsilon=self.layernorm_epsilon,
                    hidden_dropout=self.hidden_dropout, attention_dropout=self.attention_dropout, training=bool(training))


# ------------------------------------------------------------------------------------------ tokenizer
class JiebaBPETokenizer:
    """BPE tokenizer (tokenizers json) with jieba pre-segmentation, <sep> as BOS and
    <|endoftext|> as EOS/PAD (reference :42-137)."""

    def __init__(self, tokenizer_json_file):
        from tokenizers import Tokenizer
        self.tokenizer = Tokenizer.from_file(tokenizer_json_file)
        try:
            import jieba
            self._cut = lambda s: list(jieba.cut(s))
        except ImportError:  # not in this image: whitespace segmentation keeps the API usable
            self._cut = lambda s: s.split()
        self.eod_id = self.eos_id = self.pad_id = self.tokenizer.token_to_id('<|endoftext|>')
        self.bos_id = self.sep_token = self.tokenizer.token_to_id('<sep>')

    @property
    def vocab_size(self):
        return self.tokenizer.get_vocab_size(with_added_tokens=True)

    @property
    def vocab(self):
        return self.tokenizer.get_vocab(with_added_tokens=True)

    def _ids(self, text, is_code):
        if is_code:
            return self.tokenizer.encode(text, is_pretokenized=False, add_special_tokens=True).ids
        return self.tokenizer.encode(self._cut(text), is_pretokenized=True, add_special_tokens=True).ids

    def tokenize(self, text, is_code=False, add_special_tokens=True):
        ids = self._ids(text, is_code)
        return [self.bos_id] + ids + [self.eos_id] if add_special_tokens else ids

    def tokenize_prompt(self, prompt_text, text, is_code=False, add_special_tokens=True):
        return [[self.bos_id], self._ids(prompt_text, is_code), self._ids(text, is_code), [self.eos_id]]

    def detokenize(self, token_ids):
        return self.tokenizer.decode(token_ids, skip_special_tokens=True)

    eod = property(lambda self: self.eod_id)
    eos = property(lambda self: self.eos_id)
    bos = property(lambda self: self.bos_id)
    pad = property(lambda self: self.pad_id)


class BatchEncoding:
    def __init__(self, data):
        self.data = data

    def __getitem__(self, item):
        if isinstance(item, str):
            return self.data[item]
        raise KeyError("integer indexing is not available for this tokenizer")

    def __getattr__(self, item):
        try:
            return self.__dict__["data"][item]
        except KeyError:
            raise AttributeError(item)

    def __getstate__(self):
        return {"data": self.data}

    def __setstate__(self, state):
        self.__dict__["data"] = state["data"]

    def __repr__(self):
        return str(self.data)

    def keys(self):
        return self.data.keys()

    def values(self):
        return self.data.values()

    def items(self):
        return self.data.items()

    def to(self, device):
        self.data = {k: v.to(device=device) for k, v in self.data.items()}
        return self


class DistributedGPT3Tokenizer:
    def __init__(self, model_dir, sequence_length=128):
        self.tokenizer = JiebaBPETokenizer(osp.join(model_dir, 'tokenizer.json'))
        self.max_length = sequence_length

    def decode(self, tokens, **kwargs):
        if isinstance(tokens, torch.Tensor):
            tokens = tokens.detach().cpu().tolist()
        return self.tokenizer.detokenize(tokens)

    def _fit(self, ids, length):
        """pad with the pad id / cut to `length`; returns (array, number of real tokens)."""
        ids = list(ids)[:length]
        n = len(ids)
        return np.asarray(ids + [self.tokenizer.pad] * (length - n), dtype=np.int64), n

    def _fit_prompt(self, parts, length):
        bos, prompt, text, eos = parts
        if len(bos) + len(prompt) + len(text) + len(eos) > length:
            room = length - len(text) - 2
            if room >= 0 and len(prompt) >= room:   # shorten the prompt first
                prompt = prompt[:room]
            else:                                    # otherwise cut the target
                text = text[:length - 2 - len(prompt)]
        arr, n = self._fit(bos + prompt + text + eos, length)
        return arr, len(prompt), n

    def __call__(self, data, padding='longest', truncation=True, max_length=None, return_tensors='pt',
                 add_special_tokens=True, **kwargs):
        max_length = self.max_length if max_length is None else max_length
        pairs = not isinstance(data[0], str)
        if pairs:
            toks = [self.tokenizer.tokenize_prompt(p, t) for p, t in data]
            longest = max(sum(len(x) for x in t) for t in toks)
            # the reference pads pair inputs to max_length whenever truncation is on (:289-296)
            length = max_length if (truncation or padding == 'max_length') else longest
        else:
            # NB: the reference passes add_special_tokens positionally into `is_code` (:240);
            # keep the observable behaviour: text path, specials always added.
            toks = [self.tokenizer.tokenize(t) for t in data]
            longest = max(len(t) for t in toks)
            if padding == 'max_length':
                length = max_length
            else:
                length = min(longest, max_length) if truncation else longest
        ids, mask, plen = [], [], []
        for t in toks:
            if pairs:
                arr, pl, n = self._fit_prompt(t, length)
                plen.append(pl)
            else:
                arr, n = self._fit(t, length)
            m = np.zeros(length, dtype=np.int64)
            m[:n] = 1
            ids.append(arr)
            mask.append(m)
        out = dict(input_ids=np.stack(ids), attention_mask=np.stack(mask))
        if pairs:
            out["prompt_lengths"] = np.asarray(plen, dtype=np.int64)
        if return_tensors == 'pt':
            out = {k: torch.from_numpy(v).long() for k, v in out.items()}
        return BatchEncoding(out)


# ------------------------------------------------------------------------------------------ model
def _ckpt_name(mp_rank, load_dir, tag):
    return osp.join(load_dir, str(tag), 'mp_rank_{:02d}_model_states.pt'.format(mp_rank))


def pre_load(mp_rank, load_dir, tag=''):
    """{text_decoder}/model/mp_rank_00_model_states.pt['module'] (reference :431-441)."""
    ckpt = torch.load(_ckpt_name(mp_rank, load_dir, tag), map_location='cpu', weights_only=False)
    return ckpt['module']


def _check_tp1(megatron_cfg):
    if not megatron_cfg:
        return
    for k in ('tensor_model_parallel_size', 'model_parallel_size'):
        v = megatron_cfg.get(k, 1)
        if v not in (None, 1):
            raise ValueError(f"megatron_cfg.{k}={v}: the B200 path is pure data parallel; set it to 1 "
                             "(as the reference's own scripts/*.sh:13-14 and retrieval yaml do)")


# ----------------------------------------------------------------------------------------------
# Generation (SURVEY.md 8f N2): the host logic of models/modeling_distributed_gpt3.py:1369-1473,1620-1886,
# 1908-1961 on top of the KV-cache decode path of ymp.engine.
# ----------------------------------------------------------------------------------------------
def modify_logits_for_top_k_filtering(logits, top_k):
    """In place: everything below the k-th largest logit of its row becomes -inf (:1369-1373)."""
    kth = torch.topk(logits, top_k)[0][..., -1, None]
    logits.masked_fill_(logits < kth, float('-Inf'))


def modify_logits_for_top_p_filtering(logits, top_p):
    """In place nucleus filter (:1376-1395): sorted cumulative probability > top_p is dropped, shifted by
    one position so that the token crossing the threshold is kept; the best token always survives."""
    sorted_logits, sorted_indices = torch.sort(logits, descending=True)
    drop = sorted_logits.softmax(dim=-1).cumsum(dim=-1) > top_p
    drop[:, 1:] = drop[:, :-1].clone()
    drop[..., 0] = 0
    logits.masked_fill_(drop.scatter(1, sorted_indices, drop), float('-Inf'))


def sample(logits, top_k=0, top_p=0.0, temperature=1.0, vocab_size=None):
    """One token per row of logits [b, v] (:1398-1446): argmax when top_k == 1, otherwise temperature,
    top-k or top-p filtering and a multinomial draw; clamped into [0, vocab_size)."""
    assert logits.ndim == 2, 'expected the logits to be of [b, v] shape.'
    if top_k == 1:
        assert top_p == 0.0, 'cannot set both greedy and top-p samplings.'
        samples = torch.argmax(logits, dim=-1)
    else:
        logits = logits.clone()
        if temperature != 1.0:
            logits.div_(temperature)
        if top_k > 1:
            assert top_p == 0.0, 'cannot set both top-k and top-p samplings.'
            assert top_k <= logits.size(1), 'top-k is larger than logit size.'
            if vocab_size:
                assert top_k < vocab_size, 'top-k is larger than vocab size.'
            modify_logits_for_top_k_filtering(logits, top_k)
        elif top_p > 0.0:
            assert top_p <= 1.0, 'top-p should be in (0, 1].'
            modify_logits_for_top_p_filtering(logits, top_p)
        samples = torch.multinomial(logits.softmax(dim=-1), num_samples=1).view(-1)
    if vocab_size:
        samples = torch.clamp(samples, min=0, max=(vocab_size - 1))
    return samples


class InferenceParams:
    """Incremental-decoding state (:1449-1473).  The key/value memory of every layer lives in one
    ymp.engine.KVCache (packed QKV rows the attention kernels read in place); `key_value_memory_dict`
    exposes it per layer number for code that only checks for emptiness."""

    def __init__(self, max_batch_size, max_sequence_len):
        self.max_sequence_len = max_sequence_len
        self.max_batch_size = max_batch_size
        self.sequence_len_offset = 0
        self.batch_size_offset = 0
        self.key_value_memory_dict = {}
        self.cache = None
        self.token_step = None   # ymp.engine.TokenStep once this call's single-token steps have been validated

    def swap_key_value_dict(self, batch_idx):
        'swap between batches'
        if self.cache is None:
            raise ValueError('should not swap when dict in empty')
        assert len(batch_idx) == self.cache.B  # make sure batch size is the same
        self.cache.reorder(torch.as_tensor(batch_idx, device=self.cache.qkv[0].device, dtype=torch.long))
        self.key_value_memory_dict = {i + 1: t for i, t in enumerate(self.cache.qkv)}


class BeamHypotheses:
    """n-best list of finished hypotheses (:1908-1961).  score = sum_logprobs / len(hyp) ** length_penalty,
    where hyp is the (padded) token row handed in by beam_search."""

    def __init__(self, num_beams, length_penalty=1.0, early_stopping=False):
        self.length_penalty = length_penalty
        self.early_stopping = early_stopping
        self.num_beams = num_beams
        self.beams = []
        self.worst_score = 1e9

    def __len__(self):
        return len(self.beams)

    def add(self, hyp, sum_logprobs, beam_indices=None):
        score = sum_logprobs / (hyp.shape[-1] ** self.length_penalty)
        if len(self) < self.num_beams or score > self.worst_score:
            self.beams.append((score, hyp, beam_indices))
            if len(self) > self.num_beams:
                ranked = sorted((s, idx) for idx, (s, _, _) in enumerate(self.beams))
                del self.beams[ranked[0][1]]
                self.worst_score = ranked[1][0]
            else:
                self.worst_score = min(score, self.worst_score)

    def is_done(self, best_sum_logprobs, cur_len):
        if len(self) < self.num_beams:
            return False
        if self.early_stopping:
            return True
        return self.worst_score >= best_sum_logprobs / cur_len ** self.length_penalty


def run_sample(step, tokens, lengths, n_query, *, tokens_to_generate, eod_id, max_position_embeddings, top_k, top_p,
               temperature=1.0, vocab_size=None, termination_id=None, use_eod_token_for_early_termination=True,
               stop_on_double_eol=False, stop_on_eol=False):
    """DistributedGPT3.sample's loop (:1620-1741) over a decode callback.
    step(new_tokens [B, n], first) -> next-token logits [B, V] of the last position (fp32); the callback owns
    the KV cache and the visual prefix (n_query positions, fed on the first call)."""
    B = tokens.size(0)
    dev = tokens.device
    lengths = lengths.to(dev)
    tokens = torch.cat((tokens, torch.full((B, tokens_to_generate), eod_id, dtype=torch.long, device=dev)), dim=-1)
    max_len = min(tokens.size(1), max_position_embeddings)
    min_prompt = int(lengths.min().item())
    if min_prompt >= max_len:
        raise ValueError('context length + tokens_to_generate too large')
    if termination_id is None:
        termination_id = eod_id
    finished = torch.zeros(B, dtype=torch.bool, device=dev)
    prev = 0
    ctx = min_prompt
    for ctx in range(min_prompt, max_len):
        logits = step(tokens[:, prev:ctx], ctx == min_prompt)
        new = sample(logits, top_k=top_k, top_p=top_p, temperature=temperature, vocab_size=vocab_size)
        started = lengths <= ctx  # samples whose prompt has been consumed start writing their own tokens
        tokens[started, ctx] = new[started]
        prev = ctx
        if stop_on_double_eol:
            hit = ((new == 628) | ((new == 198) & (tokens[:, ctx - 1] == 198))) & started
        elif stop_on_eol:
            hit = ((new == 628) | (new == 198)) & started
        else:
            hit = (new == termination_id) & started
        finished |= hit
        if use_eod_token_for_early_termination and bool(finished.all()):
            break
    # the reference slices with the context length that still counts the prefix positions (:1740)
    return tokens[:, :ctx + n_query + 1]


def run_beam_search(step, reorder, tokens, prompt_length, n_query, *, beam_size, num_return_gen, stop_token,
                    tokens_to_generate, max_position_embeddings):
    """DistributedGPT3.beam_search's loop (:1743-1875), batch size 1, over a decode callback.
    step(new_tokens [beam, n], first) -> logits [beam, V]; reorder(idx) permutes the callback's KV cache."""
    assert tokens.size(0) == 1
    dev = tokens.device
    tokens = torch.cat((tokens, torch.full((1, tokens_to_generate), stop_token, dtype=torch.long, device=dev)), dim=-1)
    final_len = min(tokens.size(1), max_position_embeddings)
    if prompt_length >= final_len:
        raise ValueError('context length + tokens_to_generate too large')
    pool = BeamHypotheses(beam_size)
    scores = torch.zeros(beam_size, 1, dtype=torch.float32, device=dev)
    tokens = tokens.repeat(beam_size, 1)
    done = False
    prev = 0
    ctx = prompt_length
    for ctx in range(prompt_length, final_len):
        logits = step(tokens[:, prev:ctx], ctx == prompt_length)
        vocab = logits.size(-1)
        cand = torch.log_softmax(logits.float(), dim=-1) + scores
        flat = cand[0] if ctx == prompt_length else cand.view(-1)  # identical beams at the first step
        ranked_scores, ranked = torch.sort(flat, descending=True)
        ranked, ranked_scores = ranked[:2 * beam_size], ranked_scores[:2 * beam_size]
        beam_of, word_of = torch.div(ranked, vocab, rounding_mode='floor').tolist(), (ranked % vocab).tolist()
        survivors = []
        for rank, (word, beam) in enumerate(zip(word_of, beam_of)):
            if word == stop_token:
                if rank >= beam_size:  # a finished hypothesis outside the top beam_size candidates is dropped
                    continue
                pool.add(tokens[beam].clone(), ranked_scores[rank], ctx + 1 - prompt_length)
            else:
                survivors.append((word, ranked_scores[rank], beam))
            if len(survivors) == beam_size:
                break
        if pool.is_done(ranked_scores.max().item(), ctx + 1 - prompt_length):
            done = True
            break
        keep = torch.tensor([b for _, _, b in survivors], dtype=torch.long, device=dev)
        tokens = tokens[keep, :]
        tokens[:, ctx] = torch.tensor([w for w, _, _ in survivors], dtype=torch.long, device=dev)
        scores = torch.stack([sc for _, sc, _ in survivors]).reshape(-1, 1).float()
        reorder(keep)
        prev = ctx
    if not done:
        for b in range(beam_size):
            pool.add(tokens[b].clone(), scores[b], ctx + 1 - prompt_length)
    best = sorted(pool.beams, key=lambda x: float(x[0]), reverse=True)[:min(num_return_gen, len(pool.beams))]
    return AttrDict(sequences=torch.stack([h for _, h, _ in best], dim=0),
                    scores=torch.stack([torch.as_tensor(sc, device=dev).reshape(-1)[0] for sc, _, _ in best], dim=0))


def beam_chunks(prompt_lengths, per_chunk):
    """(prompt_length, sample indices) of every decode batch of run_beam_search_batch: the samples grouped by prompt
    length (groups in order of first appearance), each group cut into chunks of at most per_chunk samples."""
    groups = {}
    for i, p in enumerate(prompt_lengths):
        groups.setdefault(int(p), []).append(i)
    for p, idx in groups.items():
        for c in range(0, len(idx), per_chunk):
            yield p, idx[c:c + per_chunk]


def run_beam_search_batch(step, reorder, tokens, prompt_lengths, n_query, *, beam_size, num_return_gen, stop_token,
                          tokens_to_generate, max_position_embeddings, max_rows=64):
    """run_beam_search for every sample of tokens [B, L] at once: element i of the returned list equals
    run_beam_search on sample i alone (same ranking, same stop-token rule, same BeamHypotheses calls).

    The samples are decoded in chunks of n = max_rows // beam_size samples of equal prompt length (beam_chunks); a short
    chunk is padded to n with copies of its first sample, whose results are dropped, so every chunk has the same shape.
    Chunk row j * beam_size + b is beam b of sample samples[j].
      step(samples, new_tokens [n * beam, k], first) -> next-token logits [n * beam, V] (first: new_tokens is the whole
          prompt and the callback also feeds the visual prefix of samples[j] to its rows)
      reorder(idx) -> row r continues the history of row idx[r] (int64 [n * beam], rows of the chunk)
    One log_softmax over all rows, one top-k over [n, beam * V] and one device-to-host copy per step serve every sample.
    A sample that has finished keeps its rows: they are fed its stop token, never reordered, and their logits ignored."""
    dev = tokens.device
    beam = beam_size
    per = max_rows // beam
    if per < 1:
        raise ValueError(f"beam_size {beam} > max_rows {max_rows}")
    plens = [int(p) for p in torch.as_tensor(prompt_lengths).reshape(-1).tolist()]
    assert len(plens) == tokens.size(0)
    final_len = min(tokens.size(1) + tokens_to_generate, max_position_embeddings)
    results = [None] * tokens.size(0)
    for plen, idx in beam_chunks(plens, per):
        if plen >= final_len:
            raise ValueError('context length + tokens_to_generate too large')
        samples = idx + [idx[0]] * (per - len(idx))
        n, R = per, per * beam
        toks = torch.cat((tokens[samples].cpu(), torch.full((n, tokens_to_generate), stop_token, dtype=torch.long)), dim=-1)
        toks = toks.repeat_interleave(beam, dim=0)                     # [R, L + tokens_to_generate], host
        pools = [BeamHypotheses(beam) for _ in range(n)]
        done = [False] * n
        scores = torch.zeros(R, 1, dtype=torch.float32, device=dev)
        host_scores = torch.zeros(R, dtype=torch.float32)
        prev = 0
        ctx = plen
        for ctx in range(plen, final_len):
            first = ctx == plen
            logits = step(samples, toks[:, prev:ctx].to(dev), first)
            vocab = logits.size(-1)
            cand = torch.log_softmax(logits.float(), dim=-1) + scores
            flat = cand.view(n, beam, vocab)[:, 0] if first else cand.view(n, beam * vocab)   # identical beams at first
            top_dev, top_i = torch.topk(flat, 2 * beam, dim=-1)
            host = torch.cat([top_dev.view(torch.int32), top_i.to(torch.int32)], dim=1).cpu()
            top_s, top_i = host[:, :2 * beam].view(torch.float32), host[:, 2 * beam:].long()
            keep = list(range(R))
            for j in range(n):
                if done[j]:
                    continue
                ranked_scores = top_s[j]
                beam_of, word_of = torch.div(top_i[j], vocab, rounding_mode='floor').tolist(), (top_i[j] % vocab).tolist()
                survivors = []
                for rank, (word, b) in enumerate(zip(word_of, beam_of)):
                    if word == stop_token:
                        if rank >= beam:
                            continue
                        # the score is divided where run_beam_search divides it (on the logits' device), for the same bits
                        pools[j].add(toks[j * beam + b].clone(), top_dev[j, rank], ctx + 1 - plen)
                    else:
                        survivors.append((word, ranked_scores[rank], b))
                    if len(survivors) == beam:
                        break
                if pools[j].is_done(ranked_scores.max().item(), ctx + 1 - plen):
                    done[j] = True
                    continue
                rows = [j * beam + b for _, _, b in survivors]
                keep[j * beam:(j + 1) * beam] = rows
                block = toks[rows, :]
                block[:, ctx] = torch.tensor([w for w, _, _ in survivors], dtype=torch.long)
                toks[j * beam:(j + 1) * beam] = block
                host_scores[j * beam:(j + 1) * beam] = torch.stack([sc for _, sc, _ in survivors])
            if all(done):
                break
            scores = host_scores.view(R, 1).to(dev)
            reorder(torch.tensor(keep, dtype=torch.long, device=dev))
            prev = ctx
        for j, i in enumerate(idx):
            pool = pools[j]
            if not done[j]:
                for b in range(beam):
                    pool.add(toks[j * beam + b].clone(), scores[j * beam + b], ctx + 1 - plen)
            best = sorted(pool.beams, key=lambda x: float(x[0]), reverse=True)[:min(num_return_gen, len(pool.beams))]
            results[i] = AttrDict(sequences=torch.stack([h for _, h, _ in best], dim=0).to(dev),
                                  scores=torch.stack([torch.as_tensor(sc, device=dev).reshape(-1)[0] for sc, _, _ in best], dim=0))
    return results


class _BeamBatchDecoder:
    """Decode callbacks of DistributedGPT3.beam_search_batch over one ymp.engine.BeamBatchCache of n x beam rows.
    The first step prefills every sample into its own block of rows with exactly the calls DistributedGPT3._decode
    makes for a single beam search (so the cached prefix and the first logits are the same bits); every later step is
    one replay of the captured TokenStep over all rows, the decode attention reading its keys through the cache's row
    table, and a reorder rewrites table entries only."""

    def __init__(self, model, query_embeds, beam, n, max_len, device):
        from ymp import engine
        self.model, self.qe, self.beam, self.n = model, query_embeds, beam, n
        keys, params = model._param_list()
        self.params = params
        self.W = {k: YF.as_bf16(p) for k, p in zip(keys, params)}
        # one cache (and its captured step) per shape, kept apart from the per-sample pool so that alternating with
        # generate() recaptures nothing
        key = (n * beam, beam, max_len, str(device))
        pool = model.__dict__.setdefault("_beam_batch_pool", {})
        if key not in pool:
            pool.clear()
            pool[key] = engine.BeamBatchCache(model.config.engine_cfg(), n, beam, max_len, device)
        self.cache = pool[key]

    def _token_step(self, emb_dtype):
        from ymp import engine
        params = self.params
        sig = (params[0].data_ptr(), params[-1].data_ptr(), sum(p._version for p in params))
        ts = self.cache.token
        if ts is None or ts.sig != sig:
            static = all(p.dtype == torch.bfloat16 or not p.requires_grad for p in params)
            ts = self.cache.token = engine.TokenStep(self.cache, self.W, emb_dtype, sig, static)
        elif not ts.static:
            ts.W = self.W
        return ts

    def step(self, samples, new_tokens, first):
        from ymp import engine, ops
        c, beam, W = self.cache, self.beam, self.W
        emb = self.model.dist_model.language_model.embedding.word_embeddings(new_tokens)   # [R, k, H]
        R, n, H = emb.shape
        if not first:
            _, logits = self._token_step(emb.dtype).run(emb.reshape(R, H))
            return logits
        c.reset()
        pos = W[engine.GPT + "embedding.position_embeddings.weight"]
        out = []
        for j, s in enumerate(samples):
            ie = emb[j * beam:(j + 1) * beam]
            if self.qe is not None:
                ie = torch.cat([self.qe[s:s + 1].repeat(beam, 1, 1).to(ie.dtype), ie], dim=1)
            k = ie.size(1)
            x = (ie.float() + pos[0:k][None].float()).reshape(beam * k, H).contiguous()
            hid = engine.gpt_decode(W, x, c.block(j), k)
            out.append(ops.gemm(hid, W[engine.GPT + "embedding.word_embeddings.weight"]).float())
        c._set_len(k)
        c.start_table(k)
        return torch.cat(out)

    def reorder(self, idx):
        self.cache.reorder_table(idx)


class GPT3Model(nn.Module):
    """Parameter container with the reference's names: language_model.{embedding,encoder}...."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        H, F4, V, Lyr = config.hidden_size, config.ffn_hidden_size, config.vocab_size, config.num_hidden_layers
        std = config.init_method_std
        std_out = std / math.sqrt(2.0 * Lyr)

        def n(*shape, s=std):
            return torch.empty(*shape).normal_(0.0, s)

        lm = Holder()
        self.add_module("language_model", lm)
        lm.add_module("embedding", Holder())
        lm.embedding.add_module("word_embeddings", EmbedHolder())
        add_param(lm, "embedding.word_embeddings.weight", n(V, H))
        add_param(lm, "embedding.position_embeddings.weight", n(config.max_position_embeddings, H))
        for i in range(Lyr):
            b = f"encoder.layers.{i}."
            for nm in ("input_layernorm", "post_attention_layernorm"):
                add_param(lm, b + nm + ".weight", torch.ones(H))
                add_param(lm, b + nm + ".bias", torch.zeros(H))
            add_param(lm, b + "self_attention.query_key_value.weight", n(3 * H, H))
            add_param(lm, b + "self_attention.query_key_value.bias", torch.zeros(3 * H))
            add_param(lm, b + "self_attention.dense.weight", n(H, H, s=std_out))
            add_param(lm, b + "self_attention.dense.bias", torch.zeros(H))
            add_param(lm, b + "mlp.dense_h_to_4h.weight", n(F4, H))
            add_param(lm, b + "mlp.dense_h_to_4h.bias", torch.zeros(F4))
            add_param(lm, b + "mlp.dense_4h_to_h.weight", n(H, F4, s=std_out))
            add_param(lm, b + "mlp.dense_4h_to_h.bias", torch.zeros(H))
        add_param(lm, "encoder.final_layernorm.weight", torch.ones(H))
        add_param(lm, "encoder.final_layernorm.bias", torch.zeros(H))

    def word_embeddings_weight(self):
        return self.language_model.embedding.word_embeddings.weight


class DistributedGPT3(nn.Module):
    def __init__(self, model_dir, rank=0, path_load_tag='model', *args, **kwargs):
        super().__init__()
        _check_tp1(kwargs.pop('megatron_cfg', None))
        self.config = GPT3Config.from_pretrained(model_dir)
        self.dist_model = GPT3Model(self.config)
        kwargs.pop('checkpoint_model_parallel_size', None)
        if kwargs.pop('load_state_dict', True):
            path = _ckpt_name(0, model_dir, path_load_tag)
            if osp.exists(path):
                self.dist_model.load_state_dict(pre_load(0, model_dir, tag=path_load_tag))
            elif os.environ.get("YMP_ALLOW_RANDOM_INIT", "0") != "1":
                raise FileNotFoundError(f"{path} not found (set YMP_ALLOW_RANDOM_INIT=1 to run with "
                                        "random-initialised decoder weights, e.g. for benchmarks)")
        self.inference_params = None
        self._keys_prefix = "text_decoder.dist_model."

    def train(self, mode=True):
        if mode:
            self.inference_params = None
        return super().train(mode)

    def _param_list(self):
        return named_param_list(self.dist_model, self._keys_prefix)

    def forward(self, tokens=None, input_embeds=None, query_embeds=None, attention_mask=None,
                position_ids=None, labels=None, prompt_length=None, loss_mask=None, is_pair=(False,)):
        """Same contract as the reference (:1578-1618): returns Dict(logits, loss, losses,
        last_hidden_state).  A plain causal mask over the whole sequence and position ids
        arange(S) are always used (the reference never forwards `attention_mask` into the layers
        on this path, :1329-1332), so explicit attention_mask/position_ids are accepted only in
        that default form."""
        if tokens is not None and input_embeds is not None:
            raise ValueError("You cannot specify both decoder_input_ids and decoder_inputs_embeds at the same time")
        if tokens is None and input_embeds is None:
            raise ValueError("You have to specify either decoder_input_ids or decoder_inputs_embeds")
        if position_ids is not None:
            raise NotImplementedError("custom position_ids are not supported on the B200 path")
        if tokens is not None:
            input_embeds = self.dist_model.language_model.embedding.word_embeddings(tokens)
        if query_embeds is not None:
            input_embeds = torch.cat([query_embeds.to(input_embeds.dtype), input_embeds], dim=1)
        if labels is None:
            return self._decode(tokens, input_embeds, 0 if query_embeds is None else query_embeds.size(1))
        keys, params = self._param_list()
        logits, losses, hidden = YF.GptFn.apply(input_embeds, labels.contiguous(), self.config.engine_cfg(self.training), True,
                                                keys, *params)
        if loss_mask is None:
            loss_mask = attention_mask[:, 1:].contiguous()
        losses = losses[:, :-1].contiguous().float()
        lm = loss_mask.reshape(-1).float()
        loss = torch.sum(losses.reshape(-1) * lm) / lm.sum()
        return AttrDict(logits=logits, loss=loss, losses=losses, last_hidden_state=hidden)

    # ------------------------------------------------------------------------------------------ generation
    def _decode(self, tokens, input_embeds, n_query):
        """Inference branch of forward (:1576-1603): one incremental step over the KV cache.  input_embeds
        [B, n, H] already holds [prefix | word embeddings]; logits are returned for the LAST position only
        ([B, 1, V] fp32 - the only row sample()/beam_search() read)."""
        from ymp import engine, ops
        if self.inference_params is None:
            raise ValueError("no labels and no inference_params: call sample()/beam_search()/generate()")
        ip = self.inference_params
        B, n, H = input_embeds.shape
        ts = ip.token_step
        if ts is not None and n == 1:
            # steady state of sample() / beam_search(): nothing but the graph replay on the host path (walking the module
            # tree for the parameter list alone costs more than the whole device step; weights cannot change inside
            # one generate call - the step object was validated when this call acquired its cache)
            hid, logits = ts.run(input_embeds.reshape(B, H))
            ip.sequence_len_offset += 1
            return AttrDict(logits=logits.view(B, 1, -1), loss=None, losses=None, last_hidden_state=hid.view(B, 1, H))
        keys, params = self._param_list()
        if ip.cache is None:
            # one cache (and one captured token step) per (batch, length) is kept on the model and reused by later
            # sample() / beam_search() calls: caption evaluation decodes thousands of clips with the same shape
            key = (ip.max_batch_size, ip.max_sequence_len, str(input_embeds.device))
            pool = self.__dict__.setdefault("_decode_pool", {})
            if key not in pool:
                pool.clear()   # keep one shape resident (a 1.3B cache at beam 5 x 400 positions is 0.6 GB)
                pool[key] = engine.KVCache(self.config.engine_cfg(), ip.max_batch_size, ip.max_sequence_len, input_embeds.device)
            ip.cache = pool[key]
            ip.cache.reset()
            ip.key_value_memory_dict = {i + 1: t for i, t in enumerate(ip.cache.qkv)}
        off = ip.sequence_len_offset
        assert off == ip.cache.len and B == ip.cache.B
        if n == 1 and off > 0 and B <= ops.SKINNY_MAX_ROWS:
            # single-token step: skinny GEMMs + device-side cache length, replayed as one CUDA graph
            sig = (params[0].data_ptr(), params[-1].data_ptr(), sum(p._version for p in params))
            ts = ip.cache.token
            if ts is None or ts.sig != sig:
                # weights the graph may hold raw pointers to: bf16 parameters (used in place) and frozen fp32 ones
                # (their bf16 copy is cached until the version changes); trainable fp32 ones are re-cast every step
                static = all(p.dtype == torch.bfloat16 or not p.requires_grad for p in params)
                ts = ip.cache.token = engine.TokenStep(ip.cache, {k: YF.as_bf16(p) for k, p in zip(keys, params)},
                                                       input_embeds.dtype, sig, static)
            elif not ts.static:
                ts.W = {k: YF.as_bf16(p) for k, p in zip(keys, params)}
            if ts.static:
                ip.token_step = ts
            hid, logits = ts.run(input_embeds.reshape(B, H))
        else:
            W = {k: YF.as_bf16(p) for k, p in zip(keys, params)}
            pos = W[engine.GPT + "embedding.position_embeddings.weight"]
            x = (input_embeds.float() + pos[off:off + n][None].float()).reshape(B * n, H).contiguous()
            hid = engine.gpt_decode(W, x, ip.cache, n)
            logits = ops.gemm(hid, W[engine.GPT + "embedding.word_embeddings.weight"]).float()
        ip.sequence_len_offset += n  # tokens.size(1) + query_embeds.size(1) of the reference
        return AttrDict(logits=logits.view(B, 1, -1), loss=None, losses=None, last_hidden_state=hid.view(B, 1, H))

    def _decode_callbacks(self, query_embeds):
        def step(new_tokens, first):
            out = self(tokens=new_tokens, query_embeds=query_embeds if first else None)
            return out.logits[:, -1, :]

        def reorder(idx):
            self.inference_params.swap_key_value_dict(idx)
        return step, reorder

    @torch.no_grad()
    def sample(self, tokens, query_embeds=None, temperature=1.0, use_eod_token_for_early_termination=True,
               stop_on_double_eol=False, stop_on_eol=False, termination_id=None, **kwargs):
        """Batched greedy / top-k / top-p decoding (:1620-1741)."""
        cfg = self.config
        lengths = kwargs.pop('prompt_length', torch.tensor([tokens.size(1)], device=tokens.device))
        lengths = torch.as_tensor(lengths, device=tokens.device).reshape(-1)
        nq = 0 if query_embeds is None else query_embeds.size(1)
        max_len = min(tokens.size(1) + cfg.tokens_to_generate, cfg.max_position_embeddings)
        self.inference_params = InferenceParams(tokens.size(0), max_len + nq)
        step, _ = self._decode_callbacks(query_embeds)
        return run_sample(step, tokens, lengths, nq, tokens_to_generate=cfg.tokens_to_generate, eod_id=cfg.eod_id,
                          max_position_embeddings=cfg.max_position_embeddings, top_k=cfg.top_k, top_p=cfg.top_p,
                          temperature=temperature, vocab_size=cfg.vocab_size, termination_id=termination_id,
                          use_eod_token_for_early_termination=use_eod_token_for_early_termination,
                          stop_on_double_eol=stop_on_double_eol, stop_on_eol=stop_on_eol)

    @torch.no_grad()
    def beam_search(self, tokens, query_embeds=None, beam_size=5, num_return_gen=1, stop_token=None, **kwargs):
        """Beam search for one sample (:1743-1875): Dict(sequences [n, len], scores [n])."""
        cfg = self.config
        assert tokens.size(0) == 1
        prompt_length = int(kwargs.pop('prompt_length', tokens.size(1)))
        if stop_token is None:
            stop_token = cfg.eod_id
        nq = 0 if query_embeds is None else query_embeds.size(1)
        final_len = min(tokens.size(1) + cfg.tokens_to_generate, cfg.max_position_embeddings)
        self.inference_params = InferenceParams(beam_size, final_len + nq)
        qe = None if query_embeds is None else query_embeds.repeat(beam_size, 1, 1)
        step, reorder = self._decode_callbacks(qe)
        return run_beam_search(step, reorder, tokens, prompt_length, nq, beam_size=beam_size, num_return_gen=num_return_gen,
                               stop_token=stop_token, tokens_to_generate=cfg.tokens_to_generate,
                               max_position_embeddings=cfg.max_position_embeddings)

    @torch.no_grad()
    def beam_search_batch(self, tokens, query_embeds=None, prompt_length=None, beam_size=5, num_return_gen=1, stop_token=None):
        """beam_search for every sample of tokens [B, L] (visual prefixes query_embeds [B, Q, H], prompt lengths
        prompt_length [B]): a list of B Dict(sequences [n, len], scores [n]), element i equal to beam_search on sample i.
        Samples of equal prompt length share one decoding step: chunks of 64 // beam_size samples, each step one replay
        of the captured token step over all their beams (one weight stream instead of one per sample).  With
        beam_size <= 8 the logits are the bits of the per-sample path."""
        from ymp import ops
        cfg = self.config
        B = tokens.size(0)
        if prompt_length is None:
            prompt_length = torch.full((B,), tokens.size(1), dtype=torch.long)
        prompt_length = torch.as_tensor(prompt_length).reshape(-1)
        if stop_token is None:
            stop_token = cfg.eod_id
        nq = 0 if query_embeds is None else query_embeds.size(1)
        final_len = min(tokens.size(1) + cfg.tokens_to_generate, cfg.max_position_embeddings)
        per = ops.SKINNY_WIDE_MAX_ROWS // beam_size
        dec = _BeamBatchDecoder(self, query_embeds, beam_size, per, final_len + nq, tokens.device)
        return run_beam_search_batch(dec.step, dec.reorder, tokens, prompt_length, nq, beam_size=beam_size,
                                     num_return_gen=num_return_gen, stop_token=stop_token, tokens_to_generate=cfg.tokens_to_generate,
                                     max_position_embeddings=cfg.max_position_embeddings, max_rows=per * beam_size)

    @torch.no_grad()
    def generate(self, tokens, do_sample=True, termination_id=None, *args, **kwargs):
        """(:1878-1883)"""
        if do_sample:
            return self.sample(tokens, termination_id=termination_id, *args, **kwargs)
        return self.beam_search(tokens, stop_token=termination_id, *args, **kwargs)
