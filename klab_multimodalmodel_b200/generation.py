"""Greedy caption decoding: `transformer.generate(inputs_embeds=...)` of /root/reference/models/model.py:28 with the defaults
the reference relies on (HF/generation/utils.py:765-804,2658-2800): greedy, 20 new tokens, start id 0, EOS 1, pad 0, finished
rows keep emitting pad, stop as soon as every row has finished.

`greedy_generate` is the cached single-token path (SURVEY.md K14; HF/models/t5/modeling_t5.py:281-305, HF/cache_utils.py): per
decoder block the self-attention keys / values of the tokens emitted so far live in a preallocated [B, T_max, 3*inner] buffer
-- the q|k|v GEMM of step t writes row (b, t) of it directly through its output row stride, so "growing the cache" costs no
copy at all (HF re-allocates it with torch.cat every step) -- and the cross-attention keys / values of the encoder output are
projected once before the loop.  Every step is one token per sample: O(T) work instead of the O(T^2) of re-running the prefix.
The step for position t is a CUDA-graph region (graphs.py) over static buffers, so the launch-bound chain of small kernels
costs one graph launch per token.
`greedy_generate_recompute` is that older prefix-recompute schedule, kept as a cross-check (identical ids; tests).
`beam_generate` is beam search (`generate(num_beams=k)`) on the same cached single-token step, see below.
`sample_generate` is multinomial sampling (`generate(do_sample=True)`): greedy's state, loop and step with klab_sample_step in
place of the argmax, see below.
"""
from __future__ import annotations

import torch

from . import _lib as L
from . import ops as O


class _DecodeState:
    """Static device buffers of one decode geometry (batch, encoder length, T): token ids, finished flags, per decoder block the
    self-attention q|k|v cache and the cross-attention k|v projection.  They never move, so the kernel sequence of the
    single-token step for position t can be captured into a CUDA graph once and replayed for every later caption batch."""

    def __init__(self, tr, B, Le, T, cd, dev, rows=None):
        cfg = tr.config
        inner = cfg.num_heads * cfg.d_kv
        n = len(tr.decoder.block)
        R = B if rows is None else rows                            # decoded rows: B, or B * num_return_sequences when sampling
        self.ids = torch.empty(R, T + 1, dtype=torch.int64, device=dev)
        self.tok = torch.empty(R, 1, dtype=torch.int64, device=dev)
        self.unfinished = torch.empty(R, dtype=torch.int32, device=dev)
        self.seed = torch.zeros(1, dtype=torch.int64, device=dev)  # sampling: the call's seed, read by the kernel at run time
        self.enc = torch.empty(B * Le, cfg.d_model, dtype=cd, device=dev)
        self.cross_kv = [torch.empty(B * Le, 2 * inner, dtype=cd, device=dev) for _ in range(n)]   # once per sample
        self.self_qkv = [torch.zeros(R * T, 3 * inner, dtype=cd, device=dev) for _ in range(n)]   # row (r, t): q | k | v of token t
        self.lut, self.rz = tr.decoder.lut(T, dev)                 # covers relative positions -(T-1) .. T-1


def _decode_operands(tr, cd, mode="get"):
    """-> (per decoder block (ln0, wqkv, w_o, ln1, w_cq, w_ckv, w_co, ln2, w_i, w_ff), embedding table, LM head) in the compute
    dtype.  "get" refreshes stale bf16 copies eagerly (outside any graph); "peek" returns the buffers as they are.  The LM head
    is the embedding operand itself when tied; w_i is [wi_0; wi_1] for the gated FFN."""
    g = getattr(tr.cache, mode)
    out = []
    for blk in tr.decoder.block:
        ln0, q, k, v, o, ln1, cq, ck, cv, co, ln2, *wi, wo = blk.flat_params()
        out.append((ln0.detach(), g([q, k, v], cd), g([o], cd), ln1.detach(), g([cq], cd), g([ck, cv], cd), g([co], cd), ln2.detach(),
                    g(wi, cd), g([wo], cd)))
    return out, g([tr.shared.weight], cd), g([tr.lm_head.weight], cd)


def _decode_operands_peek(tr, cd):
    return _decode_operands(tr, cd, "peek")


def _ffn(cfg, n2, w_i, w_ff, h2):
    """Decoder FFN of one token per row, eval mode: ReLU (T5DenseActDense) or gated-GELU (T5DenseGatedActDense)."""
    if cfg.gated:
        f = O.geglu_fwd(O.linear_fwd(n2, w_i))
    else:
        f = O.linear_fwd(n2, w_i, act=L.ACT_RELU)
    return O.linear_fwd(f, w_ff, residual=h2)


def _decode_step_body(tr, st, t, B, Le, T, sample=None):
    """One token for every row: position t in, ids[:, t + 1] out.  consts only (no per-call inputs): everything it reads or
    writes lives in `st` or in the operand cache, so the region is capturable as is.  sample None: greedy (B rows, argmax);
    sample = (n, temperature, top_k, top_p): B * n rows drawn by klab_sample_step, the n rows of a sample sharing its
    cross-attention K/V."""
    cfg = tr.config
    n_rs = 1 if sample is None else sample[0]
    R = B * n_rs
    cd = st.enc.dtype
    H, dk, eps = cfg.num_heads, cfg.d_kv, cfg.layer_norm_epsilon
    inner = H * dk
    layers, tab, head = _decode_operands_peek(tr, cd)
    table = tr.decoder.block[0].layer[0].SelfAttention.relative_attention_bias.weight.detach()
    st.tok.copy_(st.ids[:, t:t + 1])
    x = O.embedding_fwd(st.tok, tab)                               # [R, d]
    for l, (ln0, wqkv, w_o, ln1, w_cq, _w_ckv, w_co, ln2, w_i, w_ff) in enumerate(layers):
        self_qkv, cross_kv = st.self_qkv[l], st.cross_kv[l]
        n0, _ = O.rmsnorm_fwd(x, ln0, eps, save_stats=False)
        row_t = self_qkv.view(R, T, 3 * inner)[:, t]               # [R, 3*inner] view, row stride T*3*inner
        O.linear_fwd(n0, wqkv, out=row_t)                          # q | k | v of the new token, written into the cache
        ctx, _ = O.t5_attention_fwd(row_t[:, :inner], self_qkv[:, inner:2 * inner], self_qkv[:, 2 * inner:], R, H, 1, T, dk,
                                    bias_table=table, lut=st.lut, rel_zero=st.rz, num_buckets=cfg.relative_attention_num_buckets,
                                    causal=True, q_offset=t)
        h1 = O.linear_fwd(ctx, w_o, residual=x)
        n1, _ = O.rmsnorm_fwd(h1, ln1, eps, save_stats=False)
        qc = O.linear_fwd(n1, w_cq)
        if n_rs == 1:
            ctx2, _ = O.t5_attention_fwd(qc, cross_kv[:, :inner], cross_kv[:, inner:], B, H, 1, Le, dk)
        else:                                                      # the n rows of a sample read its K/V (no per-row copy)
            ctx2 = O.t5_attention_decode_beam(qc, cross_kv[:, :inner], cross_kv[:, inner:], R, H, Le, dk, kv_group=n_rs)
        h2 = O.linear_fwd(ctx2, w_co, residual=h1)
        n2, _ = O.rmsnorm_fwd(h2, ln2, eps, save_stats=False)
        x = _ffn(cfg, n2, w_i, w_ff, h2)
    n, _ = O.rmsnorm_fwd(x, tr.decoder.final_layer_norm.weight, eps, save_stats=False)
    logits = O.linear_fwd(n, head, alpha=cfg.lm_head_scale, out_dtype=torch.float32)
    if sample is None:
        L.check(L.lib().klab_greedy_step(torch.cuda.current_stream().cuda_stream, B, tr.shared.weight.shape[0], logits.data_ptr(),
                                         logits.stride(0), st.ids.data_ptr(), st.ids.stride(0), t + 1, st.unfinished.data_ptr(),
                                         cfg.pad_token_id, cfg.eos_token_id))
    else:
        _, temperature, top_k, top_p = sample
        O.sample_step(logits, st.ids, t + 1, st.unfinished, st.seed, pad_id=cfg.pad_token_id, eos_id=cfg.eos_token_id,
                      temperature=temperature, top_k=top_k, top_p=top_p)
    return (st.ids,)


CHECK_EVERY = 5           # decode steps between two read-backs of the "every row has finished" flag


def _decode_state(tr, attr, tag, key, make):
    """The static state of one decode geometry, kept on the model in tr.__dict__[attr]; regions are keyed (tag, id(tr), id(st), ...)."""
    from .graphs import POOL
    states = tr.__dict__.setdefault(attr, {})
    st = states.get(key)
    if st is None:
        if len(states) >= 4:                                             # a handful of geometries at most: the caches are large
            dead = {id(o) for o in states.values()}                      # the per-position regions bake the old buffers in: drop
            POOL.drop_keys(lambda k: k[0] == tag and k[2] in dead)       # them too, or the states would never be freed
            states.clear()
        st = states[key] = make()
    return st


def _decode_run(tr, st, embeds, B, Le, T, key, sample=None):
    """Encoder, cross K|V and the cached single-token loop over the rows of `st`; -> ids [rows, n] cropped where HF stops."""
    from .graphs import POOL
    cfg = tr.config
    cd = embeds.dtype
    enc = tr.encoder.run_blocks(embeds, B, Le, tr.cache)
    O.rmsnorm_fwd(enc, tr.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon, out=st.enc, save_stats=False)
    layers, _, _ = _decode_operands(tr, cd)                                 # also validates / refreshes every operand copy
    for l, ops_l in enumerate(layers):
        O.linear_fwd(st.enc, ops_l[5], out=st.cross_kv[l])               # cross k|v, once per caption batch (modeling_t5.py:291-299)
    st.ids.fill_(cfg.pad_token_id)
    st.ids[:, 0] = cfg.decoder_start_token_id
    st.unfinished.fill_(1)
    # HF checks the stopping criteria after every token (a host round trip per step).  Finished rows only ever emit pad, so running
    # on and trimming afterwards gives the same ids: the "all rows finished" flag is read back every CHECK_EVERY steps only (the
    # queue of captured steps stays ahead of the GPU in between) and the returned length is where the last row finished.
    n_run = 0
    for t in range(T):
        # the single-token step is ~11 small kernels per block: launch bound when issued one by one, so it is a captured region
        # per position t (keys beyond t are masked by the causal bound, stale cache rows of an earlier batch never contribute)
        POOL.run(key + (t,), _decode_step_body, (), (tr, st, t, B, Le, T) + ((sample,) if sample is not None else ()))
        n_run = t + 1
        if n_run % CHECK_EVERY == 0 and n_run < T and not bool(st.unfinished.cpu().any()):
            break
    ids = st.ids[:, :n_run + 1]
    # length HF would have returned: it stops right after the step in which the last unfinished row emitted EOS
    is_eos = ids[:, 1:] == cfg.eos_token_id
    first_eos = torch.where(is_eos.any(1), is_eos.int().argmax(1) + 1, torch.full((ids.shape[0],), n_run, device=ids.device))
    n_out = 1 + int(first_eos.max().item())
    return ids[:, :n_out].clone()


@torch.no_grad()
def greedy_generate(tr, embeds, B, Le, max_new_tokens: int = 20):
    cd = embeds.dtype
    dev = embeds.device
    T = max_new_tokens                                                   # decoder positions 0 .. T-1 are ever attended to
    st = _decode_state(tr, "_klab_decode_states", "dec", (B, Le, T, cd, dev), lambda: _DecodeState(tr, B, Le, T, cd, dev))
    return _decode_run(tr, st, embeds, B, Le, T, ("dec", id(tr), id(st)))


@torch.no_grad()
def greedy_generate_recompute(tr, embeds, B, Le, max_new_tokens: int = 20):
    cfg = tr.config
    cd = embeds.dtype
    dev = embeds.device
    enc = tr.encoder.run_blocks(embeds, B, Le, tr.cache)
    enc, _ = O.rmsnorm_fwd(enc, tr.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon, save_stats=False)
    tab, head = tr.cache.get([tr.shared.weight], cd), tr.cache.get([tr.lm_head.weight], cd)
    V, d = tr.shared.weight.shape
    ids = torch.full((B, max_new_tokens + 1), cfg.pad_token_id, dtype=torch.int64, device=dev)
    ids[:, 0] = cfg.decoder_start_token_id
    unfinished = torch.ones(B, dtype=torch.int32, device=dev)
    n_out = 1
    for t in range(max_new_tokens):
        Lt = t + 1
        prefix = ids[:, :Lt].contiguous()
        x = O.embedding_fwd(prefix, tab)
        x = tr.decoder.run_blocks(x, B, Lt, tr.cache, enc_out=enc, Le=Le)
        last = x.view(B, Lt, d)[:, -1, :]                               # strided rows: the norm kernel takes a row stride
        n, _ = O.rmsnorm_fwd(last, tr.decoder.final_layer_norm.weight, cfg.layer_norm_epsilon, save_stats=False)
        logits = O.linear_fwd(n, head, alpha=cfg.lm_head_scale, out_dtype=torch.float32)
        L.check(L.lib().klab_greedy_step(torch.cuda.current_stream().cuda_stream, B, V, logits.data_ptr(), logits.stride(0),
                                         ids.data_ptr(), ids.stride(0), Lt, unfinished.data_ptr(), cfg.pad_token_id, cfg.eos_token_id))
        n_out = Lt + 1
        if not bool(unfinished.cpu().any()):                           # HF checks the stopping criteria every step too
            break
    return ids[:, :n_out]


# ------------------------------------------------------------------------------------------------------------------------------
# Beam search: GenerationMixin._beam_search of HF 5.5.0 (HF/generation/utils.py:3076-3386) on device state.  Rows are
# hypotheses, b * nb + i.  Unlike HF, the encoder output is NOT repeated per beam (the cross-attention kernel lets the nb rows
# of a sample share its K/V) and the self-attention cache is never reordered: row r writes its token-t keys / values into its
# own cache row (r, t), and the ancestry table src[r, j] (klab_beam_update) says which row holds position j of hypothesis r.
# ------------------------------------------------------------------------------------------------------------------------------
_EARLY_STOPPING = {False: 0, True: 1, "never": 2}


class _BeamState:
    """Static device buffers of one beam-search geometry (B, nb, Le, T): everything the per-position graph regions read or write."""

    def __init__(self, tr, B, nb, Le, T, cd, dev):
        cfg = tr.config
        inner = cfg.num_heads * cfg.d_kv
        n = len(tr.decoder.block)
        R = B * nb
        self.enc = torch.empty(B * Le, cfg.d_model, dtype=cd, device=dev)
        self.cross_kv = [torch.empty(B * Le, 2 * inner, dtype=cd, device=dev) for _ in range(n)]      # once per sample
        self.self_qkv = [torch.zeros(R * T, 3 * inner, dtype=cd, device=dev) for _ in range(n)]      # row (r, t)
        self.lut, self.rz = tr.decoder.lut(T, dev)
        self.src = torch.empty(2, R, T + 1, dtype=torch.int32, device=dev)
        self.run_seq = torch.empty(2, R, T + 1, dtype=torch.int64, device=dev)
        self.fin_seq = torch.empty(2, R, T + 1, dtype=torch.int64, device=dev)
        self.run_scores = torch.empty(R, dtype=torch.float32, device=dev)
        self.fin_scores = torch.empty(R, dtype=torch.float32, device=dev)
        self.fin_flag = torch.empty(R, dtype=torch.int32, device=dev)
        self.fin_len = torch.empty(R, dtype=torch.int32, device=dev)
        self.unsat = torch.empty(B, dtype=torch.int32, device=dev)
        self.done = torch.empty(B, dtype=torch.int32, device=dev)
        self.next_tok = torch.empty(R, 1, dtype=torch.int64, device=dev)
        self.cand_val = torch.empty(R, 2 * nb, dtype=torch.float32, device=dev)
        self.cand_tok = torch.empty(R, 2 * nb, dtype=torch.int32, device=dev)

    def reset(self, cfg, nb):
        """HF's initial state (:3185-3199); unused positions hold `pad_token_id or eos_token_id` (:3187), EOS for T5."""
        fill = cfg.pad_token_id or cfg.eos_token_id
        R = self.run_scores.shape[0]
        self.src.copy_(torch.arange(R, dtype=torch.int32, device=self.src.device)[None, :, None].expand_as(self.src))
        for s in (self.run_seq, self.fin_seq):
            s.fill_(fill)
            s[:, :, 0] = cfg.decoder_start_token_id
        self.run_scores.view(-1, nb).fill_(-1e9)
        self.run_scores.view(-1, nb)[:, 0] = 0.0
        self.fin_scores.fill_(-1e9)
        self.fin_flag.zero_()
        self.fin_len.zero_()
        self.unsat.fill_(1)
        self.done.zero_()
        self.next_tok.fill_(cfg.decoder_start_token_id)


def _beam_step_body(tr, st, t, B, nb, Le, T, length_penalty, early_stopping):
    """Position t for every hypothesis, then top-k and the beam update.  Reads and writes `st` and the operand cache only."""
    cfg = tr.config
    cd = st.enc.dtype
    H, dk, eps = cfg.num_heads, cfg.d_kv, cfg.layer_norm_epsilon
    inner = H * dk
    R = B * nb
    V = tr.shared.weight.shape[0]
    layers, tab, head = _decode_operands_peek(tr, cd)
    table = tr.decoder.block[0].layer[0].SelfAttention.relative_attention_bias.weight.detach()
    src = st.src[t & 1]
    x = O.embedding_fwd(st.next_tok, tab)                          # [R, d]
    for l, (ln0, wqkv, w_o, ln1, w_cq, _w_ckv, w_co, ln2, w_i, w_ff) in enumerate(layers):
        self_qkv, cross_kv = st.self_qkv[l], st.cross_kv[l]
        n0, _ = O.rmsnorm_fwd(x, ln0, eps, save_stats=False)
        row_t = self_qkv.view(R, T, 3 * inner)[:, t]
        O.linear_fwd(n0, wqkv, out=row_t)
        ctx = O.t5_attention_decode_beam(row_t[:, :inner], self_qkv[:, inner:2 * inner], self_qkv[:, 2 * inner:], R, H, T, dk,
                                         kv_group=nb, src=src, bias_table=table, lut=st.lut, rel_zero=st.rz, q_offset=t)
        h1 = O.linear_fwd(ctx, w_o, residual=x)
        n1, _ = O.rmsnorm_fwd(h1, ln1, eps, save_stats=False)
        qc = O.linear_fwd(n1, w_cq)
        ctx2 = O.t5_attention_decode_beam(qc, cross_kv[:, :inner], cross_kv[:, inner:], R, H, Le, dk, kv_group=nb)
        h2 = O.linear_fwd(ctx2, w_co, residual=h1)
        n2, _ = O.rmsnorm_fwd(h2, ln2, eps, save_stats=False)
        x = _ffn(cfg, n2, w_i, w_ff, h2)
    n, _ = O.rmsnorm_fwd(x, tr.decoder.final_layer_norm.weight, eps, save_stats=False)
    logits = O.linear_fwd(n, head, alpha=cfg.lm_head_scale, out_dtype=torch.float32)
    lib, stream = L.lib(), torch.cuda.current_stream().cuda_stream
    K = 2 * nb
    L.check(lib.klab_beam_topk(stream, R, V, K, logits.data_ptr(), logits.stride(0), st.run_scores.data_ptr(), st.cand_val.data_ptr(),
                               st.cand_tok.data_ptr()))
    L.check(lib.klab_beam_update(stream, B, nb, V, T, t, cfg.eos_token_id, float(length_penalty), _EARLY_STOPPING[early_stopping],
                                 st.cand_val.data_ptr(), st.cand_tok.data_ptr(), st.run_scores.data_ptr(), st.src.data_ptr(),
                                 st.run_seq.data_ptr(), T + 1, st.fin_scores.data_ptr(), st.fin_seq.data_ptr(), st.fin_flag.data_ptr(),
                                 st.fin_len.data_ptr(), st.unsat.data_ptr(), st.done.data_ptr(), st.next_tok.data_ptr()))
    return (st.fin_scores,)


@torch.no_grad()
def beam_generate(tr, embeds, B, Le, num_beams: int, max_new_tokens: int = 20, length_penalty: float = 1.0, early_stopping=False,
                  num_return_sequences: int = 1):
    """-> (sequences [B * num_return_sequences, n] int64, sequences_scores [B * num_return_sequences] fp32), as
    `generate(inputs_embeds, num_beams=...)` of HF 5.5.0 returns them (:3368-3376)."""
    from .graphs import POOL
    cfg = tr.config
    cd = embeds.dtype
    dev = embeds.device
    nb, T = num_beams, max_new_tokens
    states = tr.__dict__.setdefault("_klab_beam_states", {})
    key = (B, nb, Le, T, cd, dev)
    st = states.get(key)
    if st is None:
        if len(states) >= 4:                                             # as greedy_generate: a handful of geometries at most
            dead = {id(o) for o in states.values()}
            POOL.drop_keys(lambda k: k[0] == "beam" and k[2] in dead)
            states.clear()
        st = states[key] = _BeamState(tr, B, nb, Le, T, cd, dev)
    enc = tr.encoder.run_blocks(embeds, B, Le, tr.cache)
    O.rmsnorm_fwd(enc, tr.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon, out=st.enc, save_stats=False)
    layers, _, _ = _decode_operands(tr, cd)
    for l, ops_l in enumerate(layers):
        O.linear_fwd(st.enc, ops_l[5], out=st.cross_kv[l])
    st.reset(cfg, nb)
    # A sample whose finished set can no longer change is frozen on the device (klab_beam_update), so running past the step at
    # which HF stops changes nothing: the "every sample done" flag is read back every CHECK_EVERY steps only.
    n_run = 0
    for t in range(T):
        POOL.run(("beam", id(tr), id(st), t, float(length_penalty), _EARLY_STOPPING[early_stopping]), _beam_step_body, (),
                 (tr, st, t, B, nb, Le, T, length_penalty, early_stopping))
        n_run = t + 1
        if n_run % CHECK_EVERY == 0 and n_run < T and bool(st.done.cpu().all()):
            break
    nrs = num_return_sequences
    seq = st.fin_seq[n_run & 1].view(B, nb, T + 1)[:, :nrs].reshape(B * nrs, T + 1)
    scores = st.fin_scores.view(B, nb)[:, :nrs].reshape(B * nrs).clone()
    n_out = 1 + int(st.fin_len.view(B, nb)[:, :nrs].max().item())
    return seq[:, :n_out].clone(), scores


# ------------------------------------------------------------------------------------------------------------------------------
# Multinomial sampling: GenerationMixin._sample of HF 5.5.0 (HF/generation/utils.py:2658-2800) with do_sample=True and the
# temperature / top-k / top-p warpers, on the greedy machinery above.  num_return_sequences n expands sample b into the rows
# b * n + j as HF does, but the encoder output is not repeated: the n rows share the sample's cross K/V.  The draw is
# klab_sample_step's: a function of (seed, row, tokens generated so far) only, the seed one 63-bit number per call from torch's
# default CPU generator, so torch.manual_seed makes a call reproducible, whether graphs are on or off.
# ------------------------------------------------------------------------------------------------------------------------------
MAX_RETURN_SEQUENCES = 32          # rows of one sample that share its K/V in one CTA of klab_t5_attention_decode_beam


def check_sampling_options(temperature, top_k, top_p, num_return_sequences):
    """ValueError for options outside what transformers accepts (GenerationConfig.validate) or this build supports."""
    if isinstance(temperature, bool) or not isinstance(temperature, (int, float)) or not temperature > 0 or temperature == float("inf"):
        raise ValueError(f"sampling: temperature={temperature!r} must be a positive number")
    if isinstance(top_k, bool) or not isinstance(top_k, int) or top_k < 0:
        raise ValueError(f"sampling: top_k={top_k!r} must be a non-negative int (0 disables it)")
    if isinstance(top_p, bool) or not isinstance(top_p, (int, float)) or not 0.0 <= top_p <= 1.0:
        raise ValueError(f"sampling: top_p={top_p!r} must be in [0, 1]")
    n = num_return_sequences
    if isinstance(n, bool) or not isinstance(n, int) or not 1 <= n <= MAX_RETURN_SEQUENCES:
        raise ValueError(f"sampling: num_return_sequences={n!r} must be in 1..{MAX_RETURN_SEQUENCES}")


def draw_seed() -> int:
    """The seed of one sampling call: a 63-bit number from torch's default CPU generator (torch.manual_seed reproduces it)."""
    return int(torch.randint(0, 2 ** 63 - 1, (), dtype=torch.int64))


@torch.no_grad()
def sample_generate(tr, embeds, B, Le, max_new_tokens: int = 20, temperature: float = 1.0, top_k: int = 50, top_p: float = 1.0,
                    num_return_sequences: int = 1):
    """`generate(inputs_embeds, do_sample=True, ...)` -> ids [B * num_return_sequences, n] int64 (rows b * n + j), embeds
    [B * Le, d_model] bf16 or fp32 on the GPU."""
    cfg = tr.config
    if not (torch.is_tensor(embeds) and embeds.is_cuda and embeds.dtype in (torch.bfloat16, torch.float32) and embeds.dim() == 2
            and embeds.shape == (B * Le, cfg.d_model)):
        desc = f"{tuple(embeds.shape)} {embeds.dtype} on {embeds.device}" if torch.is_tensor(embeds) else type(embeds).__name__
        raise ValueError(f"sample_generate: inputs_embeds must be a CUDA bf16 / fp32 tensor [B * Le, {cfg.d_model}] (got {desc})")
    check_sampling_options(temperature, top_k, top_p, num_return_sequences)
    cd = embeds.dtype
    dev = embeds.device
    n, T = num_return_sequences, max_new_tokens
    seed = draw_seed()
    st = _decode_state(tr, "_klab_sample_states", "samp", (B, n, Le, T, cd, dev),
                       lambda: _DecodeState(tr, B, Le, T, cd, dev, rows=B * n))
    st.seed.copy_(torch.tensor([seed], dtype=torch.int64))
    sample = (n, float(temperature), int(top_k), float(top_p))
    return _decode_run(tr, st, embeds, B, Le, T, ("samp", id(tr), id(st)) + sample, sample)
