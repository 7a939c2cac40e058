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
"""
from __future__ import annotations

import torch

from . import _lib as L
from . import ops as O


class _DecodeState:
    """Static device buffers of one decode geometry (batch, encoder length, T): token ids, finished flags, per decoder block the
    self-attention q|k|v cache and the cross-attention k|v projection.  They never move, so the kernel sequence of the
    single-token step for position t can be captured into a CUDA graph once and replayed for every later caption batch."""

    def __init__(self, tr, B, Le, T, cd, dev):
        cfg = tr.config
        inner = cfg.num_heads * cfg.d_kv
        n = len(tr.decoder.block)
        self.ids = torch.empty(B, T + 1, dtype=torch.int64, device=dev)
        self.tok = torch.empty(B, 1, dtype=torch.int64, device=dev)
        self.unfinished = torch.empty(B, dtype=torch.int32, device=dev)
        self.enc = torch.empty(B * Le, cfg.d_model, dtype=cd, device=dev)
        self.cross_kv = [torch.empty(B * Le, 2 * inner, dtype=cd, device=dev) for _ in range(n)]
        self.self_qkv = [torch.zeros(B * T, 3 * inner, dtype=cd, device=dev) for _ in range(n)]   # row (b, t): q | k | v of token t
        self.lut, self.rz = tr.decoder.lut(T, dev)                 # covers relative positions -(T-1) .. T-1


def _decode_operands(tr, cd):
    g = tr.cache.get                                               # refreshes stale bf16 copies eagerly (outside any graph)
    out = []
    for blk in tr.decoder.block:
        ln0, q, k, v, o, ln1, cq, ck, cv, co, ln2, wi, wo = blk.flat_params()
        out.append((ln0.detach(), g([q, k, v], cd), g([o], cd), ln1.detach(), g([cq], cd), g([ck, cv], cd), g([co], cd), ln2.detach(),
                    g([wi], cd), g([wo], cd)))
    return out, g([tr.shared.weight], cd)


def _decode_step_body(tr, st, t, B, Le, T):
    """One token for every sample: position t in, ids[:, t + 1] out.  consts only (no per-call inputs): everything it reads or
    writes lives in `st` or in the operand cache, so the region is capturable as is."""
    cfg = tr.config
    cd = st.enc.dtype
    H, dk, d, eps = cfg.num_heads, cfg.d_kv, cfg.d_model, cfg.layer_norm_epsilon
    inner = H * dk
    layers, tab = _decode_operands_peek(tr, cd)
    table = tr.decoder.block[0].layer[0].SelfAttention.relative_attention_bias.weight.detach()
    st.tok.copy_(st.ids[:, t:t + 1])
    x = O.embedding_fwd(st.tok, tab)                               # [B, d]
    for l, (ln0, wqkv, w_o, ln1, w_cq, _w_ckv, w_co, ln2, w_i, w_ff) in enumerate(layers):
        self_qkv, cross_kv = st.self_qkv[l], st.cross_kv[l]
        n0, _ = O.rmsnorm_fwd(x, ln0, eps, save_stats=False)
        row_t = self_qkv.view(B, T, 3 * inner)[:, t]               # [B, 3*inner] view, row stride T*3*inner
        O.linear_fwd(n0, wqkv, out=row_t)                          # q | k | v of the new token, written into the cache
        ctx, _ = O.t5_attention_fwd(row_t[:, :inner], self_qkv[:, inner:2 * inner], self_qkv[:, 2 * inner:], B, H, 1, T, dk,
                                    bias_table=table, lut=st.lut, rel_zero=st.rz, num_buckets=cfg.relative_attention_num_buckets,
                                    causal=True, q_offset=t)
        h1 = O.linear_fwd(ctx, w_o, residual=x)
        n1, _ = O.rmsnorm_fwd(h1, ln1, eps, save_stats=False)
        qc = O.linear_fwd(n1, w_cq)
        ctx2, _ = O.t5_attention_fwd(qc, cross_kv[:, :inner], cross_kv[:, inner:], B, H, 1, Le, dk)
        h2 = O.linear_fwd(ctx2, w_co, residual=h1)
        n2, _ = O.rmsnorm_fwd(h2, ln2, eps, save_stats=False)
        f = O.linear_fwd(n2, w_i, act=L.ACT_RELU)
        x = O.linear_fwd(f, w_ff, residual=h2)
    n, _ = O.rmsnorm_fwd(x, tr.decoder.final_layer_norm.weight, eps, save_stats=False)
    logits = O.linear_fwd(n, tab, alpha=d ** -0.5, out_dtype=torch.float32)
    L.check(L.lib().klab_greedy_step(torch.cuda.current_stream().cuda_stream, B, tr.shared.weight.shape[0], logits.data_ptr(),
                                     logits.stride(0), st.ids.data_ptr(), st.ids.stride(0), t + 1, st.unfinished.data_ptr(),
                                     cfg.pad_token_id, cfg.eos_token_id))
    return (st.ids,)


def _decode_operands_peek(tr, cd):
    pk = tr.cache.peek
    out = []
    for blk in tr.decoder.block:
        ln0, q, k, v, o, ln1, cq, ck, cv, co, ln2, wi, wo = blk.flat_params()
        out.append((ln0.detach(), pk([q, k, v], cd), pk([o], cd), ln1.detach(), pk([cq], cd), pk([ck, cv], cd), pk([co], cd), ln2.detach(),
                    pk([wi], cd), pk([wo], cd)))
    return out, pk([tr.shared.weight], cd)


CHECK_EVERY = 5           # decode steps between two read-backs of the "every row has finished" flag


@torch.no_grad()
def greedy_generate(tr, embeds, B, Le, max_new_tokens: int = 20):
    from .graphs import POOL
    cfg = tr.config
    cd = embeds.dtype
    dev = embeds.device
    T = max_new_tokens                                                   # decoder positions 0 .. T-1 are ever attended to
    states = tr.__dict__.setdefault("_klab_decode_states", {})
    key = (B, Le, T, cd, dev)
    st = states.get(key)
    if st is None:
        if len(states) >= 4:                                             # a handful of geometries at most: the caches are large
            dead = {id(o) for o in states.values()}                      # the per-position regions bake the old buffers in: drop
            POOL.drop_keys(lambda k: k[0] == "dec" and k[2] in dead)     # them too, or the states would never be freed
            states.clear()
        st = states[key] = _DecodeState(tr, B, Le, T, cd, dev)
    enc = tr.encoder.run_blocks(embeds, B, Le, tr.cache)
    O.rmsnorm_fwd(enc, tr.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon, out=st.enc, save_stats=False)
    layers, _ = _decode_operands(tr, cd)                                 # also validates / refreshes every operand copy
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
        POOL.run(("dec", id(tr), id(st), t), _decode_step_body, (), (tr, st, t, B, Le, T))
        n_run = t + 1
        if n_run % CHECK_EVERY == 0 and n_run < T and not bool(st.unfinished.cpu().any()):
            break
    ids = st.ids[:, :n_run + 1]
    # length HF would have returned: it stops right after the step in which the last unfinished row emitted EOS
    is_eos = ids[:, 1:] == cfg.eos_token_id
    first_eos = torch.where(is_eos.any(1), is_eos.int().argmax(1) + 1, torch.full((B,), n_run, device=dev))     # tokens a row emits
    n_out = 1 + int(first_eos.max().item())
    return ids[:, :n_out].clone()


@torch.no_grad()
def greedy_generate_recompute(tr, embeds, B, Le, max_new_tokens: int = 20):
    cfg = tr.config
    cd = embeds.dtype
    dev = embeds.device
    enc = tr.encoder.run_blocks(embeds, B, Le, tr.cache)
    enc, _ = O.rmsnorm_fwd(enc, tr.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon, save_stats=False)
    tab = tr.cache.get([tr.shared.weight], cd)
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
        logits = O.linear_fwd(n, tab, alpha=d ** -0.5, out_dtype=torch.float32)
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
    H, dk, d, eps = cfg.num_heads, cfg.d_kv, cfg.d_model, cfg.layer_norm_epsilon
    inner = H * dk
    R = B * nb
    V = tr.shared.weight.shape[0]
    layers, tab = _decode_operands_peek(tr, cd)
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
        f = O.linear_fwd(n2, w_i, act=L.ACT_RELU)
        x = O.linear_fwd(f, w_ff, residual=h2)
    n, _ = O.rmsnorm_fwd(x, tr.decoder.final_layer_norm.weight, eps, save_stats=False)
    logits = O.linear_fwd(n, tab, alpha=d ** -0.5, out_dtype=torch.float32)
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
    layers, _ = _decode_operands(tr, cd)
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
