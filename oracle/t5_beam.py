"""Oracle: beam-search caption generation, `generate(inputs_embeds=..., num_beams=...)` of HF 5.5.0, restated in plain torch fp32.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  HF/ = site-packages/transformers (5.5.0).  Takes the same flat HF-style state
dict `sd` as oracle/t5.py, whose encoder / decoder stacks it runs.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch
import torch.nn.functional as F

from .t5 import T5Dims, t5_stack
# ------------------------------------------------------------------------------------------------------------------------
# Beam search: GenerationMixin._beam_search of HF 5.5.0 (HF/generation/utils.py:3076-3386 main loop, :2945-3072 top-k /
# running / finished updates, :2876-2943 stopping), restated on explicit per-step state so the CUDA build can be checked one
# step at a time.  Every top-k here takes ties to the LOWER index (stable descending sort); HF uses torch.topk, whose tie
# order is unspecified -- tests/golden/hf_beam.npz pins that the two agree on the stored cases.
# ------------------------------------------------------------------------------------------------------------------------
def _topk_desc(x: torch.Tensor, k: int):
    v, i = torch.sort(x, dim=-1, descending=True, stable=True)
    return v[..., :k], i[..., :k]


@dataclass
class BeamState:
    """Per sample b and beam slot: running sequences / scores (:3187-3195), finished sequences / scores / flags (:3192-3197),
    generated length of each finished hypothesis (the count of its non -1 `beam_indices`, :3376) and the early-stop heuristic
    flag (:3198).  `frozen[b]`: the sample can no longer change its finished set (see `beam_step`)."""
    run_seq: torch.Tensor       # [B, nb, max_length] int64
    run_scores: torch.Tensor    # [B, nb] fp32
    seq: torch.Tensor           # [B, nb, max_length] int64
    scores: torch.Tensor        # [B, nb] fp32
    fin: torch.Tensor           # [B, nb] bool
    gen_len: torch.Tensor       # [B, nb] int64
    unsat: torch.Tensor         # [B] bool
    frozen: torch.Tensor        # [B] bool


def beam_init(B: int, nb: int, max_length: int, dims: T5Dims) -> BeamState:
    # :3187 reads `pad_token_id or eos_token_id[0]`: T5's pad id 0 is falsy, so unused positions hold the EOS id
    fill = dims.pad_token_id or dims.eos_token_id
    run_seq = torch.full((B, nb, max_length), fill, dtype=torch.long)
    run_seq[:, :, 0] = dims.decoder_start_token_id
    run_scores = torch.zeros(B, nb)
    run_scores[:, 1:] = -1e9
    return BeamState(run_seq, run_scores, run_seq.clone(), torch.full((B, nb), -1e9), torch.zeros(B, nb, dtype=torch.bool),
                     torch.zeros(B, nb, dtype=torch.long), torch.ones(B, dtype=torch.bool), torch.zeros(B, dtype=torch.bool))


def beam_step(st: BeamState, logits: torch.Tensor, t: int, max_length: int, dims: T5Dims, length_penalty: float,
              early_stopping, freeze: bool = False) -> bool:
    """One iteration of the loop for the token at position t + 1 (cur_len = t + 1), logits [B * nb, V] of the running beams.
    Updates `st` in place and returns HF's "has unfinished sequences" (:2929-2943).

    freeze = True is the schedule of the CUDA build, which runs on after HF would have stopped: a sample whose heuristic flag
    dropped, or (early_stopping True) whose finished set is full, keeps its state unchanged, and once a step ends with every
    candidate of every sample hitting a stopping criterion nothing changes any more.  HF masks exactly those samples' candidates
    with -1e9 (:3048-3051), so their finished sets do not change either and both schedules return the same output.  HF's third
    stop condition, every candidate of the batch hitting a stopping criterion, needs no state of its own: such a step fills
    the finished set of every live sample with hypotheses far above the -1e9 the running beams are left with, so the heuristic
    freezes them all at the same step."""
    B, nb = st.scores.shape
    V = logits.shape[-1]
    K = 2 * nb                                                               # beams_to_keep, one EOS id (:3141)
    cur_len = t + 1
    logp = F.log_softmax(logits.float(), dim=-1).view(B, nb, V) + st.run_scores[:, :, None]      # :3278-3283
    top_v, top_i = _topk_desc(logp.reshape(B, nb * V), K)                    # :2981-2984 (ties: lower flat index)
    parent, tok = top_i // V, top_i % V
    cand_seq = torch.gather(st.run_seq, 1, parent[:, :, None].expand(B, K, max_length)).clone()
    cand_seq[:, :, cur_len] = tok
    hits = (tok == dims.eos_token_id) | (cur_len + 1 >= max_length)           # EosTokenCriteria, MaxLengthCriteria
    rv = top_v + hits.float() * -1.0e9                                       # :3012-3020
    _, ni = _topk_desc(rv, nb)
    new_run_seq = torch.gather(cand_seq, 1, ni[:, :, None].expand(B, nb, max_length))
    new_run_scores = torch.gather(rv, 1, ni)
    just = hits & (torch.arange(K) < nb)[None, :]                            # :3044-3051
    fv = top_v / ((cur_len + 1 - 1) ** length_penalty)
    fv = fv + (st.fin.all(1, keepdim=True) & (early_stopping is True)).float() * -1.0e9
    fv = fv + (~st.unsat[:, None]).float() * -1.0e9
    fv = fv + (~just).float() * -1.0e9
    m_scores = torch.cat((st.scores, fv), 1)
    m_seq = torch.cat((st.seq, cand_seq), 1)
    m_fin = torch.cat((st.fin, just), 1)
    m_len = torch.cat((st.gen_len, torch.full((B, K), t + 1, dtype=torch.long)), 1)
    _, mi = _topk_desc(m_scores, nb)                                         # :3060-3064
    new_scores = torch.gather(m_scores, 1, mi)
    new_seq = torch.gather(m_seq, 1, mi[:, :, None].expand(B, nb, max_length))
    new_fin = torch.gather(m_fin, 1, mi)
    new_len = torch.gather(m_len, 1, mi)
    # _check_early_stop_heuristic after cur_len += 1 (:2876-2915, :3351-3361)
    if early_stopping == "never" and length_penalty > 0.0:
        best_len = max_length - 1
    else:
        best_len = cur_len + 1 - 1
    best = new_run_scores[:, :1] / (best_len ** length_penalty)
    worst = torch.where(new_fin, torch.min(new_scores, dim=1, keepdim=True)[0], -1.0e9)
    new_unsat = st.unsat & torch.any(best > worst, dim=-1)
    upd = ~st.frozen if freeze else torch.ones(B, dtype=torch.bool)
    st.run_seq = torch.where(upd[:, None, None], new_run_seq, st.run_seq)
    st.run_scores = torch.where(upd[:, None], new_run_scores, st.run_scores)
    st.seq = torch.where(upd[:, None, None], new_seq, st.seq)
    st.scores = torch.where(upd[:, None], new_scores, st.scores)
    st.fin = torch.where(upd[:, None], new_fin, st.fin)
    st.gen_len = torch.where(upd[:, None], new_len, st.gen_len)
    st.unsat = torch.where(upd, new_unsat, st.unsat)
    st.frozen = st.frozen | ~st.unsat | (st.fin.all(1) & (early_stopping is True))
    # _beam_search_has_unfinished_sequences (:2929-2943), over the whole batch
    return bool(st.unsat.any()) and not (bool(st.fin.all()) and early_stopping is True) and not bool(hits.all())


def beam_output(st: BeamState, num_return_sequences: int):
    """:3368-3376: the best `num_return_sequences` finished hypotheses per sample, cropped to the longest returned one."""
    B, nb, _ = st.seq.shape
    seq = st.seq[:, :num_return_sequences].reshape(B * num_return_sequences, -1)
    scores = st.scores[:, :num_return_sequences].reshape(-1)
    n = 1 + int(st.gen_len[:, :num_return_sequences].max())
    return seq[:, :n], scores


def t5_beam_search(enc_in: torch.Tensor, sd: dict, dims: T5Dims, num_beams: int, max_new_tokens: int = 20,
                   length_penalty: float = 1.0, early_stopping=False, num_return_sequences: int = 1,
                   run_to_max_length: bool = False):
    """`generate(inputs_embeds=enc_in, num_beams=..., ...)` -> (sequences [B * nrs, n] int64, sequences_scores [B * nrs] fp32).
    The encoder output is repeated per beam as HF does (_expand_inputs_for_generation); the decoder prefix is recomputed
    every step (same arithmetic as the cache, as in t5_greedy_decode).  run_to_max_length: the freezing schedule of the CUDA
    build (see beam_step) instead of stopping where HF stops."""
    enc = t5_stack(enc_in, sd, "encoder.", dims)
    B = enc.shape[0]
    nb = num_beams
    max_length = max_new_tokens + 1
    enc_rep = enc.repeat_interleave(nb, 0)
    st = beam_init(B, nb, max_length, dims)
    for t in range(max_new_tokens):
        ids = st.run_seq[:, :, :t + 1].reshape(B * nb, t + 1)
        dec = t5_stack(F.embedding(ids, sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc_rep)
        logits = (dec[:, -1] * dims.d_model ** -0.5) @ sd["lm_head.weight"].T
        going = beam_step(st, logits, t, max_length, dims, length_penalty, early_stopping, freeze=run_to_max_length)
        if not going and not run_to_max_length:
            break
    return beam_output(st, num_return_sequences)
