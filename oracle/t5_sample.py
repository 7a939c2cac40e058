"""Oracle: multinomial-sampling caption generation, `generate(inputs_embeds=..., do_sample=True, temperature=..., top_k=...,
top_p=..., num_return_sequences=...)` of HF 5.5.0, restated in plain torch fp32.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  HF/ = site-packages/transformers (5.5.0).  Takes the same flat HF-style state
dict `sd` as oracle/t5.py, whose encoder / decoder stacks it runs.

torch.multinomial's random stream cannot be reproduced on the device, so the draw is defined instead (csrc/sampling.cu states the
same): one uniform per (row, step), `sample_uniform(seed, row, t)`, and the inverse CDF of the step's probabilities in
vocabulary order, `inverse_cdf`.  transformers with torch.multinomial replaced by that draw (tests/golden/make_sample_golden.py)
returns exactly what `t5_sample` returns.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .t5 import T5Dims, t5_stack

_M64 = (1 << 64) - 1
GOLDEN_GAMMA = 0x9E3779B97F4A7C15


def sample_uniform(seed: int, row: int, t: int) -> float:
    """u(seed, row, t) in [0, 1), t = tokens generated before this one: the splitmix64 finaliser of the Weyl counter
    seed + gamma * (1 + row * 2^16 + t) mod 2^64, top 24 bits."""
    z = (seed + GOLDEN_GAMMA * (1 + row * 65536 + t)) & _M64
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & _M64
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & _M64
    z ^= z >> 31
    return (z >> 40) * 2.0 ** -24


def inverse_cdf(probs: torch.Tensor, u) -> torch.Tensor:
    """probs [R, V] (any non-negative weights), u [R] (or a float): per row the smallest index i with
    sum_{j <= i} probs_j > u * sum(probs), in float64; the last index with a non-zero weight if rounding leaves none."""
    p = probs.double().reshape(-1, probs.shape[-1])
    u = torch.as_tensor(u, dtype=torch.float64).reshape(-1).expand(p.shape[0])
    c = p.cumsum(-1)
    tok = torch.searchsorted(c, (u * c[:, -1])[:, None], right=True)[:, 0]
    last = p.shape[1] - 1 - (p > 0).flip(-1).int().argmax(-1)
    return torch.where(tok < p.shape[1], tok, last)


def warp(logits: torch.Tensor, temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0) -> torch.Tensor:
    """The warpers `_get_logits_processor` (HF/generation/utils.py:1197-1224) appends for do_sample with num_beams 1, in its
    order and arithmetic (fp32; min_tokens_to_keep 1): TemperatureLogitsWarper (logits_process.py:236), TopKLogitsWarper
    (:536), TopPLogitsWarper (:469).  Removed tokens get -inf.  The top-p sort breaks ties in an unspecified order, as in HF."""
    scores = logits.float()
    if temperature is not None and temperature != 1.0:
        scores = scores / temperature
    if top_k is not None and top_k != 0:
        k = min(max(top_k, 1), scores.size(-1))
        scores = scores.masked_fill(scores < torch.topk(scores, k)[0][..., -1, None], -float("inf"))
    if top_p is not None and top_p < 1.0:
        sorted_logits, sorted_indices = torch.sort(scores, descending=False)
        cumulative_probs = sorted_logits.softmax(dim=-1).cumsum(dim=-1)
        remove = cumulative_probs <= (1 - top_p)
        remove[..., -1:] = 0
        scores = scores.masked_fill(remove.scatter(-1, sorted_indices, remove), -float("inf"))
    return scores


def kept_by_rule(logits: torch.Tensor, temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0):
    """The kept set as klab_sample_step defines it, in float64 over the fp32 scores (logits / temperature in fp32):
    top-k keeps s >= the k-th largest; top-p keeps token i iff the mass (softmax over the top-k set) of the tokens with a
    strictly greater score is < top_p, or s_i is the maximum -- every tied token is kept.  -> (scores fp32 [R, V],
    kept bool [R, V], top-p margin [R]: the smallest |mass_greater - top_p| over the row's distinct scores, relative, inf if
    top-p is off or 0)."""
    s = logits.float()
    if temperature != 1.0:
        s = s / temperature
    s = s.reshape(-1, s.shape[-1])
    keep = torch.ones_like(s, dtype=torch.bool)
    if top_k and top_k < s.shape[1]:
        keep &= s >= torch.topk(s, top_k, dim=-1)[0][:, -1:]
    if top_p <= 0.0:                                                   # the maximum and its ties, whatever the masses
        keep &= s == s.max(-1, keepdim=True)[0]
    margin = torch.full((s.shape[0],), float("inf"), dtype=torch.float64)
    if 0.0 < top_p < 1.0:
        d = s.double()
        w = torch.where(keep, torch.exp(d - d.max(-1, keepdim=True)[0]), torch.zeros_like(d))
        p = w / w.sum(-1, keepdim=True)
        v, idx = torch.sort(d, dim=-1, descending=True)
        ps = p.gather(1, idx)
        start = torch.ones_like(v, dtype=torch.bool)                   # first of a run of equal scores
        start[:, 1:] = v[:, 1:] != v[:, :-1]
        excl = ps.cumsum(-1) - ps
        greater = torch.where(start, excl, torch.full_like(excl, -1.0)).cummax(-1)[0]     # mass strictly above each score
        ok = (greater < top_p) | (v == v[:, :1])
        keep &= torch.empty_like(ok).scatter_(1, idx, ok)
        gap = torch.where(start & (ps > 0), (greater - top_p).abs(), torch.full_like(greater, float("inf")))
        margin = gap.min(-1)[0]
    return s, keep, margin


def t5_sample(enc_in: torch.Tensor, sd: dict, dims: T5Dims, seed: int, temperature: float = 1.0, top_k: int = 50,
              top_p: float = 1.0, num_return_sequences: int = 1, max_new_tokens: int = 20, run_to_max_length: bool = False):
    """GenerationMixin._sample (HF/generation/utils.py:2658-2800) for `generate(inputs_embeds=enc_in, do_sample=True, ...)`
    with the defined draw -> ids [B * n, len] int64, rows b * n + j.  The encoder output is repeated per row as HF does
    (_expand_inputs_for_generation); the decoder prefix is recomputed every step (same arithmetic as the cache).  Finished rows
    emit pad; the loop stops when every row has emitted EOS, or (run_to_max_length) runs all max_new_tokens steps as the CUDA
    build does before it trims to the same length."""
    enc = t5_stack(enc_in, sd, "encoder.", dims).repeat_interleave(num_return_sequences, 0)
    R = enc.shape[0]
    ids = torch.full((R, 1), dims.decoder_start_token_id, dtype=torch.long)
    unfinished = torch.ones(R, dtype=torch.bool)
    for t in range(max_new_tokens):
        dec = t5_stack(F.embedding(ids, sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc)
        logits = (dec[:, -1] * dims.d_model ** -0.5) @ sd["lm_head.weight"].T
        probs = F.softmax(warp(logits, temperature, top_k, top_p), dim=-1)
        u = torch.tensor([sample_uniform(seed, r, t) for r in range(R)], dtype=torch.float64)
        nxt = inverse_cdf(probs, u)
        nxt = torch.where(unfinished, nxt, torch.full_like(nxt, dims.pad_token_id))
        ids = torch.cat([ids, nxt[:, None]], dim=1)
        unfinished = unfinished & (nxt != dims.eos_token_id)
        if not unfinished.any() and not run_to_max_length:
            break
    if run_to_max_length:
        is_eos = ids[:, 1:] == dims.eos_token_id
        first = torch.where(is_eos.any(1), is_eos.int().argmax(1) + 1, torch.full((R,), ids.shape[1] - 1))
        return ids[:, :1 + int(first.max())]
    return ids
