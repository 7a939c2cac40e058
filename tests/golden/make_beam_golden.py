"""Generate tests/golden/hf_beam.npz: `transformers` 5.5.0 beam search, T5ForConditionalGeneration.generate(inputs_embeds=...,
num_beams=...), on the weights and inputs of make_hf_golden.case_inputs for the cases tiny_a, tiny_b and mid.

    python tests/golden/make_beam_golden.py        (needs `transformers`; the stored file comes from transformers 5.5.0)

Randomly initialised T5 almost never emits EOS, and then every hypothesis runs to the maximum length and the finished-set,
length-penalty and early-stopping logic goes untested.  So each case's EOS row of the tied embedding gets alpha * u added,
u being the mean final decoder state (after the final norm and its weight) of the case's greedy decode: the EOS logit then
rises on exactly the states the decoder visits.  alpha is tuned below until the assertions at the end hold; the modified row is
stored, so the tests do not depend on recomputing u bit for bit.

Under "<case>/": eos_row (the modified embedding row), configs (JSON list of generate() options), and per option set i
"<i>/sequences", "<i>/scores" (sequences_scores).  Option sets: every (num_beams, length_penalty, early_stopping) of
{2, 4, 8} x {1.0, 0.0, 2.0} x {False, True, "never"}, with num_return_sequences alternating between 1 and num_beams and
max_new_tokens between the default (None: 20 new tokens) and an explicit value.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.caption_model import caption_embeddings  # noqa: E402
from oracle.t5 import t5_greedy_decode, t5_stack  # noqa: E402
from oracle.t5_beam import t5_beam_search  # noqa: E402
from tests.golden.make_hf_golden import HF_CASES, case_inputs, hf_models  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
EXPLICIT_MAX_NEW = 12
ALPHAS = tuple(round(0.05 * i, 2) for i in range(1, 61))


def option_sets():
    out = []
    for nb in (2, 4, 8):
        for lp in (1.0, 0.0, 2.0):
            for es in (False, True, "never"):
                i = len(out)
                out.append(dict(num_beams=nb, length_penalty=lp, early_stopping=es, num_return_sequences=nb if i % 2 else 1,
                                max_new_tokens=None if (i // 2) % 2 == 0 else EXPLICIT_MAX_NEW))
    return out


def with_eos_row(sd, t5, row):
    """The transformer state dict with shared.weight[eos] replaced (all four tied keys keep sharing one tensor)."""
    w = sd["shared.weight"].clone()
    w[t5.eos_token_id] = torch.as_tensor(row)
    return {k: (w if v is sd["shared.weight"] else v) for k, v in sd.items()}


def case_embeds(name):
    """-> (t5 dims, transformer state dict before the EOS change, encoder inputs_embeds [B, Le, d])."""
    case, swin, t5, sds, px, src, tgt = case_inputs(name)
    with torch.no_grad():
        emb = caption_embeddings(px, src, sds, t5, swin)
    return t5, sds["transformer"], emb


def mean_decoder_state(emb, sd, t5):
    with torch.no_grad():
        ids = t5_greedy_decode(emb, sd, t5)
        enc = t5_stack(emb, sd, "encoder.", t5)
        dec = t5_stack(F.embedding(ids, sd["shared.weight"]), sd, "decoder.", t5, enc_out=enc)
    return dec.reshape(-1, dec.shape[-1]).mean(0)


def eos_stats(emb, sd, t5):
    """Fraction of returned hypotheses (num_beams 4) that end by EOS, and the output width."""
    seqs, _ = t5_beam_search(emb, sd, t5, 4, num_return_sequences=4)
    ended = (seqs[:, 1:] == t5.eos_token_id).any(1)
    return float(ended.float().mean()), seqs.shape[1]


def tuned_row(name):
    t5, sd, emb = case_embeds(name)
    u = mean_decoder_state(emb, sd, t5)
    base = sd["shared.weight"][t5.eos_token_id].clone()
    for alpha in ALPHAS:
        row = base + alpha * u
        frac, width = eos_stats(emb, with_eos_row(sd, t5, row), t5)
        print(f"{name}: alpha {alpha}: {frac:.2f} of hypotheses end by EOS, output width {width}")
        if 0.5 <= frac < 1.0:
            return row
    raise AssertionError(f"{name}: no alpha in {ALPHAS} makes half, but not all, of the hypotheses end by EOS")


def hf_generate(tr, emb, opts):
    kw = {k: v for k, v in opts.items() if v is not None}
    out = tr.generate(inputs_embeds=emb, return_dict_in_generate=True, output_scores=True, **kw)
    return out.sequences, out.sequences_scores


def main(out_dir):
    stored = {}
    stats = {False: 0, True: 0, "never": 0}
    early_stops = 0
    for name in HF_CASES:
        case, swin, t5, sds, px, src, tgt = case_inputs(name)
        row = tuned_row(name)
        _, sd, emb = case_embeds(name)
        sd = with_eos_row(sd, t5, row)
        _, _, tr = hf_models(swin, t5)
        tr.load_state_dict(sd, strict=True)
        opts = option_sets()
        stored[f"{name}/eos_row"] = row.numpy()
        stored[f"{name}/configs"] = np.array(json.dumps(opts))
        for i, o in enumerate(opts):
            with torch.no_grad():
                seqs, scores = hf_generate(tr, emb, o)
            T = o["max_new_tokens"] or 20
            ended = (seqs[:, 1:] == t5.eos_token_id).any(1)
            n_eos_early = int((ended & ((seqs[:, 1:] == t5.eos_token_id).int().argmax(1) + 1 < T)).sum())
            stats[o["early_stopping"]] += n_eos_early
            early_stops += seqs.shape[1] < T + 1
            stored[f"{name}/{i}/sequences"] = seqs.numpy()
            stored[f"{name}/{i}/scores"] = scores.numpy()
    print("hypotheses ending by EOS before the maximum length, per early_stopping:", stats, "; runs stopping early:", early_stops)
    assert all(v > 0 for v in stats.values()), stats
    assert early_stops > 0
    np.savez_compressed(os.path.join(out_dir, "hf_beam.npz"), **stored)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    torch.manual_seed(0)
    main(a.out)
