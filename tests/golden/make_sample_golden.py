"""Generate tests/golden/hf_sample.npz: `transformers` 5.5.0 multinomial sampling, T5ForConditionalGeneration.generate(
inputs_embeds=..., do_sample=True, ...), on the weights and inputs of make_hf_golden.case_inputs for the cases tiny_a, tiny_b and
mid, with each case's EOS embedding row from tests/golden/hf_beam.npz (so that rows end by EOS at varied lengths).

    python tests/golden/make_sample_golden.py        (needs `transformers`; the stored file comes from transformers 5.5.0)

torch.multinomial is replaced (unittest.mock.patch.object) by the draw this project defines: on its c-th call in a run (the
c-th generated token), row r of probs gets the token inverse_cdf(probs[r], sample_uniform(seed, r, c)) (oracle/t5_sample.py).
_sample calls it exactly once per step with probs [B * n, V], so everything else -- the warpers, the softmax, pad after EOS, the
stopping criteria, num_return_sequences -- is transformers' own.

Under "<case>/": configs (JSON list of generate() options with their seed), and per option set i "<i>/sequences".  Option
sets: every temperature of {1.0, 0.7, 1.5} x every (top_k, top_p) of {(50, 1.0) the defaults, (0, 0.9), (5, 0.8), (1, 1.0),
(0, 1.0) pure multinomial, (50, 0.5)}, num_return_sequences cycling 1, 3, 8, max_new_tokens alternating between the default
(None: 20 new tokens) and 12, seed = the set's index.
"""
import argparse
import json
import os
import sys
from unittest import mock

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.t5_sample import inverse_cdf, sample_uniform  # noqa: E402
from tests.golden.make_beam_golden import case_embeds, with_eos_row  # noqa: E402
from tests.golden.make_hf_golden import HF_CASES, case_inputs, hf_models  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
EXPLICIT_MAX_NEW = 12
WARPERS = ((50, 1.0), (0, 0.9), (5, 0.8), (1, 1.0), (0, 1.0), (50, 0.5))


def option_sets():
    out = []
    for temperature in (1.0, 0.7, 1.5):
        for top_k, top_p in WARPERS:
            i = len(out)
            out.append(dict(temperature=temperature, top_k=top_k, top_p=top_p, num_return_sequences=(1, 3, 8)[i % 3],
                            max_new_tokens=None if i % 2 == 0 else EXPLICIT_MAX_NEW, seed=i))
    return out


def golden_sd(name):
    """-> (t5 dims, transformer state dict with hf_beam.npz's EOS row, inputs_embeds [B, Le, d])."""
    t5, sd, emb = case_embeds(name)
    row = np.load(os.path.join(HERE, "hf_beam.npz"))[f"{name}/eos_row"]
    return t5, with_eos_row(sd, t5, torch.from_numpy(row)), emb


def hf_sample(tr, emb, opts):
    """transformers' generate(do_sample=True, ...) with the defined draw in place of torch.multinomial."""
    calls = []

    def draw(probs, num_samples=1, **kw):
        assert num_samples == 1 and probs.dim() == 2
        c = len(calls)
        calls.append(c)
        u = torch.tensor([sample_uniform(opts["seed"], r, c) for r in range(probs.shape[0])], dtype=torch.float64)
        return inverse_cdf(probs, u)[:, None]

    kw = {k: v for k, v in opts.items() if v is not None and k != "seed"}
    with mock.patch.object(torch, "multinomial", draw), torch.no_grad():
        return tr.generate(inputs_embeds=emb, do_sample=True, **kw)


def main(out_dir):
    stored = {}
    eos_early, early_stops = 0, 0
    for name in HF_CASES:
        case, swin, *_ = case_inputs(name)
        t5, sd, emb = golden_sd(name)
        _, _, tr = hf_models(swin, t5)
        tr.load_state_dict(sd, strict=True)
        opts = option_sets()
        stored[f"{name}/configs"] = np.array(json.dumps(opts))
        for i, o in enumerate(opts):
            seqs = hf_sample(tr, emb, o)
            T = o["max_new_tokens"] or 20
            is_eos = seqs[:, 1:] == t5.eos_token_id
            eos_early += int((is_eos.any(1) & (is_eos.int().argmax(1) + 1 < T)).sum())
            early_stops += seqs.shape[1] < T + 1
            stored[f"{name}/{i}/sequences"] = seqs.numpy()
    print("rows ending by EOS before the maximum length:", eos_early, "; runs stopping early:", early_stops)
    assert eos_early > 0 and early_stops > 0
    np.savez_compressed(os.path.join(out_dir, "hf_sample.npz"), **stored)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    main(a.out)
