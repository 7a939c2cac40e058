"""Beam search (`generate(num_beams=...)`) on the CPU: the oracle (oracle/t5_beam.py: t5_beam_search) against the stored outputs of
transformers 5.5.0 (tests/golden/hf_beam.npz, made by tests/golden/make_beam_golden.py) and against live transformers where it
imports; the run-to-max-length schedule of the CUDA build against HF's early stop; and the argument handling of
modeling.T5ForConditionalGeneration.generate, which needs no GPU."""
import json
import os

import numpy as np
import pytest
import torch

from oracle.t5_beam import t5_beam_search
from tests.golden.make_beam_golden import case_embeds, with_eos_row
from tests.golden.make_hf_golden import HF_CASES

GOLD = os.path.join(os.path.dirname(__file__), "golden", "hf_beam.npz")


def golden_case(name):
    """-> (t5 dims, transformer state dict with the stored EOS row, inputs_embeds, [(options, sequences, scores)])."""
    gold = np.load(GOLD)
    t5, sd, emb = case_embeds(name)
    sd = with_eos_row(sd, t5, torch.from_numpy(gold[f"{name}/eos_row"]))
    runs = [(o, gold[f"{name}/{i}/sequences"], gold[f"{name}/{i}/scores"])
            for i, o in enumerate(json.loads(str(gold[f"{name}/configs"])))]
    return t5, sd, emb, runs


def oracle_run(emb, sd, t5, o, **kw):
    return t5_beam_search(emb, sd, t5, o["num_beams"], o["max_new_tokens"] or 20, o["length_penalty"], o["early_stopping"],
                          o["num_return_sequences"], **kw)


@pytest.mark.parametrize("name", HF_CASES)
def test_oracle_matches_stored_transformers_beam_search(name):
    t5, sd, emb, runs = golden_case(name)
    assert len(runs) == 27
    for o, seqs, scores in runs:
        got, got_scores = oracle_run(emb, sd, t5, o)
        assert got.shape == seqs.shape and np.array_equal(got.numpy(), seqs), o
        np.testing.assert_allclose(got_scores.numpy(), scores, rtol=1e-5, atol=1e-6, err_msg=str(o))


def test_goldens_exercise_eos_and_early_stop():
    gold = np.load(GOLD)
    ended_early, short = {False: 0, True: 0, "never": 0}, 0
    for name in HF_CASES:
        for i, o in enumerate(json.loads(str(gold[f"{name}/configs"]))):
            seqs = gold[f"{name}/{i}/sequences"]
            T = o["max_new_tokens"] or 20
            eos = seqs[:, 1:] == 1
            ended_early[o["early_stopping"]] += int((eos.any(1) & (eos.argmax(1) + 1 < T)).sum())
            short += seqs.shape[1] < T + 1
    assert all(v > 0 for v in ended_early.values()) and short > 0


def test_unused_positions_hold_the_eos_id():
    """HF/generation/utils.py:3187 fills with `pad_token_id or eos_token_id[0]`; T5's pad id 0 is falsy, so the stored
    outputs pad finished hypotheses with EOS (1), not pad (0)."""
    gold = np.load(GOLD)
    seen = 0
    for name in HF_CASES:
        for i, _ in enumerate(json.loads(str(gold[f"{name}/configs"]))):
            for row in gold[f"{name}/{i}/sequences"]:
                hit = np.nonzero(row[1:] == 1)[0]
                if len(hit) and hit[0] + 2 < len(row):
                    assert (row[hit[0] + 1:] == 1).all()
                    seen += 1
    assert seen > 0


@pytest.mark.parametrize("name", HF_CASES)
def test_run_to_max_length_equals_hf_early_stop(name):
    """The CUDA build reads its "done" flag back only every few steps and runs frozen samples on: same output."""
    t5, sd, emb, runs = golden_case(name)
    for o, _, _ in runs:
        a, sa = oracle_run(emb, sd, t5, o)
        b, sb = oracle_run(emb, sd, t5, o, run_to_max_length=True)
        assert torch.equal(a, b) and torch.equal(sa, sb), o


def test_oracle_matches_live_transformers():
    transformers = pytest.importorskip("transformers")
    from tests.golden.make_beam_golden import hf_generate
    from tests.golden.make_hf_golden import case_inputs, hf_models
    for name in HF_CASES:
        t5, sd, emb, runs = golden_case(name)
        case, swin, *_ = case_inputs(name)
        _, _, tr = hf_models(swin, t5)
        tr.load_state_dict(sd, strict=True)
        for o, _, _ in runs[::4]:
            with torch.no_grad():
                seqs, scores = hf_generate(tr, emb, o)
            got, got_scores = oracle_run(emb, sd, t5, o)
            assert torch.equal(got, seqs), (name, o)
            torch.testing.assert_close(got_scores, scores, rtol=1e-5, atol=1e-6)
    assert transformers.__version__


# ---- generate() argument handling (no kernel runs) -------------------------------------------------------------------------
def _tiny():
    from klab_multimodalmodel_b200.modeling import T5Config, T5ForConditionalGeneration
    return T5ForConditionalGeneration(T5Config(vocab_size=64, d_model=64, d_ff=64, num_layers=1, num_heads=1))


def test_generation_config_defaults_follow_transformers():
    gc = _tiny().generation_config
    assert (gc.max_length, gc.max_new_tokens, gc.num_beams, gc.length_penalty, gc.early_stopping, gc.num_return_sequences) == \
        (20, None, 1, 1.0, False, 1)
    assert (gc.decoder_start_token_id, gc.eos_token_id, gc.pad_token_id) == (0, 1, 0)
    try:
        import transformers
    except ImportError:
        return
    # 5.5.0 stores None for unset fields and applies the defaults above inside generate(); the token ids come from the config
    hf = transformers.T5ForConditionalGeneration(transformers.T5Config(vocab_size=64, d_model=64, d_ff=64, num_layers=1, num_heads=1,
                                                                       decoder_start_token_id=0)).generation_config
    assert (hf.decoder_start_token_id, hf.eos_token_id, hf.pad_token_id) == (0, 1, 0)


def test_generate_dispatch(monkeypatch):
    from klab_multimodalmodel_b200 import generation
    calls = []
    monkeypatch.setattr(generation, "greedy_generate", lambda *a, **k: calls.append(("greedy", a[2:], k)) or "g")
    monkeypatch.setattr(generation, "beam_generate", lambda *a, **k: calls.append(("beam", a[2:], k)) or (torch.zeros(1, 1), None))
    tr = _tiny()
    emb = torch.zeros(2, 5, 64)
    assert tr.generate(inputs_embeds=emb) == "g"
    assert calls[-1] == ("greedy", (2, 5), {"max_new_tokens": 20})
    tr.generate(inputs_embeds=emb, max_new_tokens=7)
    assert calls[-1][2] == {"max_new_tokens": 7}
    tr.generate(inputs_embeds=emb, max_length=9)                       # explicit max_length counts the start token
    assert calls[-1][2] == {"max_new_tokens": 8}
    tr.generate(inputs_embeds=emb, num_beams=4, length_penalty=0.0, early_stopping="never", num_return_sequences=2)
    assert calls[-1] == ("beam", (2, 5), dict(num_beams=4, max_new_tokens=20, length_penalty=0.0, early_stopping="never",
                                              num_return_sequences=2))
    tr.generation_config.num_beams = 3
    tr.generate(inputs_embeds=emb)
    assert calls[-1][0] == "beam" and calls[-1][2]["num_beams"] == 3


@pytest.mark.parametrize("kw", [dict(do_sample=True), dict(num_beams=9), dict(num_beams=2, num_return_sequences=3),
                                dict(num_return_sequences=2), dict(early_stopping="sometimes"), dict(top_k=5),
                                dict(logits_processor=[object()]), dict(num_beams=0)])
def test_generate_rejects_unsupported_options(kw):
    with pytest.raises((ValueError, TypeError)):
        _tiny().generate(inputs_embeds=torch.zeros(1, 3, 64), **kw)
