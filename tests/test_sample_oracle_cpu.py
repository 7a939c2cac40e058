"""Multinomial sampling (`generate(do_sample=True)`) on the CPU: the oracle (oracle/t5_sample.py) against the stored outputs of
transformers 5.5.0 with torch.multinomial replaced by the defined draw (tests/golden/hf_sample.npz, made by
tests/golden/make_sample_golden.py) and against live transformers where it imports; the warpers against transformers' classes;
the top-p tie rule; the hash; and the argument handling of modeling.T5ForConditionalGeneration.generate, which needs no GPU."""
import json
import os

import numpy as np
import pytest
import torch

from oracle.t5 import t5_greedy_decode
from oracle.t5_sample import inverse_cdf, kept_by_rule, sample_uniform, t5_sample, warp
from tests.golden.make_hf_golden import HF_CASES
from tests.golden.make_sample_golden import golden_sd

GOLD = os.path.join(os.path.dirname(__file__), "golden", "hf_sample.npz")


def golden_case(name):
    """-> (t5 dims, transformer state dict with the stored EOS row, inputs_embeds, [(options, sequences)])."""
    gold = np.load(GOLD)
    t5, sd, emb = golden_sd(name)
    runs = [(o, gold[f"{name}/{i}/sequences"]) for i, o in enumerate(json.loads(str(gold[f"{name}/configs"])))]
    return t5, sd, emb, runs


def oracle_run(emb, sd, t5, o, **kw):
    return t5_sample(emb, sd, t5, o["seed"], o["temperature"], o["top_k"], o["top_p"], o["num_return_sequences"],
                     o["max_new_tokens"] or 20, **kw)


@pytest.mark.parametrize("name", HF_CASES)
def test_oracle_matches_stored_transformers_sampling(name):
    t5, sd, emb, runs = golden_case(name)
    assert len(runs) == 18
    for o, seqs in runs:
        got = oracle_run(emb, sd, t5, o)
        assert got.shape == seqs.shape and np.array_equal(got.numpy(), seqs), o


def test_goldens_exercise_eos_early_stop_and_every_option():
    gold = np.load(GOLD)
    ended, short, seen = 0, 0, set()
    for name in HF_CASES:
        for i, o in enumerate(json.loads(str(gold[f"{name}/configs"]))):
            seqs = gold[f"{name}/{i}/sequences"]
            T = o["max_new_tokens"] or 20
            eos = seqs[:, 1:] == 1
            ended += int((eos.any(1) & (eos.argmax(1) + 1 < T)).sum())
            short += seqs.shape[1] < T + 1
            assert seqs.shape[0] % o["num_return_sequences"] == 0
            seen.add((o["temperature"], o["top_k"], o["top_p"]))
    assert ended > 0 and short > 0 and len(seen) == 18


@pytest.mark.parametrize("name", HF_CASES)
def test_run_to_max_length_equals_early_stop(name):
    """The CUDA build reads its "all finished" flag back only every few steps, runs on and trims: same output."""
    t5, sd, emb, runs = golden_case(name)
    for o, _ in runs[::3]:
        assert torch.equal(oracle_run(emb, sd, t5, o), oracle_run(emb, sd, t5, o, run_to_max_length=True)), o


def test_oracle_matches_live_transformers():
    transformers = pytest.importorskip("transformers")
    from tests.golden.make_hf_golden import case_inputs, hf_models
    from tests.golden.make_sample_golden import hf_sample
    for name in HF_CASES:
        t5, sd, emb, runs = golden_case(name)
        case, swin, *_ = case_inputs(name)
        _, _, tr = hf_models(swin, t5)
        tr.load_state_dict(sd, strict=True)
        for o, _ in runs[::4]:
            assert torch.equal(hf_sample(tr, emb, o), oracle_run(emb, sd, t5, o)), (name, o)
    assert transformers.__version__


def test_top_k_one_is_greedy():
    t5, sd, emb, _ = golden_case("tiny_b")
    for seed in (0, 5):
        assert torch.equal(t5_sample(emb, sd, t5, seed, temperature=0.7, top_k=1), t5_greedy_decode(emb, sd, t5))


def test_hash_constants():
    # splitmix64's first output for seed 0 is 0xE220A8397B1DCDAF: its top 24 bits
    assert sample_uniform(0, 0, 0) * 2 ** 24 == 0xE220A8
    assert sample_uniform(1, 2, 3) * 2 ** 24 == 16536742
    assert sample_uniform(2 ** 63 - 1, 5, 17) * 2 ** 24 == 2570684
    assert sample_uniform(12345, 65535, 65535) * 2 ** 24 == 3705145
    assert sample_uniform(7, 1000, 0) * 2 ** 24 == 5855388


def test_inverse_cdf():
    p = torch.tensor([[0.0, 0.25, 0.0, 0.5, 0.25, 0.0]])
    for u, want in ((0.0, 1), (0.2499, 1), (0.25, 3), (0.7499, 3), (0.75, 4), (0.9999, 4)):
        assert int(inverse_cdf(p, u)) == want, u
    assert int(inverse_cdf(p * 1e-30, 1.0 - 2 ** -24)) == 4


def _rows_without_boundary_ties(n, V, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, V, generator=g) * 3
    x[:, ::7] = -float("inf")
    return x


@pytest.mark.parametrize("temperature,top_k,top_p", [(1.0, 50, 1.0), (0.7, 0, 0.9), (1.5, 5, 0.8), (1.0, 1, 1.0), (2.0, 0, 0.3),
                                                     (0.5, 300, 0.95), (1.0, 0, 1.0), (1.3, 20, 0.0)])
def test_warp_matches_transformers_warpers(temperature, top_k, top_p):
    transformers = pytest.importorskip("transformers")
    from transformers.generation.logits_process import TemperatureLogitsWarper, TopKLogitsWarper, TopPLogitsWarper
    x = _rows_without_boundary_ties(16, 257, int(temperature * 10) + top_k)
    ref = x.clone()
    if temperature != 1.0:
        ref = TemperatureLogitsWarper(temperature)(None, ref)
    if top_k:
        ref = TopKLogitsWarper(top_k)(None, ref)
    if top_p < 1.0:
        ref = TopPLogitsWarper(top_p)(None, ref)
    got = warp(x, temperature, top_k, top_p)
    assert torch.equal(got > -float("inf"), ref > -float("inf"))
    _, keep, margin = kept_by_rule(x, temperature, top_k, top_p)                # the kernel's rule: same set without ties
    assert torch.equal(keep & (x > -float("inf")), got > -float("inf"))
    assert transformers.__version__


def test_top_p_tie_rule_keeps_every_tied_token():
    x = torch.full((1, 10), -5.0)
    x[0, [2, 6]] = 1.0                                     # two tied maxima, 0.47 of the mass each
    x[0, [3, 8]] = 0.0                                     # two tied runners-up
    _, keep, _ = kept_by_rule(x, top_p=0.0)
    assert keep[0].nonzero().flatten().tolist() == [2, 6]  # top_p = 0 keeps the maximum and its ties
    _, keep, _ = kept_by_rule(x, top_p=0.5)
    assert keep[0].nonzero().flatten().tolist() == [2, 6]  # mass above the runners-up (0.85) is not < 0.5
    _, keep, _ = kept_by_rule(x, top_p=0.9)
    assert keep[0].nonzero().flatten().tolist() == [2, 3, 6, 8]
    _, keep, _ = kept_by_rule(x, top_k=3)
    assert keep[0].nonzero().flatten().tolist() == [2, 3, 6, 8]      # ties at the k-th value are kept


# ---- generate() argument handling (no kernel runs) -------------------------------------------------------------------------
def _tiny():
    from klab_multimodalmodel_b200.modeling import T5Config, T5ForConditionalGeneration
    return T5ForConditionalGeneration(T5Config(vocab_size=64, d_model=64, d_ff=64, num_layers=1, num_heads=1))


def test_sampling_defaults_follow_transformers():
    gc = _tiny().generation_config
    assert (gc.do_sample, gc.temperature, gc.top_k, gc.top_p) == (False, 1.0, 50, 1.0)


def test_generate_dispatches_sampling(monkeypatch):
    from klab_multimodalmodel_b200 import generation
    calls = []
    monkeypatch.setattr(generation, "sample_generate", lambda *a, **k: calls.append(("sample", a[2:], k)) or "s")
    monkeypatch.setattr(generation, "greedy_generate", lambda *a, **k: calls.append(("greedy", a[2:], k)) or "g")
    tr = _tiny()
    emb = torch.zeros(2, 5, 64)
    assert tr.generate(inputs_embeds=emb, do_sample=True) == "s"
    assert calls[-1] == ("sample", (2, 5), dict(max_new_tokens=20, temperature=1.0, top_k=50, top_p=1.0, num_return_sequences=1))
    tr.generate(inputs_embeds=emb, do_sample=True, temperature=0.7, top_k=0, top_p=0.9, num_return_sequences=32, max_length=9)
    assert calls[-1][2] == dict(max_new_tokens=8, temperature=0.7, top_k=0, top_p=0.9, num_return_sequences=32)
    out = tr.generate(inputs_embeds=emb, do_sample=True, return_dict_in_generate=True, output_scores=True)
    assert out.sequences == "s" and out.sequences_scores is None
    tr.generation_config.do_sample = True                          # MyModel.forward(return_loss=False) samples from here on
    tr.generation_config.top_k = 5
    tr.generate(inputs_embeds=emb)
    assert calls[-1][0] == "sample" and calls[-1][2]["top_k"] == 5
    tr.generation_config.do_sample = False
    with pytest.raises(ValueError, match="do_sample=True"):        # top_k = 5 left behind without sampling
        tr.generate(inputs_embeds=emb)
    tr.generation_config.top_k = 50
    assert tr.generate(inputs_embeds=emb) == "g"


@pytest.mark.parametrize("kw", [dict(do_sample=True, num_beams=2), dict(do_sample=True, temperature=0.0),
                                dict(do_sample=True, temperature=-1.0), dict(do_sample=True, top_k=-1),
                                dict(do_sample=True, top_k=2.5), dict(do_sample=True, top_p=1.5), dict(do_sample=True, top_p=-0.1),
                                dict(do_sample=True, num_return_sequences=0), dict(do_sample=True, num_return_sequences=33),
                                dict(temperature=0.7), dict(top_k=0), dict(top_p=0.9), dict(do_sample="yes"),
                                dict(num_return_sequences=2)])
def test_generate_rejects_bad_sampling_options(kw, monkeypatch):
    from klab_multimodalmodel_b200 import generation
    monkeypatch.setattr(generation, "sample_generate", lambda *a, **k: pytest.fail("must raise before sampling"))
    with pytest.raises(ValueError):
        _tiny().generate(inputs_embeds=torch.zeros(1, 3, 64), **kw)


@pytest.mark.parametrize("emb", [torch.zeros(3, 64), torch.zeros(3, 64, dtype=torch.float16), torch.zeros(3, 32), None])
def test_sample_generate_checks_inputs_before_any_launch(emb):
    from klab_multimodalmodel_b200.generation import sample_generate
    with pytest.raises(ValueError, match="inputs_embeds"):
        sample_generate(_tiny(), emb, 1, 3)


def test_unknown_options_still_name_logits_processors():
    with pytest.raises(ValueError, match="logits processors are not implemented"):
        _tiny().generate(inputs_embeds=torch.zeros(1, 3, 64), do_sample=True, repetition_penalty=1.2)
