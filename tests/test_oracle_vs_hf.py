"""The oracle against the real `transformers` classes the reference instantiates (its models/model.py:14-17), module by
module: Swinv2Model, T5EncoderModel, T5ForConditionalGeneration (loss, gradients, greedy generate).  CPU only.
Always against their stored outputs (tests/golden/hf_modules.npz, made by tests/golden/make_hf_golden.py with transformers
5.5.0); where `transformers` imports, also against the installed classes themselves (it is the un-vendored dependency that
holds the reference's arithmetic, SURVEY.md 8c).  Together with tests/test_oracle_golden.py (outputs of the unmodified
reference MyModel) this pins the oracle."""
import os

import numpy as np
import pytest
import torch

from oracle.swinv2 import swinv2_forward
from oracle.t5 import t5_greedy_decode, t5_lm_loss, t5_stack
from tests.golden.make_hf_golden import HF_CASES, case_inputs, hf_models, sketch

GOLD = os.path.join(os.path.dirname(__file__), "golden", "hf_modules.npz")


def _leaf_copies(sd):
    """The state dict with every tensor replaced by a fresh leaf that requires grad (tied tensors share one leaf)."""
    osd, uniq = dict(sd), {}
    for k, v in osd.items():
        if id(v) not in uniq:
            uniq[id(v)] = v.clone().requires_grad_(True)
        osd[k] = uniq[id(v)]
    return osd


def _check_against_stored(name):
    case, swin, t5, sds, px, src, tgt = case_inputs(name)
    gold = np.load(GOLD)

    def ref(key):
        return gold[f"{name}/{key}"]

    def close_by_sketch(t, key, stored, rel, what):
        """|t - stored tensor| (Frobenius, estimated through the sketch) within rel of the stored tensor's norm."""
        s = sketch(t, key)
        assert np.linalg.norm(s - stored) <= rel * np.linalg.norm(stored) + 1e-9, what

    with torch.no_grad():
        img = swinv2_forward(px, sds["image_model"], swin)
        lang = t5_stack(torch.nn.functional.embedding(src, sds["language_model"]["shared.weight"]), sds["language_model"], "encoder.", t5)
    np.testing.assert_allclose(img[:, :, :8].numpy(), ref("img_emb"), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(lang[:, :, :8].numpy(), ref("lang_emb"), rtol=1e-4, atol=1e-5)
    close_by_sketch(img, "img_emb", ref("img_sketch").astype(np.float64), 1e-4, "Swinv2Model output")
    close_by_sketch(lang, "lang_emb", ref("lang_sketch").astype(np.float64), 1e-4, "T5EncoderModel output")
    emb = torch.cat((img, lang), dim=1)
    osd = _leaf_copies(sds["transformer"])
    loss = t5_lm_loss(emb, tgt, osd, t5)
    loss.backward()
    gold_loss = float(ref("loss"))
    assert abs(loss.item() - gold_loss) <= 2e-5 * abs(gold_loss)
    names = [str(k) for k in ref("grad_names")]
    assert len(names) >= 20 and set(names) <= set(osd)
    for k, gn, gs in zip(names, ref("gnorm"), ref("gsketch")):
        g = osd[k].grad
        assert abs(g.double().norm().item() - gn) <= 1e-4 * gn + 1e-9, k
        close_by_sketch(g, k, gs.astype(np.float64), 1e-4, k)
    with torch.no_grad():
        got_ids = t5_greedy_decode(emb, sds["transformer"], t5, 20)
    gen = ref("generated")
    n = got_ids.shape[1]
    assert np.array_equal(got_ids.numpy(), gen[:, :n]) and (gen[:, n:] == 0).all()


def _check_against_installed(name):
    case, swin, t5, sds, px, src, tgt = case_inputs(name)
    lm, im, tr = hf_models(swin, t5)
    lm.load_state_dict(sds["language_model"], strict=True)
    im.load_state_dict(sds["image_model"], strict=True)
    tr.load_state_dict(sds["transformer"], strict=True)
    with torch.no_grad():
        # Swinv2Model.forward (HF/models/swinv2/modeling_swinv2.py:933-987)
        ref_img = im(pixel_values=px).last_hidden_state
        got_img = swinv2_forward(px, sds["image_model"], swin)
        torch.testing.assert_close(got_img, ref_img, rtol=1e-4, atol=1e-5)
        # T5EncoderModel.forward (HF/models/t5/modeling_t5.py:1164-1208)
        ref_lang = lm(input_ids=src).last_hidden_state
        got_lang = t5_stack(torch.nn.functional.embedding(src, sds["language_model"]["shared.weight"]), sds["language_model"], "encoder.", t5)
        torch.testing.assert_close(got_lang, ref_lang, rtol=1e-4, atol=1e-5)
    # T5ForConditionalGeneration(inputs_embeds, labels).loss + gradients (HF/models/t5/modeling_t5.py:992-1133)
    emb = torch.cat((ref_img, ref_lang), dim=1)
    ref_loss = tr(inputs_embeds=emb, labels=tgt).loss
    ref_loss.backward()
    osd = _leaf_copies(sds["transformer"])
    got_loss = t5_lm_loss(emb, tgt, osd, t5)
    got_loss.backward()
    assert abs(got_loss.item() - ref_loss.item()) <= 2e-5 * abs(ref_loss.item())
    checked = 0
    for k, p in tr.named_parameters():
        g, r = osd[k].grad, p.grad
        assert (g - r).norm().item() <= 1e-4 * r.norm().item() + 1e-9, k
        checked += 1
    assert checked >= 20
    # greedy generate (HF/generation/utils.py:2658-2800)
    with torch.no_grad():
        ref_ids = tr.generate(inputs_embeds=emb)                    # the reference's call, all defaults (models/model.py:28)
        got_ids = t5_greedy_decode(emb, sds["transformer"], t5, 20)
    n = got_ids.shape[1]
    assert torch.equal(got_ids, ref_ids[:, :n]) and (ref_ids[:, n:] == 0).all()


@pytest.mark.parametrize("name", HF_CASES)
def test_oracle_modules_match_transformers(name):
    _check_against_stored(name)
    try:
        import transformers  # noqa: F401
    except ImportError:
        return
    _check_against_installed(name)
