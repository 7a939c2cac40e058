"""T5 v1.1 / Flan-T5 on the host: the oracle against transformers 5.5.0's stored outputs (tests/golden/hf_t5v11.npz, written by
tests/golden/make_t5v11_golden.py) and live where transformers imports, and the parts of the CUDA build that need no GPU: config
parsing, the gated state-dict layout, tying / untying of the LM head by from_pretrained, save -> load of an untied model."""
import json
import os
import types

import numpy as np
import pytest
import torch

from tests.t5v11_oracle import V11Dims, beam_search, greedy_decode, lm_loss, param_shapes, sample
from tests.golden import make_t5v11_golden as G
from tests.golden.make_hf_golden import sketch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "hf_t5v11.npz"))


def _leaves(sd):
    """The state dict with one grad-requiring leaf per distinct tensor (tied keys keep sharing it)."""
    leaf = {}
    return {k: leaf.setdefault(id(v), v.clone().requires_grad_(True)) for k, v in sd.items()}


def oracle_loss_and_grads(name):
    dims = G.case_dims(name)
    sd = _leaves(G.case_state_dict(name))
    emb, lab = G.case_inputs(name)
    loss = lm_loss(emb, lab, sd, dims)
    loss.backward()
    return loss.item(), sd


@pytest.mark.parametrize("name", list(G.CASES))
def test_oracle_reproduces_golden_loss_and_gradients(name):
    loss, sd = oracle_loss_and_grads(name)
    assert loss == pytest.approx(float(GOLD[f"{name}/loss"]), rel=1e-5)
    names = list(GOLD[f"{name}/grad_names"])
    assert ("lm_head.weight" in names) == G.CASES[name]["untied"]
    for i, k in enumerate(names):
        g = sd[k].grad
        ref_norm = float(GOLD[f"{name}/gnorm"][i])
        assert g.double().norm().item() == pytest.approx(ref_norm, rel=1e-5), k
        err = np.linalg.norm(sketch(g, k) - GOLD[f"{name}/gsketch"][i].astype(np.float64))
        assert err <= 1e-5 * ref_norm + 1e-7, (k, err, ref_norm)
    if G.CASES[name]["untied"]:                                       # the head's gradient is not the embedding's
        assert not torch.allclose(sd["lm_head.weight"].grad, sd["shared.weight"].grad)


@pytest.mark.parametrize("name", list(G.CASES))
def test_oracle_reproduces_golden_ids(name):
    dims = G.case_dims(name)
    sd = G.case_state_dict(name)
    emb, _ = G.case_inputs(name)
    with torch.no_grad():
        assert torch.equal(greedy_decode(emb, sd, dims), torch.from_numpy(GOLD[f"{name}/greedy"]))
        seqs, scores = beam_search(emb, sd, dims, G.NUM_BEAMS)
        assert torch.equal(seqs, torch.from_numpy(GOLD[f"{name}/beam_sequences"]))
        assert torch.allclose(scores, torch.from_numpy(GOLD[f"{name}/beam_scores"]), rtol=1e-5, atol=1e-6)
        o = G.SAMPLE_OPTS
        ids = sample(emb, sd, dims, o["seed"], o["temperature"], o["top_k"], o["top_p"], o["num_return_sequences"])
        assert torch.equal(ids, torch.from_numpy(GOLD[f"{name}/sample"]))


@pytest.mark.parametrize("name", list(G.CASES))
def test_oracle_matches_live_transformers(name, tmp_path):
    pytest.importorskip("transformers")
    tr = G.hf_model(name, str(tmp_path / name))
    emb, lab = G.case_inputs(name)
    dims = G.case_dims(name)
    sd = G.case_state_dict(name)
    with torch.no_grad():
        assert tr(inputs_embeds=emb, labels=lab).loss.item() == pytest.approx(lm_loss(emb, lab, sd, dims).item(), rel=1e-5)
        assert torch.equal(tr.generate(inputs_embeds=emb), greedy_decode(emb, sd, dims))


def test_config_parses_flan_t5_large_and_rejects_unsupported_activations(tmp_path):
    from klab_multimodalmodel_b200.modeling import T5Config, _config_from_source
    raw = dict(G.hub_config("v11_untied"), d_model=1024, d_ff=2816, num_layers=24, num_decoder_layers=24, num_heads=16, vocab_size=32128,
               n_positions=512, output_past=True, is_encoder_decoder=True)
    (tmp_path / "config.json").write_text(json.dumps(raw))
    cfg, path = _config_from_source(T5Config, str(tmp_path))
    assert path == str(tmp_path)
    assert (cfg.d_model, cfg.d_ff, cfg.num_layers, cfg.n_dec, cfg.num_heads, cfg.vocab_size) == (1024, 2816, 24, 24, 16, 32128)
    assert cfg.gated and cfg.tie_word_embeddings is False and cfg.scale_decoder_outputs is False and cfg.lm_head_scale == 1.0
    assert cfg == T5Config(**T5Config.NAMED["google/flan-t5-large"], num_decoder_layers=24)
    # transformers' own save_pretrained stores tie_word_embeddings true with the derived scale_decoder_outputs false
    raw.update(tie_word_embeddings=True, scale_decoder_outputs=False)
    (tmp_path / "config.json").write_text(json.dumps(raw))
    assert _config_from_source(T5Config, str(tmp_path))[0].scale_decoder_outputs is False
    assert T5Config().scale_decoder_outputs is True and T5Config().lm_head_scale == 512 ** -0.5
    for bad in ("gelu", "gated-silu", "gated-relu", "silu"):
        with pytest.raises(ValueError, match="relu, gated-gelu"):
            T5Config(feed_forward_proj=bad)
    for size, arch in G.NAMED_V11.items():
        for fam in ("flan-t5", "t5-v1_1"):
            cfg = T5Config(**T5Config.NAMED[f"google/{fam}-{size}"])
            got = dict(d_model=cfg.d_model, d_ff=cfg.d_ff, num_layers=cfg.num_layers, num_heads=cfg.num_heads)
            assert got == arch and cfg.n_dec == arch["num_layers"] and cfg.d_kv == 64 and cfg.vocab_size == 32128
            assert cfg.gated and not cfg.scale_decoder_outputs


def test_gated_state_dict_keys_equal_transformers_keys():
    from klab_multimodalmodel_b200.modeling import T5Config, T5EncoderModel, T5ForConditionalGeneration
    kw = dict(G.CASES["v11_untied"]["dims"])
    ours_cfg = T5Config(**kw)
    dims = V11Dims(**kw)
    for cls, enc_only in ((T5ForConditionalGeneration, False), (T5EncoderModel, True)):
        sd = cls(ours_cfg).state_dict()
        ref = param_shapes(dims, encoder_only=enc_only)
        assert set(sd) == set(ref) and all(tuple(sd[k].shape) == tuple(ref[k]) for k in ref)
        assert any(k.endswith("DenseReluDense.wi_0.weight") for k in sd) and not any(k.endswith("DenseReluDense.wi.weight") for k in sd)
    try:
        import transformers
    except ImportError:
        return
    hf = transformers.T5ForConditionalGeneration(transformers.T5Config(
        **{k: v for k, v in G.hub_config("v11_untied").items() if k not in ("architectures", "model_type")}))
    ours = T5ForConditionalGeneration(ours_cfg)
    assert set(hf.state_dict()) == set(ours.state_dict())
    ours.load_state_dict(hf.state_dict(), strict=True)


def test_init_matches_transformers_scales():
    from klab_multimodalmodel_b200.modeling import T5Config, T5ForConditionalGeneration
    cfg = T5Config(vocab_size=64, d_model=256, d_kv=64, d_ff=1024, num_layers=1, num_heads=4, feed_forward_proj="gated-gelu",
                   tie_word_embeddings=False)
    m = T5ForConditionalGeneration(cfg)
    ff = m.encoder.block[0].layer[1].DenseReluDense
    for w, std in ((ff.wi_0.weight, 256 ** -0.5), (ff.wi_1.weight, 256 ** -0.5), (ff.wo.weight, 1024 ** -0.5)):
        assert w.std().item() == pytest.approx(std, rel=0.05)
    assert m.lm_head_tied                                          # a model built from a config is tied, as in transformers


def test_from_pretrained_ties_or_unties_like_transformers(tmp_path):
    from safetensors.torch import load_file, save_file

    from klab_multimodalmodel_b200.modeling import T5ForConditionalGeneration
    path = G.write_checkpoint("v11_untied", str(tmp_path / "untied"))
    m = T5ForConditionalGeneration.from_pretrained(path)
    sd = G.case_state_dict("v11_untied")
    assert not m.lm_head_tied and m.decoder.embed_tokens.weight is m.shared.weight
    assert torch.equal(m.lm_head.weight, sd["lm_head.weight"]) and torch.equal(m.shared.weight, sd["shared.weight"])
    assert any(p is m.lm_head.weight for p in m.parameters())
    out = m.state_dict()
    assert set(out) == set(param_shapes(G.case_dims("v11_untied")))
    assert torch.equal(out["lm_head.weight"], sd["lm_head.weight"]) and torch.equal(out["encoder.embed_tokens.weight"], sd["shared.weight"])
    # the same file with lm_head.weight equal to shared.weight, and without lm_head.weight: tied
    tensors = load_file(os.path.join(path, "model.safetensors"))
    for variant, head in (("equal", tensors["shared.weight"].clone()), ("absent", None)):
        d = tmp_path / variant
        d.mkdir()
        (d / "config.json").write_text(open(os.path.join(path, "config.json")).read())
        t = {k: v for k, v in tensors.items() if k != "lm_head.weight"}
        if head is not None:
            t["lm_head.weight"] = head
        save_file(t, str(d / "model.safetensors"))
        m2 = T5ForConditionalGeneration.from_pretrained(str(d))
        assert m2.lm_head_tied and torch.equal(m2.lm_head.weight, sd["shared.weight"])


def test_save_load_round_trips_an_untied_model(tmp_path):
    from klab_multimodalmodel_b200.modeling import Swinv2Config, T5Config
    from klab_multimodalmodel_b200.models.model import MyModel
    path = G.write_checkpoint("v11_untied", str(tmp_path / "ckpt"))
    scfg = Swinv2Config(image_size=32, embed_dim=32, depths=(1, 1, 1), num_heads=(1, 2, 4), window_size=4, pretrained_window_sizes=(0, 0, 0))
    args = types.SimpleNamespace(result_dir=str(tmp_path), language_model_name=T5Config(**G.CASES["v11_untied"]["dims"]),
                                 image_model_name=scfg, image_model_train=False, transformer_model_name=path)
    a = MyModel(args)
    assert not a.transformer.lm_head_tied
    a.save("best.pth")
    a.save_state("last.pth", step=3)
    args_b = types.SimpleNamespace(**dict(vars(args), transformer_model_name=T5Config(**G.CASES["v11_untied"]["dims"])))
    for load in ("load", "load_state"):
        b = MyModel(args_b)                                      # built from the config: tied until the untied file is loaded
        assert b.transformer.lm_head_tied
        getattr(b, load)("best.pth" if load == "load" else "last.pth")
        assert not b.transformer.lm_head_tied
        sa, sb = a.transformer.state_dict(), b.transformer.state_dict()
        assert set(sa) == set(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
