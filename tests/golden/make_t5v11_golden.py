"""Generate tests/golden/hf_t5v11.npz: `transformers` 5.5.0 T5 v1.1 / Flan-T5 models (feed_forward_proj "gated-gelu",
"tie_word_embeddings": false in config.json, so no d_model**-0.5 in front of the LM head) on seeded weights and inputs.

    python tests/golden/make_t5v11_golden.py        (needs `transformers`; the stored file comes from transformers 5.5.0)

Cases (CASES below):
  v11_tied     built from the config, as transformers builds any T5 from a config: lm_head IS shared, no scale.
  v11_untied   loaded with from_pretrained from a checkpoint directory this script writes (write_checkpoint) whose
               lm_head.weight differs from shared.weight: transformers leaves the two untied.  d_model 128 != heads * d_kv 192,
               the shape of flan-t5-small (512 vs 384).
Architectures used by the project (T5Config.NAMED) are checked against transformers' T5Config in the same run (NAMED_V11).

Under "<case>/": loss (T5ForConditionalGeneration(inputs_embeds, labels).loss, eval mode), grad_names / gnorm / gsketch (every
trainable parameter by name, see make_hf_golden.sketch), greedy (generate() defaults), beam_sequences / beam_scores
(num_beams=4, sequences_scores), sample (do_sample=True with SAMPLE_OPTS, torch.multinomial replaced by the project's defined
draw as in make_sample_golden.py).
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.t5v11_oracle import V11Dims, seeded_transformer  # noqa: E402
from tests.golden.make_hf_golden import sketch  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GATED = dict(feed_forward_proj="gated-gelu", scale_decoder_outputs=False)
CASES = {
    "v11_tied": dict(dims=dict(vocab_size=256, d_model=128, d_kv=64, d_ff=192, num_layers=2, num_heads=2, **GATED), untied=False),
    "v11_untied": dict(dims=dict(vocab_size=320, d_model=128, d_kv=64, d_ff=256, num_layers=3, num_heads=3,
                                 **GATED), untied=True),
}
BATCH, L_ENC, L_TGT = 3, 7, 6
NUM_BEAMS = 4
SAMPLE_OPTS = dict(temperature=0.8, top_k=20, top_p=0.9, num_return_sequences=2, seed=11)
# T5Config.NAMED entries of the v1.1 family: vocab 32128, d_kv 64, gated-gelu, tie_word_embeddings False
NAMED_V11 = {
    "small": dict(d_model=512, d_ff=1024, num_layers=8, num_heads=6),
    "base": dict(d_model=768, d_ff=2048, num_layers=12, num_heads=12),
    "large": dict(d_model=1024, d_ff=2816, num_layers=24, num_heads=16),
}


def case_dims(name) -> V11Dims:
    return V11Dims(**CASES[name]["dims"])


def case_state_dict(name) -> dict:
    """Seeded transformer weights (HF's initialiser scales); v11_untied: lm_head.weight has values of its own."""
    dims = case_dims(name)
    return seeded_transformer(dims, 5, style="hf", untied_head=CASES[name]["untied"])


def case_inputs(name):
    """-> (inputs_embeds [B, Le, d] fp32, labels [B, Lt] int64 with EOS last, row 1's tail ignored (-100))."""
    dims = case_dims(name)
    rng = np.random.Generator(np.random.PCG64([21, len(name)]))
    emb = rng.standard_normal(size=(BATCH, L_ENC, dims.d_model), dtype=np.float32)
    lab = rng.integers(2, dims.vocab_size - 28, size=(BATCH, L_TGT), dtype=np.int64)
    lab[:, -1] = dims.eos_token_id
    lab[1, -2:] = -100
    return torch.from_numpy(emb), torch.from_numpy(lab)


def hub_config(name) -> dict:
    """config.json as the published v1.1 checkpoints have it: `"tie_word_embeddings": false`, no scale_decoder_outputs key."""
    d = CASES[name]["dims"]
    return dict(architectures=["T5ForConditionalGeneration"], model_type="t5", vocab_size=d["vocab_size"], d_model=d["d_model"],
                d_kv=d["d_kv"], d_ff=d["d_ff"], num_layers=d["num_layers"], num_decoder_layers=d.get("num_decoder_layers", d["num_layers"]),
                num_heads=d["num_heads"], feed_forward_proj="gated-gelu", tie_word_embeddings=False, dropout_rate=0.1,
                layer_norm_epsilon=1e-6, relative_attention_num_buckets=32, relative_attention_max_distance=128, pad_token_id=0,
                eos_token_id=1, decoder_start_token_id=0)


def write_checkpoint(name, path) -> str:
    """A checkpoint directory (config.json + model.safetensors, tied tensors stored once) of case `name`."""
    from safetensors.torch import save_file
    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, "config.json"), "w") as fh:
        json.dump(hub_config(name), fh, indent=1)
    sd = case_state_dict(name)
    keep = {k: v for k, v in sd.items() if k not in ("encoder.embed_tokens.weight", "decoder.embed_tokens.weight")
            and not (k == "lm_head.weight" and v is sd["shared.weight"])}
    save_file({k: v.contiguous() for k, v in keep.items()}, os.path.join(path, "model.safetensors"))
    return path


def hf_model(name, tmp):
    """transformers' model of the case, built the way a user gets it."""
    import transformers
    if CASES[name]["untied"]:
        tr = transformers.T5ForConditionalGeneration.from_pretrained(write_checkpoint(name, tmp))
        sd = case_state_dict(name)
        assert tr.lm_head.weight is not tr.shared.weight and torch.equal(tr.lm_head.weight, sd["lm_head.weight"])
        assert torch.equal(tr.shared.weight, sd["shared.weight"])
    else:
        cfg = transformers.T5Config(**{k: v for k, v in hub_config(name).items() if k not in ("architectures", "model_type")})
        tr = transformers.T5ForConditionalGeneration(cfg)
        tr.load_state_dict(case_state_dict(name), strict=True)
        assert tr.lm_head.weight is tr.shared.weight
    assert tr.config.scale_decoder_outputs is False and tr.config.is_gated_act and tr.config.dense_act_fn == "gelu_new"
    return tr.eval()


def hf_sample(tr, emb, opts):
    from oracle.t5_sample import inverse_cdf, sample_uniform
    from unittest import mock
    calls = []

    def draw(probs, num_samples=1, **kw):
        c = len(calls)
        calls.append(c)
        u = torch.tensor([sample_uniform(opts["seed"], r, c) for r in range(probs.shape[0])], dtype=torch.float64)
        return inverse_cdf(probs, u)[:, None]

    kw = {k: v for k, v in opts.items() if k != "seed"}
    with mock.patch.object(torch, "multinomial", draw), torch.no_grad():
        return tr.generate(inputs_embeds=emb, do_sample=True, **kw)


def check_named():
    """The v1.1 architectures of T5Config.NAMED, through transformers' own config class."""
    import transformers
    for size, arch in NAMED_V11.items():
        c = transformers.T5Config(vocab_size=32128, d_kv=64, feed_forward_proj="gated-gelu", tie_word_embeddings=False, **arch)
        assert c.num_decoder_layers == arch["num_layers"] and c.is_gated_act and not c.scale_decoder_outputs
        print(f"{size}: inner {c.num_heads * c.d_kv} vs d_model {c.d_model}")


def hf_case(name, tmp) -> dict:
    tr = hf_model(name, tmp)
    emb, lab = case_inputs(name)
    loss = tr(inputs_embeds=emb, labels=lab).loss
    loss.backward()
    grads = {k: p.grad for k, p in tr.named_parameters()}
    names = sorted(grads)
    with torch.no_grad():
        greedy = tr.generate(inputs_embeds=emb)
        beam = tr.generate(inputs_embeds=emb, num_beams=NUM_BEAMS, return_dict_in_generate=True, output_scores=True)
    sample = hf_sample(tr, emb, SAMPLE_OPTS)
    print(f"{name}: loss {loss.item():.6f}, greedy {tuple(greedy.shape)}, beam {tuple(beam.sequences.shape)}, sample {tuple(sample.shape)}, "
          f"params {names}")
    return {"loss": np.float64(loss.item()), "grad_names": np.array(names),
            "gnorm": np.array([grads[k].double().norm().item() for k in names]),
            "gsketch": np.stack([sketch(grads[k], k) for k in names]).astype(np.float32),
            "greedy": greedy.numpy(), "beam_sequences": beam.sequences.numpy(), "beam_scores": beam.sequences_scores.numpy(),
            "sample": sample.numpy()}


if __name__ == "__main__":
    import tempfile
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    torch.manual_seed(0)
    check_named()
    with tempfile.TemporaryDirectory() as tmp:
        stored = {f"{name}/{k}": v for name in CASES for k, v in hf_case(name, os.path.join(tmp, name)).items()}
    np.savez_compressed(os.path.join(a.out, "hf_t5v11.npz"), **stored)
