"""Generate tests/golden/hf_modules.npz and tests/golden/hf_layout.json from the `transformers` classes the reference
instantiates (Swinv2Model, T5EncoderModel, T5ForConditionalGeneration), so that tests/test_oracle_vs_hf.py and
tests/test_abi_cpu.py check the oracle and the state-dict layout against them without `transformers` installed.

    python tests/golden/make_hf_golden.py          (needs `transformers`; the stored files come from transformers 5.5.0)

Per case of tests/test_oracle_vs_hf.py (weights seed 3, inputs seed 77), under the key prefix "<case>/":
  img_emb / lang_emb        the first 8 channels of the Swin and frozen-T5-encoder outputs, plus a sketch of each whole tensor
  loss                      T5ForConditionalGeneration(inputs_embeds, labels).loss
  grad_names, gnorm, gsketch  L2 norm and sketch of the gradient of every trainable transformer parameter, by name
  generated                 generate(inputs_embeds=...) with all defaults
A sketch is the tensor times a fixed seeded Gaussian matrix [numel, SKETCH_K] / sqrt(SKETCH_K): |sketch(a) - sketch(b)|
estimates |a - b| (Frobenius) to about +-1/sqrt(2 SKETCH_K) relative, so a whole-tensor error bound can be checked against a
few hundred stored numbers instead of the tensor.
"""
import argparse
import json
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.caption_model import seeded_inputs, seeded_state_dicts  # noqa: E402
from tests.golden.make_golden import CASES, EXTRA_CASES, dims_of  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
HF_CASES = ["tiny_a", "tiny_b", "mid"]
SKETCH_K = 64
LAYOUT_T5 = dict(vocab_size=512, d_model=128, d_ff=256, num_layers=2, num_heads=2)
LAYOUT_SWIN = dict(image_size=64, embed_dim=32, depths=(2, 2, 2), num_heads=(1, 2, 4), window_size=4)


def sketch(t: torch.Tensor, key: str) -> np.ndarray:
    g = torch.Generator().manual_seed(zlib.crc32(key.encode()))
    s = torch.randn(t.numel(), SKETCH_K, generator=g, dtype=torch.float64) / SKETCH_K ** 0.5
    return (t.detach().double().flatten() @ s).numpy()


def case_inputs(name):
    """Seeded weights and inputs of one case: -> (case, swin, t5, state dicts, pixel values, source ids, target ids)."""
    case = CASES.get(name) or EXTRA_CASES[name]
    swin, t5 = dims_of(case)
    sds = seeded_state_dicts(t5, swin, t5, seed=3)
    px, src, tgt = seeded_inputs(case["batch"], swin, t5.vocab_size, case["l_src"], case["l_tgt"], ignore_tail=case["ignore_tail"], seed=77)
    return case, swin, t5, sds, px, src, tgt


def summarize(img, lang, loss, grads, generated) -> dict:
    """The stored form of one case's outputs; grads: transformer parameter name -> gradient."""
    names = sorted(grads)
    return {"img_emb": img[:, :, :8].numpy(), "lang_emb": lang[:, :, :8].numpy(),
            "img_sketch": sketch(img, "img_emb").astype(np.float32), "lang_sketch": sketch(lang, "lang_emb").astype(np.float32),
            "loss": np.float64(loss), "generated": generated.numpy(), "grad_names": np.array(names),
            "gnorm": np.array([grads[k].double().norm().item() for k in names]),
            "gsketch": np.stack([sketch(grads[k], k) for k in names]).astype(np.float32)}


def hf_models(swin, t5):
    from transformers import Swinv2Config, Swinv2Model, T5Config, T5EncoderModel, T5ForConditionalGeneration

    def cfg():                   # one config object per model: T5EncoderModel edits the one it is given
        return T5Config(vocab_size=t5.vocab_size, d_model=t5.d_model, d_kv=t5.d_kv, d_ff=t5.d_ff, num_layers=t5.num_layers,
                        num_decoder_layers=t5.n_dec, num_heads=t5.num_heads, decoder_start_token_id=0)
    scfg = Swinv2Config(image_size=swin.image_size, patch_size=swin.patch_size, embed_dim=swin.embed_dim, depths=list(swin.depths),
                        num_heads=list(swin.num_heads), window_size=swin.window_size,
                        pretrained_window_sizes=list(swin.pretrained_window_sizes))
    return T5EncoderModel(cfg()).eval(), Swinv2Model(scfg).eval(), T5ForConditionalGeneration(cfg()).eval()


def hf_case(name) -> dict:
    case, swin, t5, sds, px, src, tgt = case_inputs(name)
    lm, im, tr = hf_models(swin, t5)
    lm.load_state_dict(sds["language_model"], strict=True)
    im.load_state_dict(sds["image_model"], strict=True)
    tr.load_state_dict(sds["transformer"], strict=True)
    with torch.no_grad():
        img = im(pixel_values=px).last_hidden_state
        lang = lm(input_ids=src).last_hidden_state
    emb = torch.cat((img, lang), dim=1)
    loss = tr(inputs_embeds=emb, labels=tgt).loss
    loss.backward()
    with torch.no_grad():
        ids = tr.generate(inputs_embeds=emb)
    return summarize(img, lang, loss.item(), {k: p.grad for k, p in tr.named_parameters()}, ids)


def hf_layout() -> dict:
    """State-dict key -> shape of the two reference classes whose layout the drop-in must carry."""
    import transformers
    t5 = transformers.T5ForConditionalGeneration(transformers.T5Config(d_kv=64, decoder_start_token_id=0, **LAYOUT_T5))
    swin = transformers.Swinv2Model(transformers.Swinv2Config(**dict(LAYOUT_SWIN, depths=list(LAYOUT_SWIN["depths"]),
                                                                      num_heads=list(LAYOUT_SWIN["num_heads"]))))
    return {"t5": {k: list(v.shape) for k, v in t5.state_dict().items()},
            "swin": {k: list(v.shape) for k, v in swin.state_dict().items()}}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    torch.manual_seed(0)
    np.savez_compressed(os.path.join(a.out, "hf_modules.npz"),
                        **{f"{name}/{k}": v for name in HF_CASES for k, v in hf_case(name).items()})
    with open(os.path.join(a.out, "hf_layout.json"), "w") as fh:
        json.dump(hf_layout(), fh, indent=0, sort_keys=True)
