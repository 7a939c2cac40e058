"""Generate tests/golden/hf_masked.npz: `transformers` 5.5.0 T5ForConditionalGeneration in TRAINING mode with every dropout
replaced by a fixed, seeded mask (random_mask below), so that the masked restatement tests/masked_oracle.py can be compared
with it exactly.

    python tests/golden/make_masked_golden.py        (needs `transformers`; the stored file comes from transformers 5.5.0)

Each dropout call of the model is attributed to its site (tests/masked_oracle.py lists them):
  nn.Dropout modules     T5Stack.dropout (first call of a forward: "input" :734, second: "final" :768),
                         T5LayerSelfAttention / T5LayerCrossAttention .dropout ("self_out" :375 / "cross_out" :406),
                         T5LayerFF.dropout ("ff_out" :149), T5DenseActDense / T5DenseGatedActDense .dropout ("ff_inner" :95 / :119);
  functional dropout     of T5Attention's probabilities (:332), attributed by wrapping each T5Attention.forward.
Cases: "relu" (the original T5: ReLU feed-forward, scaled tied LM head) and "gated" (T5 v1.1: gated-gelu, no scale).
Under "<case>/": loss, grad_names, gnorm, gsketch (see make_hf_golden.sketch), sites (every site called, in call order).
"""
import argparse
import contextlib
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.golden.make_hf_golden import sketch  # noqa: E402
from tests.t5v11_oracle import V11Dims, seeded_transformer  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
P = 0.1
CASES = {
    "relu": dict(vocab_size=256, d_model=64, d_kv=32, d_ff=96, num_layers=2, num_heads=2, feed_forward_proj="relu",
                 scale_decoder_outputs=True),
    "gated": dict(vocab_size=256, d_model=64, d_kv=32, d_ff=96, num_layers=2, num_decoder_layers=3, num_heads=3,
                  feed_forward_proj="gated-gelu", scale_decoder_outputs=False),
}
BATCH, L_ENC, L_TGT = 3, 7, 6


def case_dims(name) -> V11Dims:
    return V11Dims(**CASES[name])


def case_state_dict(name) -> dict:
    return seeded_transformer(case_dims(name), 9, style="hf")


def case_inputs(name):
    """-> (inputs_embeds [B, Le, d] fp32, labels [B, Lt] int64 with EOS last, row 1's tail ignored (-100))."""
    dims = case_dims(name)
    rng = np.random.Generator(np.random.PCG64([31, len(name)]))
    emb = rng.standard_normal(size=(BATCH, L_ENC, dims.d_model), dtype=np.float32)
    lab = rng.integers(2, dims.vocab_size - 28, size=(BATCH, L_TGT), dtype=np.int64)
    lab[:, -1] = dims.eos_token_id
    lab[1, -2:] = -100
    return torch.from_numpy(emb), torch.from_numpy(lab)


def random_mask(site, shape):
    """A fixed inverted-dropout mask per site: keep with probability 1 - P, survivors scaled by 1 / (1 - P)."""
    g = torch.Generator().manual_seed(zlib.crc32(repr(site).encode()))
    return (torch.rand(shape, generator=g) >= P).float() / (1.0 - P)


def hf_model(name):
    import transformers
    d = CASES[name]
    cfg = transformers.T5Config(vocab_size=d["vocab_size"], d_model=d["d_model"], d_kv=d["d_kv"], d_ff=d["d_ff"],
                                num_layers=d["num_layers"], num_decoder_layers=d.get("num_decoder_layers", d["num_layers"]),
                                num_heads=d["num_heads"], feed_forward_proj=d["feed_forward_proj"], dropout_rate=P,
                                tie_word_embeddings=d["scale_decoder_outputs"], decoder_start_token_id=0)
    tr = transformers.T5ForConditionalGeneration(cfg)
    tr.load_state_dict(case_state_dict(name), strict=True)
    assert tr.config.scale_decoder_outputs == d["scale_decoder_outputs"] and tr.lm_head.weight is tr.shared.weight
    return tr.train()


class _SiteDropout(torch.nn.Module):
    """Stands in for an nn.Dropout: multiplies by the site's mask (the stack's own dropout serves two sites in turn)."""

    def __init__(self, sites, mask, log):
        super().__init__()
        self.sites, self.mask, self.log, self.calls = sites, mask, log, 0

    def forward(self, x):
        site = self.sites[self.calls % len(self.sites)]
        self.calls += 1
        self.log.append(site)
        return x * self.mask(site, tuple(x.shape))


@contextlib.contextmanager
def masked(tr, mask):
    """Every dropout of `tr` (train mode) multiplies by mask(site, shape); yields the list of sites called, in order."""
    log, current, saved = [], [None], []
    functional = torch.nn.functional.dropout

    def prob_dropout(x, p=0.5, training=True, inplace=False):
        assert current[0] is not None and training and p == P, "a functional dropout outside the attention probabilities"
        log.append(current[0])
        return x * mask(current[0], tuple(x.shape))

    def wrap(attn, site):
        fwd = attn.forward

        def forward(*a, **kw):
            current[0] = site
            try:
                return fwd(*a, **kw)
            finally:
                current[0] = None
        saved.append((attn, fwd))
        attn.forward = forward

    def swap(mod, attr, sites):
        saved.append((mod, attr, getattr(mod, attr)))
        setattr(mod, attr, _SiteDropout(sites, mask, log))

    for name, st in (("encoder", tr.encoder), ("decoder", tr.decoder)):
        swap(st, "dropout", [(name, None, "input"), (name, None, "final")])
        for i, blk in enumerate(st.block):
            wrap(blk.layer[0].SelfAttention, (name, i, "self_probs"))
            swap(blk.layer[0], "dropout", [(name, i, "self_out")])
            if st.is_decoder:
                wrap(blk.layer[1].EncDecAttention, (name, i, "cross_probs"))
                swap(blk.layer[1], "dropout", [(name, i, "cross_out")])
            swap(blk.layer[-1], "dropout", [(name, i, "ff_out")])
            swap(blk.layer[-1].DenseReluDense, "dropout", [(name, i, "ff_inner")])
    torch.nn.functional.dropout = prob_dropout
    try:
        yield log
    finally:
        torch.nn.functional.dropout = functional
        for s in reversed(saved):
            if len(s) == 2:
                s[0].forward = s[1]
            else:
                setattr(*s)


def hf_case(name, mask=random_mask) -> dict:
    tr = hf_model(name)
    emb, lab = case_inputs(name)
    with masked(tr, mask) as log:
        loss = tr(inputs_embeds=emb, labels=lab).loss
    loss.backward()
    grads = {k: p.grad for k, p in tr.named_parameters()}
    names = sorted(grads)
    return {"loss": np.float64(loss.item()), "grad_names": np.array(names),
            "gnorm": np.array([grads[k].double().norm().item() for k in names]),
            "gsketch": np.stack([sketch(grads[k], k) for k in names]).astype(np.float32),
            "sites": np.array([repr(s) for s in log])}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    torch.manual_seed(0)
    stored = {}
    for name in CASES:
        out = hf_case(name)
        print(f"{name}: loss {out['loss']:.6f}, {len(out['sites'])} dropout calls, {len(out['grad_names'])} gradients")
        stored.update({f"{name}/{k}": v for k, v in out.items()})
    np.savez_compressed(os.path.join(a.out, "hf_masked.npz"), **stored)
