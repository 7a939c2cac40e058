"""The T5 transformer in TRAINING mode, restated in plain torch with every dropout replaced by a given mask.

TEST INFRASTRUCTURE ONLY.  The arithmetic is that of oracle/t5.py (the gated feed-forward and the optional LM-head scale of
tests/t5v11_oracle.py); what is added is a hook `mask(site, shape)` at each of transformers' dropout sites
(HF/models/t5/modeling_t5.py, HF/ = site-packages/transformers 5.5.0).  It returns the multiplier tensor of that site (0 or the
kept scale) or None for "no dropout".  Sites are tuples:

    (stack, None, "input")          :734   dropout of the stack input (inputs_embeds, or the decoder's embedded labels)
    (stack, i, "self_probs")        :332   attention probabilities of block i's self-attention   [B, H, Lq, Lk]
    (stack, i, "self_out")          :375   output of block i's self-attention sub-layer          [B, L, d]
    (stack, i, "cross_probs")       :332   attention probabilities of the cross-attention        [B, H, Lq, Lk]
    (stack, i, "cross_out")         :406   output of the cross-attention sub-layer               [B, L, d]
    (stack, i, "ff_inner")          :95 / gated :119   hidden layer of the feed-forward           [B, L, d_ff]
    (stack, i, "ff_out")            :149   output of the feed-forward sub-layer                  [B, L, d]
    (stack, None, "final")          :768   after the final RMSNorm

with stack "encoder" or "decoder".  With every mask None (or all ones) the functions compute exactly what oracle/t5.py and
tests/t5v11_oracle.py compute."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.swinv2 import swinv2_forward
from oracle.t5 import rms_norm, shift_right, t5_bias
from tests.t5v11_oracle import gelu_new

SITES = ("input", "self_probs", "self_out", "cross_probs", "cross_out", "ff_inner", "ff_out", "final")


def no_mask(site, shape):
    return None


def _drop(x, mask, site):
    m = mask(site, tuple(x.shape))
    return x if m is None else x * m.to(x.dtype)


def attention(x, kv_src, sd, prefix, dims, bias, causal, mask, site):
    """oracle/t5.py:t5_attention with the probability dropout (:332) between the softmax and the product with V."""
    b, lq, _ = x.shape
    lk = kv_src.shape[1]
    h, dk = dims.num_heads, dims.d_kv
    q = (x @ sd[prefix + "q.weight"].T).view(b, lq, h, dk).transpose(1, 2)
    k = (kv_src @ sd[prefix + "k.weight"].T).view(b, lk, h, dk).transpose(1, 2)
    v = (kv_src @ sd[prefix + "v.weight"].T).view(b, lk, h, dk).transpose(1, 2)
    s = q @ k.transpose(-1, -2)
    if bias is not None:
        s = s + bias[None]
    if causal:
        qi = torch.arange(lq)[:, None] + (lk - lq)
        ki = torch.arange(lk)[None, :]
        s = s + torch.where(ki > qi, torch.finfo(s.dtype).min, 0.0)
    p = torch.softmax(s.float(), dim=-1).to(s.dtype)
    p = _drop(p, mask, site)
    o = (p @ v).transpose(1, 2).reshape(b, lq, h * dk)
    return o @ sd[prefix + "o.weight"].T


def ff(x, sd, prefix, dims, mask, stack, i):
    """T5LayerFF: ReLU (T5DenseActDense :92-103) or gated-gelu (T5DenseGatedActDense :106-132), dropout of the hidden layer
    (:95 / :119) and of the sub-layer output (:149)."""
    n = rms_norm(x, sd[prefix + "layer_norm.weight"], dims.eps)
    if getattr(dims, "feed_forward_proj", "relu") == "gated-gelu":
        hdn = gelu_new(n @ sd[prefix + "DenseReluDense.wi_0.weight"].T) * (n @ sd[prefix + "DenseReluDense.wi_1.weight"].T)
    else:
        hdn = torch.relu(n @ sd[prefix + "DenseReluDense.wi.weight"].T)
    hdn = _drop(hdn, mask, (stack, i, "ff_inner"))
    return x + _drop(hdn @ sd[prefix + "DenseReluDense.wo.weight"].T, mask, (stack, i, "ff_out"))


def stack(x, sd, prefix, dims, enc_out=None, mask=no_mask):
    """T5Stack.forward (:637-792) in training mode: oracle/t5.py:t5_stack plus the eight dropout sites."""
    is_dec = enc_out is not None
    name = "decoder" if is_dec else "encoder"
    n_layers = dims.n_dec if is_dec else dims.num_layers
    l = x.shape[1]
    table = sd[f"{prefix}block.0.layer.0.SelfAttention.relative_attention_bias.weight"]
    bias = t5_bias(table, l, l, bidirectional=not is_dec, dims=dims)
    x = _drop(x, mask, (name, None, "input"))
    for i in range(n_layers):
        p = f"{prefix}block.{i}.layer."
        n = rms_norm(x, sd[p + "0.layer_norm.weight"], dims.eps)
        x = x + _drop(attention(n, n, sd, p + "0.SelfAttention.", dims, bias, is_dec, mask, (name, i, "self_probs")), mask,
                      (name, i, "self_out"))
        if is_dec:
            n = rms_norm(x, sd[p + "1.layer_norm.weight"], dims.eps)
            x = x + _drop(attention(n, enc_out, sd, p + "1.EncDecAttention.", dims, None, False, mask, (name, i, "cross_probs")),
                          mask, (name, i, "cross_out"))
            x = ff(x, sd, p + "2.", dims, mask, name, i)
        else:
            x = ff(x, sd, p + "1.", dims, mask, name, i)
    return _drop(rms_norm(x, sd[f"{prefix}final_layer_norm.weight"], dims.eps), mask, (name, None, "final"))


def lm_loss(enc_in, labels, sd, dims, mask=no_mask):
    """T5ForConditionalGeneration.forward(inputs_embeds, labels).loss in training mode (:1070-1117)."""
    enc = stack(enc_in, sd, "encoder.", dims, mask=mask)
    dec = stack(F.embedding(shift_right(labels, dims), sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc, mask=mask)
    if getattr(dims, "scale_decoder_outputs", True):
        dec = dec * dims.d_model ** -0.5
    logits = dec @ sd["lm_head.weight"].T
    return F.cross_entropy(logits.view(-1, logits.shape[-1]), labels.reshape(-1), ignore_index=-100)


def caption_loss(pixel_values, src_ids, tgt_ids, sds, lm, swin, tr, mask=no_mask):
    """models/model.py:20-26 with the transformer in training mode; the text tower and Swin stay in eval mode (as train.py
    runs them), so only the transformer's dropout sites are masked."""
    with torch.no_grad():
        lm_sd = sds["language_model"]
        lang = stack(F.embedding(src_ids, lm_sd["shared.weight"]), lm_sd, "encoder.", lm)
    img = swinv2_forward(pixel_values, sds["image_model"], swin)
    return lm_loss(torch.cat((img, lang), dim=1), tgt_ids, sds["transformer"], tr, mask)
