"""Oracle for T5 v1.1 / Flan-T5, restated in plain torch fp32: the gated-GELU feed-forward (T5DenseGatedActDense,
HF/models/t5/modeling_t5.py:106-132) and the LM head without the d_model**-0.5 scale when the config says
`scale_decoder_outputs` False (configuration_t5.py:79-83, modeling_t5.py:1105-1110).  HF/ = site-packages/transformers (5.5.0).

TEST INFRASTRUCTURE ONLY.  It builds on the original-T5 oracle (oracle/t5.py, oracle/t5_beam.py, oracle/t5_sample.py,
oracle/caption_model.py): attention, norms, position buckets, the beam-search and sampling state machines and the seeded weights
are reused as they are; only the feed-forward, the LM head and the loops that call them are restated here.  With
feed_forward_proj "relu" and scale_decoder_outputs True every function below computes what its oracle/ counterpart does.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F

from oracle.caption_model import _seeded_tensor, seeded_state_dict, swin_param_shapes, t5_param_shapes
from oracle.swinv2 import SwinDims, swinv2_forward
from oracle.t5 import T5Dims, rms_norm, shift_right, t5_attention, t5_bias
from oracle.t5_beam import beam_init, beam_output, beam_step
from oracle.t5_sample import inverse_cdf, sample_uniform, warp


@dataclass
class V11Dims(T5Dims):
    """T5Dims plus the two config fields that make a T5 v1.1 / Flan-T5 model."""
    feed_forward_proj: str = "gated-gelu"      # or "relu"
    scale_decoder_outputs: bool = False        # True for the original T5


def gelu_new(x: torch.Tensor) -> torch.Tensor:
    """NewGELUActivation, HF/activations.py: the tanh form (not the erf GELU of Swin)."""
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * torch.pow(x, 3.0))))


def ff(x, sd, prefix, dims: V11Dims):
    """T5LayerFF with T5DenseGatedActDense (gated-gelu): gelu_new(n wi_0^T) * (n wi_1^T), or T5DenseActDense (relu).  No biases."""
    n = rms_norm(x, sd[prefix + "layer_norm.weight"], dims.eps)
    if dims.feed_forward_proj == "gated-gelu":
        hdn = gelu_new(n @ sd[prefix + "DenseReluDense.wi_0.weight"].T) * (n @ sd[prefix + "DenseReluDense.wi_1.weight"].T)
    else:
        hdn = torch.relu(n @ sd[prefix + "DenseReluDense.wi.weight"].T)
    return x + hdn @ sd[prefix + "DenseReluDense.wo.weight"].T


def stack(x: torch.Tensor, sd: dict, prefix: str, dims: V11Dims, enc_out: torch.Tensor | None = None) -> torch.Tensor:
    """T5Stack.forward in eval mode (oracle/t5.py:t5_stack with `ff` as the feed-forward)."""
    is_dec = enc_out is not None
    n_layers = dims.n_dec if is_dec else dims.num_layers
    l = x.shape[1]
    table = sd[f"{prefix}block.0.layer.0.SelfAttention.relative_attention_bias.weight"]
    bias = t5_bias(table, l, l, bidirectional=not is_dec, dims=dims)
    for i in range(n_layers):
        p = f"{prefix}block.{i}.layer."
        n = rms_norm(x, sd[p + "0.layer_norm.weight"], dims.eps)
        x = x + t5_attention(n, n, sd, p + "0.SelfAttention.", dims, bias, causal=is_dec)
        if is_dec:
            n = rms_norm(x, sd[p + "1.layer_norm.weight"], dims.eps)
            x = x + t5_attention(n, enc_out, sd, p + "1.EncDecAttention.", dims, None, causal=False)
            x = ff(x, sd, p + "2.", dims)
        else:
            x = ff(x, sd, p + "1.", dims)
    return rms_norm(x, sd[f"{prefix}final_layer_norm.weight"], dims.eps)


def lm_logits(dec: torch.Tensor, sd: dict, dims: V11Dims) -> torch.Tensor:
    """HF/models/t5/modeling_t5.py:1105-1110: * d_model**-0.5 only if scale_decoder_outputs, then lm_head.weight."""
    if dims.scale_decoder_outputs:
        dec = dec * dims.d_model ** -0.5
    return dec @ sd["lm_head.weight"].T


def lm_loss(enc_in: torch.Tensor, labels: torch.Tensor, sd: dict, dims: V11Dims) -> torch.Tensor:
    """T5ForConditionalGeneration.forward(inputs_embeds, labels).loss."""
    enc = stack(enc_in, sd, "encoder.", dims)
    dec = stack(F.embedding(shift_right(labels, dims), sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc)
    logits = lm_logits(dec, sd, dims)
    return F.cross_entropy(logits.view(-1, logits.shape[-1]), labels.reshape(-1), ignore_index=-100)


def greedy_decode(enc_in: torch.Tensor, sd: dict, dims: V11Dims, max_new_tokens: int = 20) -> torch.Tensor:
    """Greedy `generate(inputs_embeds=...)` (oracle/t5.py:t5_greedy_decode with this module's stack and head)."""
    enc = stack(enc_in, sd, "encoder.", dims)
    ids = torch.full((enc_in.shape[0], 1), dims.decoder_start_token_id, dtype=torch.long)
    unfinished = torch.ones(enc_in.shape[0], dtype=torch.bool)
    for _ in range(max_new_tokens):
        dec = stack(F.embedding(ids, sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc)
        nxt = lm_logits(dec[:, -1], sd, dims).float().argmax(-1)
        nxt = torch.where(unfinished, nxt, torch.full_like(nxt, dims.pad_token_id))
        ids = torch.cat([ids, nxt[:, None]], dim=1)
        unfinished = unfinished & (nxt != dims.eos_token_id)
        if not unfinished.any():
            break
    return ids


def beam_search(enc_in: torch.Tensor, sd: dict, dims: V11Dims, num_beams: int, max_new_tokens: int = 20, length_penalty: float = 1.0,
                early_stopping=False, num_return_sequences: int = 1):
    """`generate(inputs_embeds, num_beams=...)` -> (sequences, sequences_scores) (oracle/t5_beam.py:t5_beam_search's loop)."""
    enc = stack(enc_in, sd, "encoder.", dims)
    B, nb, max_length = enc.shape[0], num_beams, max_new_tokens + 1
    enc_rep = enc.repeat_interleave(nb, 0)
    st = beam_init(B, nb, max_length, dims)
    for t in range(max_new_tokens):
        ids = st.run_seq[:, :, :t + 1].reshape(B * nb, t + 1)
        dec = stack(F.embedding(ids, sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc_rep)
        if not beam_step(st, lm_logits(dec[:, -1], sd, dims), t, max_length, dims, length_penalty, early_stopping):
            break
    return beam_output(st, num_return_sequences)


def sample(enc_in: torch.Tensor, sd: dict, dims: V11Dims, seed: int, temperature: float = 1.0, top_k: int = 50, top_p: float = 1.0,
           num_return_sequences: int = 1, max_new_tokens: int = 20):
    """`generate(inputs_embeds, do_sample=True, ...)` with the project's defined draw (oracle/t5_sample.py:t5_sample's loop)."""
    enc = stack(enc_in, sd, "encoder.", dims).repeat_interleave(num_return_sequences, 0)
    R = enc.shape[0]
    ids = torch.full((R, 1), dims.decoder_start_token_id, dtype=torch.long)
    unfinished = torch.ones(R, dtype=torch.bool)
    for t in range(max_new_tokens):
        dec = stack(F.embedding(ids, sd["shared.weight"]), sd, "decoder.", dims, enc_out=enc)
        probs = F.softmax(warp(lm_logits(dec[:, -1], sd, dims), temperature, top_k, top_p), dim=-1)
        nxt = inverse_cdf(probs, torch.tensor([sample_uniform(seed, r, t) for r in range(R)], dtype=torch.float64))
        nxt = torch.where(unfinished, nxt, torch.full_like(nxt, dims.pad_token_id))
        ids = torch.cat([ids, nxt[:, None]], dim=1)
        unfinished = unfinished & (nxt != dims.eos_token_id)
        if not unfinished.any():
            break
    return ids


def caption_loss(pixel_values, src_ids, tgt_ids, sds: dict, lm: V11Dims, swin: SwinDims, tr: V11Dims):
    """models/model.py:20-26 of the reference with gated towers: frozen text encoder, Swin, concat, loss of the transformer."""
    with torch.no_grad():
        lm_sd = sds["language_model"]
        lang = stack(F.embedding(src_ids, lm_sd["shared.weight"]), lm_sd, "encoder.", lm)
    img = swinv2_forward(pixel_values, sds["image_model"], swin)
    return lm_loss(torch.cat((img, lang), dim=1), tgt_ids, sds["transformer"], tr)


# ----------------------------------------------------------------------------------------------
# state-dict layout and seeded weights
# ----------------------------------------------------------------------------------------------
def param_shapes(d: V11Dims, encoder_only: bool = False) -> dict:
    """Key -> shape of T5ForConditionalGeneration / T5EncoderModel: gated blocks hold wi_0 and wi_1 where ReLU blocks hold wi."""
    out = {}
    for k, shape in t5_param_shapes(d, encoder_only).items():
        if d.feed_forward_proj == "gated-gelu" and k.endswith("DenseReluDense.wi.weight"):
            out[k[:-len("wi.weight")] + "wi_0.weight"] = shape
            out[k[:-len("wi.weight")] + "wi_1.weight"] = shape
        else:
            out[k] = shape
    return out


def seeded_transformer(d: V11Dims, seed: int, scope: str = "transformer", style: str = "hf", untied_head: bool = False,
                       encoder_only: bool = False) -> dict:
    """oracle/caption_model.py:seeded_state_dict over `param_shapes` (wi_0 / wi_1 get 1/sqrt(d_model), HF's std for them);
    untied_head: lm_head.weight gets values of its own (a T5 v1.1 checkpoint) instead of being shared.weight."""
    shapes = param_shapes(d, encoder_only)
    sd = seeded_state_dict(shapes, seed, scope, style, d)
    if untied_head and "lm_head.weight" in shapes:
        sd["lm_head.weight"] = _seeded_tensor(seed, scope, "lm_head.weight", shapes["lm_head.weight"], style, d)
    return sd


def seeded_state_dicts(lm: V11Dims, swin: SwinDims, tr: V11Dims, seed: int = 0, style: str = "hf", untied_head: bool = False) -> dict:
    """Weights of the three sub-models of MyModel with gated towers."""
    return {"language_model": seeded_transformer(lm, seed, "language_model", style, encoder_only=True),
            "image_model": seeded_state_dict(swin_param_shapes(swin), seed, "image_model", style, swin),
            "transformer": seeded_transformer(tr, seed, "transformer", style, untied_head=untied_head)}
