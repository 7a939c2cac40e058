"""Parameter containers with the reference's (HuggingFace) state-dict key layout, and the forward passes that run them
through the sm_100a kernels.

The module trees mirror `T5EncoderModel`, `T5ForConditionalGeneration` and `Swinv2Model` key for key (SURVEY.md 8b), so
checkpoints written by /root/reference/models/model.py:30-35 load with `load_state_dict(strict=True)` and vice versa.  The
modules only OWN parameters (ordinary fp32 `nn.Parameter`s, so DDP buckets them and `torch.optim.Adam` updates them); their
arithmetic is libklab_b200.so.  Calling anything here without an sm_100 GPU raises: there is no CPU fallback.
"""
from __future__ import annotations

import json
import math
import os
import random
import warnings
from dataclasses import asdict, dataclass

import torch
from torch import nn

from . import functional as Fn
from . import ops as O
from .functional import Ctx, OperandCache


# ------------------------------------------------------------------------------------------------
# configs (subset of HF/models/t5/configuration_t5.py:44-83, HF/models/swinv2/configuration_swinv2.py:56-73)
# ------------------------------------------------------------------------------------------------
@dataclass
class T5Config:
    vocab_size: int = 32128
    d_model: int = 512
    d_kv: int = 64
    d_ff: int = 2048
    num_layers: int = 6
    num_decoder_layers: int | None = None
    num_heads: int = 8
    relative_attention_num_buckets: int = 32
    relative_attention_max_distance: int = 128
    dropout_rate: float = 0.1
    layer_norm_epsilon: float = 1e-6
    feed_forward_proj: str = "relu"
    pad_token_id: int = 0
    eos_token_id: int = 1
    decoder_start_token_id: int = 0
    tie_word_embeddings: bool = True
    # HF/models/t5/configuration_t5.py:79-83: T5 v1.1 checkpoints say `"tie_word_embeddings": false`, and that is what switches the
    # d_model ** -0.5 scale in front of the LM head off (modeling_t5.py:1107).  None: derived from tie_word_embeddings as HF does;
    # a config.json that transformers wrote stores the derived value itself.
    scale_decoder_outputs: bool | None = None

    NAMED = {
        "t5-small": dict(d_model=512, d_ff=2048, num_layers=6, num_heads=8),
        "t5-base": dict(d_model=768, d_ff=3072, num_layers=12, num_heads=12),
        "t5-large": dict(d_model=1024, d_ff=4096, num_layers=24, num_heads=16),
        "t5-3b": dict(d_model=1024, d_kv=128, d_ff=16384, num_layers=24, num_heads=32),
        "t5-11b": dict(d_model=1024, d_kv=128, d_ff=65536, num_layers=24, num_heads=128),
        **{f"google/{family}-{size}": dict(arch, feed_forward_proj="gated-gelu", tie_word_embeddings=False)
           for family in ("flan-t5", "t5-v1_1")
           for size, arch in (("small", dict(d_model=512, d_ff=1024, num_layers=8, num_heads=6)),
                              ("base", dict(d_model=768, d_ff=2048, num_layers=12, num_heads=12)),
                              ("large", dict(d_model=1024, d_ff=2816, num_layers=24, num_heads=16)))},
    }
    FEED_FORWARD_PROJ = ("relu", "gated-gelu")

    def __post_init__(self):
        if self.feed_forward_proj not in self.FEED_FORWARD_PROJ:
            raise ValueError(f"T5Config: feed_forward_proj={self.feed_forward_proj!r} is not supported (supported: "
                             f"{', '.join(self.FEED_FORWARD_PROJ)})")
        if self.scale_decoder_outputs is None:
            self.scale_decoder_outputs = self.tie_word_embeddings is not False

    @property
    def gated(self) -> bool:
        """T5 v1.1 / Flan-T5 feed-forward: h = gelu_new(x wi_0^T) * (x wi_1^T) (HF/models/t5/modeling_t5.py:106-132)."""
        return self.feed_forward_proj == "gated-gelu"

    @property
    def lm_head_scale(self) -> float:
        """Factor on the final decoder state in front of the LM head (HF/models/t5/modeling_t5.py:1107)."""
        return self.d_model ** -0.5 if self.scale_decoder_outputs else 1.0

    @property
    def n_dec(self):
        return self.num_layers if self.num_decoder_layers is None else self.num_decoder_layers


@dataclass
class Swinv2Config:
    image_size: int = 256
    patch_size: int = 4
    num_channels: int = 3
    embed_dim: int = 128
    depths: tuple = (2, 2, 18, 2)
    num_heads: tuple = (4, 8, 16, 32)
    window_size: int = 8
    pretrained_window_sizes: tuple = (0, 0, 0, 0)
    mlp_ratio: float = 4.0
    qkv_bias: bool = True
    layer_norm_eps: float = 1e-5
    hidden_act: str = "gelu"

    NAMED = {
        "microsoft/swinv2-tiny-patch4-window8-256": dict(embed_dim=96, depths=(2, 2, 6, 2), num_heads=(3, 6, 12, 24)),
        "microsoft/swinv2-small-patch4-window8-256": dict(embed_dim=96, depths=(2, 2, 18, 2), num_heads=(3, 6, 12, 24)),
        "microsoft/swinv2-base-patch4-window8-256": dict(embed_dim=128, depths=(2, 2, 18, 2), num_heads=(4, 8, 16, 32)),
    }


def _hf_cache_roots() -> list[str]:
    """Where `transformers` keeps downloaded snapshots (HF_HUB_CACHE / TRANSFORMERS_CACHE / HF_HOME/hub / ~/.cache/huggingface/hub)."""
    roots = []
    for var in ("HF_HUB_CACHE", "HUGGINGFACE_HUB_CACHE", "TRANSFORMERS_CACHE"):
        if os.environ.get(var):
            roots.append(os.environ[var])
    home = os.environ.get("HF_HOME") or os.path.join(os.path.expanduser("~"), ".cache", "huggingface")
    roots.append(os.path.join(home, "hub"))
    return roots


_HUB_ALIASES = {"t5-small": "google-t5/t5-small", "t5-base": "google-t5/t5-base", "t5-large": "google-t5/t5-large",
                "t5-3b": "google-t5/t5-3b", "t5-11b": "google-t5/t5-11b"}


def resolve_snapshot(name: str) -> str | None:
    """A bare model name -> the newest local snapshot directory of the HF cache that holds its config.json, or None.
    The reference's `from_pretrained(name)` (/root/reference/models/model.py:14-17) finds its weights the same way when the
    hub is unreachable (HF_HUB_OFFLINE); nothing is ever downloaded here."""
    names = [name] + ([_HUB_ALIASES[name]] if name in _HUB_ALIASES else [])
    best = None
    for root in _hf_cache_roots():
        for nm in names:
            snaps = os.path.join(root, "models--" + nm.replace("/", "--"), "snapshots")
            if not os.path.isdir(snaps):
                continue
            for rev in os.listdir(snaps):
                d = os.path.join(snaps, rev)
                if os.path.exists(os.path.join(d, "config.json")):
                    m = os.path.getmtime(d)
                    if best is None or m > best[0]:
                        best = (m, d)
    return best[1] if best else None


def _config_from_dir(cls, path, overrides):
    fields = {f for f in cls.__dataclass_fields__}
    with open(os.path.join(path, "config.json")) as fh:
        raw = json.load(fh)
    kw = {k: (tuple(v) if isinstance(v, list) else v) for k, v in raw.items() if k in fields}
    kw.update(overrides)
    return cls(**kw)


def _config_from_source(cls, source, **overrides):
    """`from_pretrained`-style resolution -> (config, checkpoint directory or None):
      * a cls instance: explicit architecture, random initialisation is what the caller asked for (tests, benchmarks);
      * a local directory with config.json (+ model.safetensors / pytorch_model.bin);
      * a model name: its snapshot in the local HF cache if there is one; otherwise a KNOWN name gives the architecture but no
        weights -- the reference would fail here (no network), so this raises unless KLAB_ALLOW_RANDOM_INIT=1 opts in to a
        randomly initialised model (a loud warning is issued)."""
    if isinstance(source, cls):
        return source, None
    if isinstance(source, str) and os.path.isdir(source) and os.path.exists(os.path.join(source, "config.json")):
        return _config_from_dir(cls, source, overrides), source
    if isinstance(source, str):
        snap = resolve_snapshot(source)
        if snap is not None:
            return _config_from_dir(cls, snap, overrides), snap
        if source in cls.NAMED:
            if os.environ.get("KLAB_ALLOW_RANDOM_INIT", "0") != "1":
                raise FileNotFoundError(
                    f"{source!r}: no local checkpoint directory and no snapshot in the HF cache ({', '.join(_hf_cache_roots())}); "
                    "pass a directory with config.json + weights, or set KLAB_ALLOW_RANDOM_INIT=1 to get a RANDOMLY INITIALISED "
                    f"{cls.__name__[:-6]} model of that architecture")
            warnings.warn(f"klab_multimodalmodel_b200: {source!r} has no weights on this machine -- the model is RANDOMLY INITIALISED "
                          "(KLAB_ALLOW_RANDOM_INIT=1)", RuntimeWarning, stacklevel=3)
            kw = dict(cls.NAMED[source])
            kw.update(overrides)
            return cls(**kw), None
    raise FileNotFoundError(f"{source!r} is neither a local checkpoint directory (config.json), a cached snapshot nor a known {cls.__name__} name")


_BASE_PREFIXES = ("swinv2.", "transformer.", "model.", "encoder_model.")


def _load_checkpoint_dir(module: nn.Module, path: str, before_load=None) -> None:
    """Load model.safetensors / pytorch_model.bin of a checkpoint directory, strict on the module's own keys.  Like HF's
    `from_pretrained` it strips the base-model prefix when the file was written by a task head (the published
    microsoft/swinv2-* checkpoints are Swinv2ForImageClassification: 'swinv2.embeddings...' + 'classifier.*') and reports the
    keys it drops.  A directory without weights is an error: the reference never random-initialises silently.
    before_load(sd): called with the file's tensors before tied keys are filled in (T5ForConditionalGeneration unties its LM
    head there when the file holds a distinct one)."""
    st = os.path.join(path, "model.safetensors")
    pt = os.path.join(path, "pytorch_model.bin")
    if os.path.exists(st):
        from safetensors.torch import load_file
        sd = load_file(st)
    elif os.path.exists(pt):
        sd = torch.load(pt, map_location="cpu")
    else:
        raise FileNotFoundError(f"{path}: config.json found but neither model.safetensors nor pytorch_model.bin")
    own = module.state_dict()
    if not any(k in own for k in sd):                     # nothing matches: a task-head checkpoint of the same base model?
        for pre in _BASE_PREFIXES:
            stripped = {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
            if any(k in own for k in stripped):
                sd = {**{k: v for k, v in sd.items() if not k.startswith(pre)}, **stripped}
                break
    if before_load is not None:
        before_load(sd)
        own = module.state_dict()
    for k in own:                      # tied tensors are stored once in safetensors files
        if k not in sd:
            for alias in ("shared.weight", "encoder.embed_tokens.weight", "decoder.embed_tokens.weight", "lm_head.weight"):
                if alias in sd and own[k].shape == sd[alias].shape and k.endswith(("embed_tokens.weight", "lm_head.weight", "shared.weight")):
                    sd[k] = sd[alias]
                    break
    dropped = sorted(k for k in sd if k not in own)
    if dropped:
        warnings.warn(f"klab_multimodalmodel_b200: {path}: {len(dropped)} checkpoint tensors are not part of {type(module).__name__} "
                      f"and were ignored: {', '.join(dropped[:6])}{' ...' if len(dropped) > 6 else ''}", RuntimeWarning, stacklevel=3)
    module.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=True)


class _P(nn.Module):
    """Parameter holder shaped like nn.Linear / nn.LayerNorm / nn.Embedding (weight [+ bias])."""

    def __init__(self, *shape, bias: bool = False):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(*shape))
        if bias:
            self.bias = nn.Parameter(torch.empty(shape[0]))


def _compute_dtype(name) -> torch.dtype:
    if isinstance(name, torch.dtype):
        return name
    name = (name or os.environ.get("KLAB_DTYPE", "bf16")).lower()
    return {"bf16": torch.bfloat16, "bfloat16": torch.bfloat16, "fp32": torch.float32, "float32": torch.float32}[name]


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: tensors must live on a B200 (sm_100) device; klab_multimodalmodel_b200 has no CPU path")


def _new_seed() -> int:
    return random.getrandbits(62)


# ------------------------------------------------------------------------------------------------
# T5
# ------------------------------------------------------------------------------------------------
class _T5Attention(nn.Module):
    def __init__(self, cfg: T5Config, has_bias: bool):
        super().__init__()
        inner = cfg.num_heads * cfg.d_kv
        self.q, self.k, self.v = _P(inner, cfg.d_model), _P(inner, cfg.d_model), _P(inner, cfg.d_model)
        self.o = _P(cfg.d_model, inner)
        if has_bias:
            self.relative_attention_bias = _P(cfg.relative_attention_num_buckets, cfg.num_heads)


class _T5SelfLayer(nn.Module):
    def __init__(self, cfg, has_bias):
        super().__init__()
        self.SelfAttention = _T5Attention(cfg, has_bias)
        self.layer_norm = _P(cfg.d_model)


class _T5CrossLayer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.EncDecAttention = _T5Attention(cfg, False)
        self.layer_norm = _P(cfg.d_model)


class _T5Dense(nn.Module):
    """T5DenseActDense (wi, wo) or, gated, T5DenseGatedActDense (wi_0, wi_1, wo); HF keeps the name DenseReluDense for both."""

    def __init__(self, cfg):
        super().__init__()
        if cfg.gated:
            self.wi_0, self.wi_1 = _P(cfg.d_ff, cfg.d_model), _P(cfg.d_ff, cfg.d_model)
        else:
            self.wi = _P(cfg.d_ff, cfg.d_model)
        self.wo = _P(cfg.d_model, cfg.d_ff)

    def in_weights(self):
        """[wi] or [wi_0, wi_1]: the blocks of the one input-projection operand."""
        return [self.wi_0.weight, self.wi_1.weight] if hasattr(self, "wi_0") else [self.wi.weight]


class _T5FFLayer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.DenseReluDense = _T5Dense(cfg)
        self.layer_norm = _P(cfg.d_model)


class _T5Block(nn.Module):
    def __init__(self, cfg, is_decoder, has_bias):
        super().__init__()
        layers = [_T5SelfLayer(cfg, has_bias)]
        if is_decoder:
            layers.append(_T5CrossLayer(cfg))
        layers.append(_T5FFLayer(cfg))
        self.layer = nn.ModuleList(layers)
        self.is_decoder = is_decoder

    def flat_params(self):
        sa = self.layer[0]
        ps = [sa.layer_norm.weight, sa.SelfAttention.q.weight, sa.SelfAttention.k.weight, sa.SelfAttention.v.weight,
              sa.SelfAttention.o.weight]
        if self.is_decoder:
            ca = self.layer[1]
            ps += [ca.layer_norm.weight, ca.EncDecAttention.q.weight, ca.EncDecAttention.k.weight, ca.EncDecAttention.v.weight,
                   ca.EncDecAttention.o.weight]
        ff = self.layer[-1]
        ps += [ff.layer_norm.weight, *ff.DenseReluDense.in_weights(), ff.DenseReluDense.wo.weight]
        return ps


class T5Stack(nn.Module):
    """T5Stack (HF/models/t5/modeling_t5.py:617-792) as a parameter tree + kernel schedule."""

    def __init__(self, cfg: T5Config, is_decoder: bool, embed_tokens: _P):
        super().__init__()
        self.cfg, self.is_decoder = cfg, is_decoder
        self.embed_tokens = embed_tokens
        n = cfg.n_dec if is_decoder else cfg.num_layers
        self.block = nn.ModuleList([_T5Block(cfg, is_decoder, i == 0) for i in range(n)])
        self.final_layer_norm = _P(cfg.d_model)
        self._luts: dict = {}
        self._ctxs: dict = {}
        _STACK_COUNT[0] += 1
        self.seed_base = _STACK_COUNT[0] * 100003               # distinct dropout streams per stack / block / site

    def lut(self, L_, device):
        key = (L_, device)
        if key not in self._luts:
            lut, rz = O.t5_rel_bucket_lut(L_, L_, bidirectional=not self.is_decoder,
                                          num_buckets=self.cfg.relative_attention_num_buckets,
                                          max_distance=self.cfg.relative_attention_max_distance)
            self._luts[key] = (lut.to(device), rz)
        return self._luts[key]

    def block_ctx(self, i, B, L_, Le, p, cache, device, cd):
        """One cached Ctx per (block, shape signature): its identity keys the block's CUDA graphs."""
        key = (i, B, L_, Le, p, device, cd)
        c = self._ctxs.get(key)
        if c is None:
            cfg = self.cfg
            lut, rz = self.lut(L_, device)
            c = self._ctxs[key] = Ctx(cache=cache, is_decoder=self.is_decoder, gated=cfg.gated, B=B, L=L_, Le=Le, H=cfg.num_heads, dk=cfg.d_kv,
                                      eps=cfg.layer_norm_epsilon, num_buckets=cfg.relative_attention_num_buckets, lut=lut, rz=rz, p=p,
                                      seed=self.seed_base + 16 * (i + 1), seed_ptr=step_seed(device) if p > 0 else None)
        return c

    def run_blocks(self, x, B, L_, cache: OperandCache, enc_out=None, Le=0):
        """x: [B*L, d] in the compute dtype -> hidden state BEFORE final_layer_norm."""
        cfg = self.cfg
        p = cfg.dropout_rate if self.training else 0.0
        table = self.block[0].layer[0].SelfAttention.relative_attention_bias.weight
        if p > 0:                                                       # dropout on the stack input (:734)
            x = Fn.apply_fn(Fn.DropoutFn, x, p, self.seed_base, step_seed(x.device))
        for i, blk in enumerate(self.block):
            c = self.block_ctx(i, B, L_, Le, p, cache, x.device, x.dtype)
            x = Fn.apply_fn(Fn.T5BlockFn, c, x, enc_out, table, *blk.flat_params())
        return x


_STEP_SEEDS: dict = {}
_STACK_COUNT = [0]


def step_seed(device) -> torch.Tensor:
    """Per-device dropout counter living on the GPU: every dropout site hashes (its own constant + this counter, element
    index); `advance_step_seed` steps it once per training forward (klab_seed_advance), CUDA graphs replay unchanged."""
    key = (device.type, device.index)
    t = _STEP_SEEDS.get(key)
    if t is None:
        t = _STEP_SEEDS[key] = torch.tensor([random.getrandbits(62)], dtype=torch.int64, device=device)
    return t


def advance_step_seed(device) -> None:
    O.seed_advance(step_seed(device))


class T5EncoderModel(nn.Module):
    """Frozen text encoder of the reference (/root/reference/models/model.py:14,20-21)."""

    def __init__(self, cfg: T5Config):
        super().__init__()
        self.config = cfg
        self.shared = _P(cfg.vocab_size, cfg.d_model)
        self.encoder = T5Stack(cfg, False, self.shared)
        self.cache = OperandCache()
        init_t5_(self)

    @classmethod
    def from_pretrained(cls, source, **overrides):
        cfg, path = _config_from_source(T5Config, source, **overrides)
        m = cls(cfg)
        if path:
            _load_checkpoint_dir(m, path)
        return m.eval()

    def hidden_before_norm(self, input_ids, cd):
        """[B, L] ids -> [B*L, d] hidden state before final_layer_norm (the norm is fused into the concat)."""
        _require_cuda(input_ids, "T5EncoderModel")
        B, L_ = input_ids.shape
        tab = self.cache.get([self.shared.weight], cd)
        x = O.embedding_fwd(input_ids.contiguous(), tab)
        return self.encoder.run_blocks(x, B, L_, self.cache)


class GenerationConfig:
    """The `generation_config` fields of HF 5.5.0 (HF/generation/configuration_utils.py) that this build supports, with their
    defaults; the token ids come from the model config.  Setting `num_beams` > 1 here makes `generate()` -- and so
    `MyModel.forward(return_loss=False)` -- run beam search, as in the reference; setting `do_sample = True` makes it sample.
    The sampling defaults are those HF applies when do_sample is set (configuration_utils.py:559-561)."""

    def __init__(self, cfg: "T5Config"):
        self.max_length = 20
        self.max_new_tokens = None
        self.num_beams = 1
        self.length_penalty = 1.0
        self.early_stopping = False
        self.num_return_sequences = 1
        self.do_sample = False
        self.temperature = 1.0
        self.top_k = 50
        self.top_p = 1.0
        self.decoder_start_token_id = cfg.decoder_start_token_id
        self.eos_token_id = cfg.eos_token_id
        self.pad_token_id = cfg.pad_token_id


@dataclass
class BeamSearchOutput:
    """`generate(..., return_dict_in_generate=True, output_scores=True)`: sequences and, for beam search, the scores of the
    returned hypotheses (None for greedy decoding)."""
    sequences: torch.Tensor
    sequences_scores: torch.Tensor | None = None


_GEN_FIELDS = ("max_length", "max_new_tokens", "num_beams", "length_penalty", "early_stopping", "num_return_sequences", "do_sample",
               "temperature", "top_k", "top_p")
_SAMPLING_DEFAULTS = {"temperature": 1.0, "top_k": 50, "top_p": 1.0}
_MAX_BEAMS = 8


class T5ForConditionalGeneration(nn.Module):
    """Trainable encoder-decoder of the reference (/root/reference/models/model.py:17,26,28)."""

    def __init__(self, cfg: T5Config):
        super().__init__()
        self.config = cfg
        self.shared = _P(cfg.vocab_size, cfg.d_model)
        self.encoder = T5Stack(cfg, False, self.shared)
        self.decoder = T5Stack(cfg, True, self.shared)
        self.lm_head = _P(cfg.vocab_size, cfg.d_model)
        self.lm_head.weight = self.shared.weight                     # tied (HF/models/t5/modeling_t5.py:956-960)
        self.cache = OperandCache()
        self.generation_config = GenerationConfig(cfg)
        init_t5_(self)

    @classmethod
    def from_pretrained(cls, source, **overrides):
        """As HF's: a checkpoint whose lm_head.weight differs from shared.weight (T5 v1.1 / Flan-T5 ship their own LM head)
        gives an untied model whose lm_head holds the file's tensor; equal tensors, or no lm_head.weight, keep them tied."""
        cfg, path = _config_from_source(T5Config, source, **overrides)
        m = cls(cfg)
        if path:
            _load_checkpoint_dir(m, path, before_load=m._untie_for)
        return m.eval()

    @property
    def lm_head_tied(self) -> bool:
        return self.lm_head.weight is self.shared.weight

    def untie_lm_head(self) -> None:
        """Give lm_head a parameter of its own (initialised with a copy of shared.weight).  state_dict() keys do not change."""
        if self.lm_head_tied:
            self.lm_head.weight = nn.Parameter(self.shared.weight.detach().clone())
            # captured decode steps baked the tied operand in: drop them with their states
            from .graphs import POOL
            POOL.drop_keys(lambda k: len(k) > 1 and k[1] == id(self))
            for attr in ("_klab_decode_states", "_klab_sample_states", "_klab_beam_states"):
                self.__dict__.pop(attr, None)

    def _untie_for(self, sd) -> None:
        head, emb = sd.get("lm_head.weight"), sd.get("shared.weight")
        if head is not None and emb is not None and head.shape == emb.shape and not torch.equal(head, emb):
            self.untie_lm_head()

    def state_dict(self, *args, **kwargs):
        from .optim import wait_pending_updates
        if torch.cuda.is_available():
            wait_pending_updates(self.shared.weight.device if self.shared.weight.is_cuda else None)
        return super().state_dict(*args, **kwargs)

    def load_state_dict(self, state_dict, *args, **kwargs):
        """A state dict with a distinct lm_head.weight unties a tied model first (as from_pretrained does), so that
        MyModel.load of an untied model's file restores both tensors instead of one overwriting the other."""
        from .optim import wait_pending_updates
        if torch.cuda.is_available():
            wait_pending_updates(self.shared.weight.device if self.shared.weight.is_cuda else None)
        self._untie_for(state_dict)
        return super().load_state_dict(state_dict, *args, **kwargs)

    def loss_from_embeds(self, embeds, B, Le, labels):
        """embeds: [B*Le, d] encoder inputs_embeds (compute dtype); labels [B, Lt] int64 -> 0-dim fp32 loss
        (T5ForConditionalGeneration.forward(inputs_embeds, labels).loss, HF/models/t5/modeling_t5.py:1070-1117)."""
        cfg = self.config
        cd = embeds.dtype
        Lt = labels.shape[1]
        enc = self.encoder.run_blocks(embeds, B, Le, self.cache)
        enc = Fn.apply_fn(Fn.RMSNormFn, enc, self.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon)
        p = cfg.dropout_rate if self.training else 0.0
        sp = step_seed(embeds.device) if p > 0 else None
        if p > 0:
            enc = Fn.apply_fn(Fn.DropoutFn, enc, p, self.encoder.seed_base + 7, sp)     # :768
        labels = labels.contiguous()
        dec_in = Fn.apply_fn(Fn.DecoderEmbedFn, labels, self.shared.weight, self.cache, cd, cfg.decoder_start_token_id, cfg.pad_token_id)
        dec = self.decoder.run_blocks(dec_in, B, Lt, self.cache, enc_out=enc, Le=Le)
        return Fn.apply_fn(Fn.LMHeadLossFn, dec, self.decoder.final_layer_norm.weight, self.lm_head.weight, labels, self.cache,
                           cfg.layer_norm_epsilon, p, self.decoder.seed_base + 7, sp, cfg.lm_head_scale)

    def generate(self, inputs_embeds=None, return_dict_in_generate=False, output_scores=False, **overrides):
        """`generate(inputs_embeds=[B, Le, d], **overrides)` of HF 5.5.0 for the options in `generation_config`: greedy decoding
        (num_beams 1), beam search (num_beams 2..8) or multinomial sampling (do_sample=True, num_beams 1, with temperature, top_k
        and top_p).  The compute dtype is that of inputs_embeds (bf16 or fp32).  Returns the ids [B * num_return_sequences, n]
        int64, or with return_dict_in_generate=True a BeamSearchOutput (sequences_scores needs output_scores=True and beam
        search).  Options this build does not implement raise instead of being ignored."""
        from . import generation
        unknown = sorted(set(overrides) - set(_GEN_FIELDS))
        if unknown:
            raise ValueError(f"generate(): {', '.join(unknown)} not supported (supported: {', '.join(_GEN_FIELDS)}, "
                             "return_dict_in_generate, output_scores); logits processors are not implemented")
        gc = self.generation_config
        opt = {k: overrides.get(k, getattr(gc, k)) for k in _GEN_FIELDS}
        nb, nrs, es, sample = opt["num_beams"], opt["num_return_sequences"], opt["early_stopping"], opt["do_sample"]
        if not isinstance(nb, int) or not 1 <= nb <= _MAX_BEAMS:
            raise ValueError(f"generate(): num_beams={nb!r}; this build supports 1..{_MAX_BEAMS}")
        if not isinstance(sample, bool):
            raise ValueError(f"generate(): do_sample={sample!r} must be True or False")
        if sample:
            if nb > 1:
                raise ValueError("generate(): do_sample=True with num_beams > 1 (beam sampling) is not implemented")
            generation.check_sampling_options(opt["temperature"], opt["top_k"], opt["top_p"], nrs)
        else:
            # GenerationConfig.validate(strict=True) (HF/generation/configuration_utils.py:636-660): flags that only matter when
            # sampling.  transformers warns and ignores them; ignoring an option silently is what this build never does
            flags = [f"{k}={opt[k]!r}" for k, v in _SAMPLING_DEFAULTS.items() if opt[k] != v]
            if flags:
                raise ValueError(f"generate(): {', '.join(flags)} only apply when sampling: set do_sample=True")
            if not isinstance(nrs, int) or not 1 <= nrs <= nb:
                raise ValueError(f"generate(): num_return_sequences={nrs!r} must be in 1..num_beams ({nb})")
        if es not in (False, True, "never") or isinstance(es, int) and not isinstance(es, bool):
            raise ValueError(f"generate(): early_stopping={es!r} must be False, True or 'never'")
        # HF/generation/utils.py:1608-1640 (_prepare_generated_length) for an encoder-decoder whose decoder prompt is the start token
        if opt["max_new_tokens"] is not None:
            T = int(opt["max_new_tokens"])
        elif "max_length" in overrides or gc.max_length != 20:
            T = int(opt["max_length"]) - 1
        else:
            T = 20
        if T < 1:
            raise ValueError(f"generate(): nothing to generate (max_new_tokens {T})")
        if inputs_embeds is None or inputs_embeds.dim() != 3:
            raise ValueError("generate(): inputs_embeds [B, Le, d_model] is required")
        B, Le, d = inputs_embeds.shape
        x = inputs_embeds.reshape(B * Le, d)
        if sample:
            seqs, scores = generation.sample_generate(self, x, B, Le, max_new_tokens=T, temperature=opt["temperature"],
                                                      top_k=opt["top_k"], top_p=opt["top_p"], num_return_sequences=nrs), None
        elif nb == 1:
            seqs, scores = generation.greedy_generate(self, x, B, Le, max_new_tokens=T), None
        else:
            seqs, scores = generation.beam_generate(self, x, B, Le, num_beams=nb, max_new_tokens=T, length_penalty=float(opt["length_penalty"]),
                                                    early_stopping=es, num_return_sequences=nrs)
        if return_dict_in_generate:
            return BeamSearchOutput(seqs, scores if output_scores else None)
        return seqs


def init_t5_(m: nn.Module, seed: int | None = None):
    """T5PreTrainedModel._init_weights (HF/models/t5/modeling_t5.py:540-593), initializer_factor 1."""
    cfg = m.config
    g = torch.Generator().manual_seed(seed) if seed is not None else None
    d, dk, h, dff = cfg.d_model, cfg.d_kv, cfg.num_heads, cfg.d_ff
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.endswith("layer_norm.weight"):
                p.fill_(1.0)
            elif name == "shared.weight":
                p.normal_(0.0, 1.0, generator=g)
            elif name.endswith(".q.weight"):
                p.normal_(0.0, (d * dk) ** -0.5, generator=g)
            elif name.endswith((".k.weight", ".v.weight", "wi.weight", "wi_0.weight", "wi_1.weight", "relative_attention_bias.weight")):
                p.normal_(0.0, d ** -0.5, generator=g)
            elif name.endswith(".o.weight"):
                p.normal_(0.0, (h * dk) ** -0.5, generator=g)
            elif name.endswith("wo.weight"):
                p.normal_(0.0, dff ** -0.5, generator=g)


# ------------------------------------------------------------------------------------------------
# Swin-V2
# ------------------------------------------------------------------------------------------------
class _CPB(nn.Sequential):
    def __init__(self, heads):
        super().__init__(_P(512, 2, bias=True), nn.Identity(), _P(heads, 512))


class _SwinSelfAttention(nn.Module):
    def __init__(self, dim, heads):
        super().__init__()
        self.logit_scale = nn.Parameter(torch.empty(heads, 1, 1))
        self.continuous_position_bias_mlp = _CPB(heads)
        self.query, self.key, self.value = _P(dim, dim, bias=True), _P(dim, dim), _P(dim, dim, bias=True)


class _SwinAttention(nn.Module):
    def __init__(self, dim, heads):
        super().__init__()
        self.self = _SwinSelfAttention(dim, heads)
        self.output = nn.Module()
        self.output.dense = _P(dim, dim, bias=True)


class _SwinLayer(nn.Module):
    def __init__(self, dim, heads, mlp):
        super().__init__()
        self.attention = _SwinAttention(dim, heads)
        self.layernorm_before = _P(dim, bias=True)
        self.intermediate = nn.Module()
        self.intermediate.dense = _P(mlp, dim, bias=True)
        self.output = nn.Module()
        self.output.dense = _P(dim, mlp, bias=True)
        self.layernorm_after = _P(dim, bias=True)

    def flat_params(self):
        s = self.attention.self
        mlp = s.continuous_position_bias_mlp
        return [s.logit_scale, mlp[0].weight, mlp[0].bias, mlp[2].weight, s.query.weight, s.query.bias, s.key.weight,
                s.value.weight, s.value.bias, self.attention.output.dense.weight, self.attention.output.dense.bias,
                self.layernorm_before.weight, self.layernorm_before.bias, self.intermediate.dense.weight, self.intermediate.dense.bias,
                self.output.dense.weight, self.output.dense.bias, self.layernorm_after.weight, self.layernorm_after.bias]


class _SwinStage(nn.Module):
    def __init__(self, dim, depth, heads, mlp_ratio, downsample):
        super().__init__()
        self.blocks = nn.ModuleList([_SwinLayer(dim, heads, int(dim * mlp_ratio)) for _ in range(depth)])
        if downsample:
            self.downsample = nn.Module()
            self.downsample.reduction = _P(2 * dim, 4 * dim)
            self.downsample.norm = _P(2 * dim, bias=True)
        else:
            self.downsample = None


class Swinv2Model(nn.Module):
    """Swinv2Model (HF/models/swinv2/modeling_swinv2.py:907-987); `last_hidden_state` BEFORE the final LayerNorm is what
    `features()` returns (the final norm is fused into the concat, see functional.ConcatEmbeddingsFn)."""

    def __init__(self, cfg: Swinv2Config):
        super().__init__()
        self.config = cfg
        self.embeddings = nn.Module()
        self.embeddings.patch_embeddings = nn.Module()
        proj = _P(cfg.embed_dim, cfg.num_channels, cfg.patch_size, cfg.patch_size, bias=True)
        self.embeddings.patch_embeddings.projection = proj
        self.embeddings.norm = _P(cfg.embed_dim, bias=True)
        self.encoder = nn.Module()
        n = len(cfg.depths)
        self.encoder.layers = nn.ModuleList([
            _SwinStage(cfg.embed_dim * 2 ** s, cfg.depths[s], cfg.num_heads[s], cfg.mlp_ratio, s < n - 1) for s in range(n)])
        self.num_features = cfg.embed_dim * 2 ** (n - 1)
        self.layernorm = _P(self.num_features, bias=True)
        self.cache = OperandCache()
        self._tables: dict = {}
        self._ctxs: dict = {}
        init_swin_(self)

    @classmethod
    def from_pretrained(cls, source, **overrides):
        cfg, path = _config_from_source(Swinv2Config, source, **overrides)
        m = cls(cfg)
        if path:
            _load_checkpoint_dir(m, path)
        return m.eval()

    def tables(self, w, pw, device):
        key = (w, pw, device)
        if key not in self._tables:
            coords, index = O.swin_tables(w, pw)
            self._tables[key] = (coords.to(device), index.to(device))
        return self._tables[key]

    def features(self, pixel_values, cd):
        """(B, 3, H, W) fp32 pixels -> ([B*N_img, 8*C0] hidden state before the final LayerNorm, N_img)."""
        _require_cuda(pixel_values, "Swinv2Model")
        cfg = self.config
        B, _, Hh, Ww = pixel_values.shape
        if Hh % cfg.patch_size or Ww % cfg.patch_size or Hh != Ww:
            raise ValueError(f"image {Hh}x{Ww}: only square images divisible by the patch size are supported")
        e = self.embeddings
        x = Fn.apply_fn(Fn.PatchEmbedFn, pixel_values, e.patch_embeddings.projection.weight, e.patch_embeddings.projection.bias,
                                  e.norm.weight, e.norm.bias, self.cache, cd, cfg.patch_size, cfg.layer_norm_eps)
        res = Hh // cfg.patch_size
        for s, stage in enumerate(self.encoder.layers):
            heads = cfg.num_heads[s]
            dim = cfg.embed_dim * 2 ** s
            w = min(res, cfg.window_size)
            if res % w:
                raise ValueError(f"feature grid {res} is not a multiple of the window {w} (padding path not supported)")
            coords, index = self.tables(w, cfg.pretrained_window_sizes[s], x.device)
            for i, blk in enumerate(stage.blocks):
                shift = 0 if (i % 2 == 0 or res <= w) else cfg.window_size // 2
                key = (s, i, B, res, x.device, cd)
                c = self._ctxs.get(key)
                if c is None:
                    c = self._ctxs[key] = Ctx(cache=self.cache, B=B, res=res, heads=heads, hd=dim // heads, w=w, shift=shift, N=w * w,
                                              coords=coords, index=index, eps=cfg.layer_norm_eps)
                x = Fn.apply_fn(Fn.SwinBlockFn, c, x, *blk.flat_params())
            if stage.downsample is not None:
                d = stage.downsample
                x = Fn.apply_fn(Fn.PatchMergeFn, x, d.reduction.weight, d.norm.weight, d.norm.bias, self.cache, B, res, cfg.layer_norm_eps)
                res //= 2
        return x, res * res


def init_swin_(m: Swinv2Model, seed: int | None = None):
    """Swinv2PreTrainedModel._init_weights (HF/models/swinv2/modeling_swinv2.py:883-902), initializer_range 0.02."""
    g = torch.Generator().manual_seed(seed) if seed is not None else None
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.endswith("logit_scale"):
                p.fill_(math.log(10.0))
            elif "norm" in name.split(".")[-2]:
                p.fill_(1.0 if name.endswith("weight") else 0.0)
            elif name.endswith("bias"):
                p.zero_()
            else:
                p.normal_(0.0, 0.02, generator=g)


def config_dict(cfg) -> dict:
    return {k: (list(v) if isinstance(v, tuple) else v) for k, v in asdict(cfg).items()}
