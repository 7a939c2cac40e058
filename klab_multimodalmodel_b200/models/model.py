"""Drop-in for /root/reference/models/model.py: same class name, constructor arguments, attributes, forward signature,
checkpoint keys and error behaviour -- the arithmetic behind `forward` is libklab_b200.so (hand-written sm_100a kernels).

    reference                                      this file
    ---------------------------------------------  ----------------------------------------------------------
    T5EncoderModel.from_pretrained  (model.py:14)   modeling.T5EncoderModel.from_pretrained   (frozen)
    Swinv2Model.from_pretrained     (model.py:15)   modeling.Swinv2Model.from_pretrained
    T5ForConditionalGeneration...   (model.py:17)   modeling.T5ForConditionalGeneration.from_pretrained
    forward(images, source_encoding, target_encoding=None, return_loss=True)  (model.py:19-28)   identical
    save / load                     (model.py:30-42) identical file format ({'transformer': sd[, 'image_model': sd]})

One optional extra: `args.compute_dtype` ("bf16" default | "fp32"); the reference's argparse namespace does not have it, so
the default applies and train.py needs no change.

Data parallelism: `DistributedDataParallel(model)` (train.py:26) works unchanged.  When DDP's constructor asks the module which
parameters to ignore, the module hands it all trainable parameters but one and averages those gradients itself (reducer.py:
grouped in-place NCCL all-reduces issued block by block during backward, no bucket copies).  KLAB_GRAD_REDUCER=0 leaves
everything to DDP's own reducer.
"""
import os

import torch
import torch.distributed as dist
from torch import nn

from .. import functional as Fn
from ..graphs import POOL
from ..modeling import Swinv2Model, T5EncoderModel, T5ForConditionalGeneration, _compute_dtype, advance_step_seed
from ..optim import allow_overlap, wait_pending_updates


class MyModel(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        self.result_dir = args.result_dir

        self.language_model = T5EncoderModel.from_pretrained(args.language_model_name).requires_grad_(False)
        self.image_model = Swinv2Model.from_pretrained(args.image_model_name).requires_grad_(args.image_model_train)

        self.transformer = T5ForConditionalGeneration.from_pretrained(args.transformer_model_name)
        # forward() reads these only after wait_pending_updates(): an optimizer over exactly them (train.py:28) may run its update
        # on a side stream, under the towers of the next step
        allow_overlap(self.transformer.parameters())
        self.compute_dtype = _compute_dtype(getattr(args, "compute_dtype", None))
        self._klab_reducer = None
        self._tower_streams = {}

    # the one trainable tensor left to DDP's own reducer (DDP refuses a module that has nothing to reduce)
    _DDP_KEEPS = "transformer.decoder.final_layer_norm.weight"

    @property
    def _ddp_params_and_buffers_to_ignore(self):
        """Read by DistributedDataParallel.__init__ (torch/nn/parallel/distributed.py: `hasattr(module, ...)`).  Outside an
        initialised multi-rank process group -- or with KLAB_GRAD_REDUCER=0 -- nothing is ignored and DDP does all the work."""
        if os.environ.get("KLAB_GRAD_REDUCER", "1") == "0" or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() < 2:
            return []
        named = [(n, p) for n, p in self.named_parameters() if p.requires_grad and n != self._DDP_KEEPS]
        if self._klab_reducer is None and named:
            from ..reducer import GradReducer, broadcast_from_rank0
            broadcast_from_rank0([p for _, p in named])                # DDP broadcasts only the parameters it keeps
            self._klab_reducer = GradReducer([p for _, p in named])
            if named[0][1].is_cuda:
                # The collectives run during backward only: backward kernels hand out GEMM / T5-attention work dynamically and
                # the Swin attention kernels (static contiguous shares, for head affinity) leave the collective's SMs free -- a
                # 200 KB CTA cannot share an SM with an NCCL CTA, and a CTA that starts a wave late doubles the kernel's time.
                # Forward kernels keep the whole machine (functional.py: _backward_phase).
                Fn.DP_BACKWARD["on"] = os.environ.get("KLAB_DYNAMIC_SCHED", "1") != "0"
                Fn.DP_BACKWARD["reserve"] = int(os.environ.get("KLAB_SM_RESERVE", os.environ.get("NCCL_MAX_CTAS", "16")))
        return [n for n, _ in named]

    def _concat_embeddings(self, images, source_encoding):
        cd = self.compute_dtype
        src = source_encoding["input_ids"]
        pixel_values = images["pixel_values"]
        B = pixel_values.shape[0]
        # model.py:20-22: the frozen text encoder and the Swin encoder are independent until the concat.  The text tower is a
        # chain of small (B * L_src rows) latency-bound kernels; on a second stream it fills the SMs the Swin kernels leave idle.
        if src.is_cuda and os.environ.get("KLAB_TOWER_STREAM", "1") != "0":
            main = torch.cuda.current_stream()
            side = self._tower_streams.get(main.device)
            if side is None:
                side = self._tower_streams[main.device] = torch.cuda.Stream(main.device)
            side.wait_stream(main)
            with torch.cuda.stream(side), torch.no_grad():
                lang = self.language_model.hidden_before_norm(src, cd)
            img, n_img = self.image_model.features(pixel_values, cd)
            main.wait_stream(side)
            lang.record_stream(main)
        else:
            with torch.no_grad():
                lang = self.language_model.hidden_before_norm(src, cd)
            img, n_img = self.image_model.features(pixel_values, cd)
        d_img, d_lang, d_tr = img.shape[1], lang.shape[1], self.transformer.config.d_model
        if d_img != d_lang:        # torch.cat in the reference (model.py:23) raises the same way
            raise RuntimeError(f"Sizes of tensors must match except in dimension 1. Expected size {d_img} but got size {d_lang} "
                               "for tensor number 1 in the list.")
        if d_img != d_tr:
            raise RuntimeError(f"inputs_embeds width {d_img} does not match the transformer's d_model {d_tr}")
        lm, im = self.language_model, self.image_model
        emb = Fn.apply_fn(Fn.ConcatEmbeddingsFn, img, im.layernorm.weight, im.layernorm.bias, im.config.layer_norm_eps, lang,
                                          lm.encoder.final_layer_norm.weight, lm.config.layer_norm_epsilon, B)
        return emb, B, n_img + src.shape[1]

    def forward(self, images, source_encoding, target_encoding=None, return_loss=True):
        if self._klab_reducer is not None:
            ddp = getattr(torch.nn.parallel.DistributedDataParallel, "_active_ddp_module", None)      # set while DDP.forward runs
            self._klab_reducer.begin_step(ddp if ddp is not None and getattr(ddp, "module", None) is self else None)
        POOL.begin_step()
        if self.transformer.training and not Fn.pending_backward():
            advance_step_seed(images["pixel_values"].device)          # fresh dropout masks for this step (device-side counter)
        emb, B, Le = self._concat_embeddings(images, source_encoding)
        wait_pending_updates(emb.device)          # a fused-Adam step still running on its side stream wrote the transformer's weights
        if return_loss:
            return self.transformer.loss_from_embeds(emb, B, Le, target_encoding["input_ids"])
        else:
            with torch.no_grad():               # model.py:28 of the reference: greedy unless generation_config says otherwise
                return self.transformer.generate(inputs_embeds=emb.view(B, Le, emb.shape[-1]))

    def save(self, result_name="best.pth"):
        result_path = os.path.join(self.args.result_dir, result_name)
        checkpoints = {'transformer': self.transformer.state_dict()}
        if self.args.image_model_train:
            checkpoints['image_model'] = self.image_model.state_dict()
        torch.save(checkpoints, result_path)

    def load(self, result_name="best.pth"):
        result_path = os.path.join(self.args.result_dir, result_name)
        checkpoints = torch.load(result_path)
        self.transformer.load_state_dict(checkpoints['transformer'])
        if self.args.image_model_train:
            self.image_model.load_state_dict(checkpoints['image_model'])

    # ---- true resume (SURVEY.md 8f N4, the optional half): the reference saves weights only (train.py:88-104 never stores the
    # optimizer, the scheduler or the epoch, so a run cannot be continued).  `save_state` writes the reference's file format plus
    # three extra keys -- the reference's own `load` ignores them, so the files stay interchangeable -- and `load_state` restores
    # everything it finds.
    def save_state(self, result_name="last.pth", optimizer=None, scheduler=None, epoch=None, step=None):
        result_path = os.path.join(self.args.result_dir, result_name)
        checkpoints = {'transformer': self.transformer.state_dict()}
        if self.args.image_model_train:
            checkpoints['image_model'] = self.image_model.state_dict()
        if optimizer is not None:
            checkpoints['optimizer'] = optimizer.state_dict()
        if scheduler is not None:
            checkpoints['scheduler'] = scheduler.state_dict()
        checkpoints['progress'] = {'epoch': epoch, 'step': step}
        torch.save(checkpoints, result_path)

    def load_state(self, result_name="last.pth", optimizer=None, scheduler=None):
        """-> {'epoch': ..., 'step': ...} (None entries for a weights-only file written by the reference)."""
        result_path = os.path.join(self.args.result_dir, result_name)
        checkpoints = torch.load(result_path, map_location=next(self.transformer.parameters()).device)
        self.transformer.load_state_dict(checkpoints['transformer'])
        if self.args.image_model_train and 'image_model' in checkpoints:
            self.image_model.load_state_dict(checkpoints['image_model'])
        if optimizer is not None and 'optimizer' in checkpoints:
            optimizer.load_state_dict(checkpoints['optimizer'])
        if scheduler is not None and 'scheduler' in checkpoints:
            scheduler.load_state_dict(checkpoints['scheduler'])
        return dict(checkpoints.get('progress') or {'epoch': None, 'step': None})
