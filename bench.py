#!/usr/bin/env python
"""Headline benchmark: train samples/sec of the Swin-V2 + T5 image-caption step (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|hf_eager] [--workload 2a|3|4a|5|2b|1a|tiny] [--batch B]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step of our arm computed as DIR/<name>.npy (float32 / float64), so that two builds
run with the same arguments can be compared output for output (inputs, weights and dropout masks are seeded):
  training workloads: loss.npy (the loss the step read back) and transformer_params.npy (a fixed seeded sample of 2^20
                      elements of the transformer weights after the step's Adam update)
  decode workload 5:  generated_ids.npy (the greedy ids of the last generate() call, as float64)
Two runs agree only as far as the step is deterministic: the shared-embedding and T5 relative-bias gradients are summed with
floating-point atomics whose order varies from run to run, and over several bf16 training steps those last-bit differences
in the weights spread to every later gradient and weight update.

A "step" is exactly what /root/reference/train.py:54-71 does per batch with accumulation_steps = 1:
    (host->device copy of the batch) -> loss = model(images, src, tgt) -> loss.item() -> loss.backward() ->
    optimizer.step() (Adam over model.transformer.parameters(), train.py:28) -> optimizer.zero_grad()
with `model.transformer.train()` (T5 dropout p = 0.1 active, train.py:52) and DistributedDataParallel for N > 1.

Workload at N = 1 ("2a", BASELINE.json configs[1] realised as SURVEY.md 8d recommends because Swin-B + T5-base cannot be
concatenated, 1024 != 768): Swin-B/256/window 8 trained jointly + T5-large, bf16 tensor-core path, batch 64 per GPU,
32 source + 32 target tokens, synthetic inputs, random-init weights.  One JSON line on stdout (rank 0).

  value          : whole-job samples/s with the batch already resident in HBM (timed with CUDA events, max over ranks)
  e2e            : same through the public API with HOST (pinned) inputs: H2D copies and the loss read-back inside the timed region
  roofline       : the dominant kernel family (tcgen05 GEMM, ~97% of the FLOPs): algorithmic FLOPs of every GEMM launch of one
                   step / CUDA-event duration of those launches, against MEASURED_PEAKS.json (sustained bf16 figure)
  cpu_baseline   : the oracle port of the reference path (oracle/, plain torch fp32) on the host cores, bounded sample
  --impl reference : the reference's CPU path as its own arm: the reference is ~40 lines of glue over `transformers`
                   (/root/reference/models/model.py:19-26) and /root/reference does not exist on the GPU box, so the arm runs the
                   SAME transformers classes wired the same way (T5EncoderModel + Swinv2Model + T5ForConditionalGeneration, fp32,
                   transformer.train(), torch.optim.Adam) on the host cores; if `transformers` cannot be imported the oracle port
                   (oracle/, plain torch) stands in and the line says kind "port"
  --impl hf_eager  : informational: the same transformers modules on the B200 under torch.autocast(bfloat16) -- the eager
                   PyTorch path SURVEY.md 2.1 names as the real competitor (cuBLAS / cuDNN / ATen kernels)

At N = 1 the default run also measures BASELINE.json configs[2..4] (workloads 3, 4a and 5, each in its own process so that its
memory is gone before the headline workload runs) and reports them under "workloads" in the same JSON line, plus the step time
with the unchanged-train.py optimizer (torch.optim.Adam) under "torch_optimizer" and the HF-eager leg under "hf_eager_gpu".
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# GFLOP per sample, fwd+bwd, counted on the reference graph (BASELINE.md section 3)
WORKLOADS = {
    "2a": dict(desc="MSCOCO caption train step, Swin-B/256/w8 trained jointly + T5-large (runnable realisation of configs[1])",
               swin=dict(image_size=256, embed_dim=128, depths=(2, 2, 18, 2), num_heads=(4, 8, 16, 32), window_size=8),
               t5="t5-large", batch=64, l_src=32, l_tgt=32, train_swin=True, gflop_per_sample=422.14),
    "3": dict(desc="RedCaps span-corruption pretrain step (15% of words masked, <extra_id_n> sentinels), Swin-B/256/w8 + T5-large, 64 source + 32 target tokens (configs[2])",
              swin=dict(image_size=256, embed_dim=128, depths=(2, 2, 18, 2), num_heads=(4, 8, 16, 32), window_size=8),
              t5="t5-large", batch=64, l_src=64, l_tgt=32, train_swin=True, gflop_per_sample=511.83, span_corruption=True),
    "4a": dict(desc="high-res caption step, Swin-B/384/window 12 + T5-large, 128-token targets (runnable realisation of configs[3])",
               swin=dict(image_size=384, embed_dim=128, depths=(2, 2, 18, 2), num_heads=(4, 8, 16, 32), window_size=12),
               t5="t5-large", batch=64, l_src=32, l_tgt=128, train_swin=True, gflop_per_sample=990.98),
    "5": dict(desc="greedy caption decode, Swin-S/256/w8 + T5-base decoder with cross-attention KV cache over the Swin tokens, batch 256, 20 new tokens, single B200 (configs[4])",
              swin=dict(image_size=256, embed_dim=96, depths=(2, 2, 18, 2), num_heads=(3, 6, 12, 24), window_size=8),
              t5="t5-base", batch=256, l_src=32, l_tgt=20, train_swin=False, gflop_per_sample=0.0, decode=True),
    "2b": dict(desc="MSCOCO caption train step, Swin-S/256/w8 trained jointly + T5-base",
               swin=dict(image_size=256, embed_dim=96, depths=(2, 2, 18, 2), num_heads=(3, 6, 12, 24), window_size=8),
               t5="t5-base", batch=64, l_src=32, l_tgt=32, train_swin=True, gflop_per_sample=157.01),
    "1a": dict(desc="MSCOCO caption train step, frozen Swin-T/224/w7 + T5-base (runnable realisation of configs[0])",
               swin=dict(image_size=224, embed_dim=96, depths=(2, 2, 6, 2), num_heads=(3, 6, 12, 24), window_size=7),
               t5="t5-base", batch=2, l_src=32, l_tgt=32, train_swin=False, gflop_per_sample=87.53),
    "tiny": dict(desc="smoke-sized step", swin=dict(image_size=64, embed_dim=32, depths=(2, 2, 2), num_heads=(1, 2, 4), window_size=4),
                 t5=dict(vocab_size=512, d_model=128, d_ff=256, num_layers=2, num_heads=2), batch=4, l_src=8, l_tgt=8,
                 train_swin=True, gflop_per_sample=0.05),
}
T5_NAMED = {"t5-small": dict(d_model=512, d_ff=2048, num_layers=6, num_heads=8),
            "t5-base": dict(d_model=768, d_ff=3072, num_layers=12, num_heads=12),
            "t5-large": dict(d_model=1024, d_ff=4096, num_layers=24, num_heads=16)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(tflops=p.get("bf16_tflops_sustained", 1378.2), burst=p.get("bf16_tflops", 1632.1), hbm=p.get("hbm_gbs", 6450.3),
                    source="measured")
    return dict(tflops=1400.0, burst=1590.0, hbm=6650.0, source="fallback")


def synth_batch(w, vocab, seed, pin):
    g = torch.Generator().manual_seed(seed)
    s = w["swin"]["image_size"]
    px = torch.randn(w["batch"], 3, s, s, generator=g)
    src = torch.randint(2, vocab - 28, (w["batch"], w["l_src"]), generator=g)
    tgt = torch.randint(2, vocab - 28, (w["batch"], w["l_tgt"]), generator=g)
    tgt[:, -1] = 1
    if pin:
        px, src, tgt = px.pin_memory(), src.pin_memory(), tgt.pin_memory()
    return px, src, tgt


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def summary(self, lo, hi):
        rows = [r for r in self.rows[lo:max(hi, lo + 1)] if len(r) >= 6 and r[0].isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(int(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": reasons, "samples": len(rows)}

    def stop(self):
        if self.proc:
            self.proc.terminate()


# --------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline / hf_eager leg: the reference's own code path (transformers), or the oracle port
# --------------------------------------------------------------------------------------------------------------
def _dims(w):
    t5kw = T5_NAMED[w["t5"]] if isinstance(w["t5"], str) else w["t5"]
    sw = dict(w["swin"])
    sw.setdefault("pretrained_window_sizes", (0,) * len(sw["depths"]))
    return t5kw, sw


def hf_reference_steps(w, steps, warmup, batch, device, autocast, log=lambda *_: None):
    """The reference step with the reference's own engine: `transformers` modules wired exactly as
    /root/reference/models/model.py:14-26 (frozen T5EncoderModel under no_grad, Swinv2Model, torch.cat(dim=1),
    T5ForConditionalGeneration(inputs_embeds, labels).loss) and driven as /root/reference/train.py:52-67 does
    (transformer.train(), loss.item(), backward, torch.optim.Adam over the transformer, zero_grad).  Random-init weights
    (no checkpoints offline).  Returns per-step seconds (host clock around a synchronised step)."""
    from transformers import Swinv2Config, Swinv2Model, T5Config, T5EncoderModel, T5ForConditionalGeneration
    t5kw, sw = _dims(w)

    def tcfg():                                       # T5EncoderModel edits the config object it is given: one per model
        return T5Config(vocab_size=t5kw.get("vocab_size", 32128), d_model=t5kw["d_model"], d_kv=t5kw.get("d_kv", 64), d_ff=t5kw["d_ff"],
                        num_layers=t5kw["num_layers"], num_heads=t5kw["num_heads"], decoder_start_token_id=0)
    scfg = Swinv2Config(image_size=sw["image_size"], embed_dim=sw["embed_dim"], depths=list(sw["depths"]), num_heads=list(sw["num_heads"]),
                        window_size=sw["window_size"], pretrained_window_sizes=list(sw["pretrained_window_sizes"]))
    torch.manual_seed(0)
    with torch.device(device):
        lm = T5EncoderModel(tcfg()).requires_grad_(False).eval()
        im = Swinv2Model(scfg).requires_grad_(w["train_swin"]).eval()
        tr = T5ForConditionalGeneration(tcfg())
    tr.train()                                                       # train.py:52
    opt = torch.optim.Adam(tr.parameters(), lr=1e-4)                 # train.py:28
    wb = dict(w, batch=batch)
    px, src, tgt = synth_batch(wb, t5kw.get("vocab_size", 32128), 1234, pin=False)
    px, src, tgt = px.to(device), src.to(device), tgt.to(device)
    cuda = torch.device(device).type == "cuda"
    times = []
    for i in range(warmup + steps):
        if cuda:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.autocast(torch.device(device).type, dtype=torch.bfloat16, enabled=autocast):
            with torch.no_grad():
                lang = lm(input_ids=src).last_hidden_state
            img = im(pixel_values=px).last_hidden_state
            loss = tr(inputs_embeds=torch.cat((img, lang), dim=1), labels=tgt).loss
        lv = loss.item()
        loss.backward()
        opt.step()
        opt.zero_grad()
        if cuda:
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        log(f"hf step {i}: {dt:.3f}s loss {lv:.3f}")
        if i >= warmup:
            times.append(dt)
    return times


def hf_generate_calls(w, steps, warmup, device, log=lambda *_: None):
    """/root/reference/models/model.py:20-23,28 with the reference's engine on the GPU: frozen text encoder + Swin + concat, then
    `transformer.generate(inputs_embeds=...)` (greedy, 20 new tokens, EOS disabled for a fixed length) under bf16 autocast."""
    from transformers import Swinv2Config, Swinv2Model, T5Config, T5EncoderModel, T5ForConditionalGeneration
    t5kw, sw = _dims(w)

    def tcfg():
        return T5Config(vocab_size=t5kw.get("vocab_size", 32128), d_model=t5kw["d_model"], d_kv=t5kw.get("d_kv", 64), d_ff=t5kw["d_ff"],
                        num_layers=t5kw["num_layers"], num_heads=t5kw["num_heads"], decoder_start_token_id=0)
    scfg = Swinv2Config(image_size=sw["image_size"], embed_dim=sw["embed_dim"], depths=list(sw["depths"]), num_heads=list(sw["num_heads"]),
                        window_size=sw["window_size"], pretrained_window_sizes=list(sw["pretrained_window_sizes"]))
    torch.manual_seed(0)
    with torch.device(device):
        lm, im, tr = T5EncoderModel(tcfg()).eval(), Swinv2Model(scfg).eval(), T5ForConditionalGeneration(tcfg()).eval()
    px, src, _ = synth_batch(w, t5kw.get("vocab_size", 32128), 1234, pin=False)
    px, src = px.to(device), src.to(device)
    times = []
    for i in range(warmup + steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            emb = torch.cat((im(pixel_values=px).last_hidden_state, lm(input_ids=src).last_hidden_state), dim=1)
            ids = tr.generate(inputs_embeds=emb, max_new_tokens=w["l_tgt"], min_new_tokens=w["l_tgt"], do_sample=False)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        log(f"hf generate {i}: {dt:.3f}s ids {tuple(ids.shape)}")
        if i >= warmup:
            times.append(dt)
    return times


def oracle_port_steps(w, steps, warmup, sample_batch, log=lambda *_: None):
    """fwd + bwd + Adam step of the reference path restated in oracle/ (plain torch fp32 on the host cores); used only where
    `transformers` does not import."""
    from oracle.caption_model import caption_loss, swin_param_shapes, t5_param_shapes
    from oracle.swinv2 import SwinDims
    from oracle.t5 import T5Dims
    t5kw, sw = _dims(w)
    t5 = T5Dims(**t5kw)
    swin = SwinDims(**sw)
    g = torch.Generator().manual_seed(0)

    def make(shapes, train):
        sd, tied = {}, ("encoder.embed_tokens.weight", "decoder.embed_tokens.weight", "lm_head.weight")
        for k, shp in shapes.items():
            if k in tied:
                continue
            if len(shp) == 1 and k.endswith("weight"):
                t = torch.ones(shp)
            elif k.endswith("bias"):
                t = torch.zeros(shp)
            elif k.endswith("logit_scale"):
                t = torch.full(shp, 2.302585)
            else:
                t = torch.randn(shp, generator=g) * (1.0 if k == "shared.weight" else shp[-1] ** -0.5 * 0.5)
            sd[k] = t.requires_grad_(train)
        for k in tied:
            if k in shapes:
                sd[k] = sd["shared.weight"]
        return sd

    sds = {"language_model": make(t5_param_shapes(t5, encoder_only=True), False),
           "image_model": make(swin_param_shapes(swin), w["train_swin"]),
           "transformer": make(t5_param_shapes(t5), True)}
    params = list({id(v): v for v in sds["transformer"].values()}.values())
    opt = torch.optim.Adam(params, lr=1e-3)
    wb = dict(w, batch=sample_batch)
    px, src, tgt = synth_batch(wb, t5.vocab_size, 1234, pin=False)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss = caption_loss(px, src, tgt, sds, t5, swin, t5)
        lv = loss.item()
        loss.backward()
        opt.step()
        opt.zero_grad()
        dt = time.perf_counter() - t0
        log(f"cpu step {i}: {dt:.2f}s loss {lv:.3f}")
        if i >= warmup:
            times.append(dt)
    return times


def cpu_reference_steps(w, steps, warmup, sample_batch, log=lambda *_: None):
    """-> (per-step seconds, kind, engine): the reference's CPU path on all host threads, on a bounded sample of the workload."""
    torch.set_num_threads(os.cpu_count() or 1)
    if w.get("decode"):
        raise ValueError("the CPU arm times training workloads")
    try:
        import transformers
        times = hf_reference_steps(w, steps, warmup, sample_batch, "cpu", False, log)
        return times, "reference", (f"transformers {transformers.__version__} eager fp32 on the host cores: the reference's own engine, its three "
                                    "models wired as /root/reference/models/model.py:19-26 (that glue is restated in bench.py because "
                                    "/root/reference does not exist on the GPU box), transformer.train() (dropout on), torch.optim.Adam")
    except ImportError:
        return oracle_port_steps(w, steps, warmup, sample_batch, log), "port", "oracle/ (plain torch fp32 restatement), dropout off"


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if w.get("decode"):
        emit({"impl": "reference", "unavailable": "the CPU reference arm times the training step (workloads 2a / 3 / 4a); workload 5 is decode"})
        return
    sample = args.cpu_sample_batch
    times, kind, engine = cpu_reference_steps(w, args.steps, args.warmup, sample, log=lambda m: print(m, file=sys.stderr))
    ms = 1e3 * sum(times) / len(times)
    val = sample / (ms / 1e3)
    cores = os.cpu_count() or 1
    line = {
        "impl": "reference", "metric": "train samples/sec (Swin+T5 caption step)", "value": val, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "name": args.workload, "per_step_sample_batch": sample, "l_src": w["l_src"], "l_tgt": w["l_tgt"],
                   "dropout": "T5 p=0.1 active (train.py:52)" if kind == "reference" else "off"},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": kind, "engine": engine,
                         "sample": f"{sample} samples/step of the same model + sequence lengths, fwd+bwd+Adam, fp32, {cores} threads"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def run_hf_eager(args, w):
    """Informational leg: the reference's engine (transformers eager) on the SAME B200 under torch.autocast(bfloat16), full batch."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    try:
        import transformers
        dev = "cuda:0"
        torch.cuda.set_device(0)
        if w.get("decode"):
            times = hf_generate_calls(w, args.steps, max(args.warmup, 2), dev, log=lambda m: print(m, file=sys.stderr))
        else:
            times = hf_reference_steps(w, args.steps, max(args.warmup, 2), w["batch"], dev, True, log=lambda m: print(m, file=sys.stderr))
    except Exception as e:                                                           # noqa: BLE001  (informational: never fails the run)
        emit({"impl": "hf_eager", "unavailable": f"{type(e).__name__}: {str(e)[:200]}"})
        return
    ms = 1e3 * sum(times) / len(times)
    if w.get("decode"):
        emit({"impl": "hf_eager", "metric": "greedy decode tokens/sec (T5 decoder with cross-attention KV cache)",
              "value": w["batch"] * w["l_tgt"] / (ms / 1e3), "unit": "tokens/s", "n_gpus": 1, "steps": args.steps, "ms_per_step": ms,
              "dtype": "bf16 autocast (fp32 parameters)", "data": "synthetic",
              "config": {"workload": w["desc"], "name": args.workload, "batch_per_gpu": w["batch"], "new_tokens": w["l_tgt"], "eos": "disabled (fixed length)"},
              "engine": f"transformers {transformers.__version__} generate(inputs_embeds=...) eager + torch {torch.__version__}",
              "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)})
        return
    emit({"impl": "hf_eager", "metric": "train samples/sec (Swin+T5 caption step)", "value": w["batch"] / (ms / 1e3), "unit": "samples/s",
          "n_gpus": 1, "steps": args.steps, "ms_per_step": ms, "dtype": "bf16 autocast (fp32 parameters)", "data": "synthetic",
          "config": {"workload": w["desc"], "name": args.workload, "batch_per_gpu": w["batch"], "l_src": w["l_src"], "l_tgt": w["l_tgt"]},
          "engine": f"transformers {transformers.__version__} eager + torch {torch.__version__} (cuBLAS / cuDNN / ATen), torch.optim.Adam",
          "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)})


# --------------------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------------------
def build_model(w, device, dtype):
    import types

    from klab_multimodalmodel_b200.modeling import Swinv2Config, T5Config, init_swin_, init_t5_
    from klab_multimodalmodel_b200.models.model import MyModel
    t5kw = T5_NAMED[w["t5"]] if isinstance(w["t5"], str) else w["t5"]
    tcfg = T5Config(**t5kw)
    sw = dict(w["swin"])
    sw.setdefault("pretrained_window_sizes", (0,) * len(sw["depths"]))
    scfg = Swinv2Config(**sw)
    args = types.SimpleNamespace(result_dir="/tmp", language_model_name=tcfg, image_model_name=scfg, image_model_train=w["train_swin"],
                                 transformer_model_name=tcfg, compute_dtype=dtype)
    model = MyModel(args)
    init_t5_(model.language_model, seed=1)
    init_swin_(model.image_model, seed=2)
    init_t5_(model.transformer, seed=3)
    return model.to(device), tcfg


def _sig_operands(sig, dev, copies, seedp):
    """Operand sets for one GEMM signature: `copies` independent (A, B, out, epilogue tensors) groups."""
    M, N, K, a_mn, b_mn, od, has_bias, act, res_dt, ain_dt, has_aout, p_drop, acc, ldd = sig
    sets = []
    for _ in range(copies):
        A = torch.randn((K, M) if a_mn else (M, K), device=dev).bfloat16()
        B = torch.randn((K, N) if b_mn else (N, K), device=dev).bfloat16()
        D = torch.zeros(M, ldd, device=dev, dtype=od)[:, :N]
        kw = dict(a_mn=a_mn, b_mn=b_mn, out=D, act=act, dropout_p=p_drop, accumulate=acc, seed=5, seed_ptr=seedp if p_drop > 0 else None)
        if has_bias:
            kw["bias"] = torch.randn(N, device=dev)
        if res_dt is not None:
            kw["residual"] = torch.randn(M, N, device=dev).to(res_dt)
        if ain_dt is not None:
            kw["aux_in"] = torch.randn(M, N, device=dev).to(ain_dt)
        if has_aout:
            kw["aux_out"] = torch.empty(M, N, device=dev, dtype=od)
        sets.append((A, B, kw))
    return sets


def _sig_bytes(sig):
    """Algorithmic HBM bytes of one launch: every operand / epilogue tensor read or written once."""
    M, N, K, a_mn, b_mn, od, has_bias, act, res_dt, ain_dt, has_aout, p_drop, acc, ldd = sig
    esz = 2 if od == torch.bfloat16 else 4
    return (M * K + N * K) * 2 + M * N * esz * (1 + bool(acc) + has_aout) + (M * N * 2 if res_dt == torch.bfloat16 else M * N * 4 if res_dt is not None else 0) + \
        (M * N * 2 if ain_dt is not None else 0) + (N * 4 if has_bias else 0)


def gemm_roofline(model_step, pk, verbose=False, check=False, isolated=True):
    """Roofline of the dominant kernel family (tcgen05 GEMM, ~97 % of the FLOPs).
    (1) run one step eagerly and record the signature of EVERY GEMM launch in order (M, N, K, operand majors, output dtype and
        the fused epilogue: bias / activation / residual / aux tensors / dropout / accumulate);
    (2) SUSTAINED figure (`achieved`, `frac`): all launches of the step, in step order, each signature on its own operand set
        (together far beyond the 126 MB L2, consecutive launches never share operands), captured into ONE CUDA graph and
        replayed back to back for >= 0.4 s under CUDA events -- the GEMM work of several steps with nothing in between, i.e.
        the power / clock state of a long step.  Peak = MEASURED_PEAKS.json sustained bf16.
    (3) ISOLATED figure (`achieved_isolated`, `frac_burst`): each distinct signature replayed alone (8 launches, operands
        rotated beyond L2), idle gaps between signatures -- a kernel timed alone, so the burst peak applies.  Also gives the
        per-signature table (--verbose) that says which shapes lose."""
    import collections

    from klab_multimodalmodel_b200 import ops as O
    from klab_multimodalmodel_b200.graphs import POOL
    order = []
    orig = O.gemm

    def rec(a, b, M, N, K, **kw):
        out = orig(a, b, M, N, K, **kw)
        if a.dtype == torch.bfloat16:
            res, ain, aout = kw.get("residual"), kw.get("aux_in"), kw.get("aux_out")
            order.append((M, N, K, bool(kw.get("a_mn")), bool(kw.get("b_mn")), out.dtype, kw.get("bias") is not None, int(kw.get("act", 0)),
                          None if res is None else res.dtype, None if ain is None else ain.dtype, aout is not None,
                          float(kw.get("dropout_p", 0.0)), bool(kw.get("accumulate", False)), out.stride(0)))
        return out

    was = POOL.enabled
    O.gemm, POOL.enabled = rec, False
    try:
        model_step()
        torch.cuda.synchronize()
    finally:
        O.gemm, POOL.enabled = orig, was
    sigs = collections.Counter(order)
    dev = torch.device("cuda", torch.cuda.current_device())
    seedp = torch.zeros(1, dtype=torch.int64, device=dev)
    tot_fl = sum(2.0 * s[0] * s[1] * s[2] for s in order)
    tot_bytes = sum(_sig_bytes(s) for s in order)

    # ---- (2) sustained: the step's launch sequence, one graph, replayed continuously
    opsets = {sig: _sig_operands(sig, dev, 1, seedp)[0] for sig in sigs}
    for sig, (A, B, kw) in opsets.items():                          # eager first (per-signature autotune must not run under capture)
        orig(A, B, sig[0], sig[1], sig[2], **kw)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for sig in order:
            A, B, kw = opsets[sig]
            orig(A, B, sig[0], sig[1], sig[2], **kw)
    g.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); g.replay(); e.record()
    torch.cuda.synchronize()
    once = s.elapsed_time(e)
    reps = max(3, int(400.0 / max(once, 1e-3)) + 1)
    s.record()
    for _ in range(reps):
        g.replay()
    e.record()
    torch.cuda.synchronize()
    sus_ms = s.elapsed_time(e) / reps
    del g, opsets
    ach = tot_fl / (sus_ms * 1e-3) / 1e12 if sus_ms > 0 else 0.0

    # ---- (3) isolated per-signature timings
    iso_ms, rows = None, []
    if isolated:
        iso_ms = 0.0
        for sig, cnt in sigs.items():
            M, N, K, a_mn, b_mn, od, has_bias, act, res_dt, ain_dt, has_aout, p_drop, acc, ldd = sig
            copies = max(1, min(8, (300 << 20) // max(_sig_bytes(sig), 1)))
            sets = _sig_operands(sig, dev, copies, seedp)
            for i in range(3):
                A, B, kw = sets[i % copies]
                orig(A, B, M, N, K, **kw)
            iters = 8
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()                      # replay from a CUDA graph, as the step does: no host launch cost in the timing
            with torch.cuda.graph(g):
                for i in range(iters):
                    A, B, kw = sets[i % copies]
                    orig(A, B, M, N, K, **kw)
            g.replay()
            s.record(); g.replay(); e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / iters
            del g
            err = None
            if check and p_drop == 0.0 and not acc and act in (0, 1, 2):
                A, B, kw = sets[0]
                kw = dict(kw); D = torch.zeros(M, ldd, device=dev, dtype=od)[:, :N]; kw["out"] = D
                orig(A, B, M, N, K, **kw)
                A32 = A.float().t() if a_mn else A.float()
                B32 = B.float() if b_mn else B.float().t()
                ref = A32 @ B32
                if has_bias:
                    ref = ref + kw["bias"]
                if act == 1:
                    ref = torch.relu(ref)
                elif act == 2:
                    ref = torch.nn.functional.gelu(ref)
                if res_dt is not None:
                    ref = ref + kw["residual"].float()
                err = ((D.float() - ref).abs().max() / ref.abs().max().clamp_min(1e-6)).item()
            fl = 2.0 * M * N * K
            iso_ms += cnt * ms
            rows.append((cnt * ms, cnt, M, N, K, int(a_mn), int(b_mn), ms, fl / ms / 1e9, sig[6:13], err, _sig_bytes(sig) / ms / 1e6))
            del sets
        if verbose:
            for r in sorted(rows, reverse=True)[:(200 if check else 40)]:
                print("gemm sig: total %.2f ms  x%d  M=%d N=%d K=%d a_mn=%d b_mn=%d  %.1f us  %.0f TFLOP/s  %.0f GB/s  epi(bias,act,res,auxin,auxout,p,acc)=%s%s" %
                      (r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7] * 1e3, r[8], r[11], r[9], "" if r[10] is None else "  relerr %.2e" % r[10]),
                      file=sys.stderr)
    traffic = _gemm_traffic_from_profiles()
    out = {"bound": "tensor", "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"],
           "traffic": traffic.get("bytes_per_launch") if traffic else None, "traffic_detail": traffic,
           "kernel": "gemm_bf16_tc_kernel (tcgen05)", "launches_per_step": len(order), "distinct_shapes": len(sigs),
           "gemm_ms_per_step": sus_ms, "gemm_gflop_per_step": tot_fl / 1e9, "algorithmic_gb_per_step": tot_bytes / 1e9,
           "peak_source": pk["source"] + " bf16 SUSTAINED (applies: the launches run back to back for >= 0.4 s, like inside a long step)",
           "frac_sustained": ach / pk["tflops"], "peak_burst": pk["burst"],
           "method": "every GEMM launch of one step (shape, operand majors and fused epilogue: bias / activation / residual / aux "
                     "tensors / dropout), in step order, each signature on its own operands (working set far beyond L2), captured in one "
                     f"CUDA graph and replayed {reps}x back to back under CUDA events"}
    if iso_ms:
        ach_iso = tot_fl / (iso_ms * 1e-3) / 1e12
        out.update({"achieved_isolated": ach_iso, "frac_burst": ach_iso / pk["burst"], "gemm_ms_per_step_isolated": iso_ms,
                    "isolated_method": "each distinct signature replayed alone (8 launches from a CUDA graph, operands rotated beyond L2), idle "
                                       "gaps between signatures: a kernel timed alone, so the BURST peak applies to this figure"})
    return out


def _gemm_traffic_from_profiles():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the top GEMM signatures, from the committed `ncu --set full`
    capture (profiles/r02_gemm_top_traffic.json, written by scripts/ncu_gemm_top.py + scripts/ncu_summarise.py)."""
    path = os.path.join(ROOT, "profiles", "r02_gemm_top_traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as fh:
        return json.load(fh)


DUMP_SAMPLE = 1 << 20
DUMP_MAX_BYTES = 64 << 20


def _flat_sample(tensors, n, seed):
    """A fixed, seeded sample of n elements (drawn with replacement, in index order) of `tensors` taken as one flat vector, as
    float32 on the host; every element when they hold no more than n."""
    import numpy as np
    sizes = [t.numel() for t in tensors]
    total = sum(sizes)
    if total <= n:
        return torch.cat([t.detach().reshape(-1).float().cpu() for t in tensors]).numpy()
    idx = torch.randint(total, (n,), generator=torch.Generator().manual_seed(seed)).sort().values
    out, off, lo = [], 0, 0
    for t, s in zip(tensors, sizes):
        hi = int(torch.searchsorted(idx, off + s))
        if hi > lo:
            out.append(t.detach().reshape(-1)[(idx[lo:hi] - off).to(t.device)].float().cpu())
        off, lo = off + s, hi
    return np.concatenate([o.numpy() for o in out])


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy (float32 / float64 only, DUMP_MAX_BYTES in all)."""
    import numpy as np
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    print(f"[bench] wrote {', '.join(f'{k}.npy {tuple(a.shape)}' for k, a in arrays.items())} to {out_dir}", file=sys.stderr)


def _timed_steps(fn, k, flush, world, dev):
    """Time EXACTLY k steps as ONE region: barrier + synchronize, start event, k x (L2 flush, step), wait for every side stream the
    steps left work on (the fused Adam runs on its own stream and overlaps the NEXT step's towers), end event, synchronize; max over
    ranks.  The flush -- a 256 MiB memset, ~40 us -- sits INSIDE the region: per-step brackets with the flush outside (the earlier
    scheme) would stop the clock before the optimizer's side stream has finished and would hide it."""
    import torch.distributed as dist
    from klab_multimodalmodel_b200.optim import wait_pending_updates
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last = None
    s.record()
    for _ in range(k):
        flush.zero_()                                                   # L2 flush between timed iterations (timed)
        last = fn()
    wait_pending_updates(dev)                                           # the last optimizer step is part of the k steps
    e.record()
    torch.cuda.synchronize()
    total = s.elapsed_time(e)
    if world > 1:
        dist.barrier()
    t = torch.tensor([total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item(), last


def _timed_steps_isolated(fn, k, flush, dev):
    """Secondary figure: every step bracketed alone (flush outside, synchronize after each step, the optimizer's side stream waited
    for inside the bracket): no overlap across steps, comparable with the round-1 numbers."""
    from klab_multimodalmodel_b200.optim import wait_pending_updates
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(k):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        wait_pending_updates(dev)
        e.record()
        torch.cuda.synchronize()
        total += s.elapsed_time(e)
    return total


def dp_parity_check(model, net, w, vocab, world, rank, dev, batch):
    """Data-parallel parity (SURVEY.md section 4, "Distributed"): one dropout-off step.  Every rank runs forward + backward on
    its own shard through DDP (gradients averaged by the reducer); rank 0 then recomputes ALL shards locally with the exchange
    switched off, accumulating gradient / world -- the single-process run on the concatenated batch -- and reports the largest
    per-tensor relative difference (Frobenius) between the two."""
    import torch.distributed as dist
    was_training = model.transformer.training
    model.transformer.eval()
    params = [(n, p) for n, p in model.named_parameters() if p.requires_grad]

    def shard(r):
        px, src, tgt = synth_batch(dict(w, batch=batch), vocab, 4321 + r, pin=False)
        return {"pixel_values": px.to(dev)}, {"input_ids": src.to(dev)}, {"input_ids": tgt.to(dev)}

    for _, p in params:
        p.grad = None
    net(*shard(rank)).backward()
    torch.cuda.synchronize()
    avg = {n: p.grad.detach().clone() for n, p in params}
    dist.barrier()
    out = None
    if rank == 0:
        red = getattr(model, "_klab_reducer", None)
        if red is not None:
            red.enabled = False
        for _, p in params:
            p.grad = None
        try:
            for r in range(world):
                (model(*shard(r)) / world).backward()
        finally:
            if red is not None:
                red.enabled = True
        torch.cuda.synchronize()
        worst, name = 0.0, None
        for n, p in params:
            if p.grad is None:
                continue
            d = (p.grad.double() - avg[n].double()).norm().item() / max(p.grad.double().norm().item(), 1e-30)
            if d > worst:
                worst, name = d, n
        out = {"max_rel_err": worst, "at": name, "tensors": len(params), "batch_per_rank": batch, "ok": bool(worst <= 1e-3),
               "how": "DDP-averaged gradients of one dropout-off step vs rank 0 recomputing every rank's shard locally (sum / world)"}
    for _, p in params:
        p.grad = None
    dist.barrier()
    model.transformer.train(was_training)
    return out


def run_sub(extra_args, timeout_s):
    """Run `python bench.py <extra_args>` in its own process (GPU memory isolated) and return its JSON line (or an error dict)."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py")] + extra_args
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, cwd=ROOT, env=env)
    except subprocess.TimeoutExpired:
        return {"error": f"timed out after {timeout_s} s", "cmd": " ".join(extra_args)}
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    if r.returncode != 0 or not lines:
        return {"error": f"rc {r.returncode}: {r.stderr.strip()[-300:]}", "cmd": " ".join(extra_args)}
    try:
        return json.loads(lines[-1])
    except ValueError:
        return {"error": "unparsable output", "cmd": " ".join(extra_args)}


def run_decode(args, w):
    """Workload 5 (BASELINE.json configs[4]): `model(images, source_encoding, return_loss=False)` = Swin + frozen text tower +
    T5 encoder once, then 20 KV-cached single-token decoder steps (EOS disabled: fixed length, as SURVEY.md 8d prescribes)."""
    from klab_multimodalmodel_b200 import _lib as L
    from klab_multimodalmodel_b200 import ops as O
    from klab_multimodalmodel_b200.generation import greedy_generate
    from klab_multimodalmodel_b200.graphs import POOL
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    L.check(L.lib().klab_check_device())
    model, tcfg = build_model(w, dev, args.dtype)
    model.eval()
    model.transformer.config.eos_token_id = -1                      # never finishes early: exactly T tokens per sample
    T, B = w["l_tgt"], w["batch"]
    px_h, src_h, _ = synth_batch(w, tcfg.vocab_size, 1234, pin=True)
    px_d, src_d = px_h.to(dev), src_h.to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def api_call(px, src):
        return model({"pixel_values": px}, {"input_ids": src}, return_loss=False)

    def resident():
        return api_call(px_d, src_d)

    def e2e():
        ids = api_call(px_h.to(dev, non_blocking=True), src_h.to(dev, non_blocking=True))
        return ids.cpu()

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            ids = resident()
        torch.cuda.synchronize()
        sampler = ClockSampler(0)
        time.sleep(0.3)
        lo = sampler.mark()
        l0 = O.launch_count() + POOL.replayed_kernels
        ms_res, ids = _timed_steps(resident, args.steps, flush, 1, dev)
        launches = O.launch_count() + POOL.replayed_kernels - l0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"generated_ids": ids.cpu().double().numpy()})
        hi = sampler.mark()
        for _ in range(max(args.warmup, 3)):
            e2e()
        ms_e2e, _ = _timed_steps(e2e, args.steps, flush, 1, dev)
        clocks = sampler.summary(lo, hi)
        sampler.stop()
        # the decode loop alone (towers + encoder excluded): the HBM-bound part the roofline is about
        emb, B_, Le = model._concat_embeddings({"pixel_values": px_d}, {"input_ids": src_d})
        greedy_generate(model.transformer, emb, B_, Le, max_new_tokens=T)
        ms_loop, _ = _timed_steps(lambda: greedy_generate(model.transformer, emb, B_, Le, max_new_tokens=T), args.steps, flush, 1, dev)
    new_tokens = B * (ids.shape[1] - 1)
    cfg = tcfg
    inner, d, dff, nl, V = cfg.num_heads * cfg.d_kv, cfg.d_model, cfg.d_ff, cfg.n_dec, cfg.vocab_size
    # algorithmic HBM bytes of ONE single-token step over the whole batch (bf16): every decoder weight and the LM head streamed
    # once; the cross-attention K|V of every sample read once per block; the self-attention K|V rows written so far read once
    w_bytes = 2 * (nl * (4 * d * inner + 4 * d * inner + 2 * d * dff) + V * d)
    cross_bytes = 2 * nl * B * Le * 2 * inner
    self_bytes_avg = 2 * nl * B * ((T + 1) / 2.0) * 2 * inner
    step_bytes = w_bytes + cross_bytes + self_bytes_avg
    # the encoder-side part of a generate() call (towers + T5 encoder + cross K|V projection) is the rest of ms_res
    pk = peaks()
    ach = step_bytes * T / (ms_loop / args.steps * 1e-3) / 1e9
    line = {
        "metric": "greedy decode tokens/sec (T5 decoder with cross-attention KV cache)", "value": new_tokens / (ms_res / args.steps * 1e-3),
        "unit": "tokens/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_res / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.dtype == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "name": args.workload, "batch_per_gpu": B, "l_src": w["l_src"], "new_tokens": ids.shape[1] - 1,
                   "eos": "disabled (fixed length)", "l2_flush": "256 MiB buffer zeroed between timed iterations (inside the timed region)",
                   "step": "one generate() call through MyModel.forward(return_loss=False): Swin + text tower + T5 encoder + 20 decoder steps"},
        "e2e": {"value": new_tokens / (ms_e2e / args.steps * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": px_h.numel() * 4 + src_h.numel() * 8,
                "d2h_bytes_per_step": int(ids.numel() * 8)},
        "gpu_launches": int(launches), "clocks": clocks,
        "decode_loop_ms": ms_loop / args.steps, "decode_loop_tokens_per_s": new_tokens / (ms_loop / args.steps * 1e-3),
        "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None,
                     "kernel": "single-token decoder step (GEMV-shaped GEMMs + decode attention), whole loop",
                     "algorithmic_bytes_per_token_step": step_bytes, "of_which": {"weights": w_bytes, "cross_kv": cross_bytes, "self_kv_avg": self_bytes_avg},
                     "peak_source": pk["source"] + " HBM copy bandwidth",
                     "method": "algorithmic bytes of the 20 single-token steps / CUDA-event time of the decode loop alone (encoder side excluded)"},
        "cuda_graphs": POOL.stats(),
    }
    emit(line)


def run_ours(args, w):
    import torch.distributed as dist
    from klab_multimodalmodel_b200 import _lib as L
    from klab_multimodalmodel_b200 import ops as O
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if w.get("decode"):
        if rank == 0:
            run_decode(args, w)
        return
    # ---- N = 1, default run: the other BASELINE configs and the informational legs, each in its own process, BEFORE this
    # process touches the GPU (so their memory is gone again); their lines ride along under "workloads" / "hf_eager_gpu"
    extras, hf_leg = {}, None
    if world == 1 and not args.sub and args.workload == "2a" and not args.no_extras and not args.gemm_probe and not args.profile_range:
        k = str(min(args.steps, 10))
        for name in ("3", "4a", "5"):
            extras[name] = run_sub(["--workload", name, "--sub", "--steps", k, "--warmup", "3", "--no-cpu-baseline"], 420)
            print(f"[bench] workload {name}: {json.dumps(extras[name])[:300]}", file=sys.stderr)
        hf_leg = run_sub(["--impl", "hf_eager", "--workload", "2a", "--steps", "5", "--warmup", "2"], 420)
        print(f"[bench] hf_eager: {json.dumps(hf_leg)[:300]}", file=sys.stderr)
        if "error" not in extras.get("5", {"error": 1}):
            extras["5"]["hf_eager_gpu"] = run_sub(["--impl", "hf_eager", "--workload", "5", "--steps", "3", "--warmup", "2"], 300)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # the collective shares the GPU with the persistent tcgen05 kernels (which hand out work dynamically and simply run
        # on the SMs that are left): cap its CTAs so that it never takes more than ~10 % of the machine
        os.environ.setdefault("NCCL_MAX_CTAS", "16")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=int(os.environ.get("KLAB_NCCL_TIMEOUT_S", "600"))))
    L.check(L.lib().klab_check_device())
    model, tcfg = build_model(w, dev, args.dtype)
    model.transformer.train()                                        # train.py:52
    net = model
    if world > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP
        net = DDP(model, device_ids=[local])
    if args.optimizer == "klab":                                      # N1: fused multi-tensor Adam, same semantics as train.py:28
        from klab_multimodalmodel_b200.optim import Adam
        opt = Adam(model.transformer.parameters(), lr=1e-4)
    else:
        opt = torch.optim.Adam(model.transformer.parameters(), lr=1e-4)
    px_h, src_h, tgt_h = synth_batch(w, tcfg.vocab_size, 1234 + rank, pin=True)
    px_d, src_d, tgt_d = px_h.to(dev), src_h.to(dev), tgt_h.to(dev)
    if args.gemm_probe:
        def probe_step():
            loss = model({"pixel_values": px_d}, {"input_ids": src_d}, {"input_ids": tgt_d})
            loss.backward()
            opt.zero_grad()
        probe_step()
        r = gemm_roofline(probe_step, peaks(), verbose=True, check=True)
        emit(r)
        return
    h2d = px_h.numel() * 4 + src_h.numel() * 8 + tgt_h.numel() * 8
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)    # > 126 MB L2

    wd = int(os.environ.get("KLAB_BENCH_WATCHDOG_S", "0"))          # debugging aid: dump every thread's stack if a step stalls
    if wd:
        import faulthandler
    cur = {"opt": opt}

    def step(px, src, tgt, read_loss=True):
        if wd:
            faulthandler.dump_traceback_later(wd, exit=True)
        loss = net({"pixel_values": px}, {"input_ids": src}, {"input_ids": tgt})
        lv = loss.item() if read_loss else None                          # train.py:59 reads the loss every step
        loss.backward()
        cur["opt"].step()
        cur["opt"].zero_grad()
        return lv

    def resident_step():
        return step(px_d, src_d, tgt_d)

    # e2e: the host input path of train.py:55-59 through the drop-in's N2 pieces (klab_multimodalmodel_b200.data): every step the raw
    # fp32 [0, 1] images the reference's loader yields (loader.py:15-16) and the token ids travel from PINNED host memory to the
    # device on a side stream, one step ahead of the step that consumes them, and the image processor's rescale + normalise runs
    # on the GPU (klab_image_normalize) instead of the host; the loss is read back with .item() every step (train.py:59)
    from klab_multimodalmodel_b200.data import DevicePrefetcher, GpuImageProcessor
    raw_h = torch.rand(px_h.shape, generator=torch.Generator().manual_seed(99 + rank)).pin_memory()
    proc = GpuImageProcessor(size=tuple(px_h.shape[-2:]))

    def host_batches():
        while True:
            yield raw_h, src_h, tgt_h

    def to_device(b):
        raw, src, tgt = b
        return proc(raw, return_tensors="pt").to(dev), src.to(dev, non_blocking=True), tgt.to(dev, non_blocking=True)

    feed = DevicePrefetcher(host_batches(), dev, to_device)

    def e2e_step():
        images, src, tgt = next(feed)
        return step(images["pixel_values"], src, tgt)

    # steady state needs six steps: eager warm-up, forward capture, backward capture, then the same three for the accumulating
    # variant of the Swin backward regions (the image model's gradients are never zeroed, train.py:28)
    PRIME = 6                                             # graph construction (untimed set-up), then the W warm-up steps asked for
    for _ in range(PRIME + max(args.warmup, 3)):
        resident_step()
    e2e_step()
    torch.cuda.synchronize()
    if args.profile_range:                                # ncu --profile-from-start off: exactly the timed steps are profiled
        torch.cuda.profiler.start()
        for _ in range(args.steps):
            resident_step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local) if rank == 0 else None
    time.sleep(0.3)
    lo = sampler.mark() if sampler else 0
    from klab_multimodalmodel_b200.graphs import POOL
    l0 = O.launch_count() + POOL.replayed_kernels
    ms_res, loss_v = _timed_steps(resident_step, args.steps, flush, world, dev)
    launches = O.launch_count() + POOL.replayed_kernels - l0
    if args.dump_outputs and rank == 0:                  # before any further step changes the weights
        import numpy as np
        dump_outputs(args.dump_outputs, {"loss": np.array([loss_v], dtype=np.float64),
                                         "transformer_params": _flat_sample(list(model.transformer.parameters()), DUMP_SAMPLE, 1)})
    ms_iso = _timed_steps_isolated(resident_step, args.steps, flush, dev) if world == 1 else None
    hi = sampler.mark() if sampler else 0
    for _ in range(max(args.warmup, 3)):                 # the e2e path allocates its device batches on the prefetch stream: let the
        e2e_step()                                        # caching allocator reach its steady state (no cudaMalloc inside the timed steps)
    ms_e2e, _ = _timed_steps(e2e_step, args.steps, flush, world, dev)
    clocks = sampler.summary(lo, hi) if sampler else None
    if sampler:
        sampler.stop()
    mem_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    dp_sync, dp_par = None, None
    if world > 1:                                       # data-parallel sanity: after K averaged steps every rank holds the same weights
        probe = torch.stack([p.detach().double().sum() for p in list(model.transformer.parameters())[:8] + list(model.transformer.parameters())[-8:]])
        lo_, hi_ = probe.clone(), probe.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        dp_sync = bool(torch.equal(lo_, hi_))
        dp_par = dp_parity_check(model, net, w, tcfg.vocab_size, world, rank, dev, min(w["batch"], 8))
    # ---- the unchanged-train.py optimizer (torch.optim.Adam, train.py:28) as a second value: the operand cache then re-casts
    # the parameters it finds changed and torch's foreach Adam does the update
    torch_opt = None
    if args.optimizer == "klab" and not args.sub and not args.no_extras:
        cur["opt"] = torch.optim.Adam(model.transformer.parameters(), lr=1e-4)
        for _ in range(3):
            resident_step()
        ms_t, _ = _timed_steps(resident_step, args.steps, flush, world, dev)
        torch_opt = {"optimizer": "torch.optim.Adam (train.py:28 unchanged)", "value": world * w["batch"] / (ms_t / args.steps * 1e-3),
                     "unit": "samples/s", "ms_per_step": ms_t / args.steps}
        cur["opt"] = opt
    B = w["batch"]
    ms_step = ms_res / args.steps
    value = world * B / (ms_step * 1e-3)
    e2e_val = world * B / (ms_e2e / args.steps * 1e-3)
    pk = peaks()
    if world > 1:                                       # collectives are over: what follows is rank-0-local reporting
        dist.barrier()
        dist.destroy_process_group()
        if getattr(model, "_klab_reducer", None) is not None:
            model._klab_reducer.enabled = False
    def local_step():                                   # rank-local (no DDP collectives): only rank 0 runs the roofline probe
        loss = model({"pixel_values": px_d}, {"input_ids": src_d}, {"input_ids": tgt_d})
        loss.backward()
        opt.zero_grad()

    if wd:
        faulthandler.cancel_dump_traceback_later()
    roof = gemm_roofline(local_step, pk, verbose=args.verbose, isolated=not args.sub) if rank == 0 else None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sb = args.cpu_sample_batch
        del model, net, opt                                # (the CPU leg needs no GPU memory; keep the box quiet while it runs)
        times, kind, engine = cpu_reference_steps(w, 2, 2, sb, log=lambda m: print(m, file=sys.stderr))   # 2 warm-ups: lazy imports are cold on a fresh box
        cores = os.cpu_count() or 1
        cpu = {"value": sb / (sum(times) / len(times)), "unit": "samples/s", "cores": cores, "kind": kind, "engine": engine,
               "sample": f"{sb} samples/step of the same model + sequence lengths (2 warm-up + 2 timed steps), fwd+bwd+Adam, fp32, {cores} threads"}
    if rank == 0:
        step_tflops = value * w["gflop_per_sample"] / 1e3
        line = {
            "metric": "train samples/sec (Swin+T5 caption step)", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.dtype == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": w["desc"], "name": args.workload, "batch_per_gpu": B, "global_batch": B * world, "l_src": w["l_src"],
                       "l_tgt": w["l_tgt"], "parallelism": f"dp{world}", "optimizer": ("klab_multimodalmodel_b200.optim.Adam (fused multi-tensor kernel, torch.optim.Adam semantics)" if args.optimizer == "klab"
                                     else "torch.optim.Adam") + " over transformer params (train.py:28)",
                       "dropout": "T5 p=0.1 active (train.py:52)", "l2_flush": "256 MiB buffer zeroed between timed iterations (inside the timed region)",
                       "setup": f"{PRIME} untimed steps build the CUDA graphs (eager, capture forward / backward, then the accumulating variant of the "
                                "Swin backward regions) before the warm-up steps"},
            "e2e": {"value": e2e_val, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "path": "pinned host batch (raw fp32 images + int64 ids) -> side-stream H2D one step ahead (DevicePrefetcher) -> rescale + "
                            "normalise on the GPU (GpuImageProcessor / klab_image_normalize) -> MyModel.forward -> loss.item() -> backward -> Adam"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "step_model_tflops": step_tflops, "step_frac_of_peak": step_tflops / pk["tflops"], "step_frac_of_burst_peak": step_tflops / pk["burst"],
            "timing": "ONE event pair around the K steps (L2 flush and the optimizer's side stream inside), max over ranks",
            "ms_per_step_isolated": (ms_iso / args.steps) if ms_iso is not None else None,
            "loss": loss_v, "peak_mem_gb": round(mem_gb, 1),
            "cuda_graphs": POOL.stats(),
        }
        if torch_opt:
            line["torch_optimizer"] = torch_opt
        if extras:
            line["workloads"] = extras
        if hf_leg:
            line["hf_eager_gpu"] = hf_leg
        if world > 1:
            red = getattr(model, "_klab_reducer", None) if cpu is None else None
            line["data_parallel"] = {"weights_identical_across_ranks": dp_sync, "dp_parity": dp_par,
                                     "reducer": "klab GradReducer (grouped in-place NCCL all-reduce per bucket)" if red else "torch DDP",
                                     "buckets_per_step": getattr(red, "buckets_last_backward", None),
                                     "flat_block_buffers_per_step": getattr(red, "flats_last_backward", None), "sm_reserve": O.sm_reserve_info(),
                                     "nccl_max_ctas": os.environ.get("NCCL_MAX_CTAS")}
        emit(line)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else written to fd 1 meanwhile (e.g. NCCL's version banner) was
    diverted to stderr by `main`."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "hf_eager"])
    ap.add_argument("--workload", default="2a", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-sample-batch", type=int, default=2)
    ap.add_argument("--optimizer", default="klab", choices=["klab", "torch"],
                    help="klab = fused multi-tensor Adam (SURVEY 8f N1, same update rule); torch = stock torch.optim.Adam")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only: skip workloads 3 / 4a / 5, the torch-optimizer value and the HF-eager leg")
    ap.add_argument("--sub", action="store_true", help="internal: this process measures ONE extra workload for a parent bench run")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--profile-range", action="store_true",
                    help="for ncu --profile-from-start off: cudaProfilerStart/Stop around the K steps after warm-up, then exit (no JSON line)")
    ap.add_argument("--gemm-probe", action="store_true", help="development aid: only replay (and check) the step's GEMM signatures")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    random.seed(0)                                 # the dropout counter starts from Python's `random` (modeling.step_seed)
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                                  # libraries that print to stdout (NCCL banner) must not pollute the JSON line
    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w["batch"] = args.batch
    if args.impl == "reference":
        run_reference(args, w)
    elif args.impl == "hf_eager":
        run_hf_eager(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
