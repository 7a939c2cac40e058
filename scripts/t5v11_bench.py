"""T5 v1.1 / Flan-T5 next to the original T5 on one GPU: the caption train step, greedy decoding and the gated-GELU kernels.

    python scripts/t5v11_bench.py [--out DIR] [--steps 5] [--warmup 3] [--rounds 3]

Prints one JSON document (and writes DIR/t5v11_bench.json).  Weights are random (T5Config.NAMED architectures); the flan models
have an untied LM head, as the published checkpoints load.  Both models of a comparison live on the GPU together and are timed
in alternation, `rounds` times, `steps` calls each (CUDA events); per model the median over rounds and every round's value.
  train_step   bench.py workload 2a geometry (Swin-B/256/w8 trained jointly, B = 64, 32 + 32 tokens, bf16, dropout on, fused
               Adam over the transformer): t5-large vs google/flan-t5-large for the text tower and the transformer
  decode       bench.py workload 5 geometry (Swin-S/256/w8, B = 256, 20 new tokens, EOS disabled): t5-base vs google/flan-t5-base
  geglu_us     klab_geglu_fwd / klab_geglu_bwd per launch, bf16, d_ff 2816, at M = 6144 (encoder rows of the train step) and 2048
               (decoder rows); 4 operand sets rotated (beyond L2 at M = 6144), CUDA events over 200 launches; algorithmic bytes
               (fwd: read u, write h = 6 M d_ff; bwd: read dh and u, write du = 10 M d_ff) over 7.7 TB/s as the HBM bound
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

HBM_PEAK = 7.7e12


def timed(fn, steps, warmup):
    for _ in range(warmup):
        out = fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps, out


def build(w, t5_name, dev):
    from klab_multimodalmodel_b200.modeling import Swinv2Config, T5Config, init_swin_, init_t5_
    from klab_multimodalmodel_b200.models.model import MyModel
    tcfg = T5Config(**T5Config.NAMED[t5_name])
    sw = dict(w["swin"])
    sw.setdefault("pretrained_window_sizes", (0,) * len(sw["depths"]))
    args = types.SimpleNamespace(result_dir="/tmp", language_model_name=tcfg, image_model_name=Swinv2Config(**sw),
                                 image_model_train=w["train_swin"], transformer_model_name=tcfg, compute_dtype="bf16")
    model = MyModel(args)
    init_t5_(model.language_model, seed=1)
    init_swin_(model.image_model, seed=2)
    init_t5_(model.transformer, seed=3)
    if tcfg.gated:
        model.transformer.untie_lm_head()
    return model.to(dev), tcfg


def compare(models, make_call, steps, warmup, rounds):
    per = {m: [] for m in models}
    for m, call in models.items():                                     # capture every model's regions before timing any
        timed(call, 1, warmup)
    for _ in range(rounds):
        for m, call in models.items():
            per[m].append(timed(call, steps, 0)[0])
    return {"ms": {m: statistics.median(v) for m, v in per.items()}, "rounds_ms": per}


def train_step(steps, warmup, rounds):
    from klab_multimodalmodel_b200.optim import Adam
    w = bench.WORKLOADS["2a"]
    dev = torch.device("cuda", 0)
    calls, params = {}, {}
    for name in ("t5-large", "google/flan-t5-large"):
        model, tcfg = build(w, name, dev)
        model.train()
        opt = Adam(model.transformer.parameters(), lr=1e-5)
        px, src, tgt = [t.to(dev) for t in bench.synth_batch(w, tcfg.vocab_size, 1234, pin=False)]

        def step(model=model, opt=opt, px=px, src=src, tgt=tgt):
            loss = model({"pixel_values": px}, {"input_ids": src}, {"input_ids": tgt})
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return loss
        calls[name] = step
        params[name] = sum(p.numel() for p in model.transformer.parameters())
    r = compare(calls, None, steps, warmup, rounds)
    r.update(B=w["batch"], l_src=w["l_src"], l_tgt=w["l_tgt"], transformer_params=params,
             flan_over_t5=r["ms"]["google/flan-t5-large"] / r["ms"]["t5-large"],
             samples_per_s={m: w["batch"] / (ms * 1e-3) for m, ms in r["ms"].items()})
    return r


def decode(steps, warmup, rounds):
    w = dict(bench.WORKLOADS["5"])
    dev = torch.device("cuda", 0)
    calls = {}
    for name in ("t5-base", "google/flan-t5-base"):
        model, tcfg = build(w, name, dev)
        model.eval()
        model.transformer.config.eos_token_id = -1                     # never finishes early: exactly 20 tokens per row
        px, src, _ = [t.to(dev) for t in bench.synth_batch(w, tcfg.vocab_size, 1234, pin=False)]

        def call(model=model, px=px, src=src):
            with torch.no_grad():
                ids = model({"pixel_values": px}, {"input_ids": src}, return_loss=False)
            assert ids.shape == (w["batch"], w["l_tgt"] + 1), ids.shape
            return ids
        calls[name] = call
    r = compare(calls, None, steps, warmup, rounds)
    r.update(B=w["batch"], new_tokens=w["l_tgt"], flan_over_t5=r["ms"]["google/flan-t5-base"] / r["ms"]["t5-base"])
    return r


def geglu_us():
    from klab_multimodalmodel_b200 import ops as O
    dev = torch.device("cuda", 0)
    dff, n, copies = 2816, 200, 4
    out = {}
    for M in (6144, 2048):
        us = [torch.randn(M, 2 * dff, device=dev).bfloat16() for _ in range(copies)]
        dhs = [torch.randn(M, dff, device=dev).bfloat16() for _ in range(copies)]
        seed = torch.tensor([5], dtype=torch.int64, device=dev)
        it = [0]

        def fwd():
            it[0] += 1
            return O.geglu_fwd(us[it[0] % copies], 0.1, 7, seed)

        def bwd():
            it[0] += 1
            return O.geglu_bwd(dhs[it[0] % copies], us[it[0] % copies], 0.1, 7, seed)
        res = {}
        for name, fn, nbytes in (("fwd", fwd, 6 * M * dff), ("bwd", bwd, 10 * M * dff)):
            t = timed(fn, n, 10)[0] * 1e3
            bound = nbytes / HBM_PEAK * 1e6
            res[name] = {"us_per_launch": t, "bytes": nbytes, "hbm_bound_us": bound, "share_of_hbm_bound": bound / t,
                         "achieved_tb_s": nbytes / (t * 1e-6) / 1e12}
        out[str(M)] = res
        del us, dhs
    return {"d_ff": dff, "dtype": "bf16", "dropout_p": 0.1, "rows": out}


def release():
    """Free the models of one comparison: their captured regions pin private memory pools."""
    import gc

    from klab_multimodalmodel_b200.graphs import POOL
    POOL.drop_keys(lambda k: True)
    gc.collect()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("t5v11_bench.py measures on the GPU; there is none here")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": gpu}
    res["train_step"] = train_step(a.steps, a.warmup, a.rounds)
    release()
    res["decode"] = decode(a.steps, a.warmup, a.rounds)
    release()
    res["geglu_us"] = geglu_us()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "t5v11_bench.json"), "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
