"""Multinomial-sampling caption decoding on one GPU: the bench workload-5 geometry (Swin-S/256 + T5-base, 32 source tokens, 20 new
tokens), EOS disabled so that every call runs exactly 20 steps.

    python scripts/sample_bench.py [--out DIR] [--steps 5] [--warmup 2] [--rounds 3]

Prints one JSON document (and writes DIR/sample_bench.json).  Weights are random.
  calls_b256        one MyModel.forward(return_loss=False) at B = 256, n = 1, for greedy decoding, sampling with the transformers
                    defaults (temperature 1, top_k 50, top_p 1) and full-vocabulary nucleus sampling (top_k 0, top_p 0.9); the
                    three are alternated `rounds` times within the run, `steps` timed calls each (CUDA events); per mode the
                    median over rounds and every round's value
  calls_b64_n4      the same call with sampling defaults at B = 64, num_return_sequences 4 (256 rows)
  kernel_us         klab_sample_step per launch at R = 256 and 1024 rows of V = 32128 fp32 logits (N(0, 3^2), written once, so
                    L2-resident at R = 256: 33 MB), per warper combination, next to klab_greedy_step on the same logits; CUDA events
                    over 200 launches; hbm_bound_us = 4 R V bytes / 7.7 TB/s
  hf_eager          transformers generate(inputs_embeds, do_sample=True) under bf16 autocast on the same GPU, where it imports
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

HBM_PEAK = 7.7e12
MODES = {"greedy": dict(do_sample=False, top_k=50, top_p=1.0),
         "sample_default": dict(do_sample=True, top_k=50, top_p=1.0),
         "sample_nucleus": dict(do_sample=True, top_k=0, top_p=0.9)}
WARPERS = {"pure (T 1, k 0, p 1)": (1.0, 0, 1.0), "default (T 1, k 50, p 1)": (1.0, 50, 1.0), "nucleus (T 1, k 0, p 0.9)": (1.0, 0, 0.9),
           "all (T 0.7, k 50, p 0.9)": (0.7, 50, 0.9), "k 1": (1.0, 1, 1.0)}


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


def build(B):
    w = dict(bench.WORKLOADS["5"], batch=B)
    dev = torch.device("cuda", 0)
    model, tcfg = bench.build_model(w, dev, "bf16")
    model.eval()
    model.transformer.config.eos_token_id = -1                       # never finishes early: exactly T tokens per row
    px, src, _ = [t.to(dev) for t in bench.synth_batch(w, tcfg.vocab_size, 1234, pin=False)]
    return model, px, src, w["l_tgt"]


def set_mode(model, mode, n=1):
    gc = model.transformer.generation_config
    for k, v in MODES[mode].items():
        setattr(gc, k, v)
    gc.num_return_sequences = n


def calls(steps, warmup, rounds):
    model, px, src, T = build(256)
    call = lambda: model({"pixel_values": px}, {"input_ids": src}, return_loss=False)       # noqa: E731
    per = {m: [] for m in MODES}
    with torch.no_grad():
        for m in MODES:                                               # capture every mode's regions before timing any
            set_mode(model, m)
            timed(call, 1, warmup)
        for _ in range(rounds):
            for m in MODES:
                set_mode(model, m)
                ms, ids = timed(call, steps, 1)
                assert ids.shape == (256, T + 1), ids.shape
                per[m].append(ms)
    med = {m: statistics.median(v) for m, v in per.items()}
    out = {"B": 256, "n": 1, "new_tokens": T, "ms_per_call": med, "rounds_ms": per,
           "sample_default_over_greedy": med["sample_default"] / med["greedy"],
           "sample_nucleus_over_greedy": med["sample_nucleus"] / med["greedy"]}
    del model
    torch.cuda.empty_cache()
    model, px, src, T = build(64)
    set_mode(model, "sample_default", n=4)
    with torch.no_grad():
        _, _, Le = model._concat_embeddings({"pixel_values": px}, {"input_ids": src})
        ms, ids = timed(lambda: model({"pixel_values": px}, {"input_ids": src}, return_loss=False), steps, warmup)
    assert ids.shape == (256, T + 1), ids.shape
    b64 = {"B": 64, "n": 4, "rows": 256, "Le": Le, "ms_per_call": ms, "row_tokens_per_s": 256 * T / (ms * 1e-3)}
    del model
    torch.cuda.empty_cache()
    return out, b64


def kernel_us():
    from klab_multimodalmodel_b200 import _lib as L
    from klab_multimodalmodel_b200 import ops as O
    dev = torch.device("cuda", 0)
    V, n = 32128, 200
    out = {}
    g = torch.Generator(device=dev).manual_seed(0)
    for R in (256, 1024):
        logits = torch.randn(R, V, device=dev, generator=g) * 3
        ids = torch.zeros(R, 21, dtype=torch.int64, device=dev)
        unf = torch.ones(R, dtype=torch.int32, device=dev)
        seed = torch.tensor([12345], dtype=torch.int64, device=dev)
        s = torch.cuda.current_stream().cuda_stream
        res = {}

        def greedy():                                                 # EOS -1: every row stays unfinished, as in the sampling launches
            L.check(L.lib().klab_greedy_step(s, R, V, logits.data_ptr(), V, ids.data_ptr(), 21, 1, unf.data_ptr(), 0, -1))
        res["greedy_step"] = timed(greedy, n, 10)[0] * 1e3
        for name, (temp, k, p) in WARPERS.items():
            res[name] = timed(lambda: O.sample_step(logits, ids, 1, unf, seed, pad_id=0, eos_id=-1, temperature=temp, top_k=k,
                                                    top_p=p), n, 10)[0] * 1e3
        out[str(R)] = {"us_per_launch": res, "hbm_bound_us": 4 * R * V / HBM_PEAK * 1e6}
        del logits
    return {"V": V, "rows": out}


def run_hf(B, Le, steps):
    try:
        import transformers
    except ImportError as e:
        return {"unavailable": str(e)}
    w = bench.WORKLOADS["5"]
    from klab_multimodalmodel_b200.modeling import T5Config
    c = T5Config(**T5Config.NAMED[w["t5"]])
    cfg = transformers.T5Config(vocab_size=c.vocab_size, d_model=c.d_model, d_kv=c.d_kv, d_ff=c.d_ff, num_layers=c.num_layers,
                                num_heads=c.num_heads, decoder_start_token_id=0)
    dev = torch.device("cuda", 0)
    m = transformers.T5ForConditionalGeneration(cfg).to(dev).eval()
    emb = torch.randn(B, Le, c.d_model, device=dev)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        ms, ids = timed(lambda: m.generate(inputs_embeds=emb, do_sample=True, max_new_tokens=20, eos_token_id=None), steps, 1)
    assert ids.shape == (B, 21), ids.shape
    return {"B": B, "generate_ms": ms, "row_tokens_per_s": B * 20 / (ms * 1e-3),
            "engine": f"transformers {transformers.__version__} eager, do_sample=True (top_k 50), bf16 autocast, fp32 parameters, "
                      "encoder on random inputs_embeds"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench.py measures on the GPU; there is none here")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": gpu}
    res["calls_b256"], res["calls_b64_n4"] = calls(a.steps, a.warmup, a.rounds)
    res["kernel_us"] = kernel_us()
    try:
        res["hf_eager"] = run_hf(256, res["calls_b64_n4"]["Le"], max(2, a.steps // 2))
    except Exception as e:                                              # noqa: BLE001  (informational)
        res["hf_eager"] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "sample_bench.json"), "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
