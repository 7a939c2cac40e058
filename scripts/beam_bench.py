"""Beam-search caption decoding on one GPU: the bench workload-5 geometry (Swin-S/256 + T5-base, 32 source tokens, 20 new tokens)
with num_beams 4, at B = 64 samples (256 hypothesis rows, the row count of the greedy workload) and B = 256 (1024 rows).

    python scripts/beam_bench.py [--out DIR] [--steps 5] [--warmup 2]

Prints one JSON document (and writes DIR/beam_bench.json).  Weights are random and EOS is disabled, so every call runs exactly
20 steps; the script asserts that the output has 21 columns on both our side and the transformers side, so the work is equal.
  generate_ms       one MyModel.forward(return_loss=False) with generation_config.num_beams = 4 (towers, encoder, decode loop)
  loop_ms           the decode loop alone: beam_generate minus its encoder side (T5 encoder + norm + cross K|V projection),
                    both timed separately with CUDA events
  bytes_per_step    algorithmic HBM bytes of one decode step, from shapes (bf16 operands): decoder + LM-head weights once,
                    self K|V of the positions written so far (average over the 20 steps) per hypothesis, cross K|V ONCE PER
                    SAMPLE, the fp32 logits written by the LM head and read by the top-k kernel, the ancestry / sequence tables
  hbm_share         bytes_per_step * 20 / loop time, over the 7.7 TB/s of the B200 data sheet
  cross_attn_us     one cross-attention launch (one block) at B = 64 samples, num_beams 1, 2, 4, 8
  hf_eager          transformers generate(inputs_embeds, num_beams=4) under bf16 autocast on the same GPU, where it imports
L2 is not flushed between timed calls (the 2 x 126 MB working set of a step exceeds it only at B = 256).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

HBM_PEAK = 7.7e12
NB = 4


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


def step_bytes(cfg, B, nb, Le, T):
    inner, d, dff, nl, V = cfg.num_heads * cfg.d_kv, cfg.d_model, cfg.d_ff, cfg.n_dec, cfg.vocab_size
    R = B * nb
    weights = 2 * (nl * (4 * d * inner + 4 * d * inner + 2 * d * dff) + V * d)
    self_kv = 2 * nl * R * ((T + 1) / 2.0) * 2 * inner
    cross_kv = 2 * nl * B * Le * 2 * inner
    logits = 2 * 4 * R * V
    tables = R * (T + 1) * (4 + 8 + 8) * 2
    return {"weights": weights, "self_kv_avg": self_kv, "cross_kv": cross_kv, "logits_round_trip": logits, "beam_tables": tables,
            "total": weights + self_kv + cross_kv + logits + tables}


def run_ours(B, steps, warmup):
    from klab_multimodalmodel_b200 import ops as O
    from klab_multimodalmodel_b200.generation import beam_generate
    w = dict(bench.WORKLOADS["5"], batch=B)
    dev = torch.device("cuda", 0)
    model, tcfg = bench.build_model(w, dev, "bf16")
    model.eval()
    model.transformer.config.eos_token_id = -1                       # never finishes early: exactly T tokens per hypothesis
    model.transformer.generation_config.num_beams = NB
    tr, cfg, T = model.transformer, model.transformer.config, w["l_tgt"]
    px, src, _ = [t.to(dev) for t in bench.synth_batch(w, tcfg.vocab_size, 1234, pin=False)]
    with torch.no_grad():
        gen_ms, ids = timed(lambda: model({"pixel_values": px}, {"input_ids": src}, return_loss=False), steps, warmup)
        assert ids.shape == (B, T + 1), ids.shape
        emb, B_, Le = model._concat_embeddings({"pixel_values": px}, {"input_ids": src})
        full_ms, _ = timed(lambda: beam_generate(tr, emb, B_, Le, NB, T), steps, warmup)
        st = tr._klab_beam_states[(B, NB, Le, T, emb.dtype, dev)]

        def encoder_side():
            enc = tr.encoder.run_blocks(emb, B_, Le, tr.cache)
            O.rmsnorm_fwd(enc, tr.encoder.final_layer_norm.weight, cfg.layer_norm_epsilon, out=st.enc, save_stats=False)
            for blk, ckv in zip(tr.decoder.block, st.cross_kv):
                ca = blk.layer[1].EncDecAttention
                O.linear_fwd(st.enc, tr.cache.get([ca.k.weight, ca.v.weight], emb.dtype), out=ckv)
        enc_ms, _ = timed(encoder_side, steps, warmup)
    loop_ms = full_ms - enc_ms
    by = step_bytes(cfg, B, NB, Le, T)
    rows = B * NB
    return {"B": B, "num_beams": NB, "hypothesis_rows": rows, "Le": Le, "new_tokens": T, "generate_ms": gen_ms,
            "beam_generate_ms": full_ms, "encoder_side_ms": enc_ms, "loop_ms": loop_ms,
            "hypothesis_tokens_per_s": rows * T / (gen_ms * 1e-3), "loop_hypothesis_tokens_per_s": rows * T / (loop_ms * 1e-3),
            "bytes_per_step": by, "hbm_share": by["total"] * T / (loop_ms * 1e-3) / HBM_PEAK,
            "logits_share_of_bytes": by["logits_round_trip"] / by["total"]}, model


def cross_attention_us(model, B, Le, steps):
    from klab_multimodalmodel_b200 import ops as O
    cfg = model.transformer.config
    H, dk = cfg.num_heads, cfg.d_kv
    inner = H * dk
    dev = torch.device("cuda", 0)
    kv = torch.randn(B * Le, 2 * inner, device=dev, dtype=torch.bfloat16)
    out = {}
    for nb in (1, 2, 4, 8):
        q = torch.randn(B * nb, inner, device=dev, dtype=torch.bfloat16)
        ms, _ = timed(lambda: O.t5_attention_decode_beam(q, kv[:, :inner], kv[:, inner:], B * nb, H, Le, dk, kv_group=nb), 50 * steps, 5)
        out[str(nb)] = ms * 1e3
    return {"B": B, "Le": Le, "us_per_launch": out,
            "kv_bytes_per_launch": B * Le * 2 * inner * 2}


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
        ms, ids = timed(lambda: m.generate(inputs_embeds=emb, num_beams=NB, max_new_tokens=20, eos_token_id=None), steps, 1)
    assert ids.shape == (B, 21), ids.shape
    return {"B": B, "num_beams": NB, "generate_ms": ms, "hypothesis_tokens_per_s": B * NB * 20 / (ms * 1e-3),
            "engine": f"transformers {transformers.__version__} eager, bf16 autocast, fp32 parameters, encoder on random inputs_embeds"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("beam_bench.py measures on the GPU; there is none here")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": gpu, "runs": []}
    model = None
    for B in (64, 256):
        r, model = run_ours(B, a.steps, a.warmup)
        res["runs"].append(r)
        Le = r["Le"]
        if B == 64:
            res["cross_attention"] = cross_attention_us(model, 64, Le, a.steps)
        del model
        torch.cuda.empty_cache()
    try:
        res["hf_eager"] = run_hf(64, res["runs"][0]["Le"], max(2, a.steps // 2))
    except Exception as e:                                              # noqa: BLE001  (informational)
        res["hf_eager"] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "beam_bench.json"), "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
