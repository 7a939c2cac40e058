"""Multinomial sampling on the B200: klab_sample_step (csrc/sampling.cu) against the float64 statement of its definition
(oracle/t5_sample.py: kept_by_rule, sample_uniform, inverse_cdf), its distribution over 2^16 draws, and
`generate(do_sample=True, ...)` end to end against the stored transformers outputs (tests/golden/hf_sample.npz)."""
import numpy as np
import pytest
import torch

from oracle.t5_sample import kept_by_rule, sample_uniform
from tests.test_sample_oracle_cpu import golden_case

pytestmark = pytest.mark.gpu
DEV = "cuda"
MARGIN = 1e-5


def run_step(logits, t, seed, temperature=1.0, top_k=0, top_p=1.0, unfinished=None, eos_id=1, pad_id=0):
    from klab_multimodalmodel_b200 import ops as O
    R = logits.shape[0]
    ids = torch.full((R, t + 1), -7, dtype=torch.int64, device=DEV)
    unf = torch.ones(R, dtype=torch.int32, device=DEV) if unfinished is None else unfinished.to(DEV, torch.int32).clone()
    O.sample_step(logits.to(DEV).contiguous(), ids, t, unf, torch.tensor([seed], dtype=torch.int64, device=DEV), pad_id=pad_id,
                  eos_id=eos_id, temperature=temperature, top_k=top_k, top_p=top_p)
    torch.cuda.synchronize()
    assert (ids[:, :t] == -7).all()                                   # only column t is written
    return ids[:, t].cpu(), unf.cpu()


def reference_draw(x, t, seed, temperature, top_k, top_p):
    """-> (token [R], margin [R], kept [R, V]): the defined draw in float64, and how far (relative) the row is from a decision boundary --
    u * Z from the nearest cumulative boundary, and the top-p mass from its threshold."""
    s, keep, pmargin = kept_by_rule(x, temperature, top_k, top_p)
    d = s.double()
    w = torch.where(keep, torch.exp(d - d.max(-1, keepdim=True)[0]), torch.zeros_like(d))
    c = w.cumsum(-1)
    Z = c[:, -1]
    u = torch.tensor([sample_uniform(seed, r, t - 1) for r in range(x.shape[0])], dtype=torch.float64)
    target = u * Z
    tok = torch.searchsorted(c, target[:, None], right=True)[:, 0].clamp_max(x.shape[1] - 1)
    hi = c.gather(1, tok[:, None])[:, 0]
    lo = torch.where(tok > 0, c.gather(1, (tok - 1).clamp_min(0)[:, None])[:, 0], torch.zeros_like(hi))
    dmargin = torch.minimum(hi - target, target - lo) / Z
    return tok, torch.minimum(dmargin, pmargin), keep


def logits_rows(R, V, seed):
    """LM-head-like rows: a broad N(0, 2^2) background and 64 plausible tokens per row 20..30 above it.  (On a flat row of 32128
    tokens each token holds ~3e-5 of the mass, so most draws would sit within the 1e-5 margin of a boundary.)"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(R, V, generator=g) * 2
    x.scatter_add_(1, torch.randint(0, V, (R, 64), generator=g), 20 + 10 * torch.rand(R, 64, generator=g))
    x[1, ::5] = -float("inf")                                         # -inf entries
    x[2, [3, V // 2, V - 1]] = x[2].max() + 2.0                       # three tied maxima (top-k and top-p keep them all)
    x[3, 1] = x[3].max() + 40.0                                       # EOS all but certain: clears unfinished
    x[4, : V // 3] = -float("inf")
    return x


@pytest.mark.parametrize("temperature", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("V", [300, 1000, 32128])
def test_kernel_matches_defined_draw(V, temperature):
    R = 64
    x = logits_rows(R, V, V + int(temperature * 10))
    checked = total = 0
    for top_k in (0, 1, 7, 50, V + 5):
        for top_p in (1.0, 0.9, 0.3, 0.0):
            seed = 1000 * top_k + int(top_p * 10) + V
            t = 1 + (top_k + int(top_p * 10)) % 19
            unf = torch.ones(R, dtype=torch.int32)
            unf[5:7] = 0                                              # finished rows: pad, unfinished stays 0
            got, got_unf = run_step(x, t, seed, temperature, top_k, top_p, unfinished=unf)
            ref, margin, keep = reference_draw(x, t, seed, temperature, top_k, top_p)
            ok = margin > MARGIN
            ok[5:7] = False
            checked += int(ok.sum())
            total += R - 2
            msg = (V, temperature, top_k, top_p)
            assert torch.equal(got[ok], ref[ok]), (msg, got[ok][got[ok] != ref[ok]], ref[ok][got[ok] != ref[ok]])
            assert (got[5:7] == 0).all() and (got_unf[5:7] == 0).all(), msg
            assert torch.equal(got_unf.bool(), unf.bool() & (got != 1)), msg
            assert got[3] == 1 and got_unf[3] == 0, msg                           # the EOS draw
            live = torch.arange(R) != 5
            live[6] = False
            assert keep[live].gather(1, got[live][:, None]).all(), msg           # never outside the kept set
            if top_k == 1 or top_p == 0.0:
                assert int(got[2]) in (3, V // 2, V - 1), msg                          # ties at the top are drawn among
    assert checked >= 0.99 * total, (checked, total)


def test_tied_maxima_are_all_drawn_with_top_k_one():
    V = 500
    x = torch.randn(1, V) * 0.1
    x[0, [7, 100, 499]] = 5.0
    x = x.repeat(3000, 1)
    got, _ = run_step(x, 3, 11, top_k=1)
    assert set(got.tolist()) == {7, 100, 499}


def test_distribution_chi_square():
    from scipy import stats
    V, N, temperature, top_p = 1000, 1 << 16, 1.3, 0.95
    g = torch.Generator().manual_seed(3)
    row = torch.randn(1, V, generator=g) * 2.5
    got, _ = run_step(row.expand(N, V), 1, 20261020, temperature, 0, top_p)
    _, keep, margin = kept_by_rule(row, temperature, 0, top_p)
    assert float(margin[0]) > MARGIN
    s = (row.float() / temperature).double()[0]
    p = torch.where(keep[0], torch.exp(s - s.max()), torch.zeros_like(s))
    p = p / p.sum()
    assert keep[0][got].all()                                          # not one draw outside the kept set
    counts = torch.bincount(got, minlength=V).double()
    exp = p * N
    big = exp >= 5
    obs = torch.cat([counts[big], counts[~big].sum()[None]])
    ex = torch.cat([exp[big], exp[~big].sum()[None]])
    if ex[-1] == 0:
        obs, ex = obs[:-1], ex[:-1]
    chi = stats.chisquare(obs.numpy(), ex.numpy())
    print(f"chi-square over {len(obs)} bins: {chi.statistic:.1f}, p = {chi.pvalue:.3g}")
    assert chi.pvalue > 1e-6


def test_bad_arguments_return_an_error_code():
    from klab_multimodalmodel_b200 import _lib as L
    lib = L.lib()
    x = torch.zeros(2, 70000, device=DEV)                              # more than shared memory holds
    ids = torch.zeros(2, 4, dtype=torch.int64, device=DEV)
    unf = torch.ones(2, dtype=torch.int32, device=DEV)
    seed = torch.zeros(1, dtype=torch.int64, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    args = lambda V, t, temp, k, p, sp: (s, 2, V, x.data_ptr(), x.stride(0), ids.data_ptr(), 4, t, unf.data_ptr(), 0, 1, temp, k, p, sp)
    assert lib.klab_sample_step(*args(70000, 1, 1.0, 0, 1.0, seed.data_ptr())) != 0
    assert b"shared memory" in lib.klab_last_error()
    for bad in (args(100, 0, 1.0, 0, 1.0, seed.data_ptr()), args(100, 4, 1.0, 0, 1.0, seed.data_ptr()),
                args(100, 1, 0.0, 0, 1.0, seed.data_ptr()), args(100, 1, 1.0, -1, 1.0, seed.data_ptr()),
                args(100, 1, 1.0, 0, -0.5, seed.data_ptr()), args(100, 1, 1.0, 0, 1.0, None)):
        assert lib.klab_sample_step(*bad) != 0
    torch.cuda.synchronize()


# ---- end to end ------------------------------------------------------------------------------------------------------------
def _transformer(t5, sd):
    from klab_multimodalmodel_b200.modeling import T5Config, T5ForConditionalGeneration
    tr = T5ForConditionalGeneration(T5Config(vocab_size=t5.vocab_size, d_model=t5.d_model, d_kv=t5.d_kv, d_ff=t5.d_ff,
                                             num_layers=t5.num_layers, num_decoder_layers=t5.num_decoder_layers, num_heads=t5.num_heads))
    tr.load_state_dict(sd, strict=True)
    return tr.to(DEV).eval()


def _opts(o):
    return {k: v for k, v in o.items() if v is not None and k != "seed"}


@pytest.fixture
def fixed_seed(monkeypatch):
    """generate() draws its seed from torch's CPU generator; the goldens were made with seed = the option set's index."""
    from klab_multimodalmodel_b200 import generation
    box = {}
    monkeypatch.setattr(generation, "draw_seed", lambda: box["seed"])
    return box


@pytest.mark.parametrize("name", ["tiny_a", "tiny_b", "mid"])
def test_generate_fp32_matches_transformers(name, fixed_seed):
    t5, sd, emb, runs = golden_case(name)
    tr = _transformer(t5, sd)
    for o, seqs in runs:
        fixed_seed["seed"] = o["seed"]
        got = tr.generate(inputs_embeds=emb.to(DEV), do_sample=True, **_opts(o)).cpu()
        assert got.shape == seqs.shape and np.array_equal(got.numpy(), seqs), (name, o, got, seqs)


def test_mymodel_forward_samples_from_generation_config(fixed_seed):
    from tests.test_beam_search_gpu import _mymodel
    model, (t5, sd, emb, _), px, src = _mymodel("tiny_a", "fp32")
    _, _, _, runs = golden_case("tiny_a")
    gc = model.transformer.generation_config
    for o, seqs in (runs[1], runs[8], runs[16]):
        fixed_seed["seed"] = o["seed"]
        gc.do_sample, gc.temperature, gc.top_k, gc.top_p = True, o["temperature"], o["top_k"], o["top_p"]
        gc.num_return_sequences, gc.max_new_tokens = o["num_return_sequences"], o["max_new_tokens"]
        got = model({"pixel_values": px}, {"input_ids": src}, return_loss=False).cpu()
        assert np.array_equal(got.numpy(), seqs), o


def test_graphs_geometry_and_seeds():
    from klab_multimodalmodel_b200.graphs import POOL
    t5, sd, emb, _ = golden_case("mid")
    tr = _transformer(t5, sd)
    o = dict(do_sample=True, temperature=1.5, top_k=0, top_p=0.9, num_return_sequences=3)
    for dtype in (torch.float32, torch.bfloat16):
        e = emb.to(DEV, dtype)

        def gen(x=e, **kw):
            torch.manual_seed(7)
            return tr.generate(inputs_embeds=x, **dict(o, **kw)).cpu()
        a = gen()
        b = gen(num_return_sequences=8)                                 # another n in between
        c = gen(x=e[:1])                                                # and another batch size
        again = gen()
        POOL.enabled = False
        try:
            eager, eager_b = gen(), gen(num_return_sequences=8)
        finally:
            POOL.enabled = True
        assert torch.equal(a, again) and torch.equal(a, eager) and torch.equal(b, eager_b)
        assert c.shape[0] == 3 and b.shape[0] == 8 * emb.shape[0] and a.shape[0] == 3 * emb.shape[0]
        torch.manual_seed(8)                                            # another seed, another output
        other = tr.generate(inputs_embeds=e, **o).cpu()
        assert other.shape != a.shape or not torch.equal(other, a)


@pytest.mark.parametrize("name", ["tiny_b", "mid"])
def test_bf16_top_k_one_is_greedy_and_rows_differ(name):
    from klab_multimodalmodel_b200.generation import greedy_generate
    t5, sd, emb, _ = golden_case(name)
    tr = _transformer(t5, sd)
    B, Le, d = emb.shape
    e = emb.to(DEV, torch.bfloat16)
    got = tr.generate(inputs_embeds=e, do_sample=True, top_k=1, temperature=0.7).cpu()
    assert torch.equal(got, greedy_generate(tr, e.reshape(B * Le, d), B, Le).cpu())
    hot = tr.generate(inputs_embeds=e, do_sample=True, temperature=2.0, num_return_sequences=8).cpu()
    assert hot.shape[0] == 8 * B
    for b in range(B):
        rows = hot[8 * b:8 * b + 8]
        assert not (rows == rows[0]).all(), (name, b)
