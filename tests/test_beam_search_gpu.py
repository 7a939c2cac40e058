"""Beam search on the B200: the two beam kernels (csrc/beam_search.cu) against torch and the oracle's step function, the
beam-aware decode attention (klab_t5_attention_decode_beam) against the existing decode kernels on explicitly gathered K/V,
and `generate(num_beams=...)` end to end against the oracle and the stored transformers outputs (tests/golden/hf_beam.npz)."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.t5_beam import beam_init, beam_step
from tests.golden.make_hf_golden import HF_CASES, case_inputs
from tests.test_beam_oracle_cpu import golden_case, oracle_run

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _lib():
    from klab_multimodalmodel_b200 import _lib as L
    return L.lib()


def _s():
    return torch.cuda.current_stream().cuda_stream


def run_topk(logits, scores, k):
    R, V = logits.shape
    val = torch.empty(R, k, device=DEV)
    tok = torch.empty(R, k, dtype=torch.int32, device=DEV)
    assert _lib().klab_beam_topk(_s(), R, V, k, logits.data_ptr(), logits.stride(0), scores.data_ptr(), val.data_ptr(), tok.data_ptr()) == 0
    return val, tok


@pytest.mark.parametrize("nb,V", [(2, 300), (4, 1000), (8, 32128)])
def test_topk_kernel_matches_log_softmax_topk(nb, V):
    g = torch.Generator().manual_seed(nb)
    R, k = 6 * nb, 2 * nb
    logits = torch.randn(R, V, generator=g) * 4
    logits[0, 5:9] = logits[0].max() + 1.0                            # planted ties at the top: lower index first
    logits[1, ::3] = -float("inf")
    logits[2, 10] = logits[2, 20] = logits[2, 30] = 50.0
    scores = torch.randn(R, generator=g)
    scores[3::nb] = -1e9                                               # the initial state of beams 1.. (:3194)
    val, tok = run_topk(logits.to(DEV), scores.to(DEV), k)
    acc = F.log_softmax(logits, -1) + scores[:, None]
    ref_v, ref_i = torch.sort(acc, dim=-1, descending=True, stable=True)
    torch.testing.assert_close(val.cpu(), ref_v[:, :k], rtol=2e-6, atol=2e-5)
    live = scores > -1e8                                               # -1e9 rows: the sum rounds most values to the same float
    assert torch.equal(tok.cpu().long()[live], ref_i[:, :k][live])
    assert torch.equal(tok.cpu().long()[0, :4], torch.arange(5, 9)) and torch.equal(tok.cpu().long()[2, :3], torch.tensor([10, 20, 30]))


class DevBeam:
    """The device state klab_beam_update works on, for the kernel-level test."""

    def __init__(self, B, nb, T):
        R = B * nb
        self.B, self.nb, self.T = B, nb, T
        self.src = torch.arange(R, dtype=torch.int32, device=DEV)[None, :, None].repeat(2, 1, T + 1)
        self.run_seq = torch.ones(2, R, T + 1, dtype=torch.long, device=DEV)
        self.run_seq[:, :, 0] = 0
        self.fin_seq = self.run_seq.clone()
        self.run_scores = torch.full((B, nb), -1e9, device=DEV)
        self.run_scores[:, 0] = 0
        self.run_scores = self.run_scores.flatten()
        self.fin_scores = torch.full((R,), -1e9, device=DEV)
        self.fin_flag = torch.zeros(R, dtype=torch.int32, device=DEV)
        self.fin_len = torch.zeros(R, dtype=torch.int32, device=DEV)
        self.unsat = torch.ones(B, dtype=torch.int32, device=DEV)
        self.done = torch.zeros(B, dtype=torch.int32, device=DEV)
        self.next_tok = torch.zeros(R, dtype=torch.long, device=DEV)

    def step(self, logits, t, lp, es):
        val, tok = run_topk(logits, self.run_scores, 2 * self.nb)
        rc = _lib().klab_beam_update(_s(), self.B, self.nb, logits.shape[1], self.T, t, 1, lp, {False: 0, True: 1, "never": 2}[es],
                                     val.data_ptr(), tok.data_ptr(), self.run_scores.data_ptr(), self.src.data_ptr(),
                                     self.run_seq.data_ptr(), self.T + 1, self.fin_scores.data_ptr(), self.fin_seq.data_ptr(),
                                     self.fin_flag.data_ptr(), self.fin_len.data_ptr(), self.unsat.data_ptr(), self.done.data_ptr(),
                                     self.next_tok.data_ptr())
        assert rc == 0


@pytest.mark.parametrize("es", [False, True, "never"])
@pytest.mark.parametrize("lp", [1.0, 0.0, 2.0])
def test_update_kernel_matches_oracle_step(es, lp):
    from oracle.t5 import T5Dims
    dims = T5Dims()
    B, nb, V, T = 5, 4, 97, 12
    g = torch.Generator().manual_seed(int(lp * 10) + len(str(es)))
    dev = DevBeam(B, nb, T)
    ref = beam_init(B, nb, T + 1, dims)
    for t in range(T):
        logits = torch.randn(B * nb, V, generator=g) * 2
        logits[:, 1] += torch.rand(B * nb, generator=g) * 4                   # EOS often near the top
        dev.step(logits.to(DEV), t, lp, es)
        beam_step(ref, logits, t, T + 1, dims, lp, es, freeze=True)
        buf = (t + 1) & 1
        msg = f"step {t}"
        assert torch.equal(dev.done.cpu().bool(), ref.frozen), msg
        assert torch.equal(dev.unsat.cpu().bool(), ref.unsat), msg
        assert torch.equal(dev.fin_seq[buf].cpu().view(B, nb, -1), ref.seq), msg
        assert torch.equal(dev.fin_flag.cpu().bool().view(B, nb), ref.fin), msg
        assert torch.equal(dev.fin_len.cpu().long().view(B, nb), ref.gen_len), msg
        torch.testing.assert_close(dev.fin_scores.cpu().view(B, nb), ref.scores, rtol=1e-6, atol=1e-5)
        live = ~ref.frozen
        assert torch.equal(dev.run_seq[buf].cpu().view(B, nb, -1)[live], ref.run_seq[live]), msg
        assert torch.equal(dev.next_tok.cpu().view(B, nb)[live], ref.run_seq[live][:, :, t + 1]), msg
    # ancestry: every cache row a hypothesis reads belongs to its own sample
    src = dev.src[T & 1].cpu().long()
    assert ((src // nb) == (torch.arange(B * nb) // nb)[:, None]).all()


def _gather_self(cache, src, T, t):
    """cache [R*T, w] -> [R*(t+1), w]: row (r, j) = cache row src[r, j] * T + j."""
    j = torch.arange(t + 1, device=DEV)
    return cache[(src[:, :t + 1].long() * T + j).reshape(-1)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("dk,H", [(64, 2), (32, 3), (128, 1)])
def test_beam_self_attention_matches_gathered_decode(dtype, dk, H):
    from klab_multimodalmodel_b200 import ops as O
    B, nb, T = 3, 4, 19
    R, inner = B * nb, H * dk
    g = torch.Generator().manual_seed(dk)
    qkv = torch.randn(R * T, 3 * inner, generator=g).to(DEV, dtype)
    table = torch.randn(32, H, generator=g).to(DEV)
    lut, rz = O.t5_rel_bucket_lut(T, T, False, 32, 128)
    lut = lut.to(DEV)
    for t in (0, 5, 16, T - 1):
        parent = torch.randint(0, nb, (R, T + 1), generator=g) + (torch.arange(R) // nb * nb)[:, None]
        parent[:, t] = torch.arange(R)
        src = parent.to(DEV, torch.int32)
        q = qkv.view(R, T, 3 * inner)[:, t, :inner]
        got = O.t5_attention_decode_beam(q, qkv[:, inner:2 * inner], qkv[:, 2 * inner:], R, H, T, dk, kv_group=nb, src=src,
                                         bias_table=table, lut=lut, rel_zero=rz, q_offset=t)
        kg = _gather_self(qkv[:, inner:2 * inner], src, T, t)
        vg = _gather_self(qkv[:, 2 * inner:], src, T, t)
        ref, _ = O.t5_attention_fwd(q.contiguous(), kg, vg, R, H, 1, t + 1, dk, bias_table=table, lut=lut, rel_zero=rz, causal=True,
                                    q_offset=t)
        # different summation order from the reference kernels: fp32 within 1e-5, bf16 outputs within two bf16 ulps
        tol = dict(rtol=1e-5, atol=1e-5) if dtype == torch.float32 else dict(rtol=1.6e-2, atol=1.6e-2)
        torch.testing.assert_close(got.float(), ref.float(), **tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("group", [1, 2, 4, 8])
def test_beam_cross_attention_shares_kv(dtype, group):
    from klab_multimodalmodel_b200 import ops as O
    B, H, dk, Le = 5, 2, 64, 77
    R, inner = B * group, H * dk
    g = torch.Generator().manual_seed(group)
    kv = torch.randn(B * Le, 2 * inner, generator=g).to(DEV, dtype)
    q = torch.randn(R, inner, generator=g).to(DEV, dtype)
    got = O.t5_attention_decode_beam(q, kv[:, :inner], kv[:, inner:], R, H, Le, dk, kv_group=group)
    rep = kv.view(B, Le, 2 * inner).repeat_interleave(group, 0).reshape(R * Le, 2 * inner)       # HF's per-beam copy
    ref, _ = O.t5_attention_fwd(q, rep[:, :inner], rep[:, inner:], R, H, 1, Le, dk)
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == torch.float32 else dict(rtol=1.6e-2, atol=1.6e-2)
    torch.testing.assert_close(got.float(), ref.float(), **tol)


# ---- end to end ------------------------------------------------------------------------------------------------------------
def _transformer(t5, sd, dtype=torch.float32):
    from klab_multimodalmodel_b200.modeling import T5Config, T5ForConditionalGeneration
    tr = T5ForConditionalGeneration(T5Config(vocab_size=t5.vocab_size, d_model=t5.d_model, d_kv=t5.d_kv, d_ff=t5.d_ff,
                                             num_layers=t5.num_layers, num_decoder_layers=t5.num_decoder_layers, num_heads=t5.num_heads))
    tr.load_state_dict(sd, strict=True)
    return tr.to(DEV).eval()


def _gen(tr, emb, o, dtype=torch.float32):
    out = tr.generate(inputs_embeds=emb.to(DEV, dtype), return_dict_in_generate=True, output_scores=True,
                      **{k: v for k, v in o.items() if v is not None})
    return out.sequences.cpu(), out.sequences_scores.cpu()


@pytest.mark.parametrize("name", HF_CASES)
def test_generate_fp32_matches_transformers_and_oracle(name):
    t5, sd, emb, runs = golden_case(name)
    tr = _transformer(t5, sd)
    for o, seqs, scores in runs:
        got, got_scores = _gen(tr, emb, o)
        assert np.array_equal(got.numpy(), seqs), (name, o, got, seqs)
        np.testing.assert_allclose(got_scores.numpy(), scores, rtol=1e-4, atol=1e-4, err_msg=str(o))
    for o, _, _ in runs[::5]:                                          # the oracle, which equals them (tests/test_beam_oracle_cpu.py)
        ref, ref_scores = oracle_run(emb, sd, t5, o)
        got, got_scores = _gen(tr, emb, o)
        assert torch.equal(got, ref)
        torch.testing.assert_close(got_scores, ref_scores, rtol=1e-4, atol=1e-4)


def _mymodel(name, dtype):
    from klab_multimodalmodel_b200.modeling import Swinv2Config, T5Config
    from klab_multimodalmodel_b200.models.model import MyModel
    t5, sd, emb, runs = golden_case(name)
    case, swin, _, sds, px, src, tgt = case_inputs(name)
    tcfg = T5Config(vocab_size=t5.vocab_size, d_model=t5.d_model, d_kv=t5.d_kv, d_ff=t5.d_ff, num_layers=t5.num_layers,
                    num_decoder_layers=t5.num_decoder_layers, num_heads=t5.num_heads)
    scfg = Swinv2Config(image_size=swin.image_size, embed_dim=swin.embed_dim, depths=tuple(swin.depths), num_heads=tuple(swin.num_heads),
                        window_size=swin.window_size, pretrained_window_sizes=tuple(swin.pretrained_window_sizes))
    args = types.SimpleNamespace(result_dir="/tmp", language_model_name=tcfg, image_model_name=scfg, image_model_train=False,
                                 transformer_model_name=tcfg, compute_dtype=dtype)
    model = MyModel(args)
    model.language_model.load_state_dict(sds["language_model"], strict=True)
    model.image_model.load_state_dict(sds["image_model"], strict=True)
    model.transformer.load_state_dict(sd, strict=True)
    return model.to(DEV).eval(), (t5, sd, emb, runs), px.to(DEV), src.to(DEV)


def test_mymodel_forward_runs_beam_search_from_generation_config():
    model, (t5, sd, emb, runs), px, src = _mymodel("tiny_a", "fp32")
    o = dict(num_beams=4, max_new_tokens=None, length_penalty=1.0, early_stopping=False, num_return_sequences=1)
    model.transformer.generation_config.num_beams = 4
    got = model({"pixel_values": px}, {"input_ids": src}, return_loss=False).cpu()
    ref, _ = oracle_run(emb, sd, t5, o)
    assert torch.equal(got, ref)
    model.transformer.generation_config.num_beams = 1
    from klab_multimodalmodel_b200.generation import greedy_generate
    emb_d, B, Le = model._concat_embeddings({"pixel_values": px}, {"input_ids": src})
    assert torch.equal(model({"pixel_values": px}, {"input_ids": src}, return_loss=False).cpu(),
                       greedy_generate(model.transformer, emb_d, B, Le).cpu())


def test_graphs_off_and_geometry_switches_give_identical_output():
    from klab_multimodalmodel_b200.graphs import POOL
    t5, sd, emb, runs = golden_case("mid")
    tr = _transformer(t5, sd)
    o = dict(num_beams=4, length_penalty=1.0, early_stopping=False, num_return_sequences=4)
    for dtype in (torch.float32, torch.bfloat16):
        a = _gen(tr, emb, o, dtype)
        b = _gen(tr, emb, dict(o, num_beams=2, num_return_sequences=1), dtype)         # another geometry in between
        c = _gen(tr, emb[:1], o, dtype)                                                    # and another batch size
        again = _gen(tr, emb, o, dtype)
        POOL.enabled = False
        try:
            eager = _gen(tr, emb, o, dtype)
            eager_b = _gen(tr, emb, dict(o, num_beams=2, num_return_sequences=1), dtype)
        finally:
            POOL.enabled = True
        for x, y in ((a, again), (a, eager), (b, eager_b)):
            assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])
        assert c[0].shape[0] == 4


def test_num_beams_one_is_greedy():
    from klab_multimodalmodel_b200.generation import greedy_generate
    t5, sd, emb, runs = golden_case("tiny_b")
    tr = _transformer(t5, sd)
    B, Le, d = emb.shape
    x = emb.to(DEV).reshape(B * Le, d)
    assert torch.equal(tr.generate(inputs_embeds=emb.to(DEV), num_beams=1).cpu(), greedy_generate(tr, x, B, Le).cpu())


@pytest.mark.parametrize("name", HF_CASES)
def test_bf16_scores_equal_teacher_forced_nll(name):
    """bf16 hypotheses may differ from fp32 ones, but each returned score must be what the bf16 model assigns to its own
    hypothesis: sequences_scores * len ** length_penalty = -(summed token NLL) of the teacher-forced loss."""
    t5, sd, emb, runs = golden_case(name)
    tr = _transformer(t5, sd)
    for lp in (1.0, 2.0):
        o = dict(num_beams=4, length_penalty=lp, early_stopping=False, num_return_sequences=4)
        seqs, scores = _gen(tr, emb, o, torch.bfloat16)
        ref, _ = oracle_run(emb, sd, t5, dict(o, max_new_tokens=None))
        diff = (seqs[:, :min(seqs.shape[1], ref.shape[1])] != ref[:, :min(seqs.shape[1], ref.shape[1])]).any(0).nonzero()
        print(f"{name} lp={lp}: first position where bf16 ids differ from the fp32 oracle: "
              f"{int(diff[0]) if len(diff) else 'none'}")
        B, Le, d = emb.shape
        for r in range(seqs.shape[0]):
            row = seqs[r, 1:]
            eos = (row == 1).nonzero()
            n = int(eos[0]) + 1 if len(eos) else len(row)
            labels = row[:n][None].to(DEV)
            e = emb[r // 4].to(DEV, torch.bfloat16).reshape(Le, d)
            with torch.no_grad():
                nll = float(tr.loss_from_embeds(e, 1, Le, labels)) * n
            want = -nll / n ** lp
            assert abs(float(scores[r]) - want) <= 1e-2 * abs(want), (name, lp, r, float(scores[r]), want)
