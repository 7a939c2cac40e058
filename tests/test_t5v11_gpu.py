"""T5 v1.1 / Flan-T5 on the B200: the gated-GELU kernels (csrc/geglu.cu) against a float64 statement, and the gated, unscaled
models end to end -- loss, every gradient, greedy / beam / sampled ids -- against transformers 5.5.0's stored outputs
(tests/golden/hf_t5v11.npz) and the oracle, then MyModel with gated towers, its training with an untied LM head."""
import dataclasses
import math
import types

import numpy as np
import pytest
import torch

from oracle.caption_model import seeded_inputs
from oracle.t5 import t5_lm_loss
from tests.golden import make_t5v11_golden as G
from tests.golden.make_golden import CASES, dims_of
from tests.golden.make_hf_golden import sketch
from tests.t5v11_oracle import V11Dims, caption_loss, seeded_state_dicts
from tests.test_t5v11_oracle_cpu import GOLD, oracle_loss_and_grads

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ---------------------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------------------
def _gelu_new64(x):
    t = torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3))
    return 0.5 * x * (1.0 + t), 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * math.sqrt(2.0 / math.pi) * (1.0 + 3 * 0.044715 * x * x)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("dff", [2816, 64])
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_geglu_kernels_match_float64(dff, dtype, p):
    from klab_multimodalmodel_b200 import ops as O
    M = 333
    g = torch.Generator().manual_seed(dff)
    u = (torch.randn(M, 2 * dff, generator=g) * 2).to(DEV, dtype)
    dh = torch.randn(M, dff, generator=g).to(DEV, dtype)
    counter = torch.tensor([12345], dtype=torch.int64, device=DEV)
    seed = 77
    # the mask klab_dropout_apply draws for a contiguous [M, d_ff] tensor with the same seed and device counter
    mask = O.dropout_apply(torch.ones(M, dff, dtype=dtype, device=DEV), p, seed, counter).double().cpu() if p else 1.0
    h = O.geglu_fwd(u, p, seed, counter if p else None)
    du = O.geglu_bwd(dh, u, p, seed, counter if p else None)
    u64, dh64 = u.double().cpu(), dh.double().cpu() * mask
    a, b = u64[:, :dff], u64[:, dff:]
    ga, dga = _gelu_new64(a)
    ref_h = ga * b * mask
    ref_du = torch.cat([dh64 * b * dga, dh64 * ga], 1)
    # fp32: h to 1e-4; du to 2e-3, since 1 - t^2 of gelu_new' cancels in fp32 where tanh saturates (as in torch's own fp32 autograd
    # of gelu_new); observed on a B200: 5.8e-4
    for got, ref, tol in ((h, ref_h, 1e-4), (du, ref_du, 2e-3)):
        tol = tol if dtype == torch.float32 else 8e-3
        got = got.double().cpu()
        assert got.shape == ref.shape
        err = (got - ref).abs() / (ref.abs() + 1e-2)
        assert err.max().item() <= tol, (dff, dtype, p, err.max().item())
    if p:
        dropped = mask == 0
        assert (h.cpu()[dropped] == 0).all() and (h.cpu()[~dropped & ((ga * b).abs() > 1e-3)] != 0).all()
        assert 0.05 < dropped.double().mean().item() < 0.15
        counter += 1                                                   # a replay after klab_seed_advance: another mask
        assert not torch.equal(O.geglu_fwd(u, p, seed, counter).cpu() == 0, h.cpu() == 0)


def test_geglu_rejects_d_ff_not_multiple_of_8():
    from klab_multimodalmodel_b200 import ops as O
    with pytest.raises(RuntimeError, match="multiple of 8"):
        O.geglu_fwd(torch.zeros(4, 24, device=DEV))


# ---------------------------------------------------------------------------------------------------------------------------
# gated models against transformers and the oracle
# ---------------------------------------------------------------------------------------------------------------------------
def _tcfg(dims):
    from klab_multimodalmodel_b200.modeling import T5Config
    return T5Config(vocab_size=dims.vocab_size, d_model=dims.d_model, d_kv=dims.d_kv, d_ff=dims.d_ff, num_layers=dims.num_layers,
                    num_decoder_layers=dims.num_decoder_layers, num_heads=dims.num_heads, feed_forward_proj=dims.feed_forward_proj,
                    tie_word_embeddings=dims.scale_decoder_outputs)


def transformer(name, tmp_path):
    """(a) built from the config and loaded (tied), (b) from_pretrained of the checkpoint directory (untied)."""
    from klab_multimodalmodel_b200.modeling import T5ForConditionalGeneration
    if G.CASES[name]["untied"]:
        tr = T5ForConditionalGeneration.from_pretrained(G.write_checkpoint(name, str(tmp_path / name)))
    else:
        tr = T5ForConditionalGeneration(_tcfg(G.case_dims(name)))
        tr.load_state_dict(G.case_state_dict(name), strict=True)
    assert tr.lm_head_tied != G.CASES[name]["untied"] and tr.config.gated and not tr.config.scale_decoder_outputs
    return tr.to(DEV).eval()


def _loss_and_grads(tr, name, dtype):
    emb, lab = G.case_inputs(name)
    B, Le, d = emb.shape
    tr.zero_grad(set_to_none=True)
    loss = tr.loss_from_embeds(emb.reshape(B * Le, d).to(DEV, dtype), B, Le, lab.to(DEV))
    loss.backward()
    return loss.item(), {k: p.grad.detach().cpu() for k, p in tr.named_parameters()}


@pytest.mark.parametrize("name", list(G.CASES))
def test_fp32_loss_and_every_gradient(name, tmp_path):
    tr = transformer(name, tmp_path)
    _, osd = oracle_loss_and_grads(name)
    for _ in range(2):                                                 # eager, then a captured replay of the blocks
        loss, grads = _loss_and_grads(tr, name, torch.float32)
        assert loss == pytest.approx(float(GOLD[f"{name}/loss"]), rel=1e-4)
        names = list(GOLD[f"{name}/grad_names"])
        assert sorted(grads) == names
        for i, k in enumerate(names):
            ref_norm = float(GOLD[f"{name}/gnorm"][i])
            assert grads[k].double().norm().item() == pytest.approx(ref_norm, rel=1e-4), k
            assert np.linalg.norm(sketch(grads[k], k) - GOLD[f"{name}/gsketch"][i]) <= 1e-4 * ref_norm + 1e-6, k
            o = osd[k].grad.double()
            assert (grads[k].double() - o).norm().item() <= 1e-4 * o.norm().item() + 1e-6, k


def test_bf16_loss_and_gradients(tmp_path):
    name = "v11_untied"
    tr = transformer(name, tmp_path)
    loss, grads = _loss_and_grads(tr, name, torch.bfloat16)
    ref_loss, osd = oracle_loss_and_grads(name)
    assert loss == pytest.approx(ref_loss, rel=1e-2)
    errs = {k: (g.double() - osd[k].grad.double()).norm().item() / osd[k].grad.double().norm().item() for k, g in grads.items()}
    worst = max(errs, key=errs.get)
    print("bf16 relative gradient errors: median", float(np.median(list(errs.values()))), "worst", worst, errs[worst])
    assert errs[worst] <= 1e-1 and float(np.median(list(errs.values()))) <= 3e-2
    assert errs["lm_head.weight"] <= 3e-2 and errs["shared.weight"] <= 5e-2


@pytest.fixture
def graphs_off():
    from klab_multimodalmodel_b200.graphs import POOL
    was = POOL.enabled

    def set_(on):
        POOL.enabled = on and was
    yield set_
    POOL.enabled = was


@pytest.mark.parametrize("graphs", [True, False])
@pytest.mark.parametrize("name", list(G.CASES))
def test_fp32_greedy_beam_and_sample_ids(name, graphs, tmp_path, graphs_off, monkeypatch):
    from klab_multimodalmodel_b200 import generation
    graphs_off(graphs)
    tr = transformer(name, tmp_path)
    emb, _ = G.case_inputs(name)
    e = emb.to(DEV)
    for _ in range(2):                                                 # first call captures, the second replays
        assert np.array_equal(tr.generate(inputs_embeds=e).cpu().numpy(), GOLD[f"{name}/greedy"])
        out = tr.generate(inputs_embeds=e, num_beams=G.NUM_BEAMS, return_dict_in_generate=True, output_scores=True)
        assert np.array_equal(out.sequences.cpu().numpy(), GOLD[f"{name}/beam_sequences"])
        assert np.allclose(out.sequences_scores.cpu().numpy(), GOLD[f"{name}/beam_scores"], rtol=1e-4, atol=1e-5)
        o = dict(G.SAMPLE_OPTS)
        monkeypatch.setattr(generation, "draw_seed", lambda: o["seed"])
        got = tr.generate(inputs_embeds=e, do_sample=True, **{k: v for k, v in o.items() if k != "seed"})
        assert np.array_equal(got.cpu().numpy(), GOLD[f"{name}/sample"])
    B, Le, d = emb.shape
    rec = generation.greedy_generate_recompute(tr, e.reshape(B * Le, d), B, Le)
    assert np.array_equal(rec.cpu().numpy(), GOLD[f"{name}/greedy"])


# ---------------------------------------------------------------------------------------------------------------------------
# MyModel: gated frozen text tower and gated transformer with its own LM head
# ---------------------------------------------------------------------------------------------------------------------------
def gated_mymodel(dtype="fp32"):
    from klab_multimodalmodel_b200.modeling import Swinv2Config
    from klab_multimodalmodel_b200.models.model import MyModel
    case = CASES["tiny_a"]
    swin, t5 = dims_of(case)
    t5 = V11Dims(**dataclasses.asdict(t5))                       # gated-gelu, no LM-head scale
    sds = seeded_state_dicts(t5, swin, t5, seed=0, style="hf", untied_head=True)
    scfg = Swinv2Config(image_size=swin.image_size, embed_dim=swin.embed_dim, depths=tuple(swin.depths), num_heads=tuple(swin.num_heads),
                        window_size=swin.window_size, pretrained_window_sizes=tuple(swin.pretrained_window_sizes))
    args = types.SimpleNamespace(result_dir="/tmp", language_model_name=_tcfg(t5), image_model_name=scfg, image_model_train=False,
                                 transformer_model_name=_tcfg(t5), compute_dtype=dtype)
    model = MyModel(args)
    model.language_model.load_state_dict(sds["language_model"], strict=True)
    model.image_model.load_state_dict(sds["image_model"], strict=True)
    model.transformer.load_state_dict(sds["transformer"], strict=True)         # the distinct lm_head.weight unties the head
    assert not model.transformer.lm_head_tied
    return model.cuda().eval(), sds, case, swin, t5


def test_mymodel_gated_caption_loss_fp32():
    model, sds, case, swin, t5 = gated_mymodel()
    px, src, tgt = seeded_inputs(case["batch"], swin, t5.vocab_size, case["l_src"], case["l_tgt"], seed=5)
    for _ in range(2):
        loss = model({"pixel_values": px.cuda()}, {"input_ids": src.cuda()}, {"input_ids": tgt.cuda()})
        ref = caption_loss(px, src, tgt, sds, t5, swin, t5)
        assert loss.item() == pytest.approx(ref.item(), rel=1e-4)


@pytest.mark.parametrize("optimizer", ["klab", "torch"])
def test_training_tracks_oracle_and_updates_head_and_embedding_separately(optimizer):
    model, sds, case, swin, t5 = gated_mymodel()
    tr = model.transformer
    lr, steps = 5e-4, 3
    params = list(tr.parameters())
    assert any(p is tr.lm_head.weight for p in params) and any(p is tr.shared.weight for p in params)
    if optimizer == "klab":
        from klab_multimodalmodel_b200.optim import Adam
        opt = Adam(params, lr=lr)
    else:
        opt = torch.optim.Adam(params, lr=lr)
    osd = {k: dict(v) for k, v in sds.items()}
    uniq = {}
    for k, v in osd["transformer"].items():
        osd["transformer"][k] = uniq.setdefault(id(v), v.clone().requires_grad_(True))
    oopt = torch.optim.Adam(list(uniq.values()), lr=lr)
    head0, emb0 = tr.lm_head.weight.detach().clone(), tr.shared.weight.detach().clone()
    got, ref = [], []
    for s in range(steps):
        px, src, tgt = seeded_inputs(case["batch"], swin, t5.vocab_size, case["l_src"], case["l_tgt"], ignore_tail=True, seed=100 + s % 2)
        loss = model({"pixel_values": px.cuda()}, {"input_ids": src.cuda()}, {"input_ids": tgt.cuda()})
        got.append(loss.item())
        loss.backward()
        opt.step()
        opt.zero_grad()
        rl = caption_loss(px, src, tgt, osd, t5, swin, t5)
        ref.append(rl.item())
        rl.backward()
        oopt.step()
        oopt.zero_grad()
    for s, (a, b) in enumerate(zip(got, ref)):
        assert abs(a - b) <= 1e-4 * (1 + 2 * s) * abs(b), (optimizer, s, got, ref)
    from klab_multimodalmodel_b200.optim import wait_pending_updates
    wait_pending_updates()
    head, emb = tr.lm_head.weight.detach().cpu(), tr.shared.weight.detach().cpu()
    assert not torch.equal(head, head0.cpu()) and not torch.equal(emb, emb0.cpu())
    for got_w, key in ((head, "lm_head.weight"), (emb, "shared.weight")):
        want = osd["transformer"][key].detach()
        assert (got_w - want).norm().item() <= 1e-3 * want.norm().item(), key
    assert (head - emb).norm().item() > 0.1 * emb.norm().item()


def test_relu_tied_model_reads_shared_as_head():
    """The original T5 path is untouched: lm_head IS shared, the scale is d_model**-0.5, the FFN weight is wi."""
    from klab_multimodalmodel_b200.modeling import T5Config, T5ForConditionalGeneration
    tr = T5ForConditionalGeneration(T5Config(vocab_size=256, d_model=128, d_ff=256, num_layers=1, num_heads=2)).to(DEV).eval()
    assert tr.lm_head_tied and tr.config.lm_head_scale == 128 ** -0.5 and not tr.config.gated
    emb = torch.randn(2, 5, 128, device=DEV)
    lab = torch.randint(2, 200, (2, 4), device=DEV)
    sd = {k: v.detach().cpu() for k, v in tr.state_dict().items()}
    from oracle.t5 import T5Dims
    dims = T5Dims(vocab_size=256, d_model=128, d_ff=256, num_layers=1, num_heads=2)
    ref = t5_lm_loss(emb.cpu(), lab.cpu(), sd, dims).item()
    assert tr.loss_from_embeds(emb.reshape(10, 128), 2, 5, lab).item() == pytest.approx(ref, rel=1e-4)
