"""The training step with T5 dropout on (p = 0.1, model.transformer.train() as train.py runs it), against the masked restatement
tests/masked_oracle.py fed with the masks the library draws.  Every mask is a pure function of (site seed + device step counter,
element index), so with the counter pinned the mask of any site is dropout_apply over a tensor of ones of the site's shape.  The
site seeds are those of modeling.py / functional.py, read from each stack's `seed_base`:

    seed_base                     stack input (:734)
    base + 0 / + 1                self-attention probabilities (:332) / self-attention output (:375)
    base + 2 / + 3                cross-attention probabilities (:332) / cross-attention output (:406)
    base + 4 / + 5                FFN inner (:95, gated :119) / FFN output (:149)
    seed_base + 7                 after the final norm (:768)
with base = seed_base + 16 (i + 1) for block i.  A site wired to the wrong seed, a missing or misplaced site, or a backward
kernel that regenerates a different mask than its forward twin moves some gradient far beyond the bounds."""
import numpy as np
import pytest
import torch

from oracle.caption_model import seeded_inputs
from tests import masked_oracle as MO
from tests.golden import make_t5v11_golden as G11
from tests.golden.make_golden import CASES, EXTRA_CASES
from tests.test_step_parity_gpu import build

pytestmark = pytest.mark.gpu

P = 0.1
PINNED = 123456789
_OFFSET = {"self_probs": 0, "self_out": 1, "cross_probs": 2, "cross_out": 3, "ff_inner": 4, "ff_out": 5}


def site_seed(tr, site):
    stack, i, kind = site
    base = getattr(tr, stack).seed_base
    if kind == "input":
        return base
    if kind == "final":
        return base + 7
    return base + 16 * (i + 1) + _OFFSET[kind]


def device_masks(tr, ctr):
    """mask(site, shape) for the masked oracle: the multipliers the kernels of site `site` apply with the counter `ctr`."""
    from klab_multimodalmodel_b200 import ops as O
    seen = set()

    def mask(site, shape):
        seen.add(site[2])
        return O.dropout_apply(torch.ones(shape, device=ctr.device), P, site_seed(tr, site), ctr).cpu()
    mask.seen = seen
    return mask


def _leaves(sds, case):
    sds = {k: dict(v) for k, v in sds.items()}
    leaves = {}
    for scope in ("transformer", "image_model"):
        uniq = {}
        for k, v in sds[scope].items():
            if id(v) not in uniq:
                uniq[id(v)] = v.clone().requires_grad_(scope == "transformer" or case["train_swin"])
            sds[scope][k] = uniq[id(v)]
            leaves[(scope, k)] = uniq[id(v)]
    return sds, leaves


def masked_oracle_grads(case, sds, swin, t5, px, src, tgt, mask, autocast=False):
    sds, leaves = _leaves(sds, case)
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
        loss = MO.caption_loss(px, src, tgt, sds, t5, swin, t5, mask)
    loss.backward()
    return loss.item(), leaves


def model_grads(model):
    return {(scope, k): p.grad.detach().float().cpu() for scope, mod in (("transformer", model.transformer), ("image_model", model.image_model))
            for k, p in mod.named_parameters() if p.grad is not None}


def check_fp32(loss, grads, ref_loss, leaves, what):
    assert abs(loss - ref_loss) <= 1e-4 * abs(ref_loss), (what, loss, ref_loss)
    failures = []
    for key, g in grads.items():                               # tied keys of the reference share one leaf
        ref = leaves[key]
        err = (g - ref.grad).norm().item() / max(ref.grad.norm().item(), 1e-12)
        if err > 2e-4 and (g - ref.grad).norm().item() > 1e-5:
            failures.append((err, ".".join(key)))
    failures.sort(reverse=True)
    assert not failures, f"{what}: {len(failures)} gradient tensors beyond 2e-4: {failures[:8]}"
    assert len(grads) >= 50


@pytest.mark.parametrize("graphs", [True, False])
@pytest.mark.parametrize("name", ["mid", "tiny_a"])
def test_fp32_training_step_matches_masked_oracle(name, graphs):
    """MyModel in training mode, fp32: loss within 1e-4 relative and every gradient within 2e-4 Frobenius-relative of the masked
    oracle, on the warm-up step, the captured step and its replay (graphs on) or eagerly (graphs off).  Covers all eight
    dropout sites of both stacks: the stack-input and final-norm DropoutFn / LMHeadLossFn masks, and inside T5BlockFn the
    attention-probability masks of every attention kernel the shapes select, the o-projection and FFN GEMM epilogues, the
    rmsnorm_bwd(drop=...) masks of the sub-layer outputs and the ReLU-backward dgrad.  After one seed_advance the masks and
    the loss change."""
    from klab_multimodalmodel_b200 import ops as O
    from klab_multimodalmodel_b200.graphs import POOL
    from klab_multimodalmodel_b200.modeling import step_seed
    case = CASES.get(name) or EXTRA_CASES[name]
    model, sds, swin, t5 = build(case, "fp32", style="hf")
    model.transformer.train()
    was = POOL.enabled
    POOL.enabled = graphs and was
    try:
        px, src, tgt = seeded_inputs(case["batch"], swin, t5.vocab_size, case["l_src"], case["l_tgt"], ignore_tail=True)
        batch = ({"pixel_values": px.cuda()}, {"input_ids": src.cuda()}, {"input_ids": tgt.cuda()})
        ctr = step_seed(px.cuda().device)
        ref = None
        for step in range(3 if POOL.enabled else 1):                 # warm-up, capture, replay
            model.zero_grad(set_to_none=True)
            ctr.fill_(PINNED)                                        # the forward advances it once: the same masks every step
            loss = model(*batch)
            loss.backward()
            if ref is None:
                mask = device_masks(model.transformer, ctr)
                ref = masked_oracle_grads(case, sds, swin, t5, px, src, tgt, mask)
                assert mask.seen == set(MO.SITES)
            check_fp32(loss.item(), model_grads(model), *ref, f"{name} step {step}")
        # one more forward advances the counter again: other masks, another loss
        first = O.dropout_apply(torch.ones(4096, device="cuda"), P, site_seed(model.transformer, ("decoder", 0, "ff_inner")), ctr).cpu()
        l2 = model(*batch).item()
        again = O.dropout_apply(torch.ones(4096, device="cuda"), P, site_seed(model.transformer, ("decoder", 0, "ff_inner")), ctr).cpu()
        assert not torch.equal(first, again)
        assert abs(l2 - ref[0]) > 1e-4 * abs(ref[0])
    finally:
        POOL.enabled = was


def test_fp32_gated_training_step_matches_masked_oracle(tmp_path):
    """The gated-GELU T5 v1.1 transformer (hf_t5v11 case v11_untied: unscaled untied LM head, d_model != heads * d_kv) in training
    mode: the klab_geglu_fwd / klab_geglu_bwd masks (FFN inner site) and all other sites, loss 1e-4 and every gradient 2e-4
    against the masked oracle, eager and replayed."""
    from klab_multimodalmodel_b200.modeling import step_seed
    from tests.test_t5v11_gpu import transformer
    name = "v11_untied"
    tr = transformer(name, tmp_path).train()
    dims = G11.case_dims(name)
    emb, lab = G11.case_inputs(name)
    B, Le, d = emb.shape
    ctr = step_seed(torch.device("cuda", torch.cuda.current_device()))
    ctr.fill_(PINNED)
    mask = device_masks(tr, ctr)
    leaf = {}
    sd = {k: leaf.setdefault(id(v), v.clone().requires_grad_(True)) for k, v in G11.case_state_dict(name).items()}
    ref_loss = MO.lm_loss(emb, lab, sd, dims, mask)
    ref_loss.backward()
    assert mask.seen == set(MO.SITES)
    for step in range(3):                                             # eager, capture, replay of the blocks
        tr.zero_grad(set_to_none=True)
        loss = tr.loss_from_embeds(emb.reshape(B * Le, d).cuda(), B, Le, lab.cuda())
        loss.backward()
        assert abs(loss.item() - ref_loss.item()) <= 1e-4 * abs(ref_loss.item()), (step, loss.item(), ref_loss.item())
        for k, p in tr.named_parameters():
            r = sd[k].grad.double()
            err = (p.grad.detach().double().cpu() - r).norm().item() / max(r.norm().item(), 1e-12)
            assert err <= 2e-4 or (p.grad.detach().double().cpu() - r).norm().item() <= 1e-5, (step, k, err)


def test_bf16_training_step_matches_masked_oracle():
    """bf16 tensor-core path on `mid` in training mode: loss within 1e-2 of the fp32 masked oracle; every gradient within 4x the
    error of the masked oracle under torch.autocast(bfloat16) + 2e-2 (+ 5e-2 for the cancellation-dominated logit_scale /
    CPB-MLP gradients), the rule of test_bf16_loss_and_all_gradients."""
    from klab_multimodalmodel_b200.modeling import step_seed
    case = EXTRA_CASES["mid"]
    model, sds, swin, t5 = build(case, "bf16", style="hf")
    model.transformer.train()
    px, src, tgt = seeded_inputs(case["batch"], swin, t5.vocab_size, case["l_src"], case["l_tgt"], ignore_tail=True)
    ctr = step_seed(px.cuda().device)
    ctr.fill_(PINNED)
    loss = model({"pixel_values": px.cuda()}, {"input_ids": src.cuda()}, {"input_ids": tgt.cuda()})
    loss.backward()
    mask = device_masks(model.transformer, ctr)
    ref_loss, leaves = masked_oracle_grads(case, sds, swin, t5, px, src, tgt, mask)
    _, ac_leaves = masked_oracle_grads(case, sds, swin, t5, px, src, tgt, mask, autocast=True)
    assert abs(loss.item() - ref_loss) <= 1e-2 * abs(ref_loss), (loss.item(), ref_loss)
    grads, failures, ratios = model_grads(model), [], []
    for key in grads:
        ref = leaves[key]
        nref = max(ref.grad.norm().item(), 1e-12)
        err = (grads[key] - ref.grad).norm().item() / nref
        err_ac = (ac_leaves[key].grad.float() - ref.grad).norm().item() / nref
        ratios.append(err / max(err_ac, 1e-3))
        noisy = "logit_scale" in key[1] or "continuous_position_bias" in key[1]
        if err > 4.0 * err_ac + (5e-2 if noisy else 2e-2):
            failures.append((err, ".".join(key), err_ac))
    failures.sort(reverse=True)
    assert not failures, f"{len(failures)} gradient tensors worse than 4x the autocast error + 2e-2: {failures[:8]}"
    print(f"[mid/bf16 train] loss {loss.item():.5f} (masked fp32 oracle {ref_loss:.5f}); median (err / autocast err) {float(np.median(ratios)):.2f}")
