"""The masked training-mode restatement of the T5 transformer (tests/masked_oracle.py) on the host: with all-ones masks it is
oracle/t5.py (and tests/t5v11_oracle.py) exactly; with random masks it reproduces transformers 5.5.0 in training mode with every
dropout replaced by the same masks -- stored (tests/golden/hf_masked.npz, written by tests/golden/make_masked_golden.py) and
live where transformers imports.  The GPU test of the training step (tests/test_training_dropout_gpu.py) uses it as yardstick."""
import os

import numpy as np
import pytest
import torch

from oracle.t5 import t5_lm_loss
from tests import masked_oracle as MO
from tests import t5v11_oracle as V11
from tests.golden import make_masked_golden as G
from tests.golden.make_hf_golden import sketch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "hf_masked.npz"))


def _leaves(sd):
    leaf = {}
    return {k: leaf.setdefault(id(v), v.clone().requires_grad_(True)) for k, v in sd.items()}


def _loss_and_grads(fn, name):
    sd = _leaves(G.case_state_dict(name))
    emb, lab = G.case_inputs(name)
    loss = fn(emb, lab, sd)
    loss.backward()
    return loss, sd


def _site_log():
    log = []

    def mask(site, shape):
        log.append(repr(site))
        return G.random_mask(site, shape)
    return mask, log


@pytest.mark.parametrize("name", list(G.CASES))
def test_all_ones_masks_are_the_eval_oracle(name):
    """Every site multiplied by ones: loss and every gradient bit-identical to oracle/t5.py (ReLU, scaled head) or
    tests/t5v11_oracle.py (gated-gelu, unscaled head)."""
    dims = G.case_dims(name)
    ones = lambda site, shape: torch.ones(shape)                                     # noqa: E731
    got, gsd = _loss_and_grads(lambda e, l, sd: MO.lm_loss(e, l, sd, dims, ones), name)
    if name == "relu":
        ref, rsd = _loss_and_grads(lambda e, l, sd: t5_lm_loss(e, l, sd, dims), name)
    else:
        ref, rsd = _loss_and_grads(lambda e, l, sd: V11.lm_loss(e, l, sd, dims), name)
    assert torch.equal(got, ref)
    for k in gsd:
        assert torch.equal(gsd[k].grad, rsd[k].grad), k


@pytest.mark.parametrize("name", list(G.CASES))
def test_masked_oracle_reproduces_golden(name):
    """All eight dropout sites, every block of both stacks: the sites the restatement visits are the ones transformers called,
    in the same order; loss and every gradient (norm and sketch) equal transformers' under the same masks."""
    dims = G.case_dims(name)
    mask, log = _site_log()
    loss, sd = _loss_and_grads(lambda e, l, sd: MO.lm_loss(e, l, sd, dims, mask), name)
    assert log == list(GOLD[f"{name}/sites"])
    assert {eval(s)[2] for s in log} == set(MO.SITES)
    assert loss.item() == pytest.approx(float(GOLD[f"{name}/loss"]), rel=1e-5)
    names = list(GOLD[f"{name}/grad_names"])
    assert set(names) <= set(sd)
    for i, k in enumerate(names):
        g = sd[k].grad
        ref_norm = float(GOLD[f"{name}/gnorm"][i])
        assert g.double().norm().item() == pytest.approx(ref_norm, rel=1e-5), k
        err = np.linalg.norm(sketch(g, k) - GOLD[f"{name}/gsketch"][i].astype(np.float64))
        assert err <= 1e-5 * ref_norm + 1e-7, (k, err, ref_norm)
    # the masks matter: without them the loss moves well beyond the tolerance
    plain, _ = _loss_and_grads(lambda e, l, sd: MO.lm_loss(e, l, sd, dims), name)
    assert abs(plain.item() - loss.item()) > 1e-3 * abs(loss.item())


@pytest.mark.parametrize("name", list(G.CASES))
def test_masked_oracle_matches_live_transformers(name):
    pytest.importorskip("transformers")
    dims = G.case_dims(name)
    live = G.hf_case(name)
    mask, log = _site_log()
    loss, sd = _loss_and_grads(lambda e, l, sd: MO.lm_loss(e, l, sd, dims, mask), name)
    assert log == list(live["sites"])
    assert loss.item() == pytest.approx(float(live["loss"]), rel=1e-5)
    for i, k in enumerate(live["grad_names"]):
        assert sd[k].grad.double().norm().item() == pytest.approx(float(live["gnorm"][i]), rel=1e-5), k
        err = np.linalg.norm(sketch(sd[k].grad, k) - live["gsketch"][i].astype(np.float64))
        assert err <= 1e-5 * float(live["gnorm"][i]) + 1e-7, k
