"""The autograd restatement of the criterion (oracle/criterion.py) against vectors produced by the unmodified reference
HungarianMatcher + SetCriterion (tests/golden/criterion.npz, tools/gen_golden_criterion.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import criterion as oc

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "criterion.npz"))
CASES = ["train_b3", "eval_b2"]


def run_oracle(name):
    seed, B, Q, training = (int(v) for v in GOLD[f"{name}.cfg"])
    out, padded = oc.synthetic_case(seed, B, Q)
    leaves = {}
    for layer, d in [("main", out)] + [(f"aux{i}", a) for i, a in enumerate(out["aux_outputs"])]:
        for k in list(d):
            if torch.is_tensor(d[k]):
                d[k] = d[k].clone().requires_grad_(True)
                leaves[f"{layer}.{k}"] = d[k]
    losses, indices = oc.set_criterion(out, padded, training=bool(training))
    w = oc.weight_dict()
    total = sum(losses[k] * w[k] for k in losses if k in w)
    total.backward()
    return losses, indices, total, leaves


@pytest.mark.parametrize("name", CASES)
def test_losses_matching_and_gradients_match_the_reference(name):
    losses, indices, total, leaves = run_oracle(name)
    keys = [k[len(name) + 6:] for k in GOLD.files if k.startswith(f"{name}.loss.")]
    assert sorted(keys) == sorted(losses)                                   # same dict keys as SetCriterion.forward
    for k in keys:
        np.testing.assert_allclose(float(losses[k]), float(GOLD[f"{name}.loss.{k}"]), rtol=2e-6, atol=1e-7, err_msg=k)
    np.testing.assert_allclose(float(total), float(GOLD[f"{name}.total"]), rtol=2e-6)
    for l, ind in enumerate(indices):
        for b, (i, j) in enumerate(ind):
            assert np.array_equal(i.numpy(), GOLD[f"{name}.match.{l}.{b}.src"]) and np.array_equal(j.numpy(), GOLD[f"{name}.match.{l}.{b}.tgt"])
    for k, t in leaves.items():
        got = t.grad.numpy() if t.grad is not None else np.zeros(tuple(t.shape), np.float32)
        assert_grad_matches_golden(got, f"{name}.grad.{k}", rtol=1e-5, atol_rel=1e-6)


def assert_grad_matches_golden(got, key, rtol, atol_rel):
    """Tolerance atol = 1e-9 + atol_rel * max|golden|.  A dense gradient map is stored as max|grad| + a seeded sample."""
    if key in GOLD.files:
        g = GOLD[key]
        np.testing.assert_allclose(got, g, rtol=rtol, atol=1e-9 + atol_rel * np.abs(g).max(), err_msg=key)
        return
    gmax = float(GOLD[key + ".absmax"])
    np.testing.assert_allclose(np.abs(got).max(), gmax, rtol=rtol, atol=1e-9 + atol_rel * gmax, err_msg=key + " max")
    np.testing.assert_allclose(got.reshape(-1)[GOLD[key + ".idx"]], GOLD[key + ".val"], rtol=rtol, atol=1e-9 + atol_rel * gmax, err_msg=key)
