"""CPU: host-side contract of the product model (no compute): state_dict keys/shapes equal the reference's,
trainability rule, aliasing, and that the forward fails loudly without CUDA (no CPU fallback)."""
import json
import os
import sys
import types

import pytest
import torch

from monodetr_b200 import build_monodetr
from monodetr_b200.monodetr import DEFAULT_MODEL_CFG
from oracle import monodetr_torch as om

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def model():
    torch.manual_seed(0)
    m, crit = build_monodetr(DEFAULT_MODEL_CFG)
    assert crit is None
    return m


def test_state_dict_contract(model):
    sd = model.state_dict()
    spec = om.with_aliases({k: torch.empty(s) for k, s in om.state_dict_spec().items()})
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in spec.items()}
    assert len(sd) == 582                                                    # SURVEY.md 8b
    assert sum(p.numel() for p in model.parameters()) == 37675220
    trainable = [p for p in model.parameters() if p.requires_grad]
    assert len(trainable) == 328 and sum(p.numel() for p in trainable) == 37452739


def test_aliases_are_the_same_objects(model):
    assert model.depthaware_transformer.decoder.bbox_embed is model.bbox_embed
    assert model.depthaware_transformer.decoder.dim_embed is model.dim_embed_3d


def test_frozen_rule(model):
    for name, p in model.named_parameters():
        if name.startswith("backbone.0.body."):
            assert p.requires_grad == any(s in name for s in ("layer2", "layer3", "layer4")), name
    assert not model.depth_predictor.depth_bin_values.requires_grad


def test_init_rules(model):
    assert torch.allclose(model.class_embed[0].bias, torch.full((3,), -4.59511985))
    assert torch.all(model.bbox_embed[0].layers[-1].bias[2:] == -2.0)
    m = model.depthaware_transformer.encoder.layers[0].self_attn
    assert not m.sampling_offsets.weight.any() and not m.attention_weights.weight.any()
    assert float(m.sampling_offsets.bias.abs().max()) == 4.0


def test_strict_load_of_reference_shaped_checkpoint(model):
    sd = om.with_aliases(om.deterministic_state_dict())
    sd["backbone.0.body.bn1.num_batches_tracked"] = torch.tensor(0)           # dropped like the reference (backbone.py:41-50)
    model.load_state_dict(sd, strict=True)


def test_forward_requires_cuda(model):
    images, calibs, sizes = om.synthetic_inputs(1, 0, H=96, W=320)
    with pytest.raises(RuntimeError, match="CUDA"):
        model(images, calibs, None, sizes)


def _reference_spec():
    with open(os.path.join(ROOT, "tests", "golden", "reference_model_spec.json")) as f:
        return json.load(f)


def test_state_dict_matches_unmodified_reference(model):
    spec = _reference_spec()
    assert [k for k, _ in spec["state_dict"]] == list(model.state_dict().keys())
    assert {k: tuple(s) for k, s in spec["state_dict"]} == {k: tuple(v.shape) for k, v in model.state_dict().items()}
    assert set(spec["trainable"]) == {n for n, p in model.named_parameters() if p.requires_grad}


def test_build_returns_the_reference_criterion_when_importable(monkeypatch):
    """B2: build_monodetr(cfg) -> (model, criterion) like monodetr.py:550-614; with the reference package importable
    (as inside tools/train_val.py) the criterion is the reference's SetCriterion, built with what the reference's build()
    passes it (stored in tests/golden/reference_model_spec.json).  A stand-in `lib.models.monodetr` records the call."""
    spec = _reference_spec()
    cfg = spec["model_cfg"]

    class SetCriterion(torch.nn.Module):
        def __init__(self, num_classes, matcher, weight_dict, focal_alpha, losses):
            super().__init__()
            self.num_classes, self.matcher, self.weight_dict, self.focal_alpha, self.losses = \
                num_classes, matcher, weight_dict, focal_alpha, losses

    matcher = object()
    pkg = {name: types.ModuleType(name) for name in ("lib", "lib.models", "lib.models.monodetr",
                                                      "lib.models.monodetr.matcher", "lib.models.monodetr.monodetr")}
    pkg["lib.models.monodetr.matcher"].build_matcher = lambda c: matcher if c == cfg else None
    pkg["lib.models.monodetr.monodetr"].SetCriterion = SetCriterion
    for name, mod in pkg.items():
        monkeypatch.setitem(sys.modules, name, mod)
    _, crit = build_monodetr(cfg)
    assert type(crit) is SetCriterion and crit.matcher is matcher
    ref = spec["criterion"]
    assert crit.weight_dict == ref["weight_dict"] and crit.losses == ref["losses"]
    assert crit.focal_alpha == ref["focal_alpha"] and crit.num_classes == ref["num_classes"]
    # without loss weights in the cfg (stand-alone model use) there is nothing to build a criterion from
    assert build_monodetr(DEFAULT_MODEL_CFG)[1] is None
