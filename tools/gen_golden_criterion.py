"""Golden vectors for the training criterion, produced by the UNMODIFIED reference classes (lib/models/monodetr/matcher.py
HungarianMatcher, lib/models/monodetr/monodetr.py SetCriterion incl. DDNLoss) run on CPU through in-memory shims
(tools/ref_shims.py + the three below; no reference file is edited):  `Tensor.cuda()` -> identity and `torch.tensor(...,
device='cuda')` -> CPU, because loss_angles / loss_depth_map hard-code the device (monodetr.py:443,462).
The gradient of the depth-map logits (a dense B x 81 x 24 x 80 map) is stored as max|grad| and a seeded sample of
DEPTH_MAP_SAMPLE entries, which keeps the fixture small.
    python tools/gen_golden_criterion.py  -> tests/golden/criterion.npz"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ref_shims  # noqa: E402
from oracle import criterion as oc  # noqa: E402

ref = ref_shims.install()
torch.Tensor.cuda = lambda self, *a, **k: self
_tensor = torch.tensor
torch.tensor = lambda *a, **k: _tensor(*a, **{kk: vv for kk, vv in k.items() if kk != "device"})
from lib.models.monodetr.matcher import HungarianMatcher  # noqa: E402
from lib.models.monodetr.monodetr import SetCriterion  # noqa: E402

DEPTH_MAP_SAMPLE = 4096

matcher = HungarianMatcher(cost_class=2, cost_bbox=5, cost_giou=2, cost_3dcenter=10)
losses = ["labels", "boxes", "cardinality", "depths", "dims", "angles", "center", "depth_map"]
crit = SetCriterion(3, matcher=matcher, weight_dict=oc.weight_dict(), focal_alpha=0.25, losses=losses)

out = {}
CASES = {"train_b3": (21, 3, 550, True), "eval_b2": (22, 2, 50, False)}
for name, (seed, B, Q, training) in CASES.items():
    o, padded = oc.synthetic_case(seed, B, Q)
    leaves = []

    def req(d):
        for k in list(d):
            if torch.is_tensor(d[k]):
                d[k] = d[k].clone().requires_grad_(True)
                leaves.append((k, d[k]))
    req(o)
    for a in o["aux_outputs"]:
        req(a)
    targets = oc.prepare_targets(padded)
    crit.train(training)
    ld = crit(o, targets)
    total = sum(ld[k] * crit.weight_dict[k] for k in ld if k in crit.weight_dict)
    total.backward()
    out[f"{name}.cfg"] = np.array([seed, B, Q, int(training)], np.int64)
    for k, v in ld.items():
        out[f"{name}.loss.{k}"] = np.asarray(float(v), np.float64)
    out[f"{name}.total"] = np.asarray(float(total), np.float64)
    for i, (k, t) in enumerate(leaves):
        layer = "main" if i < 6 else f"aux{(i - 6) // 5}"
        g = t.grad.numpy() if t.grad is not None else np.zeros(t.shape, np.float32)
        if k == "pred_depth_map_logits":
            idx = np.sort(np.random.default_rng(seed).choice(g.size, DEPTH_MAP_SAMPLE, replace=False)).astype(np.int64)
            out[f"{name}.grad.{layer}.{k}.idx"], out[f"{name}.grad.{layer}.{k}.val"] = idx, g.reshape(-1)[idx]
            out[f"{name}.grad.{layer}.{k}.absmax"] = np.abs(g).max()
        else:
            out[f"{name}.grad.{layer}.{k}"] = g
    g = 11 if training else 1
    for l, od in enumerate([o] + o["aux_outputs"]):
        ind = matcher({k: v.detach() for k, v in od.items() if k != "aux_outputs"}, targets, group_num=g)
        for b, (i, j) in enumerate(ind):
            out[f"{name}.match.{l}.{b}.src"] = i.numpy()
            out[f"{name}.match.{l}.{b}.tgt"] = j.numpy()
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "criterion.npz"), **out)
print(len(out), "arrays;", {k: float(v) for k, v in out.items() if k.startswith("train_b3.loss.")})
