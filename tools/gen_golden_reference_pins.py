"""Generate the fixtures that pin the oracle and the model's host contract to the UNMODIFIED reference (CPU), so that the
tests which compare with it run anywhere:

  tests/golden/reference_model_spec.json  state_dict keys (in order) and shapes, trainable parameter names, the `model`
                                          section of configs/monodetr.yaml and the criterion build_monodetr() assembles
  tests/golden/reference_model_forward.npz  forward outputs, eval and train mode, deterministic weights (base_seed 1),
                                          1x3x192x640 input; the depth-map logits as a seeded sample of SAMPLE entries
  tests/golden/reference_model_grads.npz  parameter gradients of the surrogate loss, train mode, deterministic weights,
                                          1x3x96x320 input: per parameter max|grad| and GRAD_SAMPLE entries (incl. the argmax)
  tests/golden/reference_adamw.npz        five steps of the reference AdamW class (lib/helpers/optimizer_helper.py)

    python tools/gen_golden_reference_pins.py        (needs the reference, see tools/ref_shims.py)
"""
import json
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
warnings.filterwarnings("ignore")
import ref_shims  # noqa: E402
from oracle import monodetr_torch as om  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
OUT_KEYS = ("pred_logits", "pred_boxes", "pred_3d_dim", "pred_depth", "pred_angle", "pred_depth_map_logits")
SAMPLE = 2048
GRAD_SAMPLE = 32


def _reference_model(pkg, cfg, dropout):
    cfg = dict(cfg, dropout=dropout)
    torch.manual_seed(0)
    model, crit = pkg.build_monodetr(cfg)
    if dropout == 0.0:   # the depth encoder hard-codes dropout=0.1 (depth_predictor.py:49-50): neutralise in memory
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):
                m.p = 0.0
            if isinstance(m, torch.nn.MultiheadAttention):
                m.dropout = 0.0
    return model, crit


def spec(pkg, cfg):
    model, crit = _reference_model(pkg, cfg, cfg["dropout"])
    d = {"state_dict": [[k, list(v.shape)] for k, v in model.state_dict().items()],
         "trainable": [n for n, p in model.named_parameters() if p.requires_grad],
         "model_cfg": cfg,
         "criterion": {"weight_dict": crit.weight_dict, "losses": crit.losses, "focal_alpha": crit.focal_alpha,
                       "num_classes": crit.num_classes}}
    with open(os.path.join(OUT, "reference_model_spec.json"), "w") as f:     # one list entry per line
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: [\n" + ",\n".join(json.dumps(e) for e in v) + "\n]" if isinstance(v, list)
                                   else f"{json.dumps(k)}: {json.dumps(v)}" for k, v in d.items()) + "\n}\n")


def forward(pkg, cfg):
    model, _ = _reference_model(pkg, cfg, 0.0)
    model.load_state_dict(om.with_aliases(om.deterministic_state_dict(base_seed=1)))
    images, calibs, sizes = om.synthetic_inputs(1, 0, H=192, W=640)
    arrs = {"B": 1, "H": 192, "W": 640, "seed": 0, "base_seed": 1}
    for mode, training in (("eval", False), ("train", True)):
        model.train(training)
        with torch.no_grad():
            out = model(images, calibs, None, sizes)
        for k in OUT_KEYS:
            a = out[k].numpy()
            if k == "pred_depth_map_logits":
                idx = np.sort(np.random.default_rng(7).choice(a.size, SAMPLE, replace=False)).astype(np.int64)
                arrs[f"{mode}.{k}.idx"], arrs[f"{mode}.{k}.val"] = idx, a.reshape(-1)[idx]
                arrs[f"{mode}.{k}.absmax"] = np.abs(a).max()
            else:
                arrs[f"{mode}.{k}"] = a
        for i, aux in enumerate(out["aux_outputs"]):
            for k, v in aux.items():
                arrs[f"{mode}.aux{i}.{k}"] = v.numpy()
    np.savez_compressed(os.path.join(OUT, "reference_model_forward.npz"), **arrs)


def grads(pkg, cfg):
    model, _ = _reference_model(pkg, cfg, 0.0)
    sd0 = om.deterministic_state_dict()
    model.load_state_dict(om.with_aliases(sd0))
    model.train(True)
    images, calibs, sizes = om.synthetic_inputs(1, 0, H=96, W=320)
    om.surrogate_loss(model(images, calibs, None, sizes)).backward()
    names, scale, idx, val = [], [], [], []
    rng = np.random.default_rng(11)
    for name, p in model.named_parameters():
        if p.grad is None or name not in sd0:
            continue
        g = p.grad.numpy().reshape(-1)
        pick = {int(np.abs(g).argmax())}
        if g.size > 1:
            pick.update(int(i) for i in rng.choice(g.size, min(GRAD_SAMPLE, g.size) - 1, replace=False))
        pick = np.array(sorted(pick), np.int64)
        names.append(name)
        scale.append(np.abs(g).max())
        idx.append(pick)
        val.append(g[pick])
    np.savez_compressed(os.path.join(OUT, "reference_model_grads.npz"), names=np.array(names), scale=np.array(scale, np.float32),
                        offsets=np.cumsum([0] + [len(i) for i in idx]), idx=np.concatenate(idx), val=np.concatenate(val),
                        B=1, H=96, W=320, seed=0)


def adamw():
    if ref_shims.REF_ROOT not in sys.path:
        sys.path.insert(0, ref_shims.REF_ROOT)
    from lib.helpers.optimizer_helper import build_optimizer
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.LayerNorm(5), torch.nn.Linear(5, 3))
    opt = build_optimizer({"type": "adamw", "lr": 2e-4, "weight_decay": 1e-4}, model)
    arrs = {"names": np.array([n for n, _ in model.named_parameters()]), "lr": 2e-4, "weight_decay": 1e-4}
    for i, p in enumerate(model.parameters()):
        arrs[f"param.0.{i}"] = p.detach().numpy().copy()
    for step in range(1, 6):
        for i, p in enumerate(model.parameters()):
            p.grad = torch.randn_like(p)
            arrs[f"grad.{step}.{i}"] = p.grad.numpy().copy()
        opt.step()
        for i, p in enumerate(model.parameters()):
            arrs[f"param.{step}.{i}"] = p.detach().numpy().copy()
    np.savez_compressed(os.path.join(OUT, "reference_adamw.npz"), **arrs)


def main():
    pkg = ref_shims.install()
    cfg = ref_shims.load_cfg()["model"]
    spec(pkg, cfg)
    forward(pkg, cfg)
    grads(pkg, cfg)
    adamw()


if __name__ == "__main__":
    main()
