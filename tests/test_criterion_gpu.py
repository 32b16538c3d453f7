"""Device criterion (csrc/criterion.cu through monodetr_b200.criterion) against the autograd oracle (oracle/criterion.py, CPU,
scipy assignment) and the golden vectors of the unmodified reference HungarianMatcher + SetCriterion."""
import os

import numpy as np
import pytest
import torch

from oracle import criterion as oc
from test_oracle_criterion import assert_grad_matches_golden

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "criterion.npz"))
CFG = {"num_classes": 3, "cls_loss_coef": 2, "focal_alpha": 0.25, "bbox_loss_coef": 5, "giou_loss_coef": 2, "3dcenter_loss_coef": 10,
       "dim_loss_coef": 1, "angle_loss_coef": 1, "depth_loss_coef": 1, "depth_map_loss_coef": 1, "set_cost_class": 2, "set_cost_bbox": 5,
       "set_cost_giou": 2, "set_cost_3dcenter": 10, "aux_loss": True, "dec_layers": 3}


def _to_cuda(out, padded, nhwc_depth=False):
    def mv(d):
        return {k: (v.cuda().requires_grad_(True) if torch.is_tensor(v) else v) for k, v in d.items() if k != "aux_outputs"}
    o = mv(out)
    if nhwc_depth:                   # the model hands over a permuted view of NHWC storage (monodetr.py:147)
        base = out["pred_depth_map_logits"].permute(0, 2, 3, 1).contiguous().cuda().requires_grad_(True)
        o["pred_depth_map_logits"] = base.permute(0, 3, 1, 2)
        o["_depth_base"] = base
    o["aux_outputs"] = [mv(a) for a in out["aux_outputs"]]
    return o, {k: v.cuda() for k, v in padded.items()}


def _run(out, padded, training, nhwc_depth=False, as_list=False):
    from monodetr_b200.criterion import build_criterion
    crit = build_criterion(CFG).cuda().train(training)
    o, p = _to_cuda(out, padded, nhwc_depth)
    targets = oc.prepare_targets(p) if as_list else p
    losses = crit(o, targets)
    total = sum(losses[k] * crit.weight_dict[k] for k in losses if k in crit.weight_dict)
    total.backward()
    torch.cuda.synchronize()
    return crit, o, losses, total


def _matches(crit, padded):
    """(L, B, group, Gmax) device result -> per layer / image (query indices, target indices) in the reference's order."""
    m = crit.last_indices.cpu().numpy()
    mask = padded["mask_2d"].numpy().astype(bool)
    res = []
    for l in range(m.shape[0]):
        per = []
        for b in range(m.shape[1]):
            n = int(mask[b].sum())
            src, tgt = [], []
            for g in range(m.shape[2]):
                pairs = sorted((int(m[l, b, g, j]), j) for j in range(n) if m[l, b, g, j] >= 0)     # scipy returns rows sorted
                src += [q for q, _ in pairs]
                tgt += [j for _, j in pairs]
            per.append((np.array(src, np.int64), np.array(tgt, np.int64)))
        res.append(per)
    return res


@pytest.mark.parametrize("name", ["train_b3", "eval_b2"])
def test_against_reference_golden(name):
    seed, B, Q, training = (int(v) for v in GOLD[f"{name}.cfg"])
    out, padded = oc.synthetic_case(seed, B, Q)
    crit, o, losses, total = _run(out, padded, bool(training))
    keys = [k[len(name) + 6:] for k in GOLD.files if k.startswith(f"{name}.loss.")]
    assert sorted(keys) == sorted(losses)
    for l, per in enumerate(_matches(crit, padded)):
        for b, (src, tgt) in enumerate(per):
            assert np.array_equal(src, GOLD[f"{name}.match.{l}.{b}.src"]) and np.array_equal(tgt, GOLD[f"{name}.match.{l}.{b}.tgt"]), (l, b)
    for k in keys:
        np.testing.assert_allclose(float(losses[k]), float(GOLD[f"{name}.loss.{k}"]), rtol=2e-5, atol=1e-6, err_msg=k)
    np.testing.assert_allclose(float(total), float(GOLD[f"{name}.total"]), rtol=2e-5)
    for layer, d in [("main", o)] + [(f"aux{i}", a) for i, a in enumerate(o["aux_outputs"])]:
        for k, t in d.items():
            if not torch.is_tensor(t) or k.startswith("_"):
                continue
            got = t.grad.cpu().numpy() if t.grad is not None else np.zeros(tuple(t.shape), np.float32)
            assert_grad_matches_golden(got, f"{name}.grad.{layer}.{k}", rtol=2e-4, atol_rel=2e-5)


@pytest.mark.parametrize("seed,B,Q,training,kw", [(31, 8, 550, True, {}), (32, 5, 50, False, {}), (33, 2, 550, True, {"max_gt": 50}),
                                                   (34, 3, 64, False, {"max_gt": 1, "n_aux": 0}), (35, 1, 550, True, {"n_aux": 1}),
                                                   (36, 2, 55, True, {})])      # 36: 5 queries per group < objects (transposed problem)
def test_against_oracle(seed, B, Q, training, kw):
    out, padded = oc.synthetic_case(seed, B, Q, **kw)
    crit, o, losses, total = _run(out, padded, training, nhwc_depth=True, as_list=(seed % 2 == 0))
    ref_out = {k: (v.clone().requires_grad_(True) if torch.is_tensor(v) else v) for k, v in out.items() if k != "aux_outputs"}
    ref_out["aux_outputs"] = [{k: v.clone().requires_grad_(True) for k, v in a.items()} for a in out["aux_outputs"]]
    ref_losses, ref_idx = oc.set_criterion(ref_out, padded, training=training)
    w = oc.weight_dict()
    ref_total = sum(ref_losses[k] * w[k] for k in ref_losses if k in w)
    ref_total.backward()
    assert sorted(losses) == sorted(ref_losses)
    padded_for_match = padded
    if seed % 2 == 0:        # list-of-dicts input: the valid targets were compacted to a prefix before packing
        n = padded["mask_2d"].sum(1)
        padded_for_match = {"mask_2d": torch.arange(padded["mask_2d"].shape[1])[None] < n[:, None]}
        padded_for_match["mask_2d"] = padded_for_match["mask_2d"][:, :max(int(n.max()), 1)]
    for l, per in enumerate(_matches(crit, padded_for_match)):
        for b, (src, tgt) in enumerate(per):
            assert np.array_equal(src, ref_idx[l][b][0].numpy()) and np.array_equal(tgt, ref_idx[l][b][1].numpy()), (l, b)
    for k in ref_losses:
        np.testing.assert_allclose(float(losses[k]), float(ref_losses[k]), rtol=2e-5, atol=1e-6, err_msg=k)
    pairs = [(o, ref_out)] + list(zip(o["aux_outputs"], ref_out["aux_outputs"]))
    for li, (d, r) in enumerate(pairs):
        for k, t in r.items():
            if not torch.is_tensor(t):
                continue
            g = t.grad.numpy() if t.grad is not None else np.zeros(tuple(t.shape), np.float32)
            src = d["_depth_base"].grad.permute(0, 3, 1, 2) if k == "pred_depth_map_logits" else d[k].grad
            got = src.cpu().numpy() if src is not None else np.zeros_like(g)
            np.testing.assert_allclose(got, g, rtol=2e-4, atol=1e-9 + 2e-5 * np.abs(g).max(), err_msg=f"layer {li} {k}")


def test_determinism_no_targets_and_errors():
    from monodetr_b200.criterion import HungarianMatcher, build_criterion
    out, padded = oc.synthetic_case(41, 2, 550)
    a = _run(out, padded, True)[2]
    b = _run(out, padded, True)[2]
    for k in a:
        assert torch.equal(a[k], b[k]), k                                   # fixed-order reductions: bit-identical
    padded["mask_2d"][:] = False                                            # a batch without objects (monodetr.py:508 clamps num_boxes to 1)
    crit, o, losses, total = _run(out, padded, True)
    assert float(losses["loss_bbox"]) == 0.0 and float(losses["class_error"]) == 100.0 and torch.isfinite(total)
    assert float(o["pred_boxes"].grad.abs().max()) == 0.0 and float(o["pred_logits"].grad.abs().max()) > 0.0
    crit = build_criterion(CFG).cuda()
    with pytest.raises(RuntimeError):
        crit({k: v for k, v in out.items() if k != "aux_outputs"}, padded)      # CPU tensors
    big, pb = oc.synthetic_case(43, 1, 100, n_aux=0)
    with pytest.raises(RuntimeError):                                            # 100 queries in one group: beyond the matcher's 64
        crit.eval()(_to_cuda(big, pb)[0], {k: v.cuda() for k, v in pb.items()})
    out2, padded2 = oc.synthetic_case(42, 2, 50)
    o, p = _to_cuda(out2, padded2)
    m = HungarianMatcher(2, 10, 5, 2).cuda()
    ind = m(o, p, group_num=1)
    ref = oc.hungarian_match({k: v for k, v in out2.items() if k != "aux_outputs"}, oc.prepare_targets(padded2), 1)
    for (i, j), (ri, rj) in zip(ind, ref):
        order = np.argsort(i.cpu().numpy())
        assert np.array_equal(i.cpu().numpy()[order], ri.numpy()) and np.array_equal(j.cpu().numpy()[order], rj.numpy())


def test_model_outputs_through_the_criterion():
    """MonoDETR.forward (train mode) -> device criterion -> backward into the model: finite losses and parameter gradients."""
    from monodetr_b200 import build_monodetr
    from monodetr_b200.monodetr import DEFAULT_MODEL_CFG
    from oracle import monodetr_torch as om
    torch.manual_seed(0)
    cfg = dict(DEFAULT_MODEL_CFG, **CFG, criterion="device", device="cuda")
    model, crit = build_monodetr(cfg)
    model, crit = model.cuda().train(), crit.cuda().train()
    images, calibs, sizes = om.synthetic_inputs(2, 3, H=384, W=1280)
    _, padded = oc.synthetic_case(51, 2, 550)
    out = model(images.cuda(), calibs.cuda(), None, sizes.cuda())
    losses = crit(out, {k: v.cuda() for k, v in padded.items()})
    total = sum(losses[k] * crit.weight_dict[k] for k in losses if k in crit.weight_dict)
    total.backward()
    torch.cuda.synchronize()
    assert torch.isfinite(total) and len(losses) == 26
    n = sum(1 for p in model.parameters() if p.grad is not None and torch.isfinite(p.grad).all() and float(p.grad.abs().max()) > 0)
    assert n > 300
    ref_losses, _ = oc.set_criterion({k: (v.detach().float().cpu() if torch.is_tensor(v) else
                                          [{kk: vv.detach().float().cpu() for kk, vv in a.items()} for a in v]) for k, v in out.items()},
                                     padded, training=True)
    for k in ref_losses:
        np.testing.assert_allclose(float(losses[k]), float(ref_losses[k]), rtol=5e-5, atol=1e-6, err_msg=k)
