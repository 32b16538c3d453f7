"""CPU: the AdamW restatement in oracle/optim.py against five steps of the UNMODIFIED reference class
(lib/helpers/optimizer_helper.py), stored by tools/gen_golden_reference_pins.py in tests/golden/reference_adamw.npz."""
import os

import numpy as np
import torch

from oracle.optim import adamw_reference_step


def test_adamw_port_matches_reference_class(golden_dir):
    g = np.load(os.path.join(golden_dir, "reference_adamw.npz"))
    names = [str(n) for n in g["names"]]
    lr, wd = float(g["lr"]), float(g["weight_decay"])
    mine = [torch.from_numpy(g[f"param.0.{i}"].copy()) for i in range(len(names))]
    ms = [torch.zeros_like(p) for p in mine]
    vs = [torch.zeros_like(p) for p in mine]
    wds = [0.0 if "bias" in n else wd for n in names]
    for step in range(1, 6):
        grads = [torch.from_numpy(g[f"grad.{step}.{i}"]) for i in range(len(names))]
        adamw_reference_step(mine, grads, ms, vs, step, lr, 0.9, 0.999, 1e-8, wds)
        for i, p in enumerate(mine):
            assert torch.equal(p, torch.from_numpy(g[f"param.{step}.{i}"])), (step, names[i])
