"""Generate tests/golden/reference_msda_kernels.npz: the reference's own CUDA kernels (oracle/_ref/libref_msda.so, built by
`make -C oracle` where the reference is present) on the full-size inputs of tests/test_msda_gpu.py::
test_full_size_against_oracle_and_reference_kernels.  Per Lq and result: max|x| and a seeded sample of SAMPLE entries.

    python tools/gen_golden_msda_ref_kernels.py [OUT.npz]          (needs a CUDA device)
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref_gpu  # noqa: E402
from test_msda_gpu import FULL_SHAPES, full_size_case  # noqa: E402

SAMPLE = 1024


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "reference_msda_kernels.npz")
    assert ref_gpu.available(), "oracle/_ref/libref_msda.so not built"
    rng = np.random.default_rng(5)
    arrs = {}
    for Lq in (50, 550, 10200):
        dv = [t.cuda() for t in full_size_case(Lq)]
        res = (ref_gpu.forward(*dv[:5]),) + ref_gpu.backward(*dv)
        torch.cuda.synchronize()
        for name, t in zip(("out", "grad_value", "grad_loc", "grad_attn"), res):
            a = t.cpu().numpy().reshape(-1)
            idx = np.sort(rng.choice(a.size, SAMPLE, replace=False)).astype(np.int32)
            arrs[f"Lq{Lq}.{name}.idx"], arrs[f"Lq{Lq}.{name}.val"] = idx, a[idx]
            arrs[f"Lq{Lq}.{name}.absmax"] = np.abs(a).max()
    np.savez_compressed(out_path, levels=np.array(FULL_SHAPES), **arrs)
    print("wrote", out_path, len(arrs), "arrays")


if __name__ == "__main__":
    main()
