import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    items.sort(key=_rank)                                   # stable: keeps the in-file order


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(autouse=True)
def _seed_global_generators():
    """Every test starts from the same global torch / numpy generator state (CPU and, when present, CUDA), so a draw that
    does not pass its own `generator=` is still reproducible run to run and independent of which tests ran before it."""
    import numpy as np
    import torch
    torch.manual_seed(20250924)
    np.random.seed(20250924)
    yield


# Run order for `pytest -x`: the parity suites of the path's own operators first (MSDA, tensor-core conv/linear, whole
# model), host/oracle checks next, everything else after -- so that one late failure cannot hide the main parity evidence.
_ORDER = ["test_msda_gpu", "test_msda_reference_generators_gpu", "test_conv_gemm_gpu", "test_elementwise_gpu",
          "test_attn_norm_gpu", "test_heads_gpu", "test_optim_gpu", "test_decode_gpu", "test_preprocess_gpu", "test_criterion_gpu", "test_model_gpu", "test_model_grad_gpu"]


def _rank(item):
    name = os.path.splitext(os.path.basename(str(item.fspath)))[0]
    return _ORDER.index(name) if name in _ORDER else len(_ORDER)
