import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "voiceprintrecognition-paddlepaddle_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with `-m gpu` on the GPU box)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def ref_head():
    """tests/golden/ref_head.npz with every classifier gradient dW_<tag> rebuilt from the span coefficients dWspan_<tag>
    that tests/golden/make_ref_fixtures.py stores for it (dW = emb^T c[:-1] + W * c[-1])."""
    import numpy as np
    g = np.load(os.path.join(GOLDEN, "ref_head.npz"))
    d = {k: g[k] for k in g.files}
    for k in [k for k in d if k.startswith("dWspan_")]:
        c = d.pop(k)
        d["dW_" + k[len("dWspan_"):]] = d["emb"].T @ c[:-1] + d["W"][:, :c.shape[1]] * c[-1]
    return d


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device: the ppvector hot path has no CPU fallback")
    return torch.device("cuda:0")
