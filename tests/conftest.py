import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with `-m gpu` under gpurun)")


@pytest.fixture(scope="session", autouse=True)
def _no_grad():
    torch.set_grad_enabled(False)
    yield


@pytest.fixture(scope="session", autouse=True)
def _golden_threads():
    """The thread count tests/golden/ was generated with, whatever the host's core count: the CPU oracle then
    reproduces the goldens' bits (oracle.GOLDEN_THREADS)."""
    from oracle import GOLDEN_THREADS
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="session")
def prop_sd():
    from oracle import weights
    return weights.make_prop_state_dict(1234)


@pytest.fixture(scope="session")
def fuse_sd():
    from oracle import weights
    return weights.make_fusion_state_dict(4321)


@pytest.fixture(scope="session")
def golden():
    def load(name):
        return np.load(os.path.join(GOLDEN, name))
    return load


@pytest.fixture(scope="session")
def dev():
    assert torch.cuda.is_available(), "gpu tests need CUDA"
    return torch.device("cuda:0")


@pytest.fixture(scope="session", params=["tf32", "fp16"])
def nets(request, prop_sd, fuse_sd, dev):
    """mivos_b200 networks loaded with the seeded oracle weights (top_k 20 and 50) + FusionNet, once
    per activation type: every network-level parity test runs on the TF32 path and on the fp16 path."""
    import mivos_b200
    import torch
    out = {"act": request.param}
    for k in (20, 50):
        n = mivos_b200.PropagationNetwork(top_k=k, act_dtype=torch.float16 if request.param == "fp16" else torch.float32)
        n.load_state_dict(prop_sd, strict=True)
        out[k] = n.to(dev)
    f = mivos_b200.FusionNet()
    f.load_state_dict(fuse_sd, strict=True)
    out["fuse"] = f.to(dev)
    return out
