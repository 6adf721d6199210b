import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")


def pytest_collection_modifyitems(config, items):
    has_gpu = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def fixture_sd():
    return torch.load(os.path.join(GOLDEN, "weights_fixture.pt"))


@pytest.fixture(scope="session")
def golden_dgcnn():
    return torch.load(os.path.join(GOLDEN, "golden_dgcnn.pt"))


@pytest.fixture(scope="session")
def golden_episodes():
    return torch.load(os.path.join(GOLDEN, "golden_episodes.pt"))
