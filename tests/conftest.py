import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "vrp-gym_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (sm_100) GPU; run with `-m gpu` on the GPU box")


def pytest_collection_modifyitems(config, items):
    import torch

    have_gpu = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device in this container"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
