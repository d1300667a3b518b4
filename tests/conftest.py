import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device")


def pytest_collection_modifyitems(config, items):
    """`gpu`-marked tests are skipped (not errored) on a box without a CUDA device, so a plain `pytest tests` is green
    on the CPU as well."""
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_rotated():
    from gpu_helpers import load_fixture
    return load_fixture("rotated_g24.pt")


@pytest.fixture(scope="session")
def golden_general():
    from gpu_helpers import load_fixture
    return load_fixture("general_g20.pt")


@pytest.fixture(scope="session")
def golden_init():
    from gpu_helpers import load_fixture
    return load_fixture("init_g24.pt")
