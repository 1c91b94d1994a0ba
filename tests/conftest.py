import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def known():
    return dict(np.load(os.path.join(GOLDEN, "known_answers.npz"), allow_pickle=False))


@pytest.fixture(scope="session")
def refout():
    return dict(np.load(os.path.join(GOLDEN, "reference_outputs.npz"), allow_pickle=False))


@pytest.fixture(scope="session")
def refsig():
    with open(os.path.join(GOLDEN, "reference_signatures.json")) as f:
        return json.load(f)
