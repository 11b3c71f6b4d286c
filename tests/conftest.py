import gzip
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    with gzip.open(os.path.join(GOLDEN, name + ".json.gz"), "rt") as f:
        return json.load(f)


@pytest.fixture(scope="session")
def golden_models():
    return load_golden("models")


@pytest.fixture(scope="session")
def golden_ops():
    return load_golden("ops_1") + load_golden("ops_2")        # one list, stored in two halves of under 1 MB


@pytest.fixture(scope="session")
def golden_orders():
    return load_golden("orders")


@pytest.fixture(scope="session")
def golden_synth():
    return load_golden("synthetic")
