import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
CONV_FIXTURES = ["c1_norte", "c1_rte", "rand_t3r4_dk4", "rand_dk25", "mag_mini_dk50", "oag_mini", "hub_h2"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def load_golden(name):
    import torch
    return torch.load(os.path.join(GOLDEN_DIR, name + ".pt"), map_location="cpu", weights_only=False)


def load_record():
    """tests/golden/reference_record.json: parameter inventories of the reference and digests of its larger outputs."""
    import json
    with open(os.path.join(GOLDEN_DIR, "reference_record.json")) as f:
        return json.load(f)


@pytest.fixture(params=CONV_FIXTURES)
def conv_fixture(request):
    fx = load_golden(request.param)
    fx["name"] = request.param
    return fx
