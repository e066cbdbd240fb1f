"""pytest configuration: the `gpu` marker, import path and shared fixtures."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
if GOLDEN_DIR not in sys.path:
    sys.path.insert(0, GOLDEN_DIR)
from golden_weights import load, state_digest  # noqa: E402,F401  (tests/golden/)

GOLDEN_NAMES = ["simplevit_tiny", "vit_tiny_cls", "vit_tiny_mean_nonsquare", "vit_tiny_tokens"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    return load(os.path.join(GOLDEN_DIR, name + ".pt"))


@pytest.fixture(params=GOLDEN_NAMES)
def golden(request):
    return load_golden(request.param)


def reference_init(name: str, cls):
    """`cls` built under the seed and keywords of reference_surface.pt's `init[name]`, after checking that it draws
    bit-identical parameters to the reference's constructor (key order, shapes, values)."""
    spec = load_golden("reference_surface")["init"][name]
    torch.manual_seed(spec["seed"])
    m = cls(**spec["kwargs"])
    assert list(state_digest(m.state_dict()).items()) == list(spec["digest"].items()), name
    return m
