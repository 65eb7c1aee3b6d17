import gzip
import json
import lzma
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
if os.path.join(ROOT, "tests") not in sys.path:
    sys.path.insert(0, os.path.join(ROOT, "tests"))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    """gpu-marked tests are skipped (not failed) on a host without a CUDA device; the product itself raises there."""
    gpu_items = [it for it in items if it.get_closest_marker("gpu")]
    if not gpu_items:
        return
    try:
        import torch
        have = torch.cuda.is_available()
    except Exception:
        have = False
    if not have:
        skip = pytest.mark.skip(reason="no CUDA device on this host")
        for it in gpu_items:
            it.add_marker(skip)


def load_golden(name):
    with gzip.open(os.path.join(GOLDEN, name), "rt") as f:
        g = json.load(f)
    if "tape_file" in g:
        # a long RNG tape is kept beside the fixture as xz-compressed little-endian float64: as JSON text it would make the
        # fixture larger than 1 MB
        with lzma.open(os.path.join(GOLDEN, g.pop("tape_file"))) as f:
            g["tape"] = np.frombuffer(f.read(), dtype="<f8").tolist()
    return g


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = load_golden(name)
        return cache[name]

    return get


@pytest.fixture(scope="session", autouse=True)
def _built_library(request):
    """GPU tests call through the C-ABI: (re)build libbsr_b200.so when it is missing or older than its sources."""
    if any(item.get_closest_marker("gpu") and not any(m.name == "skip" for m in item.iter_markers()) for item in request.session.items):
        import __graft_entry__ as g
        g.build()
    yield
