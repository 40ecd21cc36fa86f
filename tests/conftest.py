import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_cuda():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def manifest():
    with open(os.path.join(GOLDEN, "manifest.json")) as f:
        m = json.load(f)
    # round-2 additions (tests/golden/make_golden_r2.py): negative / edge vectors and four more fixtures
    with open(os.path.join(GOLDEN, "manifest_r2.json")) as f:
        r2 = json.load(f)
    m["png"] += r2["png"]
    m["gz"] += r2["gz"]
    m["fixtures"].update(r2["fixtures"])
    return m


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def ctx():
    """The product: libdebigulator_b200.so on cuda:0. No fallback."""
    import debigulator_b200 as d
    from debigulator_b200.build import build_library
    build_library()
    c = d.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def ref():
    """What the product is compared with: the unmodified reference (oracle/_ref/libref.so) where its sources are at
    hand, else the plain-C restatement (oracle/debig_oracle.c), which tests/test_oracle.py pins to the reference's
    own outputs, with stb-shaped PNG and zlib streams from the corpus's encoder (oracle/checker.py)."""
    from oracle import checker
    checker._impl().lib()
    return checker
