import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "single-stable-dreamfusion_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_report_header(config):
    from oracle import ref_ext as r
    built = all(os.path.exists(os.path.join(r.REF_DIR, n + ".so")) for n in ("_gridencoder", "_raymarching", "_freqencoder"))
    return "ref_ext tests compare against: " + ("the reference's own CUDA extensions (oracle/_ref)" if built else
                                                "the C oracle stand-in (oracle/ref_standin.py; oracle/_ref is not built)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def ref_ext():
    """The reference's own CUDA extensions (oracle/_ref) when they were built, else the C oracle behind the same calls
    (oracle/ref_standin.py), which test_golden.py pins to stored outputs of those extensions."""
    from oracle import ref_ext as r
    from oracle import ref_standin
    return r.load() or ref_standin.load()
