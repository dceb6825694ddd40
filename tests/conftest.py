import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _cuda_device_count():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


def pytest_collection_modifyitems(config, items):
    """Tests marked `gpu` need a device: on a CPU-only host they are skipped (the product itself has no CPU path and
    fails loudly there), so a plain `pytest tests` stays green without -m."""
    if _cuda_device_count() > 0:
        return
    skip = pytest.mark.skip(reason="no CUDA device: the classification path has no CPU fallback")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session", autouse=True)
def built():
    """Make sure the product library and the C oracle exist (compiles only when stale or missing)."""
    from pheniqs_b200.build import build
    build()
    from oracle import oracle
    if not os.path.exists(oracle.PORT_LIBRARY):
        oracle.build("port")
    reference = os.environ.get("PHENIQS_REFERENCE")         # the upstream Pheniqs sources, to build oracle/_ref from
    if not oracle.ref_available() and reference and os.path.exists(os.path.join(reference, "pamld.cpp")):
        subprocess.run(["make", "-s", "-C", oracle.HERE, "ref", "REFERENCE=" + reference], check=True)
    return True
