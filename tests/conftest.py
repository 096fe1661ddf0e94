import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _cuda_usable():
    """A CUDA device and the engine library: without them `gpu`-marked tests are skipped, not failed."""
    try:
        import torch
        if not torch.cuda.is_available():
            return False
    except Exception:
        return False
    return os.path.exists(os.path.join(ROOT, "mcl_3dl_b200", "libmcl3dl_b200.so"))


def pytest_collection_modifyitems(config, items):
    if any(it.get_closest_marker("gpu") for it in items) and not _cuda_usable():
        skip = pytest.mark.skip(reason="needs a CUDA device (run on the B200 box with -m gpu)")
        for it in items:
            if it.get_closest_marker("gpu"):
                it.add_marker(skip)


@pytest.fixture(scope="session")
def port():
    """The repo-owned CPU restatement (oracle/libmcl3dl_oracle.so), built on demand."""
    from oracle import cpu_checker as cc
    cc.build("port")
    return cc.CpuChecker("port")


@pytest.fixture(scope="session")
def reference():
    """The original project's own CPU models, as answers recorded from its build (tests/recorded_reference.py).
    MCL3DL_RECORD_REFERENCE=1 records them afresh from the live build in oracle/_ref (tests/golden/make_golden.py)."""
    from recorded_reference import recording, replaying
    if not os.environ.get("MCL3DL_RECORD_REFERENCE"):
        yield replaying()
        return
    from oracle import cpu_checker as cc
    ref, store = recording(cc.CpuChecker("reference"))
    yield ref
    store.save()


def golden(name):
    import numpy as np
    return np.load(os.path.join(GOLDEN, name))
