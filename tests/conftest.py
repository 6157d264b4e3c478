import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _cuda_device_count():
    """Devices the CUDA driver reports (0 without a driver).  Deliberately not torch: the tests drive the C-ABI."""
    import ctypes
    try:
        cu = ctypes.CDLL("libcuda.so.1")
        n = ctypes.c_int(0)
        if cu.cuInit(0) != 0 or cu.cuDeviceGetCount(ctypes.byref(n)) != 0:
            return 0
        return n.value
    except OSError:
        return 0


def pytest_collection_modifyitems(config, items):
    # A plain `pytest tests` on a CPU-only box skips the gpu-marked tests instead of failing in speechPlayer_initialize.
    # With a device present nothing is skipped: a missing or broken library must fail loudly there.
    if _cuda_device_count() > 0:
        return
    skip = pytest.mark.skip(reason="no CUDA device (the engine has no CPU path)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement (oracle/klatt_oracle.c); built on demand (gcc only)."""
    from oracle import oracle
    if not oracle.have_port():
        oracle.build(quiet=True)
    return oracle.PortLib()


@pytest.fixture(scope="session")
def reflib():
    """The compiled reference with Philox noise: oracle/_ref, built from the NVSpeechPlayer checkout NVSP_REFERENCE_DIR names."""
    from oracle import oracle
    if not oracle.have_ref() and not oracle.build(quiet=True):
        pytest.skip("oracle/_ref not built and NVSP_REFERENCE_DIR names no NVSpeechPlayer checkout")
    return oracle.RefLib(philox=True)


@pytest.fixture(scope="session")
def golden_scenarios():
    return np.load(os.path.join(GOLDEN, "scenarios.npz"))


@pytest.fixture(scope="session")
def golden_config1():
    return np.load(os.path.join(GOLDEN, "config1.npz"))
