import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")
    config.addinivalue_line("markers", "slow: CPU test that takes more than a few seconds")
    config.addinivalue_line("markers", "gpu_next: CUDA cases written after the round's last GPU session; "
                                       "not part of -m gpu until they have run on a B200 once")


def golden(name):
    """The arrays of tests/golden/<name>.npz.  Where <name>_V.npz exists it holds the integrals
    V[p,q,r,s], packed by make_golden.py::pack_integrals, and they are rebuilt here exactly."""
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))
    packed = os.path.join(GOLDEN, name + "_V.npz")
    if os.path.exists(packed):
        g["V"] = _unpack_integrals(np.load(packed, allow_pickle=False))
    return g


def _unpack_integrals(packed):
    """V from its non-zeros with p <= r and q <= s, mirrored by V[p,q,r,s] = V[r,q,p,s] = V[p,s,r,q]."""
    n = int(packed["n"])
    keep = np.unpackbits(packed["mask"], count=n ** 4).astype(bool).reshape((n,) * 4)
    p, q, r, s = np.nonzero(keep)
    V = np.zeros((n,) * 4)
    for idx in ((p, q, r, s), (r, q, p, s), (p, s, r, q), (r, s, p, q)):
        V[idx] = packed["val"]
    return V


@pytest.fixture
def cpu_abi(monkeypatch):
    """Host tensors + numpy emulation of the C ABI (tests/abi_emulator.py): checks the
    host logic of pymes_b200 without a GPU.  Never active in -m gpu tests."""
    from tests import abi_emulator
    return abi_emulator.install(monkeypatch)


@pytest.fixture(autouse=True)
def _quiet_logs():
    from pymes_b200 import log
    log.set_quiet(True)
    yield
    log.set_quiet(False)
