import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def orc():
    """The CPU oracle (test infrastructure only)."""
    from oracle import cpu
    cpu.build()
    return cpu


@pytest.fixture(scope="session")
def ref_root():
    """A MoCoPCI checkout to import the reference's own Python from (baseline/fetch_ref.py: the
    one MOCOPCI_REFERENCE names, or its copy under baseline/_ref). The repository does not carry
    the reference, so the tests that run its model, dataset class and module patching skip without
    one. The parity tests compare with restatements of the reference's torch helpers
    (oracle/torch_port.py), the C oracle and a stored kernel snapshot (tests/kernel_snapshot.py)."""
    from baseline import fetch_ref
    root = fetch_ref.root()
    if root is None:
        pytest.skip("no MoCoPCI checkout (set MOCOPCI_REFERENCE or run baseline/fetch_ref.py)")
    return root
