import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Before any test touches torch: the CPU oracle is held to reference-made fixtures bit for bit, which holds only
# under the host-independent CPU arithmetic the fixtures were written with (oracle/numerics.py).
from oracle import numerics  # noqa: E402

numerics.pin()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")
