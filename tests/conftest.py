import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Stated floating-point tolerance of the path (DESIGN.md "Parity"): a logit may differ from the
# CPU oracle by at most TOL_SIGMA x (std of that model's logits).  Measured noise floor between two
# legitimate builds of the SAME reference source is ~1.5e-3 sigma (SURVEY.md s.8c).
TOL_SIGMA = 5e-3
# KV-cache entries are fp16-rounded fp32 values: allow two half ulps of the entry magnitude + abs floor.
KV_RTOL = 2e-3
KV_ATOL = 2e-4


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle_pkg():
    """Builds (if needed) and returns the oracle package.  The tests compare with stored outputs of the reference
    (tests/golden/); its binaries in oracle/_ref/ exist only where build() found the reference sources."""
    import oracle

    oracle.build(ref=False)
    return oracle


def golden(name):
    import numpy as np

    return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
