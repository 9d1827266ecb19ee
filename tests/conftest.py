"""pytest configuration: the ``gpu`` marker, golden fixtures, and the shared device context."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "hotpath_golden.npz")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def golden():
    """Reference outputs from the fixture file plus the seeded inputs they were computed from, regenerated."""
    from golden.make_golden import golden_inputs, inputs_sha1

    z = np.load(GOLDEN)
    out = {k: z[k] for k in z.files}
    inputs = golden_inputs()
    if not np.array_equal(inputs_sha1(inputs), out.pop("inputs_sha1")):
        raise RuntimeError("the seeded golden inputs no longer regenerate bit for bit (NumPy random stream changed?)")
    out.update(inputs)
    return out


def golden_cases(prefix):
    """Names below ``prefix/`` in the fixture file (collected at import time for parametrisation)."""
    z = np.load(GOLDEN)
    names = sorted({k[len(prefix) + 1:].rsplit("/", 1)[0] for k in z.files if k.startswith(prefix + "/")})
    return names


@pytest.fixture(scope="session")
def ctx():
    """Process-wide device context.  Fails loudly when the CUDA library or the GPU is missing."""
    from linalg_b200 import default_context

    return default_context()
