import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "stanford-ctc_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_ctc():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "ctc_cases.npz"))


@pytest.fixture(scope="session")
def golden_brnn():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "brnn_cases.npz"))


@pytest.fixture(scope="session")
def golden_rnnetcpu():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "rnnetcpu_ref.npz"))


@pytest.fixture(scope="session")
def golden_bf():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "blankforce_cases.npz"))


@pytest.fixture(scope="session")
def golden_rnn():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "rnn_cases.npz"))


@pytest.fixture(scope="session")
def golden_ref():
    import numpy as np
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "ctc_reference_exact.npz")))


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible (there is no CPU fallback)")
    torch.cuda.set_device(0)
    return torch
