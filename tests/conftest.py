import math
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    import oracle as om
    om.build()
    return om.Oracle()


@pytest.fixture(scope="session")
def watref():
    import oracle as om
    om.build()
    if not om.WatRef.available():
        pytest.skip("oracle/_ref/libwatref.so not built (needs WATFFT_REFERENCE, a wat-fft checkout, at build time)")
    return om.WatRef()


@pytest.fixture(scope="session")
def reference():
    """The reference modules: transpiled (oracle/_ref/libwatref.so) when built, otherwise the outputs stored from them,
    which answer for the stored inputs only (backends.StoredWatRef)."""
    import oracle as om
    from backends import StoredWatRef
    om.build()
    return om.WatRef() if om.WatRef.available() else StoredWatRef()


@pytest.fixture(scope="session")
def wf():
    """The product package; fails loudly when the CUDA library is missing."""
    import watfft_b200
    watfft_b200._cabi.lib()
    return watfft_b200


def f32_bound(n):
    """north_star: max |err| / ||x||_2 <= 2e-6 * log2(N) for f32."""
    return 2e-6 * math.log2(n)


def f64_bound(n):
    """north_star: 1e-14 * log2(N) for f64."""
    return 1e-14 * math.log2(n)


def rel_err(a, b, x):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    nx = np.linalg.norm(np.asarray(x, np.float64).ravel())
    return float(np.max(np.abs(a - b)) / (nx if nx > 0 else 1.0))
