import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session", autouse=True)
def built_extension():
    """The CUDA library is a build artefact (git-ignored): make sure it exists and is not older
    than its sources before any test imports it.  Building is not a fallback -- if nvcc is missing
    this raises and the tests fail loudly."""
    from quantized_distillation_b200 import build as qd_build
    if qd_build.is_stale():
        qd_build.build()
    try:                                            # optional compiled front door: never a reason to fail the suite
        if qd_build.fast_is_stale():
            qd_build.build_fast()
    except Exception:
        pass
    return qd_build.OUT


@pytest.fixture(scope="session")
def golden():
    import golden_store
    path = os.path.join(ROOT, "tests", "golden", "reference_vectors.npz")
    data = golden_store.load(path)
    cases = {}
    for row in data["meta"]:
        family, key, kind, n, b, s = str(row).split("|")
        cases.setdefault(family, []).append(dict(key=key, kind=kind, n=int(n), bucket=None if int(b) < 0 else int(b), s=int(s)))
    return data, cases


@pytest.fixture(scope="session")
def golden_options():
    """Reference outputs for the options only the NMT loop passes (subtract_mean, max_element, stochastic
    rounding with the reference's own draws): tests/golden/make_golden_options.py."""
    import golden_store
    path = os.path.join(ROOT, "tests", "golden", "reference_vectors_options.npz")
    data = golden_store.load(path)
    cases = {}
    for row in data["meta"]:
        family, key, kind, n, b, s, sub, mx = str(row).split("|")
        cases.setdefault(family, []).append(dict(key=key, kind=kind, n=int(n), bucket=None if int(b) < 0 else int(b), s=int(s),
                                                 subtract_mean=bool(int(sub)), max_element=False if mx == "no" else float(mx)))
    return data, cases
