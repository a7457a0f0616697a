import os
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    """Plain `pytest tests` on a box without a CUDA device: the gpu-marked tests are skipped (they would all fail in
    kb200_create — backend='cuda' has no CPU fallback), so the host tests keep showing real regressions."""
    if not any("gpu" in it.keywords for it in items):
        return
    from pykrige_b200 import _cabi
    if _cabi.device_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device (backend='cuda' has no CPU fallback)")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def ref_goldens():
    return np.load(os.path.join(GOLDEN, "reference_goldens.npz"))


@pytest.fixture(scope="session")
def ref_cases():
    return np.load(os.path.join(GOLDEN, "ref_cases.npz"))


@pytest.fixture(scope="session")
def ref_pinv():
    """Reference outputs with pseudo_inv=True (make_golden.py pinv)."""
    return np.load(os.path.join(GOLDEN, "ref_pinv.npz"))


@pytest.fixture(scope="session")
def ref_custom():
    """Reference outputs for variogram_model='custom' callables (make_golden.py custom)."""
    return np.load(os.path.join(GOLDEN, "ref_custom.npz"))


@pytest.fixture(scope="session")
def ref_scenarios():
    """Reference outputs of the whole-chain scenarios (make_golden.py scenarios)."""
    return np.load(os.path.join(GOLDEN, "ref_scenarios.npz"))


@pytest.fixture(scope="session")
def ref_ctor():
    """Reference outputs of core._initialize_variogram_model / core._find_statistics (make_golden.py ctor)."""
    return np.load(os.path.join(GOLDEN, "ref_ctor.npz"))


@pytest.fixture(scope="session")
def ref_native():
    """Outputs of the reference's compiled cok.pyx twins on cases.NATIVE_INPUTS (make_golden_native.py)."""
    return np.load(os.path.join(GOLDEN, "ref_native.npz"))


def assert_parity(out, ref, R, what=""):
    """SURVEY.md §8(d): allclose(out, ref, rtol=R, atol=R*max|ref|)."""
    out = np.asarray(np.ma.getdata(out), dtype=np.float64)
    ref = np.asarray(np.ma.getdata(ref), dtype=np.float64)
    assert out.shape == ref.shape, (what, out.shape, ref.shape)
    atol = R * float(np.max(np.abs(ref))) if ref.size else 0.0
    bad = ~np.isclose(out, ref, rtol=R, atol=atol)
    if bad.any():
        i = np.argmax(np.abs(out - ref))
        raise AssertionError("%s: %d/%d outside rtol=%g atol=%g; worst |d|=%g at %d (out=%r ref=%r)" % (
            what, int(bad.sum()), out.size, R, atol, float(np.abs(out - ref).flat[i]), i,
            float(out.flat[i]), float(ref.flat[i])))
