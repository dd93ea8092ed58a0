import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

# The reference package (bayes_opt) drives the drop-in tests.  build() vendors it, unmodified, into the
# git-ignored oracle/_ref (oracle/vendor_ref.py), which stays with the built tree; the tests only read it.  The
# product package imports `bayes_opt` from sys.path like any user environment.
from oracle.vendor_ref import ref_dir  # noqa: E402

_REF = ref_dir()
if _REF and _REF not in sys.path:
    sys.path.insert(0, _REF)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


_NEEDS_REF = ("ExpectedImprovement", "UpperConfidenceBound", "ProbabilityOfImprovement", "ConstantLiar", "GPHedge",
              "ConstraintModel", "AcquisitionFunction", "bayes_opt", "TS(")


def _skip_without_reference(items):
    """The acquisition-seam classes ARE bayes_opt's classes: without the (vendored) reference package they cannot be
    imported.  Tests that touch them are skipped with a loud reason instead of erroring; the GP seam / C-ABI tests
    still run."""
    try:
        import bayes_opt  # noqa: F401

        return
    except ImportError:
        pass
    import inspect

    skip = pytest.mark.skip(reason="bayes_opt not importable: build() vendors it into oracle/_ref "
                                   "(oracle/vendor_ref.py) where the reference source tree is present")
    for item in items:
        try:
            src = inspect.getsource(item.function)
        except (OSError, TypeError, AttributeError):
            continue
        if any(tok in src for tok in _NEEDS_REF) or "ref" in getattr(item, "fixturenames", ()):
            item.add_marker(skip)


def pytest_collection_modifyitems(config, items):
    _skip_without_reference(items)
    try:
        import torch

        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        # a checkout without the built library (the .so is git-ignored): compile it once, loudly
        from bayesianoptimization_b200._build import LIB, build_library

        if not os.path.exists(LIB):
            build_library(force=True)
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))


@pytest.fixture(scope="session")
def golden():
    return load_golden


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference package."""
    try:
        import bayes_opt
    except ImportError:
        pytest.skip("reference package bayes_opt not importable (build() vendors it with oracle/vendor_ref.py)")
    return bayes_opt
