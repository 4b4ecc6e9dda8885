import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_SRC = os.environ.get("SIMPLEX_REF", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def ref_cases():
    with open(os.path.join(GOLDEN, "reference_cases.json")) as fh:
        return json.load(fh)["cases"]


@pytest.fixture(scope="session")
def cfg_digests():
    with open(os.path.join(GOLDEN, "cfg_digests.json")) as fh:
        return json.load(fh)


@pytest.fixture(scope="session")
def reference_module():
    """The original project's simplex.py, loaded from $SIMPLEX_REF (its src/ directory), or None when that is not set.
    Its sources are not part of this repository: the tests that take it compare with records in tests/golden/ and,
    given the module, with the original itself too."""
    if not REF_SRC:
        return None
    path = os.path.join(REF_SRC, "simplex.py")
    if not os.path.exists(path):
        raise FileNotFoundError(f"$SIMPLEX_REF is set but {path} does not exist")
    import importlib.util
    spec = importlib.util.spec_from_file_location("reference_simplex", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="session")
def dantzig_cases():
    """The extension entering rule (most negative, lowest index on ties), driven through the reference itself by
    tests/golden/make_golden.py dantzig."""
    with open(os.path.join(GOLDEN, "dantzig_cases.json")) as fh:
        return json.load(fh)["cases"]
