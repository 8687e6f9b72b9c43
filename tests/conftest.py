import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from oracle.ref_loader import reference_path  # noqa: E402

GOLDEN = os.path.join(REPO, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_meta():
    import json
    with open(os.path.join(GOLDEN, "golden_meta.json")) as f:
        return json.load(f)


NO_REFERENCE = "needs the original project's sources: $VQA_REFERENCE or oracle/_ref/reference.zip"


def have_reference():
    return reference_path() is not None


@pytest.fixture(scope="session")
def reference_modules(tmp_path_factory):
    """Import the original project from where oracle/ref_loader.py finds it (a source directory or the archive
    tools/stage_reference.sh stages); skipped where neither is present."""
    path = reference_path()
    if path is None:
        pytest.skip(NO_REFERENCE)
    os.chdir(tmp_path_factory.mktemp("refcwd"))  # utils.config mkdirs relative to CWD (SURVEY T9)
    if path not in sys.path:
        sys.path.insert(0, path)
    import importlib
    return importlib
