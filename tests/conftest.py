"""pytest configuration: registers the `gpu` marker and builds the checkers once per session."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.oracle import Oracle, build

    build()
    return Oracle()


@pytest.fixture(scope="session")
def reference():
    """The compiled reference; only where oracle/_ref has been built (the build container, or a GPU box
    that received the prebuilt .so)."""
    from oracle.oracle import REF_SO, Reference, build

    build()
    if not os.path.exists(REF_SO):
        pytest.skip("oracle/_ref not built (no /root/reference here)")
    return Reference()


@pytest.fixture(scope="session")
def ref_vectors():
    return json.load(open(os.path.join(GOLDEN, "ref_vectors.json")))


@pytest.fixture(scope="session")
def ref_vectors_r02():
    return json.load(open(os.path.join(GOLDEN, "ref_vectors_r02.json")))


@pytest.fixture(scope="session")
def archive_stdout():
    return json.load(open(os.path.join(GOLDEN, "archive_stdout.json")))


@pytest.fixture(scope="session")
def sha_examples():
    return json.load(open(os.path.join(GOLDEN, "sha_examples.json")))


@pytest.fixture(scope="session")
def reference_archive():
    return json.load(open(os.path.join(GOLDEN, "reference_archive.json")))
