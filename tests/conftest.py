import os
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


class GoldenVectors(dict):
    """Name -> array, with the `files` list of an NpzFile."""
    @property
    def files(self):
        return list(self)


@pytest.fixture(scope="session")
def golden():
    """tests/golden/reference_vectors*.npz (tests/golden/make_golden.py), kept in parts of less than 1 MB"""
    out = GoldenVectors()
    for name in ("reference_vectors.npz", "reference_vectors_blob_lists.npz", "reference_vectors_live.npz"):
        with np.load(os.path.join(ROOT, "tests", "golden", name)) as part:
            out.update((k, part[k]) for k in part.files)
    return out


@pytest.fixture(scope="session")
def oracle():
    """The CPU restatement (oracle/visfd_oracle.cpp) -- the checker, never the product."""
    from oracle.pyoracle import Oracle
    return Oracle("port")


@pytest.fixture(scope="session")
def ref_oracle():
    """The unmodified reference (oracle/_ref), when it has been built and shipped."""
    from oracle.pyoracle import Oracle, have
    if not have("reference"):
        pytest.skip("oracle/_ref/libvisfd_ref.so not present")
    return Oracle("reference")


@pytest.fixture(scope="session")
def ctx():
    """A CUDA context on cuda:0; fails loudly (no fallback) if the library or GPU is missing."""
    import visfd_b200
    c = visfd_b200.Context(0)
    yield c
    c.close()
