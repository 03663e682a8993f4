import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O
    O.lib()
    return O


def digest(arrays):
    """sha256 over the bytes of one array or of a tuple of arrays, in order."""
    h = hashlib.sha256()
    for a in arrays if isinstance(arrays, tuple) else (arrays,):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


class Reference:
    """What the reference's own code (oracle/_ref) returns.  Where oracle/_ref is built, check() runs it and also holds
    the recorded digest to it; elsewhere check() compares with the digest recorded in golden/reference_digests.json."""

    def __init__(self, oracle):
        self.live = oracle.ref_lib() is not None
        with open(os.path.join(GOLDEN, "reference_digests.json")) as f:
            self.digests = json.load(f)

    def check(self, key, got, ref_fn):
        """`got` (an array or a tuple of arrays) must be bit-identical to the reference's result `ref_fn()`."""
        d = digest(got)
        if self.live:
            assert d == digest(ref_fn()), key
            assert self.digests.get(key) == d, "reference_digests.json is stale for %s: the reference gives %s" % (key, d)
        else:
            assert d == self.digests[key], key


@pytest.fixture(scope="session")
def reference(oracle):
    return Reference(oracle)


@pytest.fixture(scope="session")
def views():
    return {v: np.load(os.path.join(GOLDEN, "views", v + ".npz"))["xyz"] for v in ("cheff000", "cheff001", "cheff002")}


@pytest.fixture(scope="session")
def golden():
    return {v: np.load(os.path.join(GOLDEN, "golden_%s.npz" % v)) for v in ("cheff000", "cheff001", "cheff002")}


def forest_path(name="synthetic-T100-D15"):
    return os.path.join(GOLDEN, "forests", name + ".yaml.gz")


@pytest.fixture(scope="session")
def main_forest(oracle):
    return oracle.load_forest_yaml(forest_path())


@pytest.fixture(scope="session")
def kpl():
    """The product library through its ctypes binding; building it is part of the fixture."""
    from keypoint_learning_b200 import build as B
    B.build_lib()
    import keypoint_learning_b200 as K
    K.load_library()
    return K
