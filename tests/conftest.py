import hashlib
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


class GoldenArrays(dict):
    """Every access returns a fresh array, as np.load's NpzFile does: a test that writes into one cannot change what
    the next test reads."""

    def __getitem__(self, name):
        return dict.__getitem__(self, name).copy()


@pytest.fixture(scope="session")
def golden():
    """Stored arrays plus the seeded inputs, regenerated from their recipes and checked against their digests."""
    from signals import from_recipe
    with np.load(os.path.join(HERE, "golden", "golden_v1.npz")) as npz:
        arrays = GoldenArrays({name: npz[name] for name in npz.files})
    with open(os.path.join(HERE, "golden", "golden_v1.json")) as fh:
        meta = json.load(fh)
    for name, recipe in meta["inputs"].items():
        x = from_recipe(recipe)
        assert hashlib.sha256(x.tobytes()).hexdigest() == recipe["sha256"], f"{name}: tests/signals.py has drifted"
        arrays[name] = x
    return arrays, meta


@pytest.fixture(scope="session")
def oracle():
    from oracle_lib import Oracle
    return Oracle()


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    return a.tobytes() == b.tobytes()
