import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pytorch-nmf_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle import golden_inputs  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class Fixture(dict):
    """{"<case>/<field>": array} of one fixture file, keyed like np.load's result (`files` included)."""

    @property
    def files(self):
        return list(self)


def load_npz(fname):
    """A fixture written by oracle/make_golden.py, with the inputs it stores as seeded recipes regenerated and checked."""
    with np.load(os.path.join(GOLDEN, fname), allow_pickle=False) as z:
        return Fixture(golden_inputs.unpack({k: z[k] for k in z.files}))


def load_golden(fname="reference_small.npz"):
    """Return {case_name: {field: value}} from a fixture written by oracle/make_golden.py."""
    z = load_npz(fname)
    cases = {}
    for key in z.files:
        name, field = key.split("/", 1)
        v = z[key]
        if field in ("V", "W0", "H0", "W", "H"):
            v = torch.from_numpy(v.copy())
        elif field == "kind":
            v = str(v)
        elif field == "losses":
            v = [float(x) for x in v]
        else:
            v = float(v)
            if field in ("n_iter", "max_iter") or (field in ("trainable_W", "trainable_H")):
                v = int(v)
        cases.setdefault(name, {})[field] = v
    return cases


@pytest.fixture(scope="session")
def golden():
    return load_golden()


def has_cuda():
    return torch.cuda.is_available()
