"""pytest configuration.

* ``-m "not gpu"``: oracle vs golden vectors, host logic, C-ABI load/export
  checks, world_size-2 gloo tests -- runs anywhere in a few minutes.
* ``-m gpu``: the parity tests proper; they call the CUDA path through the
  C ABI (ctypes) and compare with the oracle / golden fixtures.  They read
  nothing outside the repository.
"""
import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line(
        "markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle_cpu():
    from oracle import cpu
    cpu.lib()
    return cpu


def load_golden(name):
    """Arrays of fixture `name`: ``name.npz`` plus, for a fixture stored in
    parts to keep every file below 1 MB, ``name.part1.npz``, ... ."""
    paths = [os.path.join(GOLDEN, name + ".npz")] + sorted(
        glob.glob(os.path.join(GOLDEN, glob.escape(name) + ".part*.npz")))
    out = {}
    for path in paths:
        with np.load(path) as z:
            out.update({k: z[k] for k in z.files})
    return out


def canon_index(ranks_bev, ranks_depth, ranks_feat):
    """Canonical order of a point index: by voxel rank, then point id.  The
    reference's argsort leaves the order inside a voxel unspecified
    (view_transformer.py:590), so index tensors are compared in this form."""
    k = np.lexsort((ranks_depth, ranks_bev))
    return ranks_bev[k], ranks_depth[k], ranks_feat[k]
