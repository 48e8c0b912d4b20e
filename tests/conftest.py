import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')
    config.addinivalue_line('markers', 'needs_reference: needs the unmodified reference (see oracle/refharness.py)')


def pytest_collection_modifyitems(config, items):
    from oracle import refharness
    if refharness.available():
        return
    skip_ref = pytest.mark.skip(reason='the unmodified reference is neither at NW_REFERENCE_SRC nor staged under oracle/_ref/')
    for item in items:
        if 'needs_reference' in item.keywords:
            item.add_marker(skip_ref)


def make_case(n_points=4000, n_geo=6, radius=500.0, seed=3, dtype=np.float32, shape=None, scale=1.2):
    """Seeded (mesh, points, sigma) triple shared by oracle and GPU tests."""
    from ch_shrinkwrap_b200 import minimesh, synth
    shape = shape or synth.Sphere(radius)
    pts, sig = synth.smlm_cloud(shape, n_points, seed=seed, dtype=dtype)
    mesh = synth.star_mesh(shape, n_geo, scale=scale)
    return mesh, pts, sig


@pytest.fixture
def case_small():
    return make_case()
