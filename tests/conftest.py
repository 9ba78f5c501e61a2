import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name + '.npz')) as z:
        g = {k: z[k] for k in z.files}
    if 'w_linspace' in g:
        # the axis was stored as np.linspace(start, stop, num), which rebuilds it bit for bit (make_golden.py)
        start, stop, num = g.pop('w_linspace')
        g['w'] = np.linspace(start, stop, int(num))
    return g


@pytest.fixture
def golden():
    return load_golden


class PeakRec:
    pass


def peaks_from_golden(g):
    """Peak records (loc, width, area, height, bounds) stored with a golden case."""
    out = []
    for loc, width, area, height in zip(g['peak_loc'], g['peak_width'], g['peak_area'], g['peak_height']):
        p = PeakRec()
        p.loc, p.width, p.area, p.height = float(loc), float(width), float(area), float(height)
        p.bounds = [p.loc - 2 * p.width, p.loc + 2 * p.width]
        out.append(p)
    return out


def relerr(got, want):
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    return float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-300)))
