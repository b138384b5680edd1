import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "practical-path-guiding_b200"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "slow: long-running statistical test")
    # Mitsuba's rough-transmittance tables (data/microfacet/*.dat, 2 MB each) and Hosek-Wilkie sky coefficients (skymodeldata.h) are not
    # part of the repository: the tests read what they need of them from tests/golden (tools/make_golden.py).
    from common import load_rough_transmittance, load_sky_tables
    from ppg_b200 import rtrans, sunsky
    for dist in ("beckmann", "ggx"):
        rtrans._cache[dist] = load_rough_transmittance(dist)
    sunsky._tables = load_sky_tables()
