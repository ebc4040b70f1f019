import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = os.path.join(ROOT, "gr-uwspr_b200")
if PKG not in sys.path:
    sys.path.insert(0, PKG)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")
    config.addinivalue_line("markers", "reference: compares with the reference (live where oracle/_ref is built, else recorded)")


@pytest.fixture(scope="session")
def golden():
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden.npz"))
    return g


@pytest.fixture(scope="session")
def golden_windows():
    d = os.path.join(ROOT, "tests", "golden")
    return {n: np.load(os.path.join(d, "win_%s.npy" % n)) for n in ("ve3emb_c2", "test_1500", "rec_150613", "mix_whales")}


def case_window(name, golden_windows):
    """input samples of a golden case (fixtures from disk, synthetic ones regenerated from their seed)"""
    from oracle import testdata as td
    if name in golden_windows:
        return golden_windows[name]
    from tests.golden.make_golden import SYNTH_CASES
    for n, stream, window, snr, md in SYNTH_CASES:
        if n == name:
            return td.synth_window(stream, window, snr_db=snr)[0]
    raise KeyError(name)
