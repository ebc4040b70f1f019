"""Argument checks of the device decoder's entry points that fail before any CUDA call (no GPU needed)."""
import numpy as np
import pytest

import uwspr_b200 as ub
from uwspr_b200.binding import _p

E_PARAM = 1


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    return ub.load_library()


def test_decode_device_null_context(lib):
    refined = np.zeros(4, ub.REFINED_DTYPE)
    jig = np.zeros((4, 17), ub.JIG_DTYPE)
    soft = np.zeros((4, 17, 162), np.uint8)
    dec, msg = np.zeros(4, np.uint8), np.zeros((4, 7), np.int8)
    assert lib.uwspr_b200_decode_device(None, _p(refined), _p(jig), _p(soft), 0, 4, 17, _p(dec), _p(msg), None, None) == -E_PARAM
    assert lib.uwspr_b200_decode_device(None, None, None, None, 0, 0, 17, _p(dec), _p(msg), None, None) == -E_PARAM


@pytest.mark.parametrize("nbits,delta,maxcycles", [(81, 60, 10000), (31, 60, 10000), (82, 60, 10000), (81, 0, 10000),
                                                   (81, -60, 10000), (81, 60, 0), (81, 60, 441870)])
def test_fano_batch_null_context_and_domain(lib, nbits, delta, maxcycles):
    sym = np.zeros((2, 162), np.uint8)
    out = [np.zeros(2, np.int32)] + [np.zeros(2, np.uint32) for _ in range(3)] + [np.zeros((2, 11), np.uint8)]
    st = lib.uwspr_b200_fano_batch(None, _p(sym), 0, 2, nbits, delta, maxcycles, *(_p(a) for a in out))
    assert st == E_PARAM
    assert not any(a.any() for a in out)
