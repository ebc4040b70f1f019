"""Argument checks of the array receiver and the front-end stream that fail with E_PARAM before any CUDA call
(no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

import uwspr_b200 as ub
from uwspr_b200.binding import Input, Params, _p

E_PARAM = 1


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    return ub.load_library()


TAPS = np.ones(33, np.float32)


def params(**kw):
    p = dict(fs=375, fl=45000, spb=256, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10, device=0,
             max_windows=0, max_candidates=0, nonlinear_intended_t=0)
    p.update(kw)
    return Params(*p.values())


def audio_input(**kw):
    a = dict(kind=2, taps=_p(TAPS), ntaps=len(TAPS), complex_taps=0, decim=32, delay=0, fc=1500.0, fs_in=12000.0)
    a.update(kw)
    return Input(*a.values())


BAD = {
    "nchan 0": dict(nchan=0),
    "nchan negative": dict(nchan=-3),
    "batch 0": dict(batch=0),
    "shift*fs 0": dict(shift=0),
    "shift*fs negative": dict(shift=-1),
    "shift*fs > fl": dict(shift=121),
    "fs 0": dict(prm=dict(fs=0)),
    "kind -1": dict(inp=dict(kind=-1)),
    "kind 3": dict(inp=dict(kind=3)),
    "fs_in/decim != fs": dict(inp=dict(fs_in=12001.0)),
    "decim != fs_in/fs": dict(inp=dict(decim=16)),
    "fs_in 0": dict(inp=dict(fs_in=0.0)),
    "ntaps 0": dict(inp=dict(ntaps=0)),
    "ntaps 16385": dict(inp=dict(ntaps=16385)),
    "decim 0": dict(inp=dict(decim=0)),
    "negative delay": dict(inp=dict(delay=-1)),
    "NULL taps": dict(inp=dict(taps=None)),
    "float32 kind, ntaps 0": dict(inp=dict(kind=1, ntaps=0)),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_array_receiver_create_rejects(lib, case):
    c = BAD[case]
    prm = params(**c.get("prm", {}))
    inp = audio_input(**c.get("inp", {}))
    h = C.c_void_p(1)
    st = lib.uwspr_b200_array_receiver_create(C.byref(prm), C.byref(inp), c.get("nchan", 2), c.get("shift", 9), c.get("batch", 4),
                                              C.byref(h))
    assert st == E_PARAM
    assert h.value is None


def test_array_receiver_null_pointers(lib):
    prm, inp, h = params(), audio_input(), C.c_void_p()
    assert lib.uwspr_b200_array_receiver_create(None, C.byref(inp), 2, 9, 4, C.byref(h)) == E_PARAM
    assert lib.uwspr_b200_array_receiver_create(C.byref(prm), None, 2, 9, 4, C.byref(h)) == E_PARAM
    assert lib.uwspr_b200_array_receiver_create(C.byref(prm), C.byref(inp), 2, 9, 4, None) == E_PARAM
    x = np.zeros((2, 8), np.int16)
    assert lib.uwspr_b200_array_receiver_push(None, _p(x), 0, 8, 8, 0) == E_PARAM
    assert lib.uwspr_b200_array_receiver_pop(None, None, None, None, None) == 0
    assert lib.uwspr_b200_array_receiver_windows(None) == 0
    assert lib.uwspr_b200_array_receiver_launch_count(None) == 0
    lib.uwspr_b200_array_receiver_destroy(None)


def test_complex_input_ignores_the_front_end_fields(lib):
    """kind 0 has no front-end: its taps / decim are not checked, so the create gets as far as the device"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    prm, h = params(), C.c_void_p()
    inp = audio_input(kind=0, taps=None, ntaps=0, decim=0, fs_in=0.0)
    assert lib.uwspr_b200_array_receiver_create(C.byref(prm), C.byref(inp), 2, 9, 4, C.byref(h)) == 2   # E_CUDA


@pytest.mark.parametrize("nchan,fmt,ntaps,decim,delay,fs_in", [(0, 0, 33, 32, 0, 12000.0), (70000, 0, 33, 32, 0, 12000.0),
                                                               (2, 2, 33, 32, 0, 12000.0), (2, 0, 0, 32, 0, 12000.0),
                                                               (2, 0, 16385, 32, 0, 12000.0), (2, 1, 33, 0, 0, 12000.0),
                                                               (2, 1, 33, 4097, 0, 12000.0), (2, 0, 33, 32, -1, 12000.0),
                                                               (2, 0, 33, 32, 0, 0.0)])
def test_frontend_stream_create_rejects(lib, nchan, fmt, ntaps, decim, delay, fs_in):
    taps = np.ones(max(ntaps, 1), np.float32)
    h = C.c_void_p(1)
    assert lib.uwspr_b200_frontend_stream_create(0, nchan, fmt, _p(taps), ntaps, 0, decim, delay, 1500.0, fs_in, C.byref(h)) == E_PARAM
    assert h.value is None


def test_frontend_stream_null_pointers(lib):
    h = C.c_void_p()
    assert lib.uwspr_b200_frontend_stream_create(0, 2, 0, None, 33, 0, 32, 0, 1500.0, 12000.0, C.byref(h)) == E_PARAM
    assert lib.uwspr_b200_frontend_stream_create(0, 2, 0, _p(TAPS), 33, 0, 32, 0, 1500.0, 12000.0, None) == E_PARAM
    x, out, n = np.zeros((2, 64), np.float32), np.zeros((2, 4), np.complex64), C.c_int64(7)
    assert lib.uwspr_b200_frontend_stream_push(None, _p(x), 0, 64, 64, _p(out), 0, 4, 4, C.byref(n)) == E_PARAM
    assert n.value == 0
    assert lib.uwspr_b200_frontend_stream_outputs(None) == 0
    lib.uwspr_b200_frontend_stream_destroy(None)
