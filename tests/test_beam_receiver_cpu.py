"""Delay-and-sum beams without a GPU: every argument check of uwspr_b200_beamform and
uwspr_b200_array_receiver_create_beams that returns E_PARAM before any CUDA call, and plane_wave_steering against
hand-computed delays and phases."""
import ctypes as C

import numpy as np
import pytest

import uwspr_b200 as ub
from uwspr_b200.binding import Beams, Input, Params, _p

E_PARAM = 1


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    return ub.load_library()


def params(**kw):
    p = dict(fs=375, fl=45000, spb=256, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10, device=0,
             max_windows=0, max_candidates=0, nonlinear_intended_t=0)
    p.update(kw)
    return Params(*p.values())


TAPS = np.ones(33, np.float32)


def audio_input(**kw):
    a = dict(kind=2, taps=_p(TAPS), ntaps=len(TAPS), complex_taps=0, decim=32, delay=0, fc=1500.0, fs_in=12000.0)
    a.update(kw)
    return Input(*a.values())


def tables(nbeam, nchan, weight=1.0 + 0.5j, delay=3):
    w = np.full((nbeam, nchan), weight, np.complex64)
    d = np.full((nbeam, nchan), delay, np.int32)
    return w, d


# ---- uwspr_b200_beamform ---------------------------------------------------------------------------------------------
BAD_BEAMFORM = {
    "nchan 0": dict(nchan=0),
    "nchan 1025": dict(nchan=1025),
    "nbeam 0": dict(nbeam=0),
    "nbeam 1025": dict(nbeam=1025),
    "delay -1": dict(delay=-1),
    "delay 8193": dict(delay=8193),
    "NaN weight": dict(weight=complex(np.nan, 0.0)),
    "NaN imaginary weight": dict(weight=complex(0.0, np.nan)),
    "inf weight": dict(weight=complex(np.inf, 0.0)),
    "-inf imaginary weight": dict(weight=complex(0.0, -np.inf)),
    "n negative": dict(n=-1),
    "in_stride < n": dict(in_stride=63),
    "out_stride < n": dict(out_stride=63),
    "space_in 2": dict(space_in=2),
    "space_in -1": dict(space_in=-1),
    "space_out 2": dict(space_out=2),
    "NULL in": dict(null="in"),
    "NULL out": dict(null="out"),
    "NULL weights": dict(null="weights"),
    "NULL delays": dict(null="delays"),
}


@pytest.mark.parametrize("case", sorted(BAD_BEAMFORM))
def test_beamform_rejects(lib, case):
    c = BAD_BEAMFORM[case]
    nchan, nbeam, n = c.get("nchan", 3), c.get("nbeam", 2), c.get("n", 64)
    w, d = tables(max(nbeam, 1), max(nchan, 1), c.get("weight", 1.0 + 0.5j), c.get("delay", 3))
    w[-1, -1] = c.get("weight", w[-1, -1])   # one bad entry, at the end, is enough
    x = np.zeros((max(nchan, 1), 64), np.complex64)
    y = np.zeros((max(nbeam, 1), 64), np.complex64)
    ptrs = {"in": _p(x), "out": _p(y), "weights": _p(w), "delays": _p(d)}
    if "null" in c:
        ptrs[c["null"]] = None
    st = lib.uwspr_b200_beamform(0, ptrs["in"], c.get("space_in", 0), c.get("in_stride", 64), nchan, n, ptrs["weights"],
                                 ptrs["delays"], nbeam, ptrs["out"], c.get("space_out", 0), c.get("out_stride", 64))
    assert st == E_PARAM
    assert not y.any()


def test_beamform_bad_single_entries(lib):
    """a single bad weight or delay anywhere in the matrix is found"""
    x = np.zeros((5, 16), np.complex64)
    y = np.zeros((4, 16), np.complex64)
    for bad in ("delay", "weight"):
        for b, c in ((0, 0), (2, 3), (3, 4)):
            w, d = tables(4, 5)
            if bad == "delay":
                d[b, c] = 8193
            else:
                w[b, c] = complex(np.inf, 1.0)
            assert lib.uwspr_b200_beamform(0, _p(x), 0, 16, 5, 16, _p(w), _p(d), 4, _p(y), 0, 16) == E_PARAM, (bad, b, c)


def test_beamform_binding_checks_shapes():
    x = np.zeros((3, 10), np.complex64)
    with pytest.raises(ValueError):
        ub.beamform(x, np.ones((2, 4), np.complex64), np.zeros((2, 4), np.int32))
    with pytest.raises(ValueError):
        ub.beamform(x, np.ones((2, 3), np.complex64), np.zeros((2, 2), np.int32))


# ---- uwspr_b200_array_receiver_create_beams ----------------------------------------------------------------------------
BAD_CREATE = dict(BAD_BEAMFORM)
for k in ("n negative", "in_stride < n", "out_stride < n", "space_in 2", "space_in -1", "space_out 2", "NULL in", "NULL out"):
    del BAD_CREATE[k]
BAD_CREATE.update({
    "NULL beams": dict(null="beams"),
    "NULL params": dict(null="params"),
    "NULL input": dict(null="input"),
    "NULL out": dict(null="handle"),
    "nbeam * batch > INT_MAX / 2": dict(nbeam=1024, batch=(2 ** 31 - 1) // 2 // 1024 + 1),
    "batch 0": dict(batch=0),
    "shift*fs > fl": dict(shift=121),
    "kind 3": dict(inp=dict(kind=3)),
    "fs_in/decim != fs": dict(inp=dict(fs_in=12001.0)),
    "ntaps 0": dict(inp=dict(ntaps=0)),
})


@pytest.mark.parametrize("case", sorted(BAD_CREATE))
def test_create_beams_rejects(lib, case):
    c = BAD_CREATE[case]
    nchan, nbeam = c.get("nchan", 3), c.get("nbeam", 2)
    w, d = tables(max(nbeam, 1), max(nchan, 1), c.get("weight", 1.0 + 0.5j), c.get("delay", 3))
    w[-1, -1] = c.get("weight", w[-1, -1])
    bm = Beams(nbeam, None if c.get("null") == "weights" else _p(w), None if c.get("null") == "delays" else _p(d))
    prm, inp = params(), audio_input(**c.get("inp", {}))
    h = C.c_void_p(1)
    args = {"params": C.byref(prm), "input": C.byref(inp), "beams": C.byref(bm), "handle": C.byref(h)}
    if c.get("null") in args:
        args[c["null"]] = None
    st = lib.uwspr_b200_array_receiver_create_beams(args["params"], args["input"], nchan, args["beams"], c.get("shift", 9),
                                                    c.get("batch", 4), args["handle"])
    assert st == E_PARAM
    if c.get("null") != "handle":
        assert h.value is None


def test_create_beams_in_domain_reaches_the_device(lib):
    """the largest accepted matrix passes every check, so the create gets as far as the device"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    w, d = tables(1024, 1024, 0.03 + 0.0j, 8192)
    bm, prm, inp, h = Beams(1024, _p(w), _p(d)), params(), audio_input(), C.c_void_p()
    assert lib.uwspr_b200_array_receiver_create_beams(C.byref(prm), C.byref(inp), 1024, C.byref(bm), 9, 4, C.byref(h)) == 2
    x = np.zeros((1024, 1), np.complex64)
    y = np.zeros((1024, 1), np.complex64)
    assert lib.uwspr_b200_beamform(0, _p(x), 0, 1, 1024, 1, _p(w), _p(d), 1024, _p(y), 0, 1) == 2   # E_CUDA


# ---- plane_wave_steering ------------------------------------------------------------------------------------------------
# A line of three hydrophones on the x axis.  With sound_speed == fc == 1500, the carrier phase of a delay of
# x metres of path is exactly x cycles, and 375 sps make one sample 4 m.
LINE = np.array([[0.0, 0.0], [7.3, 0.0], [20.1, 0.0]])


def test_steering_broadside():
    w, d = ub.plane_wave_steering(LINE, [[0.0, 1.0]])
    assert d.tolist() == [[0, 0, 0]]
    assert np.allclose(w, np.full((1, 3), 1 / np.sqrt(3)), atol=1e-7)


def test_steering_endfire():
    # source towards +x: hydrophone x hears it x/1500 s early, so it is delayed by x/1500 s to line up with the origin:
    # 7.3 m = 1.825 samples -> 2, 20.1 m = 5.025 -> 5; the phase removes x cycles: e^{-2 pi i frac(x)}
    w, d = ub.plane_wave_steering(LINE, [[1.0, 0.0], [-1.0, 0.0]])
    assert d.tolist() == [[0, 2, 5], [5, 3, 0]]
    want = np.array([[1.0, np.exp(-2j * np.pi * 0.3), np.exp(-2j * np.pi * 0.1)],
                     # source towards -x: the origin is the earliest, 20.1 m ahead of the last; 12.8 m = 3.2 -> 3
                     [np.exp(-2j * np.pi * 0.1), np.exp(-2j * np.pi * 0.8), 1.0]]) / np.sqrt(3)
    assert np.allclose(w, want, atol=1e-6)
    assert w.dtype == np.complex64 and d.dtype == np.int32


def test_steering_oblique_and_3d():
    # 60 degrees off the axis: path differences x cos 60 = x/2 metres
    u = [[0.5, np.sqrt(3) / 2]]
    w, d = ub.plane_wave_steering(LINE, u)
    align = LINE[:, 0] / 2.0          # metres; the origin hears it last
    assert d.tolist() == [np.rint(align / 4.0).astype(int).tolist()]
    assert np.allclose(w[0], np.exp(-2j * np.pi * align) / np.sqrt(3), atol=1e-6)
    # the same line in 3-D, the source straight above: broadside again
    p3 = np.c_[LINE, np.zeros(3)]
    w3, d3 = ub.plane_wave_steering(p3, [[0.0, 0.0, 1.0]])
    assert d3.tolist() == [[0, 0, 0]] and np.allclose(w3, 1 / np.sqrt(3), atol=1e-7)


def test_steering_normalised_and_other_speeds():
    rng = np.random.default_rng(4)
    pos = rng.uniform(0.0, 200.0, (16, 2))
    ang = np.linspace(0, 2 * np.pi, 12, endpoint=False)
    w, d = ub.plane_wave_steering(pos, np.c_[np.cos(ang), np.sin(ang)])
    assert w.shape == d.shape == (12, 16)
    assert np.allclose((np.abs(w.astype(np.complex128)) ** 2).sum(axis=1), 1.0, atol=1e-6)
    assert (d.min(axis=1) == 0).all() and d.max() <= 71     # 283 m of aperture at most: 71 samples
    # halving the sound speed doubles every delay before rounding
    w2, d2 = ub.plane_wave_steering(LINE, [[1.0, 0.0]], sound_speed=750.0, fc=1000.0, fs=375.0)
    assert d2.tolist() == [[0, 4, 10]]
    assert np.allclose(w2[0], np.exp(-2j * np.pi * 1000.0 * LINE[:, 0] / 750.0) / np.sqrt(3), atol=1e-6)
    with pytest.raises(ValueError):
        ub.plane_wave_steering(pos, [[1.0, 0.0, 0.0]])
