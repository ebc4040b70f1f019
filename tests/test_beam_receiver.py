"""Delay-and-sum beams on the device: the one-shot beamformer against a float64 restatement and exact identities, the
beam receiver against the plain receiver fed the one-shot beams, and the array gain on a plane wave that no single
hydrophone decodes."""
import ctypes

import numpy as np
import pytest

from oracle import port_binding as ob
from oracle import testdata as td

pytestmark = pytest.mark.gpu

import uwspr_b200 as ub  # noqa: E402
from uwspr_b200 import synth  # noqa: E402

STRIDE = 9 * 375
FL = 45000


def dev(a):
    """a contiguous CUDA copy of a numpy array and the (pointer, dtype, shape) tuple the bindings take"""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t, (ctypes.c_void_p(t.data_ptr()), a.dtype, a.shape)


def splits(n, sizes, rng=None):
    """cut points of n samples into pieces of the given sizes (cycled), or a seeded random split"""
    cuts, at, i = [0], 0, 0
    while at < n:
        at = min(n, at + (int(rng.integers(1, 50000)) if rng is not None else sizes[i % len(sizes)]))
        cuts.append(at)
        i += 1
    return cuts


def cnoise(rng, shape, scale=1.0):
    return ((rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) * scale).astype(np.complex64)


def restate(x, w, d):
    """y_b[n] = sum_c w[b, c] x_c[n - d[b, c]] in float64"""
    nchan, n = x.shape
    y = np.zeros((w.shape[0], n), np.complex128)
    xd = x.astype(np.complex128)
    for b in range(w.shape[0]):
        for c in range(nchan):
            k = int(d[b, c])
            if k < n:
                y[b, k:] += complex(w[b, c]) * xd[c, :n - k]
    return y


def restate_fast(x, w, d):
    """restate() for many beams: one pass per channel and distinct delay"""
    nchan, n = x.shape
    y = np.zeros((w.shape[0], n), np.complex128)
    for c in range(nchan):
        xc = x[c].astype(np.complex128)
        for k in np.unique(d[:, c]):
            rows = np.flatnonzero(d[:, c] == k)
            if k < n:
                y[rows, k:] += w[rows, c].astype(np.complex128)[:, None] * xc[None, :n - k]
    return y


# ---- 1. one-shot against float64 ------------------------------------------------------------------------------------
# (nchan, nbeam, delays): "zero", "max" (all 8192) or "random" (0..8192, with 0 and 8192 present); n is no multiple of
# the 128-sample tile, and nbeam 7 / 1024 leave partial and many 32-beam groups
CASES = [(1, 1, "zero", 1001), (1, 1024, "random", 9301), (5, 7, "random", 9301), (5, 64, "max", 9301),
         (64, 64, "random", 9301), (64, 7, "zero", 1001), (64, 1, "max", 8300), (300, 1, "random", 9301),
         (300, 1024, "random", 1001), (300, 64, "zero", 4097)]


def case_data(nchan, nbeam, delays, n, seed):
    rng = np.random.default_rng(seed)
    x = cnoise(rng, (nchan, n))
    w = cnoise(rng, (nbeam, nchan), 1.0 / np.sqrt(2 * nchan))
    if delays == "zero":
        d = np.zeros((nbeam, nchan), np.int32)
    elif delays == "max":
        d = np.full((nbeam, nchan), 8192, np.int32)
    else:
        # most delays short (an array's fan of beams), some anywhere in the domain, both ends present
        d = rng.integers(0, 300, (nbeam, nchan)).astype(np.int32)
        far = rng.random((nbeam, nchan)) < 0.1
        d[far] = rng.integers(0, 8193, int(far.sum()))
        d.flat[0], d.flat[-1] = 0, 8192
    return x, w, d


@pytest.mark.parametrize("nchan,nbeam,delays,n", CASES)
def test_one_shot_against_float64(nchan, nbeam, delays, n):
    x, w, d = case_data(nchan, nbeam, delays, n, seed=nchan * 7 + nbeam)
    got = ub.beamform(x, w, d)
    want = (restate if nbeam * nchan <= 400 else restate_fast)(x, w, d)
    assert got.shape == (nbeam, n)
    # the error's rms over each beam against the beam's rms: a few fp32 roundings of the running sum per channel.
    # (Its largest sample, at the beam's peaks, reaches about 3e-6 of the rms; one wrong or missing sample would be
    # 1e-2 of it.)
    err = got.astype(np.complex128) - want
    rms = np.sqrt((np.abs(want) ** 2).mean(axis=1))
    err_rms = np.sqrt((np.abs(err) ** 2).mean(axis=1))
    assert (err_rms <= 1e-6 * rms).all(), (err_rms / np.maximum(rms, 1e-30)).max()
    assert (np.abs(err).max(axis=1) <= 2e-5 * rms).all()
    # device input and output: the same floats
    import torch
    tx, arg = dev(x)
    out = torch.zeros((nbeam, n + 3, 2), dtype=torch.float32, device="cuda")
    assert ub.beamform(arg, w, d, out_device_ptr=out.data_ptr(), out_stride=n + 3) == n
    torch.cuda.synchronize()
    dgot = out.cpu().numpy().view(np.complex64)[..., 0][:, :n]
    assert np.array_equal(dgot.view(np.uint32), got.view(np.uint32))


# ---- 2. exact identities -------------------------------------------------------------------------------------------
def test_exact_identities():
    import torch
    rng = np.random.default_rng(12)
    nchan, n = 6, 5000
    x = cnoise(rng, (nchan, n))
    # one-hot rows, delay 0: the channels themselves
    w = np.eye(nchan, dtype=np.complex64)
    d = np.zeros((nchan, nchan), np.int32)
    assert np.array_equal(ub.beamform(x, w, d), x)
    # one-hot rows with delays: each channel shifted, the leading samples zero
    shifts = [0, 1, 31, 129, 4999, 8192]
    w = np.zeros((len(shifts), nchan), np.complex64)
    d = rng.integers(0, 8193, (len(shifts), nchan)).astype(np.int32)   # the zero-weight entries' delays do not matter
    for b, k in enumerate(shifts):
        w[b, b] = 1.0
        d[b, b] = k
    got = ub.beamform(x, w, d)
    for b, k in enumerate(shifts):
        want = np.zeros(n, np.complex64)
        want[k:] = x[b, :max(0, n - k)]
        assert np.array_equal(got[b], want), k
    # host and device buffers give the same floats
    tx, arg = dev(x)
    out = torch.zeros((len(shifts), n, 2), dtype=torch.float32, device="cuda")
    ub.beamform(arg, w, d, out_device_ptr=out.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.complex64)[..., 0].view(np.uint32), got.view(np.uint32))


# ---- 3./4. the receiver ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def five_channels():
    """5 channels x 20 windows at shift 9 s: frames at different frequencies and times, channel 2 all zeros,
    channel 4 carries two overlapping frames (as tests/test_array_receiver.py builds them)"""
    nwin = 20
    n = FL + (nwin - 1) * STRIDE
    rng = np.random.default_rng(3)
    x = ((rng.standard_normal((5, n)) + 1j * rng.standard_normal((5, n))) * np.sqrt(0.15 / 10 ** (-1.2) / 2.0))
    x[2] = 0
    plan = {0: [(5000, -4.0, 1)], 1: [(30000, 6.3, 2), (60000, -1.1, 3)], 3: [(52000, 2.2, 4)],
            4: [(12000, -3.0, 5), (20000, 3.5, 6)]}
    for c, frames in plan.items():
        for start, f0, seed in frames:
            msg = td.message_bytes(np.random.default_rng(seed))
            x[c, start:start + 162 * 256] += td.modulate(ob.channel_symbols(msg), f0=f0, drift=0.0, start=0, fl=162 * 256)
    return x.astype(np.complex64), nwin


def run_receiver(rx, data, cuts):
    got = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        got += rx.push(data[:, lo:hi])
    got += rx.push(data[:, :0], flush=True)
    return [(c, w, bytes(m), cand.tobytes()) for c, w, m, cand in got]


def mixed_beams():
    """4 beams of the 5 channels: one channel delayed, two channels in phase, all channels at random, the silent one"""
    rng = np.random.default_rng(17)
    w = np.zeros((4, 5), np.complex64)
    d = np.zeros((4, 5), np.int32)
    w[0, 0], d[0, 0] = 1.0, 700
    w[1, 1], w[1, 3], d[1, 3] = 0.7, 0.7j, 37
    w[2] = cnoise(rng, 5, 0.3)
    d[2] = rng.integers(0, 400, 5)
    w[3, 2], d[3, 2] = 1.0, 8192
    return w, d


@pytest.fixture(scope="module")
def beam_reference(five_channels):
    """the plain receiver on the one-shot beams"""
    x, nwin = five_channels
    w, d = mixed_beams()
    y = ub.beamform(x, w, d)
    rx = ub.ArrayReceiver(4, shift=9, batch_windows=7)
    want = run_receiver(rx, y, splits(y.shape[1], [y.shape[1]]))
    assert rx.windows_done() == nwin
    rx.close()
    return want


@pytest.mark.parametrize("batch", [1, 3, 7, 64])
def test_stream_equals_one_shot(five_channels, beam_reference, batch):
    x, nwin = five_channels
    w, d = mixed_beams()
    want = beam_reference
    assert {c for c, *_ in want} >= {0, 1, 2} and 3 not in {c for c, *_ in want}   # the silent beam decodes nothing
    n = x.shape[1]
    for cuts in (splits(n, [1, 31, 4096]), splits(n, None, np.random.default_rng(batch))):
        rx = ub.ArrayReceiver(5, shift=9, batch_windows=batch, beams=(w, d))
        assert run_receiver(rx, x, cuts) == want, (batch, len(cuts))
        assert rx.windows_done() == nwin
        rx.close()


def test_stream_equals_one_shot_audio():
    """int16 audio through the front-end: the beams of the front-end's streams"""
    rng = np.random.default_rng(9)
    pos = rng.uniform(0.0, 200.0, (4, 2))
    nwin = 3
    pcm, truth = synth.gen_plane_wave_audio(pos, [0.6, 0.8], 4, (FL + (nwin - 1) * STRIDE) * 32 / 12000.0 / 60.0, -12.0,
                                            seed=5, f0=-3.0)
    taps = ub.flowgraph_taps()
    w, d = ub.plane_wave_steering(pos, [[0.6, 0.8], [-0.8, 0.6]])
    streams = ub.frontend(pcm, taps=taps, delay=0)
    y = ub.beamform(streams, w, d)
    rx = ub.ArrayReceiver(2, shift=9, batch_windows=2)
    want = run_receiver(rx, y, splits(y.shape[1], [y.shape[1]]))
    rx.close()
    assert truth["msg"] in {m for c, _, m, _ in want if c == 0}
    rx = ub.ArrayReceiver(4, shift=9, batch_windows=2, input="int16", taps=taps, delay=0, beams=(w, d))
    got = run_receiver(rx, pcm, splits(pcm.shape[1], [99_991, 7, 300_001]))
    assert rx.windows_done() == nwin
    assert got == want
    rx.close()
    # the same audio resident on the device
    rx = ub.ArrayReceiver(4, shift=9, batch_windows=3, input="int16", taps=taps, delay=0, beams=(w, d))
    t, arg = dev(pcm)
    got = rx.push(arg, flush=True)
    assert [(c, k, bytes(m), cand.tobytes()) for c, k, m, cand in got] == want
    rx.close()


def test_identity_beams_reproduce_the_array_receiver(five_channels):
    x, nwin = five_channels
    rx = ub.ArrayReceiver(5, shift=9, batch_windows=7)
    want = run_receiver(rx, x, splits(x.shape[1], [10_000]))
    rx.close()
    rx = ub.ArrayReceiver(5, shift=9, batch_windows=7, beams=(np.eye(5, dtype=np.complex64), np.zeros((5, 5), np.int32)))
    got = run_receiver(rx, x, splits(x.shape[1], [10_000]))
    assert rx.windows_done() == nwin
    rx.close()
    assert got == want and len(want) >= 5


# ---- 5. array gain ----------------------------------------------------------------------------------------------------
# Calibrated once on a B200 with this geometry and source (16 hydrophones in a 200 m square, source from 40 degrees,
# 2.2 minutes of int16 audio, seeds 1..4, per-channel SNR in 2500 Hz from -42 to -28 dB in 2 dB steps): the plain
# receiver decoded nothing on any hydrophone up to -32 dB, the text on some hydrophones of every seed at -30 dB and on
# all 16 at -28 dB.  The beam steered at the source decoded it in 1 of 4 seeds at -42 dB and in every seed from -40 dB
# up (about -28 dB on the beam, 12 dB of array gain), with a spectral SNR of 4.5-5.0 dB at -36 dB.  -36 dB leaves
# 4 dB of margin on both sides.
GAIN_SNR_DB = -36.0
GAIN_DIR = [np.cos(np.radians(40.0)), np.sin(np.radians(40.0))]


@pytest.mark.parametrize("seed", [1, 2])
def test_array_gain(seed):
    rng = np.random.default_rng(100 + seed)
    pos = rng.uniform(0.0, 200.0, (16, 2))
    pcm, truth = synth.gen_plane_wave_audio(pos, GAIN_DIR, 16, 2.2, GAIN_SNR_DB, seed=seed, f0=1.5)
    taps = ub.flowgraph_taps()
    ang = np.radians([40.0, 130.0, 220.0, 310.0])
    w, d = ub.plane_wave_steering(pos, np.c_[np.cos(ang), np.sin(ang)])
    assert d[0].max() >= 20   # the integer delays matter
    plain = ub.ArrayReceiver(16, shift=9, batch_windows=2, input="int16", taps=taps, delay=0)
    heard_plain = plain.push(pcm, flush=True)
    plain.close()
    beams = ub.ArrayReceiver(16, shift=9, batch_windows=2, input="int16", taps=taps, delay=0, beams=(w, d))
    heard = beams.push(pcm, flush=True)
    beams.close()
    assert heard_plain == [], [(c, bytes(m)) for c, _, m, _ in heard_plain]
    u = ub.WSPR_unpacker()
    texts = {u.unpack(m)[1] for c, _, m, _ in heard if c == 0}
    assert truth["text"] in texts, heard


# ---- 6. launches ------------------------------------------------------------------------------------------------------
def test_launches_per_batch_do_not_grow_with_beams_or_channels(five_channels):
    x, _ = five_channels
    per_batch = {}
    for nchan, nbeam in ((1, 1), (8, 8), (8, 64), (64, 3)):
        data = np.repeat(x[:1], nchan, axis=0)
        w = np.zeros((nbeam, nchan), np.complex64)
        w[:, 0] = 1.0                       # every beam is channel 0: the same candidates on every beam
        d = np.zeros((nbeam, nchan), np.int32)
        d[:, 1:] = 50
        rx = ub.ArrayReceiver(nchan, shift=9, batch_windows=4, beams=(w, d))
        counts = []
        for k in range(3):   # each push completes one more batch of 4 windows
            lo = 0 if k == 0 else FL + (4 * k - 1) * STRIDE
            rx.push(data[:, lo:FL + (4 * k + 3) * STRIDE])
            counts.append(rx.launch_count())
            assert rx.windows_done() == 4 * (k + 1)
        per_batch[(nchan, nbeam)] = np.diff(counts).tolist()
        rx.close()
    first = per_batch[(1, 1)]
    assert all(v == first for v in per_batch.values()) and first[0] > 0, per_batch
