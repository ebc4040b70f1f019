"""The streaming front-end and the multi-channel receiver on the device.

Correctness is equality with entry points that already exist and are tested: the stream's outputs with the one-shot
front-end bit for bit, the receiver's messages with a per-channel Context.coarse_fine over the same 375-sps stream
followed by the host decoder."""
import ctypes

import numpy as np
import pytest

from oracle import port_binding as ob
from oracle import testdata as td

pytestmark = pytest.mark.gpu

import uwspr_b200 as ub  # noqa: E402

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


# ---- 1. the front-end stream equals the one-shot front-end, bit for bit -------------------------------------------
@pytest.fixture(scope="module")
def audio3():
    rng = np.random.default_rng(5)
    n = 260_000
    t = np.arange(n) / 12000.0
    a = 0.3 * rng.standard_normal((3, n)) + 0.2 * np.cos(2 * np.pi * (1500.0 + np.array([[-7.0], [2.0], [9.0]])) * t)
    return {"float32": a.astype(np.float32), "int16": np.clip(np.round(a * 32768.0), -32768, 32767).astype(np.int16)}


TAPS = {"real": (lambda: ub.lowpass_taps(), None), "complex": (lambda: ub.flowgraph_taps(), 0)}


@pytest.mark.parametrize("fmt", ["float32", "int16"])
@pytest.mark.parametrize("taps_kind", ["real", "complex"])
def test_stream_equals_one_shot(audio3, fmt, taps_kind):
    audio = audio3[fmt]
    make, delay = TAPS[taps_kind]
    taps = make()
    d = (len(taps) - 1) // 2 if delay is None else delay
    want = ub.frontend(audio, taps=taps, delay=d)          # one-shot over all samples
    ntaps = len(taps)
    cases = [(1, 3000), (31, None), (32, None), (33, None), (ntaps - 1, None), (ntaps, None), (100_000, None), ("random", None)]
    for size, limit in cases:
        n = limit or audio.shape[1] - 40_000   # the one-shot sees 40 000 samples more: every streamed output is in it
        cuts = splits(n, [size]) if size != "random" else splits(n, None, np.random.default_rng(11))
        fs = ub.FrontendStream(3, taps=taps, delay=d, fmt=audio.dtype)
        got = np.concatenate([fs.push(audio[:, lo:hi]) for lo, hi in zip(cuts[:-1], cuts[1:])], axis=1)
        m = max(0, (n - d + 31) // 32)   # #{m: 32 m + delay < n}
        assert got.shape == (3, m) and fs.outputs() == m, size
        assert np.array_equal(got.view(np.uint32), want[:, :m].view(np.uint32)), size
        fs.close()
    # every combination of audio and output on the host and on the device, odd pieces
    import torch
    n = audio.shape[1] - 40_000
    m = max(0, (n - d + 31) // 32)
    cuts = splits(n, [4097, 77, 50_000])
    for audio_on_device, out_on_device in ((True, True), (False, True), (True, False)):
        fs = ub.FrontendStream(3, taps=taps, delay=d, fmt=audio.dtype)
        out = torch.zeros((3, m + 5, 2), dtype=torch.float32, device="cuda")
        parts, done = [], 0
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            t, arg = dev(audio[:, lo:hi]) if audio_on_device else (None, audio[:, lo:hi])
            if out_on_device:
                done += fs.push(arg, out_device_ptr=out.data_ptr() + 8 * done, out_stride=m + 5)
            else:
                parts.append(fs.push(arg))
        if out_on_device:
            assert done == m
            torch.cuda.synchronize()
            got = out.cpu().numpy().view(np.complex64)[..., 0][:, :m]
        else:
            got = np.concatenate(parts, axis=1)
        assert got.shape == (3, m)
        assert np.array_equal(got.view(np.uint32), want[:, :m].view(np.uint32)), (audio_on_device, out_on_device)
        fs.close()


# ---- 2./3. complex input against a per-channel reference ------------------------------------------------------------
def reference(streams, nwin):
    """per channel: Context.coarse_fine over that channel's stream (stride 3375, 17 jiggles) and the host decoder;
    the list in (window, channel, candidate) order"""
    ctx = ub.Context(maxdrift=0, max_windows=nwin)
    per = []
    for x in streams:
        npk, cands, refined, jig, soft = ctx.coarse_fine(x, nwin=nwin, stride=STRIDE)
        base = np.concatenate([[0], np.cumsum(npk)])
        win = np.repeat(np.arange(nwin), npk)
        per.append([(int(win[g]), g - int(base[win[g]]), bytes(m), cands[g].tobytes())
                    for g, m, _ in ub.decode_candidates(refined, jig, soft)])
    ctx.close()
    out = []
    for k in range(nwin):
        for c in range(len(streams)):
            out += [(c, k, m, cb) for w, j, m, cb in per[c] if w == k]
    return out


def run_receiver(rx, data, cuts):
    got = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        got += rx.push(data[:, lo:hi])
    got += rx.push(data[:, :0], flush=True)
    return [(c, w, bytes(m), cand.tobytes()) for c, w, m, cand in got]


@pytest.fixture(scope="module")
def five_channels():
    """5 channels x 20 windows at shift 9 s: frames at different frequencies and times, channel 2 all zeros,
    channel 4 carries two overlapping frames"""
    nwin = 20
    n = FL + (nwin - 1) * STRIDE
    rng = np.random.default_rng(3)
    x = ((rng.standard_normal((5, n)) + 1j * rng.standard_normal((5, n))) * np.sqrt(0.15 / 10 ** (-1.2) / 2.0))
    x[2] = 0
    plan = {0: [(5000, -4.0, 1)], 1: [(30000, 6.3, 2), (60000, -1.1, 3)], 3: [(52000, 2.2, 4)],
            4: [(12000, -3.0, 5), (20000, 3.5, 6)]}
    truth = set()
    for c, frames in plan.items():
        for start, f0, seed in frames:
            msg = td.message_bytes(np.random.default_rng(seed))
            x[c, start:start + 162 * 256] += td.modulate(ob.channel_symbols(msg), f0=f0, drift=0.0, start=0, fl=162 * 256)
            truth.add(bytes(msg))
    x = x.astype(np.complex64)
    return x, nwin, reference(list(x), nwin), truth


def test_complex_input_against_per_channel_reference(five_channels):
    x, nwin, want, truth = five_channels
    rx = ub.ArrayReceiver(5, shift=9, batch_windows=7)
    got = run_receiver(rx, x, splits(x.shape[1], [10_000]))
    assert rx.windows_done() == nwin
    assert got == want
    heard = {m for _, _, m, _ in want}
    assert heard <= truth and len(heard) >= 5
    assert not [1 for c, *_ in want if c == 2]   # the silent channel decodes nothing
    rx.close()


@pytest.mark.parametrize("batch", [1, 3, 7, 64])
def test_batch_size_and_push_split_change_nothing(five_channels, batch):
    x, nwin, want, _ = five_channels
    n = x.shape[1]
    for cuts in (splits(n, [n]), splits(n, [1, 3375, 45_001]), splits(n, None, np.random.default_rng(batch))):
        rx = ub.ArrayReceiver(5, shift=9, batch_windows=batch)
        assert run_receiver(rx, x, cuts) == want, (batch, len(cuts))
        assert rx.windows_done() == nwin
        rx.close()


# ---- 4./5. audio end to end -----------------------------------------------------------------------------------------
TEXTS = [("VE3EMB", "FN25", 30), ("W1AW", "FN31", 23), ("K1ABC", "FN42", 37), ("G4ABC", "IO91", 20)]


@pytest.fixture(scope="module")
def audio4():
    """4 channels of int16 12 kHz audio, one known type-1 text each, in noise; 4 windows per channel at shift 9 s"""
    fs_in, nwin = 12000.0, 4
    n = (FL + (nwin - 1) * STRIDE) * 32
    rng = np.random.default_rng(21)
    audio = np.zeros((4, n))
    for c, (call, grid, dbm) in enumerate(TEXTS):
        sym = ub.channel_symbols(ub.pack_type1(call, grid, dbm)).astype(np.float64)
        f0 = (2.7, -5.2, 0.6, 4.4)[c]
        start = int((0.8 + 0.5 * c + 9.0 * (c % 2)) * fs_in)
        f = 1500.0 + f0 + (np.repeat(sym, 8192) - 1.5) * 375.0 / 256.0
        audio[c, start:start + 162 * 8192] = 0.1 * np.cos(2 * np.pi * np.cumsum(f) / fs_in)
        audio[c] += 0.2 * rng.standard_normal(n)
    pcm = np.clip(np.round(audio * 32768.0), -32768, 32767).astype(np.int16)
    taps = ub.flowgraph_taps()
    streams = ub.frontend(pcm, taps=taps, delay=0)   # one-shot front-end: the reference's 375-sps streams
    return pcm, taps, nwin, reference(list(streams), nwin)


def test_audio_end_to_end(audio4):
    pcm, taps, nwin, want = audio4
    rx = ub.ArrayReceiver(4, shift=9, batch_windows=3, input="int16", taps=taps, delay=0)
    got = run_receiver(rx, pcm, splits(pcm.shape[1], [99_991, 7, 300_001]))
    assert rx.windows_done() == nwin
    assert got == want
    u = ub.WSPR_unpacker()
    for c, (call, grid, dbm) in enumerate(TEXTS):
        heard = {u.unpack(np.frombuffer(m, np.uint8))[1] for ch, _, m, _ in got if ch == c}
        assert "%s %s %2d" % (call, grid, dbm) in heard, c


def test_device_audio_equals_host_audio(audio4):
    pcm, taps, nwin, want = audio4
    rx = ub.ArrayReceiver(4, shift=9, batch_windows=2, input="int16", taps=taps, delay=0)
    got = []
    cuts = splits(pcm.shape[1], [123_457, 1_000_003])
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        t, arg = dev(pcm[:, lo:hi])
        got += rx.push(arg)
    got += rx.push(pcm[:, :0], flush=True)
    assert [(c, w, bytes(m), cand.tobytes()) for c, w, m, cand in got] == want
    # float32 audio through the same path equals the one-shot float front-end's streams
    a32 = pcm.astype(np.float32) / 32768.0
    rx32 = ub.ArrayReceiver(4, shift=9, batch_windows=4, input="float32", taps=taps, delay=0)
    t, arg = dev(a32)
    got32 = rx32.push(arg, flush=True)
    want32 = reference(list(ub.frontend(a32, taps=taps, delay=0)), nwin)
    assert [(c, w, bytes(m), cand.tobytes()) for c, w, m, cand in got32] == want32


# ---- 6. one submission per batch ---------------------------------------------------------------------------------
def test_launches_per_batch_do_not_grow_with_channels(five_channels):
    x, _, _, _ = five_channels
    per_batch = {}
    for nchan in (1, 8):
        data = np.repeat(x[:1], nchan, axis=0)   # the same candidates on every channel
        rx = ub.ArrayReceiver(nchan, shift=9, batch_windows=4)
        counts = []
        for k in range(3):   # each push completes one more batch of 4 windows
            lo = 0 if k == 0 else FL + (4 * k - 1) * STRIDE
            rx.push(data[:, lo:FL + (4 * k + 3) * STRIDE])
            counts.append(rx.launch_count())
            assert rx.windows_done() == 4 * (k + 1)
        per_batch[nchan] = np.diff(counts).tolist()
        rx.close()
    assert per_batch[1] == per_batch[8] and per_batch[1][0] > 0, per_batch


# ---- 7. status paths that need the device ------------------------------------------------------------------------
def test_status_paths():
    # 63*4096 + 16384 complex samples of staging do not fit shared memory
    with pytest.raises(ub.UwsprError) as e:
        ub.ArrayReceiver(2, input="float32", taps=np.ones(16384, np.float32), decim=4096, fs_in=375.0 * 4096, delay=0)
    assert e.value.status == 1
    with pytest.raises(ub.UwsprError) as e:
        ub.FrontendStream(2, taps=np.ones(16384, np.float32), decim=4096, fs_in=375.0 * 4096, delay=0)
    assert e.value.status == 1
    # more candidates than max_candidates: the batch's status comes back, and the receiver refuses further pushes
    rng = np.random.default_rng(8)
    x = np.zeros((2, FL), np.complex64)
    for c in range(2):
        msg = td.message_bytes(rng)
        x[c, 1000:1000 + 162 * 256] = td.modulate(ob.channel_symbols(msg), f0=-3.0 + 5 * c, drift=0.0, start=0, fl=162 * 256)
    rx = ub.ArrayReceiver(2, shift=9, batch_windows=1, max_candidates=1)
    with pytest.raises(ub.UwsprError) as e:
        rx.push(x)
    assert e.value.status == 3
    with pytest.raises(ub.UwsprError) as e:
        rx.push(x)
    assert e.value.status == 5
    rx.close()
    # a push whose outputs exceed the caller's capacity consumes nothing
    fs = ub.FrontendStream(1, delay=0)
    lib = ub.load_library()
    a = np.zeros(640, np.float32)
    out = np.zeros(4, np.complex64)
    got = ctypes.c_int64()
    st = lib.uwspr_b200_frontend_stream_push(fs.h, a.ctypes.data_as(ctypes.c_void_p), 0, 640, 640,
                                             out.ctypes.data_as(ctypes.c_void_p), 0, 4, 4, ctypes.byref(got))
    assert st == 3 and fs.outputs() == 0
    # strides shorter than a channel's samples or outputs are E_PARAM for one channel too, and consume nothing
    big = np.zeros(64, np.complex64)
    for stride, ostride in ((0, 64), (639, 64), (640, 63)):
        st = lib.uwspr_b200_frontend_stream_push(fs.h, a.ctypes.data_as(ctypes.c_void_p), 0, stride, 640,
                                                 big.ctypes.data_as(ctypes.c_void_p), 0, ostride, 64, ctypes.byref(got))
        assert st == 1 and fs.outputs() == 0, (stride, ostride)
    assert fs.push(a).shape == (1, 20)
    rx1 = ub.ArrayReceiver(1, shift=9, batch_windows=1)
    xs = np.zeros(FL, np.complex64)
    for stride in (0, FL - 1):
        assert lib.uwspr_b200_array_receiver_push(rx1.h, xs.ctypes.data_as(ctypes.c_void_p), 0, stride, FL, 0) == 1
    assert rx1.windows_done() == 0
    rx1.push(xs.reshape(1, -1))
    assert rx1.windows_done() == 1
    rx1.close()
