"""What the comparisons with the reference compute, on both sides, as plain arrays.

Each case is a function case(ref) -> {key: array}.  With ref=True it asks the reference (oracle/_ref: the unmodified
upstream sources compiled against oracle/stubs); with ref=False it asks this repository's code (the oracle's C
restatement, or the product library for the unpacker and the message log) the same questions on the same inputs.
The tests require the two dictionaries to be equal.  Where oracle/_ref is built the reference side is computed live;
elsewhere it is read from recorded_cases.npz, written by `python tests/golden/make_golden.py --reference-cases`,
whose `source` entry says which implementation answered.  Long byte streams (spectrograms, call traces, decoder
records, hash tables) are kept as SHA-256 digests so that the file stays small; the comparison stays exact."""
import hashlib
import os
import tempfile

import numpy as np

from oracle import port_binding as ob
from oracle import ref_binding as rb
from oracle import testdata as td

RECORDED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "recorded_cases.npz")

PIPELINE_PARAMS = [(0, 10, 10), (4, 10, 10), (2, 40, 3), (1, 100, 1000000)]


def _sha(b):
    return np.frombuffer(hashlib.sha256(bytes(b)).digest(), np.uint8)


def _calls_sha(calls):
    return _sha(b"".join(bytes(c) for c in calls))


def _fanos_sha(fanos):
    # byte 172 = data[10], never written by the reference decoder (Fano.cc:243-247)
    return _sha(b"".join(bytes(f)[:172] + bytes(f)[176:] for f in fanos))


def _chain(out, key, cands, blobs, calls, fanos):
    out[key + "cands"] = td.canon_cands(cands).view(np.uint8).reshape(-1, 48)
    out[key + "blobs"] = np.asarray(blobs, np.uint8).reshape(-1, 7)
    out[key + "n_calls"], out[key + "calls_sha"] = np.array([len(calls)]), _calls_sha(calls)
    out[key + "n_fanos"], out[key + "fanos_sha"] = np.array([len(fanos)]), _fanos_sha(fanos)


def pipeline(ref, maxdrift, hbw, thr):
    """FDR -> sync_and_demodulate on four seeded synthetic windows from -8 to -28.5 dB"""
    out = {}
    if ref:
        f, sd = rb.RefFDR(maxdrift=maxdrift, halfbandwidth=hbw, threshold=thr), rb.RefSD(maxdrift=maxdrift)
    else:
        f = ob.OracleFDR(maxdrift=maxdrift, halfbandwidth=hbw, threshold=thr)
    out["geometry"] = np.array([f.n, f.size, f.hpbm, f.m, f.df, f.min_snr], np.float64)
    out["window"] = np.asarray(f.window())
    for w, snr in enumerate([-8.0, -19.0, -25.0, -28.5]):
        x, _ = td.synth_window(11, w, snr_db=snr)
        if ref:
            cands, ps, psavg = f.transform(x, want_ps=True)
            blobs, calls, fanos = sd.demodulate(x, cands)
        else:
            ps = f.spectrogram(x)
            c0, psavg, _ = f.normalize_peaks(ps)
            cands = f.coarse(ps, c0)
            blobs, calls, fanos = ob.demodulate(x, cands)
        out["w%d/ps_shape" % w], out["w%d/ps_sha" % w] = np.array(ps.shape), _sha(np.ascontiguousarray(ps, np.float32))
        out["w%d/psavg" % w] = np.asarray(psavg)
        _chain(out, "w%d/" % w, cands, blobs, calls, fanos)
    return out


def two_signals_and_noise(ref):
    """two transmissions in one window, noise alone, all zeros (hbw 40)"""
    a, _ = td.synth_window(3, 0, snr_db=-12.0, f0=-20.0)
    b, _ = td.synth_window(3, 1, snr_db=-15.0, f0=17.0)
    n, _ = td.synth_window(3, 2, snr_db=-60.0)
    out = {}
    if ref:
        f, sd = rb.RefFDR(halfbandwidth=40), rb.RefSD()
    else:
        f = ob.OracleFDR(halfbandwidth=40)
    for k, x in enumerate((a + b, n, np.zeros(45000, np.complex64))):
        cands = f.transform(x)
        blobs, calls, fanos = sd.demodulate(x, cands) if ref else ob.demodulate(x, cands)
        _chain(out, "x%d/" % k, cands, blobs, calls, fanos)
    return out


def sync_and_demodulate_direct(ref):
    """sync_and_demodulate() itself: both drift models, every mode, lags that run off both ends of the buffer"""
    sd = rb.RefSD() if ref else None
    x, _ = td.synth_window(5, 0, snr_db=-15.0, f0=2.2, drift=1.7, start=500)
    rng = np.random.default_rng(5)
    cand = np.zeros(1, ob.CAND_DTYPE)
    out = {}
    for trial in range(12):
        nonlinear = trial % 3 == 2
        cand["m_type"] = 1 if nonlinear else 0
        if nonlinear:
            cand["V1"], cand["V2"], cand["p1"], cand["p2"] = ob.slm_trajectory(int(rng.integers(0, 125)))
        f1 = float(rng.uniform(-5, 5))
        shift = int(rng.integers(-400, 4000))
        drift = 0.0 if nonlinear else float(rng.choice([0.0, 1.0, -2.5, 0.5]))
        mode = trial % 3 if not nonlinear else int(rng.integers(0, 3))
        kw = dict(ifmin=-2, ifmax=2, fstep=0.25, lagmin=shift - 128, lagmax=shift + 128, lagstep=64)
        r = sd.eval(cand[0], x, f1, shift, drift, mode, **kw) if ref else ob.sync_and_demodulate(cand[0], x, f1, shift, drift, mode, **kw)
        out["t%d/f1" % trial] = np.array([r[0]], np.float32)
        out["t%d/shift" % trial] = np.array([r[1]], np.int64)
        out["t%d/sync" % trial] = np.array([r[2]], np.float32)
        out["t%d/symbols" % trial] = np.asarray(r[3], np.uint8)
    return out


def slm_exhaustive(ref):
    """the SLM drift model for all 125 trajectories at t = 0..119"""
    f = rb.slm_frequency_drift if ref else ob.slm_frequency_drift
    tab = np.zeros((125, 120), np.float32)
    for k in range(125):
        V1, V2, p1, p2 = ob.slm_trajectory(k)
        for t in range(120):
            tab[k, t] = f(V1, V2, p1, p2, 1500.0, float(t))
    return dict(table=tab)


def code_tables_and_decoder(ref):
    """the sync vector, and the Fano decoder on decodable words with corrupted symbols and on noise (time-outs)"""
    out = dict(pr3=np.asarray(rb.pr3() if ref else ob.sync_vector(), np.uint8))
    rng = np.random.default_rng(9)
    for trial in range(20):
        if trial % 2:
            soft = rng.integers(0, 256, 162).astype(np.uint8)  # times out
        else:  # a decodable word with a few corrupted symbols
            data = np.zeros(11, np.uint8)
            data[:7] = td.message_bytes(rng)
            soft = np.where(ob.encode(data)[:162] == 1, 190, 66).astype(np.uint8)
            soft[rng.integers(0, 162, 12)] = 128
        r = rb.fano_decode(soft, maxcycles=200) if ref else ob.fano(soft, maxcycles=200)
        out["t%d/result" % trial] = np.array([r[0], r[2], r[3], r[4]], np.int64)
        # on a time-out the reference returns uninitialised heap for unvisited nodes
        out["t%d/data" % trial] = np.asarray(r[1][:10], np.uint8) if r[0] == 0 else np.zeros(10, np.uint8)
    return out


def sliding_window(ref):
    """sliding_window_stream_to_pdu (fs 375, fl 45000, shift 9 s) fed 1125 samples per work() call"""
    rng = np.random.default_rng(1)
    stream = (rng.standard_normal(45000 + 3 * 3375) + 1j * rng.standard_normal(45000 + 3 * 3375)).astype(np.complex64)
    if ref:
        sw = rb.lib().ref_sw_new(375, 45000, 9, 2)
        out_w = np.zeros(45000, np.complex64)
        wins, pos = [], 0
        while pos < len(stream):
            n = min(1125, len(stream) - pos)
            chunk = np.ascontiguousarray(stream[pos:pos + n])
            if rb.lib().ref_sw_work(sw, chunk.ctypes.data, n, out_w.ctypes.data):
                wins.append(out_w.copy())
            pos += n
        rb.lib().ref_sw_free(sw)
    else:   # window k = stream[k*shift*fs, +fl), one per work() call at most
        wins = [stream[k * 3375:k * 3375 + 45000] for k in range(ob.sliding_window_count(len(stream), 1125))]
    return dict(count=np.array([len(wins)]), windows_sha=np.stack([_sha(w.tobytes()) for w in wins]))


def message_log(ref, golden, golden_windows):
    """the text appended to messagelog.txt for the decodes of two fixtures (a nonlinear and a linear candidate),
    without the clock lines"""
    frames = []
    for name in ("ve3emb_c2", "mix_whales"):
        cands = golden[name + "/cands"].view(ob.CAND_DTYPE).reshape(-1)
        frames.append((name, cands))
    if ref:
        with tempfile.TemporaryDirectory() as d:
            sd = rb.RefSD(logdir=d)
            for name, cands in frames:
                blobs, _, _ = sd.demodulate(golden_windows[name], cands)
                assert len(blobs) == 1
            text = open(os.path.join(d, "messagelog.txt")).read()
            del sd
        # drop the "Start time" line and its blank line, and the per-frame clock lines
        got = "".join(l + "\n" for l in text.split("\n")[2:] if not l.startswith(("Handoff time", "Elapsed time")))
        text = got.rstrip("\n") + "\n\n"
    else:
        from uwspr_b200.binding import format_message_log
        # in both fixtures the first candidate is the one that decodes, and the reference run published one blob
        text = "".join(format_message_log(k + 1, cands[0], golden[name + "/blobs"][0]) for k, (name, cands) in enumerate(frames))
    return dict(text=np.frombuffer(text.encode("latin1"), np.uint8))


def unpacker(ref):
    """random 50-bit payloads (a third with a valid type-1 callsign) through the unpacker: status and text of each,
    and the callsign hash table it builds on the way (type 2 and 3 messages)"""
    import uwspr_b200 as ub
    u = rb.RefUnpacker() if ref else ub.WSPR_unpacker()
    rng = np.random.default_rng(50)
    n = 20000
    status, text = np.zeros(n, np.int64), np.zeros((n, 32), np.uint8)
    for trial in range(n):
        m = rng.integers(0, 256, 7).astype(np.uint8)
        m[6] &= 0xC0
        if trial % 3 == 0:
            m[:4] = np.frombuffer(bytes.fromhex("d42c73eb"), np.uint8)
            m[3] = (m[3] & 0xF0) | int(rng.integers(0, 16))
        s, t = u.unpack(m)
        b = t.encode("latin1")
        assert len(b) < text.shape[1], t
        status[trial] = s
        text[trial, :len(b)] = np.frombuffer(b, np.uint8)
    return dict(status=status, text=text, hashtab_sha=_sha(np.asarray(u.hashtab, np.uint8).tobytes()))


def texts(d):
    return [bytes(r).rstrip(b"\0").decode("latin1") for r in d["text"]]


CASES = dict([("pipeline_md%d_hbw%d_thr%d" % p, (pipeline, p)) for p in PIPELINE_PARAMS] + [
    ("two_signals_and_noise", (two_signals_and_noise, ())), ("sync_and_demodulate_direct", (sync_and_demodulate_direct, ())),
    ("slm_exhaustive", (slm_exhaustive, ())), ("code_tables_and_decoder", (code_tables_and_decoder, ())),
    ("sliding_window", (sliding_window, ())), ("message_log", (message_log, "golden")), ("unpacker", (unpacker, ()))])


def compute(name, ref, golden=None, golden_windows=None):
    fn, args = CASES[name]
    return fn(ref, golden, golden_windows) if args == "golden" else fn(ref, *args)


def reference(name, golden=None, golden_windows=None):
    """the reference's side of case `name`: live where oracle/_ref is built, else as recorded"""
    if rb.available():
        return compute(name, True, golden, golden_windows)
    rec = np.load(RECORDED)
    p = name + "/"
    return {k[len(p):]: rec[k] for k in rec.files if k.startswith(p)}


def assert_same(got, want):
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for k in want:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.shape == b.shape and np.array_equal(a, b), k
