"""CPU-side checks of the product: the C-ABI library builds for sm_100a, loads, exports every
symbol include/uwspr_b200.h declares, fails loudly without a GPU; the host-side decoder
(deinterleave, Fano, peak-up/decode loop) matches the oracle and the golden vectors."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import uwspr_b200 as ub
from oracle import port_binding as ob
from oracle import testdata as td
from tests.golden import reference_cases as rc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    return ub.load_library()


def test_header_symbols_all_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "uwspr_b200.h")).read()
    declared = sorted(set(re.findall(r"UWSPR_B200_API\s+[\w\s\*]+?\b(uwspr_b200_\w+)\s*\(", hdr)))
    assert declared == sorted(ub.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name


def test_struct_layouts_match_reference_candidate_t():
    assert ub.CAND_DTYPE.itemsize == 48
    assert [ub.CAND_DTYPE.fields[n][1] for n in ("freq", "snr", "drift", "sync", "shift", "m_type", "lin_drift", "V1", "V2", "p1", "p2")] == \
        [0, 4, 8, 12, 16, 20, 24, 24, 32, 40, 44]
    assert ub.REFINED_DTYPE.itemsize == 24 and ub.JIG_DTYPE.itemsize == 16


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(ub.UwsprError) as e:
        ub.Context()
    assert e.value.status == 2  # UWSPR_B200_E_CUDA


def test_parameter_domain_checked_before_cuda(lib):
    for kw in (dict(halfbandwidth=188), dict(spb=128), dict(fl=1000), dict(maxfreqs=0)):
        with pytest.raises(ub.UwsprError) as e:
            ub.Context(**kw)
        assert e.value.status == 1, kw


def test_host_decoder_matches_oracle(lib, golden):
    assert np.array_equal(ub.deinterleave(np.arange(162, dtype=np.uint8)), golden["kat/deinterleave_of_iota"])
    rng = np.random.default_rng(11)
    for trial in range(30):
        if trial % 3 == 0:
            soft = rng.integers(0, 256, 162).astype(np.uint8)
        else:
            data = np.zeros(11, np.uint8)
            data[:7] = td.message_bytes(rng)
            soft = np.where(ob.encode(data)[:162] == 1, 185, 71).astype(np.uint8)
            soft[rng.integers(0, 162, 5 * (trial % 7))] = rng.integers(0, 256)
        a = ub.fano(soft, maxcycles=300)
        b = ob.fano(soft, maxcycles=300)
        assert a[0] == b[0] and a[2:] == b[2:]
        assert np.array_equal(a[1][:10], b[1][:10])


def test_decode_loop_on_golden_fano_records(lib, golden):
    """the decoder records of the reference run: same verdict, metric, cycles, message"""
    for name in golden["case_names"]:
        for rec in golden[str(name) + "/fanos"]:
            sym = rec[:162]
            r, data, metric, cycles, maxnp = ub.fano(sym)
            want = np.frombuffer(rec[176:192].tobytes(), dtype=np.uint32)
            assert r == int(np.frombuffer(rec[176:180].tobytes(), np.int32)[0])
            assert (metric, cycles, maxnp) == (int(want[1]), int(want[2]), int(want[3]))
            if r == 0:
                assert np.array_equal(data[:10], rec[162:172])


def test_shard_ranges():
    from uwspr_b200.sharding import shard_range, stream_span
    for n in (0, 1, 7, 100000):
        for world in (1, 2, 4, 8):
            parts = [shard_range(n, r, world) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == n
            assert all(parts[i][1] == parts[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in parts]
            assert max(sizes) - min(sizes) <= 1
    assert stream_span(2, 5, 22500, 45000) == (45000, 4 * 22500 + 45000)


def test_message_log_text_matches_reference_file(lib, golden, golden_windows):
    """the reference block appends to ./messagelog.txt on every decode (sync_and_demodulate_impl.cc:507-526);
    the same candidates and blobs through uwspr_b200_format_message_log give the same lines (the reference's
    file live where oracle/_ref is built, else as recorded)"""
    want = rc.reference("message_log", golden, golden_windows)
    rc.assert_same(rc.compute("message_log", False, golden, golden_windows), want)
    assert bytes(want["text"]).decode("latin1").count("Frame: ") == 2


def test_unpacker_known_answers(lib):
    u = ub.WSPR_unpacker()
    f = lambda h: np.frombuffer(bytes.fromhex(h), np.uint8)  # noqa: E731
    assert u.unpack(f("d42c73eb3a7780")) == (0, "VE3EMB FN25 30")   # examples/VE3EMB.c2, test_1500_Hz.wav
    assert u.unpack(f("d42c73eb0d1840")) == (0, "VE3EMB FN42 33")   # examples/150613_1920.wav


def test_unpacker_against_reference_all_message_types(lib):
    """random 50-bit payloads cover type 1, type 2 (prefix/suffix) and type 3 (hashed call) paths, with the
    callsign hash table evolving identically on both sides (lib/helpers.cc:494-590); the reference answers live
    where oracle/_ref is built, else as recorded"""
    want = rc.reference("unpacker")
    rc.assert_same(rc.compute("unpacker", False), want)
    kinds = {"3" if t.startswith("<") else "2" if "/" in t else "1" for t in rc.texts(want) if t}
    assert kinds == {"1", "2", "3"}


def test_decode_batch_equals_candidate_loop_for_any_thread_count(lib):
    """uwspr_b200_decode_batch == one uwspr_b200_decode_candidate per candidate == the oracle's decoder
    driven by the reference's gate (sync_and_demodulate_impl.cc:457-490), for 1, 3 and all host threads"""
    rng = np.random.default_rng(5)
    n, nj = 150, 17
    refined = np.zeros(n, ub.REFINED_DTYPE)
    jig = np.zeros((n, nj), ub.JIG_DTYPE)
    soft = rng.integers(0, 256, (n, nj, 162)).astype(np.uint8)
    sent = np.zeros((n, 7), np.uint8)
    refined["worth_a_try"] = rng.random(n) < 0.9
    jig["gate"] = rng.random((n, nj)) < 0.7
    for g in range(n):
        data = np.zeros(11, np.uint8)
        data[:7] = sent[g] = td.message_bytes(rng)
        clean = np.where(ob.encode(data)[:162] == 1, 200, 56).astype(np.uint8)
        # interleave: the decoder de-interleaves what it is handed
        tx = np.zeros(162, np.uint8)
        tx[ub.deinterleave(np.arange(162, dtype=np.uint8))] = clean
        first_good = rng.integers(0, nj + 6)          # >= nj: never decodable
        for t in range(first_good, nj):
            s = tx.copy()
            hit = rng.integers(0, 162, rng.integers(0, 12))
            s[hit] = rng.integers(0, 256, len(hit))
            soft[g, t] = s
    want = {}
    for g in range(n):
        if not refined["worth_a_try"][g]:
            continue
        for t in range(nj):
            if not jig["gate"][g, t]:
                continue
            r, data, *_ = ob.fano(ub.deinterleave(soft[g, t]))
            if r == 0:
                want[g] = (bytes(data[:7]), t)
                break
    assert 30 < len(want) < n
    L = lib
    single = {}
    for g in range(n):
        msg = np.zeros(7, np.int8)
        idt = C.c_int32()
        if L.uwspr_b200_decode_candidate(ub.binding._p(refined[g:g + 1]), ub.binding._p(jig[g]), ub.binding._p(soft[g]),
                                         nj, ub.binding._p(msg), C.byref(idt), None):
            single[g] = (msg.tobytes(), idt.value)
    assert single == want
    for nthreads in (1, 3, 0):
        got = {g: (m.tobytes(), t) for g, m, t in ub.decode_candidates(refined, jig, soft, nthreads=nthreads)}
        assert got == want
    assert ub.decode_candidates(refined[:0], jig[:0], soft[:0]) == []


def test_packer_and_channel_symbols_round_trip(lib, golden):
    """transmit direction: text -> message -> channel symbols.  Known answers from the reference fixtures,
    the encoder against the oracle's restatement of lib/Fano.cc, and text -> pack -> unpack == text with both
    this library's unpacker and the compiled reference's"""
    assert ub.pack_type1("VE3EMB", "FN25", 30).tobytes().hex() == "d42c73eb3a7780"
    assert ub.pack_type1("ve3emb", "fn42", 33).tobytes().hex() == "d42c73eb0d1840"
    assert np.array_equal(ub.channel_symbols(golden["kat/encode_in"][:7]), ob.channel_symbols(golden["kat/encode_in"][:7]))
    rng = np.random.default_rng(3)
    letters = "ABCDEFGHIJKLMNOPQRSTUVWXYZ"
    u = ub.WSPR_unpacker()
    from oracle import ref_binding as rb
    ru = rb.RefUnpacker() if rb.available() else None
    for trial in range(300):
        n_suffix = int(rng.integers(1, 4))
        if trial % 2:   # digit second: "K1ABC"
            call = letters[rng.integers(26)] + str(rng.integers(10)) + "".join(letters[rng.integers(26)] for _ in range(n_suffix))
        else:           # digit third: "VE3EMB"
            call = letters[rng.integers(26)] + letters[rng.integers(26)] + str(rng.integers(10)) + \
                "".join(letters[rng.integers(26)] for _ in range(n_suffix))
        grid = letters[rng.integers(18)] + letters[rng.integers(18)] + str(rng.integers(10)) + str(rng.integers(10))
        dbm = int(rng.choice([0, 3, 7, 10, 13, 17, 20, 23, 27, 30, 33, 37, 40, 43, 47, 50, 53, 57, 60]))
        msg = ub.pack_type1(call, grid, dbm)
        assert msg[6] & 0x3f == 0
        want = "%s %s %2d" % (call, grid, dbm)   # the reference prints the power two wide
        assert u.unpack(msg) == (0, want)
        if ru is not None:
            assert ru.unpack(msg)[1] == want
        assert np.array_equal(ub.channel_symbols(msg), ob.channel_symbols(msg))
    for bad in (("TOOLONGCALL", "FN25", 30), ("VE3EMB", "ZZ99", 30), ("VE3EMB", "FN25", 31), ("ABCDEF", "FN25", 30)):
        with pytest.raises(ub.UwsprError):
            ub.pack_type1(*bad)


def test_c2_reader(lib, golden_windows, tmp_path):
    """uwspr.c2file_source's reader: header fields, conjugation on load (c2file_source_impl.cc:91), short files refused"""
    import struct
    x = golden_windows["ve3emb_c2"]
    raw = np.empty((45000, 2), "<f4")
    raw[:, 0], raw[:, 1] = x.real, -x.imag     # what the file holds: the reader flips the sign back
    path = tmp_path / "t.c2"
    path.write_bytes(struct.pack("<14sid", b"150426_0918.c2", 2, 10.1387) + raw.tobytes())
    iq, name, typ, freq = ub.read_c2(str(path))
    assert (name, typ, freq) == ("150426_0918.c2", 2, 10.1387)
    assert iq.tobytes() == x.tobytes()
    (tmp_path / "short.c2").write_bytes(path.read_bytes()[:-8])
    with pytest.raises(ub.UwsprError):
        ub.read_c2(str(tmp_path / "short.c2"))
    with pytest.raises(ub.UwsprError):
        ub.read_c2(str(tmp_path / "missing.c2"))


def test_frontend_and_batch_decoder_argument_checks(lib):
    """argument errors are statuses, reported before any CUDA call (so they can be checked without a GPU)"""
    audio = np.zeros(64, np.float32)
    taps = np.ones(4, np.float32)
    with pytest.raises(ub.UwsprError):
        ub.frontend(audio, taps=np.zeros(0, np.float32))          # no taps
    with pytest.raises(ub.UwsprError):
        ub.frontend(audio, taps=taps, decim=0)                     # bad decimation
    with pytest.raises(ub.UwsprError):
        ub.frontend(audio, taps=taps, fs_in=0.0)                   # bad rate
    with pytest.raises(ub.UwsprError):
        ub.frontend(audio, taps=taps, delay=-1)
    L = lib
    r = np.zeros(1, ub.REFINED_DTYPE)
    j = np.zeros((1, 17), ub.JIG_DTYPE)
    s = np.zeros((1, 17, 162), np.uint8)
    d = np.zeros(1, np.uint8)
    m = np.zeros(7, np.int8)
    P = ub.binding._p
    assert L.uwspr_b200_decode_batch(P(r), P(j), P(s), 1, 18, 0, P(d), P(m), None, None) < 0     # jig_count > 17
    assert L.uwspr_b200_decode_batch(P(r), P(j), P(s), -1, 17, 0, P(d), P(m), None, None) < 0
    assert L.uwspr_b200_decode_batch(None, None, None, 0, 17, 0, None, None, None, None) == 0   # nothing to do
    assert L.uwspr_b200_decode_batch(P(r), P(j), P(s), 1, 17, 0, None, P(m), None, None) < 0     # no output
    assert L.uwspr_b200_decode_batch(P(r), P(j), P(s), 1, 17, 2, P(d), P(m), None, None) == 0 and d[0] == 0
