"""The Fano decoder on the device (uwspr_b200_fano_batch, uwspr_b200_decode_device) against the host decoder
(uwspr_b200_fano, uwspr_b200_decode_batch), byte for byte: every counter, the partial path of a time-out, and the
per-candidate outputs of the peak-up/decode loop, early stop included."""
import ctypes as C

import numpy as np
import pytest

from oracle import port_binding as ob
from oracle import testdata as td
from tests.conftest import case_window

pytestmark = pytest.mark.gpu

import uwspr_b200 as ub  # noqa: E402
from uwspr_b200.binding import _p  # noqa: E402

E_PARAM, E_CAPACITY, E_STATE = 1, 3, 5
TIMEOUT_CYCLES = 10000 * 81 + 2   # cycles a decode reports when it gives up at maxcycles 10000


@pytest.fixture(scope="module")
def ctx():
    c = ub.Context(maxdrift=4, max_windows=256, max_candidates=4096)
    yield c
    c.close()


def host_rows(sym, delta=60, maxcycles=10000, nbits=81):
    out = [ub.fano(s, delta=delta, maxcycles=maxcycles, nbits=nbits) for s in sym]
    return (np.array([o[0] for o in out], np.int32), np.stack([o[1] for o in out]),
            np.array([o[2] for o in out], np.uint32), np.array([o[3] for o in out], np.uint32),
            np.array([o[4] for o in out], np.uint32))


def assert_rows_equal(got, want):
    for name, a, b in zip(("status", "data11", "metric", "cycles", "maxnp"), got, want):
        assert a.dtype == b.dtype and np.array_equal(a, b), name


def encoded_rows(rng, n, clean_hi=200, clean_lo=56, max_hits=60):
    """random messages through the encoder (decoder order, no interleaving), 0..max_hits symbols corrupted"""
    rows = np.zeros((n, 162), np.uint8)
    for k in range(n):
        data = np.zeros(11, np.uint8)
        data[:7] = td.message_bytes(rng)
        rows[k] = np.where(ob.encode(data)[:162] == 1, clean_hi, clean_lo)
        hit = rng.integers(0, 162, rng.integers(0, max_hits + 1))
        rows[k, hit] = rng.integers(0, 256, len(hit))
    return rows


def test_fano_batch_on_the_golden_decoder_records(ctx, golden):
    """every decoder call of the recorded reference runs"""
    sym = np.concatenate([golden[str(name) + "/fanos"][:, :162] for name in golden["case_names"]])
    assert len(sym) > 0
    assert_rows_equal(ub.fano_batch(ctx, sym), host_rows(sym))


@pytest.mark.parametrize("maxcycles", [300, 10000])
def test_fano_batch_on_seeded_sequences(ctx, maxcycles):
    """2 000 rows: half encoded messages with 0..60 corrupted symbols, half uniformly random (time-outs with their
    partial paths)"""
    rng = np.random.default_rng(100 + maxcycles)
    sym = np.concatenate([encoded_rows(rng, 1000), rng.integers(0, 256, (1000, 162)).astype(np.uint8)])
    got = ub.fano_batch(ctx, sym, maxcycles=maxcycles)
    want = host_rows(sym, maxcycles=maxcycles)
    assert_rows_equal(got, want)
    assert (want[0] == 0).sum() > 100 and (want[0] == -1).sum() > 100


@pytest.mark.parametrize("nbits", [32, 50, 81])
@pytest.mark.parametrize("delta", [30, 60, 120])
def test_fano_batch_code_lengths_steps_and_constant_inputs(ctx, nbits, delta):
    rng = np.random.default_rng(nbits * 1000 + delta)
    sym = np.concatenate([np.zeros((1, 162), np.uint8), np.full((1, 162), 255, np.uint8), encoded_rows(rng, 94, max_hits=30),
                          rng.integers(0, 256, (32, 162)).astype(np.uint8)])
    assert_rows_equal(ub.fano_batch(ctx, sym, delta=delta, maxcycles=300, nbits=nbits),
                      host_rows(sym, delta=delta, maxcycles=300, nbits=nbits))


def test_fano_batch_device_input_and_domain(ctx):
    import torch
    rng = np.random.default_rng(7)
    sym = np.concatenate([encoded_rows(rng, 64), rng.integers(0, 256, (64, 162)).astype(np.uint8)])
    t = torch.from_numpy(sym).cuda()
    assert_rows_equal(ub.fano_batch(ctx, t, maxcycles=300), host_rows(sym, maxcycles=300))
    for kw in (dict(nbits=31), dict(nbits=82), dict(delta=0), dict(delta=-60), dict(maxcycles=0),
               dict(maxcycles=441870)):   # (441 870*81 + 1)*60 >= 2^31: the threshold would not fit in int32
        with pytest.raises(ub.UwsprError) as e:
            ub.fano_batch(ctx, sym[:4], **kw)
        assert e.value.status == E_PARAM, kw
    assert ub.fano_batch(ctx, sym[:0])[0].size == 0


# ---------------------------------------------------------------------------------------- candidate form
def synthetic_candidates(rng, n, nj):
    """as test_decode_batch_equals_candidate_loop_for_any_thread_count, plus candidates with every gate off: the
    first decodable jiggle varies (or there is none), so early stop shows in idt_used and fano_cycles"""
    refined = np.zeros(n, ub.REFINED_DTYPE)
    jig = np.zeros((n, nj), ub.JIG_DTYPE)
    soft = rng.integers(0, 256, (n, nj, 162)).astype(np.uint8)
    refined["worth_a_try"] = rng.random(n) < 0.9
    jig["gate"] = rng.random((n, nj)) < 0.7
    jig["gate"][rng.random(n) < 0.05] = 0
    inter = ub.deinterleave(np.arange(162, dtype=np.uint8))
    for g in range(n):
        data = np.zeros(11, np.uint8)
        data[:7] = td.message_bytes(rng)
        clean = np.where(ob.encode(data)[:162] == 1, 200, 56).astype(np.uint8)
        tx = np.zeros(162, np.uint8)
        tx[inter] = clean      # the decoder de-interleaves what it is handed
        first_good = rng.integers(0, nj + 2)
        for t in range(first_good, nj):
            s = tx.copy()
            hit = rng.integers(0, 162, rng.integers(0, 12))
            s[hit] = rng.integers(0, 256, len(hit))
            soft[g, t] = s
    return refined, jig, soft


def host_decode(refined, jig, soft):
    n, nj = jig.shape[0], jig.shape[1] if jig.ndim == 2 else 0
    dec, msg, idt, cyc = np.zeros(n, np.uint8), np.zeros((n, 7), np.int8), np.zeros(n, np.int32), np.zeros(n, np.uint32)
    got = ub.load_library().uwspr_b200_decode_batch(_p(refined), _p(jig), _p(soft), n, nj, 0, _p(dec), _p(msg), _p(idt), _p(cyc))
    assert got >= 0
    return got, dec, msg, idt, cyc


def device_decode(ctx, refined, jig, soft, n=None, nj=None, space=ub.binding.HOST):
    """uwspr_b200_decode_device; refined/jig/soft None: the results on the device; else numpy arrays or CUDA tensors"""
    if refined is None:
        args = (None, None, None)
    elif space == ub.binding.DEVICE:
        args = tuple(C.c_void_p(a.data_ptr()) for a in (refined, jig, soft))
    else:
        args = (_p(refined), _p(jig), _p(soft))
    m = max(n, 1)
    dec, msg, idt, cyc = np.zeros(m, np.uint8), np.zeros((m, 7), np.int8), np.zeros(m, np.int32), np.zeros(m, np.uint32)
    got = ctx.L.uwspr_b200_decode_device(ctx.h, *args, space, n, nj, _p(dec), _p(msg), _p(idt), _p(cyc))
    return got, dec[:n], msg[:n], idt[:n], cyc[:n]


def assert_decodes_equal(got, want):
    assert got[0] == want[0]
    for name, a, b in zip(("decoded", "messages7", "idt_used", "fano_cycles"), got[1:], want[1:]):
        assert np.array_equal(a, b), name


@pytest.mark.parametrize("nj", [1, 5, 17])
def test_decode_device_equals_decode_batch(ctx, nj):
    rng = np.random.default_rng(40 + nj)
    refined, jig, soft = synthetic_candidates(rng, 2000, nj)
    want = host_decode(refined, jig, soft)
    got = device_decode(ctx, refined, jig, soft, 2000, nj)
    assert_decodes_equal(got, want)
    assert 200 < want[0] < 2000
    if nj > 1:   # candidates decoded at a later jiggle after earlier gated time-outs: early stop had work to skip
        assert ((want[3] > 0) & (want[4] > TIMEOUT_CYCLES)).any()


def test_decode_device_all_jiggles_time_out(ctx):
    rng = np.random.default_rng(64)
    refined = np.zeros(64, ub.REFINED_DTYPE)
    refined["worth_a_try"] = 1
    jig = np.zeros((64, 17), ub.JIG_DTYPE)
    jig["gate"] = 1
    soft = rng.integers(0, 256, (64, 17, 162)).astype(np.uint8)
    want = host_decode(refined, jig, soft)
    assert want[0] == 0 and np.all(want[4] == np.uint32(17 * TIMEOUT_CYCLES))
    assert_decodes_equal(device_decode(ctx, refined, jig, soft, 64, 17), want)


def test_decode_device_device_pointers_and_empty(ctx):
    import torch
    rng = np.random.default_rng(9)
    refined, jig, soft = synthetic_candidates(rng, 300, 17)
    want = host_decode(refined, jig, soft)
    t = [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).cuda() for a in (refined, jig, soft)]
    assert_decodes_equal(device_decode(ctx, *t, 300, 17, space=ub.binding.DEVICE), want)
    got = ctx.decode(*t, cycles=True)
    assert [(g, bytes(m), i) for g, m, i in got[0]] == \
        [(g, want[2][g].tobytes(), int(want[3][g])) for g in np.flatnonzero(want[1])]
    assert np.array_equal(got[1], want[4])
    assert device_decode(ctx, refined[:0], jig[:0], soft[:0], 0, 17)[0] == 0
    assert ctx.decode(refined[:0], jig[:0], soft[:0]) == []


# ------------------------------------------------------------------ the results of the fine path, on the device
def host_chain(ctx, samples, **kw):
    npk, cands, refined, jig, soft = ctx.coarse_fine(samples, **kw)
    return npk, cands, host_decode(refined, jig, soft)


def test_resident_decode_on_a_synthetic_batch(ctx):
    """coarse_fine without soft symbols + decode_device on what it left == coarse_fine + the host decoder, for
    host-fed and device-resident samples"""
    import torch
    xs, metas = td.synth_batch(256, stream=61)
    npk, cands, want = host_chain(ctx, xs)
    assert want[0] >= 200
    total = ctx.coarse_fine(xs, fetch=False)
    assert total == len(cands)
    assert_decodes_equal(device_decode(ctx, None, None, None, total, 17), want)
    t = torch.from_numpy(xs.reshape(-1).view(np.float32)).cuda()
    assert ctx.coarse_fine((t.data_ptr(), xs.size), nwin=256, fetch=False) == total
    assert_decodes_equal(device_decode(ctx, None, None, None, total, 17), want)
    msgs = ctx.decode()
    assert [(g, bytes(m), i) for g, m, i in msgs] == [(g, want[2][g].tobytes(), int(want[3][g])) for g in np.flatnonzero(want[1])]
    # staged jiggles: the results of fine() on the list coarse() left
    ctx.coarse(xs)
    refined, jig, soft = ctx.fine(xs, jig_first=1, jig_count=16)
    want16 = host_decode(refined[:total], jig[:total], soft[:total])
    assert_decodes_equal(device_decode(ctx, None, None, None, total, 16), want16)


def test_resident_decode_on_the_golden_windows(golden, golden_windows):
    names = ["ve3emb_c2", "test_1500", "rec_150613", "mix_whales"]
    c = ub.Context(maxdrift=0, max_windows=1)
    for name in names:
        x = case_window(name, golden_windows).reshape(1, -1)
        npk, cands, want = host_chain(c, x)
        total = c.coarse_fine(x, fetch=False)
        got = device_decode(c, None, None, None, total, 17)
        assert_decodes_equal(got, want)
        assert got[2][got[1] == 1].tobytes() == golden[name + "/blobs"].tobytes(), name
    c.close()


def test_decode_device_errors():
    c = ub.Context(maxdrift=0, max_windows=24, max_candidates=400)
    assert device_decode(c, None, None, None, 0, 17)[0] == -E_STATE        # no fine call yet
    xs, _ = td.synth_batch(24, stream=52)
    total = c.coarse_fine(xs, fetch=False)
    assert total > 0
    assert device_decode(c, None, None, None, total + 1, 17)[0] == -E_PARAM
    assert device_decode(c, None, None, None, total, 16)[0] == -E_PARAM
    assert device_decode(c, None, None, None, total, 18)[0] == -E_PARAM
    out = c.result_buffers(24)
    c.submit(xs, out)
    assert device_decode(c, None, None, None, total, 17)[0] == -E_STATE    # a submission is outstanding
    c.wait()
    assert device_decode(c, None, None, None, total, 17)[0] >= 0
    rng = np.random.default_rng(3)
    refined, jig, soft = synthetic_candidates(rng, 401, 1)
    assert device_decode(c, refined, jig, soft, 401, 1)[0] == -E_CAPACITY
    assert device_decode(c, refined[:400], jig[:400], soft[:400], 400, 1)[0] >= 0
    # host inputs replace the results of the last fine call on the device
    assert device_decode(c, None, None, None, total, 17)[0] == -E_STATE
    c.coarse(xs)   # a candidate list without fine results
    assert device_decode(c, None, None, None, total, 17)[0] == -E_STATE
    with pytest.raises(ub.UwsprError) as e:
        c.decode()
    assert e.value.status == E_STATE
    c.close()
