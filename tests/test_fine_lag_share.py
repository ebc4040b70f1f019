"""The lag searches of the fine path (stages A and D) evaluate their rotating points with one tone table per
(symbol, tone) shared by every lag (k_fine_lagshare).  UWSPR_B200_NO_LAG_SHARE, read when a context is created,
sends them back through the per-point kernel.  Both must give the same bytes: refined records, jiggles and soft
symbols, and the decoded messages of a multi-channel receiver."""
import numpy as np
import pytest

from oracle import port_binding as ob
from oracle import testdata as td

pytestmark = pytest.mark.gpu

import uwspr_b200 as ub  # noqa: E402


def both(monkeypatch, make, run):
    """run(make()) without, then with the lag-sharing kernel; returns both results and both launch counts"""
    out = {}
    for share in (False, True):
        if share:
            monkeypatch.delenv("UWSPR_B200_NO_LAG_SHARE", raising=False)
        else:
            monkeypatch.setenv("UWSPR_B200_NO_LAG_SHARE", "1")
        obj = make()
        l0 = obj.launch_count()
        res = run(obj)
        out[share] = (res, obj.launch_count() - l0)
        obj.close()
    return out[False], out[True]


def assert_same(a, b):
    assert len(a) == len(b)
    for u, v in zip(a, b):
        assert np.asarray(u).tobytes() == np.asarray(v).tobytes()


def fine_pair(monkeypatch, x, cands, ctx_kw, **fine_kw):
    x = np.asarray(x).reshape(-1, 45000) if np.asarray(x).ndim == 1 else x
    npk = np.array([len(cands)], np.int32)
    (off, loff), (on, lon) = both(monkeypatch, lambda: ub.Context(**ctx_kw),
                                  lambda c: c.fine(x, npk, cands, **fine_kw))
    assert_same(off, on)
    assert lon > loff   # the lag-sharing kernel ran
    return on


def test_seeded_maxdrift4_batch(monkeypatch):
    xs, _ = td.synth_batch(48, stream=31)
    (off, loff), (on, lon) = both(monkeypatch, lambda: ub.Context(maxdrift=4, max_windows=48),
                                  lambda c: c.coarse_fine(xs))
    assert_same(off, on)
    assert lon > loff
    assert on[2]["worth_a_try"].any()
    assert (on[1]["lin_drift"] != 0).any() and (on[1]["lin_drift"] == 0).any()   # rotating and table-path points


def test_shifts_off_both_ends(monkeypatch):
    x, _ = td.synth_window(21, 0, snr_db=-12.0, start=375)
    cands = np.zeros(6, ub.CAND_DTYPE)
    for g, (sh, dr) in enumerate([(-300, 0.5), (-300, 0.0), (0, 1.0), (3200, -2.0), (3700, 3.0), (3700, 0.0)]):
        cands[g]["freq"], cands[g]["sync"], cands[g]["shift"], cands[g]["m_type"], cands[g]["lin_drift"] = 1.4648438, 0.3, sh, 0, dr
    fine_pair(monkeypatch, x, cands, dict(maxdrift=4))


@pytest.mark.parametrize("intended_t", [0, 1])
def test_nonlinear_candidates(monkeypatch, golden_windows, intended_t):
    """t == 0 makes nonlinear points constant-frequency (table path); the intended t makes them rotate"""
    x = golden_windows["ve3emb_c2"]
    cands = np.zeros(3, ub.CAND_DTYPE)
    for g, k in enumerate([0, 57, 124]):
        cands[g]["freq"], cands[g]["sync"], cands[g]["shift"], cands[g]["m_type"] = -0.7324219, 0.5, 256, 1
        cands[g]["V1"], cands[g]["V2"], cands[g]["p1"], cands[g]["p2"] = ob.slm_trajectory(k)
    fine_pair(monkeypatch, x, cands, dict(nonlinear_intended_t=intended_t))


def test_drift0_and_drifting_mix_in_one_call(monkeypatch):
    """one slice holds candidates of both kinds, so each lag-stage kernel skips the other's"""
    xs = np.stack([td.synth_window(40 + w, 0, snr_db=-8.0)[0] for w in range(3)])
    cands = np.zeros(3 * 12, ub.CAND_DTYPE)
    rng = np.random.default_rng(5)
    for g in range(len(cands)):
        cands[g]["freq"] = np.float32(rng.uniform(-20, 20))
        cands[g]["sync"] = 0.3
        cands[g]["shift"] = int(rng.integers(-2, 30)) * 128
        cands[g]["lin_drift"] = 0.0 if g % 3 == 0 else np.float32(rng.uniform(-4, 4))
    npk = np.array([12, 12, 12], np.int32)
    (off, loff), (on, lon) = both(monkeypatch, lambda: ub.Context(maxdrift=4, max_windows=3),
                                  lambda c: c.fine(xs, npk, cands))
    assert_same(off, on)
    assert lon > loff


def test_odd_stride_stream(monkeypatch):
    """windows 9 s apart on one stream: odd sample offsets, windows not 16-byte aligned"""
    stride, nwin = 9 * 375, 9
    n = 45000 + (nwin - 1) * stride
    rng = np.random.default_rng(8)
    stream = ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * np.sqrt(0.15 / 10 ** (-1.2) / 2.0))
    msg = td.message_bytes(np.random.default_rng(4))
    stream[7001:7001 + 162 * 256] += td.modulate(ob.channel_symbols(msg), f0=2.5, drift=0.0, start=0, fl=162 * 256)
    stream = stream.astype(np.complex64)
    (off, loff), (on, lon) = both(monkeypatch, lambda: ub.Context(maxdrift=2, max_windows=nwin),
                                  lambda c: c.coarse_fine(stream, nwin=nwin, stride=stride))
    assert_same(off, on)
    assert lon > loff
    assert on[0].sum() > 0


def test_staged_first_jiggle(monkeypatch):
    xs, _ = td.synth_batch(24, stream=77)
    ctx = ub.Context(maxdrift=4, max_windows=24)
    npk, cands = ctx.coarse(xs)
    ctx.close()
    (off, loff), (on, lon) = both(monkeypatch, lambda: ub.Context(maxdrift=4, max_windows=24),
                                  lambda c: c.fine(xs, npk, cands, jig_first=0, jig_count=1))
    assert_same(off, on)
    assert lon > loff


def test_array_receiver_messages(monkeypatch):
    nwin, stride = 12, 9 * 375
    n = 45000 + (nwin - 1) * stride
    rng = np.random.default_rng(12)
    x = ((rng.standard_normal((3, n)) + 1j * rng.standard_normal((3, n))) * np.sqrt(0.15 / 10 ** (-1.2) / 2.0))
    for c, (start, f0, seed) in enumerate([(5000, -4.0, 1), (30000, 6.3, 2), (38000, 2.2, 4)]):
        msg = td.message_bytes(np.random.default_rng(seed))
        x[c, start:start + 162 * 256] += td.modulate(ob.channel_symbols(msg), f0=f0, drift=0.0, start=0, fl=162 * 256)
    x = x.astype(np.complex64)

    def run(rx):
        got = []
        for lo in range(0, n, 20_000):
            got += rx.push(x[:, lo:lo + 20_000])
        got += rx.push(x[:, :0], flush=True)
        return [(c, w, bytes(m), cand.tobytes()) for c, w, m, cand in got]

    (off, loff), (on, lon) = both(monkeypatch, lambda: ub.ArrayReceiver(3, maxdrift=2, shift=9, batch_windows=5), run)
    assert off == on
    assert len(on) >= 3
    assert lon > loff
