"""Parity of the device chain across the parameter domain uwspr_b200_create accepts, and across the fine path's
slices of 16 384 candidates.

Part 1: one context per row (cf, fs, maxdrift, threshold, halfbandwidth, maxfreqs at and near the edges of what
create accepts).  Every candidate record of seeded windows equals the oracle's post-FFT chain on the GPU's own
spectrogram; up to 8 candidates per context, plus hand-made nonlinear ones, equal the oracle's refinement, every
jiggle and all 162 soft symbols, with nonlinear_intended_t 0 and 1.  Each row asserts, through ctx.info, that it
reached the kernel path it is there for.  The largest accepted values are found by stepping a parameter up until
create refuses it, and checked against a restatement of build_tables' rules (capi.cu).

Part 2: the fine path runs a chunk's candidates in slices of 16 384 on one workspace.  Chunks of more than 2.5
slices, device-resident and host-fed, equal one small call on the same windows copy for copy; a caller-supplied
list of more candidates per window than the context's maxcand is refined in full; slices whose candidate counts
are 1 and 15 modulo 16 (the lag-sharing kernel pairs symbols 160 and 161 of 16 candidates) equal the oracle.
"""
import math

import numpy as np
import pytest

from oracle import port_binding as ob
from oracle import testdata as td
from oracle.verify import cands_equal_exact, oracle_on_gpu_ps

pytestmark = pytest.mark.gpu

import uwspr_b200 as ub  # noqa: E402

SLICE = 16384                 # candidates per fine-path slice (capi.cu: uw_fine_work_alloc)
HZ_PER_BIN = 375.0 / 512.0    # bin width of the synthetic 375-sps signals, whatever fs the context is told

# refusal texts of build_tables (capi.cu)
R_FINPB = "fewer than 3 pass-band bins"
R_IFR = "reaches past the spectrum"
R_BIN = "bin offsets depend on the bin"
R_SPAN = "drift hypotheses span too many bins"
R_TILE = "too many bins / sequences for one tile"
R_RANGE = "would index outside the spectrum"


# ---------------------------------------------------------------------------------------------------------------
# build_tables restated: the offset sequences of every drift hypothesis and the rules that refuse a parameter set


def _slm_drift(V1, V2, p2, cf, t):
    """slm_frequency_drift_host (capi.cu) with p1 = 0: double inside, fp32 result"""
    q1, q2 = V1 * t, V2 * t + p2
    sign = 1.0 if (q1 * V1 + q2 * V2) > 0 else -1.0
    num, den = abs(V1 * q1 + V2 * q2), math.sqrt(q1 * q1 + q2 * q2)
    if den == 0:
        return np.float32(0.0)
    return np.float32(-sign * num / den * float(np.float32(cf)) / 1500.0)


def tables(fs=375, spb=256, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, **_):
    """what build_tables makes of these parameters: a dict (n_unique, tile_w, maxcand, the set of distinct offset
    sequences ...) or the text of the rule that refuses them"""
    size = 2 * spb
    df = np.float32(np.float32(fs) / np.float32(size))
    m = size // 2
    hpbm = int(math.ceil(np.float32(np.float32(halfbandwidth) / df)))
    if 2 * hpbm < 3:
        return R_FINPB
    maxcand = min(maxfreqs, (2 * hpbm - 1) // 2)
    ifr = np.arange(m - hpbm - 1, m + hpbm + 1)
    if ifr[0] < 0:
        return R_IFR
    k = np.arange(162)
    seqs = []
    for h in range(2 * maxdrift + 1):
        # FDR_impl.cc:353, a double expression truncated
        x = ((k - 81.0) / 81.0 * float(h - maxdrift)) / (2.0 * float(df))
        seqs.append(np.trunc(ifr[:, None] + x[None, :]).astype(np.int64) - ifr[:, None])
    t = (k * 111 // 162).astype(np.float64)
    for tr in range(125):
        V1, V2, p2 = float((tr // 5) % 5) - 2.0, float(tr // 25) - 2.0, (tr % 5) * 200 + 50
        q = np.array([_slm_drift(V1, V2, p2, cf, tt) for tt in t], np.float32) / df          # :384-385, fp32
        s = (ifr[:, None].astype(np.float32) + q[None, :]).astype(np.float32)
        seqs.append(np.trunc(s).astype(np.int64) - ifr[:, None])
    for off in seqs:
        if (off != off[0]).any():
            return R_BIN
    seqs = [tuple(off[0]) for off in seqs]
    every = np.array(seqs)
    if np.abs(every).max() > 100:
        return R_SPAN
    uniq = set(seqs)
    off_min, off_max = min(0, int(every.min())), max(0, int(every.max()))
    tile_w = 11 + off_max - off_min
    if tile_w > 40 or len(uniq) > 192:
        return R_TILE
    lo = min(m - hpbm - 3, (m - hpbm + 1) - 5 + off_min)
    hi = max(m + hpbm + 2, (m + hpbm - 2) + 5 + off_max)
    if lo < 0 or hi > size - 1:
        return R_RANGE
    return dict(n_unique=len(uniq), seqs=uniq, tile_w=tile_w, maxcand=maxcand, n_lin=2 * maxdrift + 1, hpbm=hpbm,
                df=float(df))


def refusal(**kw):
    """None when create accepts the parameters, else the text of its E_PARAM refusal"""
    try:
        ctx = ub.Context(**kw)
    except ub.UwsprError as e:
        assert e.status == 1, str(e)
        return str(e)
    ctx.close()
    return None


_bounds = {}


def last_accepted(name, start, step, **kw):
    """Steps `name` up from `start` until create refuses it for a rule that bounds it from above; isolated values
    whose offsets depend on the bin (hazard H6) are refused on the way and stepped over.  Coarse steps of `step`,
    then steps of 1.  Returns (largest accepted value below the first such refusal, that refusal's value, text)."""
    key = (name, start, step, tuple(sorted(kw.items())))
    if key in _bounds:
        return _bounds[key]
    assert refusal(**{name: start}, **kw) is None
    v = start
    while True:
        why = refusal(**{name: v + step}, **kw)
        if why is not None and R_BIN not in why:
            break
        v += step
    last, first_bad = None, None
    for u in range(v, v + step + 1):
        why = refusal(**{name: u}, **kw)
        if why is None:
            last = u
        elif R_BIN not in why:
            first_bad = u
            break
    assert last is not None and first_bad is not None
    _bounds[key] = (last, first_bad, why)
    return _bounds[key]


# ---------------------------------------------------------------------------------------------------------------
# inputs and checks


def window(seed, f0s, drifts, snr_db=-10.0):
    """seeded window: one WSPR frame per (f0, drift), independent payloads and starts, in complex AWGN (2500 Hz
    SNR convention of oracle/testdata.py for a unit-amplitude frame)"""
    rng = np.random.default_rng([20240611, seed])
    x = np.zeros(45000, np.complex128)
    for f0, dr in zip(f0s, drifts):
        msg = td.message_bytes(rng)
        x += td.modulate(ob.channel_symbols(msg), f0=float(f0), drift=float(dr), start=int(rng.integers(0, 2600)))
    s2 = (375.0 / 2500.0) / 10 ** (snr_db / 10.0)
    x += np.sqrt(s2 / 2.0) * (rng.standard_normal(45000) + 1j * rng.standard_normal(45000))
    return x.astype(np.complex64)


def spread(seed, hpbm, maxdrift, nsig):
    """nsig signals spread over the pass band of a context with hpbm half-band bins; drifts up to maxdrift Hz"""
    band = hpbm * HZ_PER_BIN - 4.0
    f0s = np.linspace(-band, band, nsig) if nsig > 1 and band > 0 else np.zeros(1)
    rng = np.random.default_rng(seed)
    drifts = rng.uniform(-1.0, 1.0, len(f0s)) * min(maxdrift, 8)
    return window(seed, f0s, drifts)


def assert_fine_rows(refined, jig, soft, x, cands, cf):
    """refined records, jiggles and soft symbols of `cands` (all from window x) equal the oracle's, bit for bit"""
    o_ref, o_jigs = ob.demodulate_full(x, cands, cf=cf)
    for g in range(len(cands)):
        assert refined["f1"][g].tobytes() == o_ref[g, 0].tobytes()
        assert refined["shift1"][g] == int(o_ref[g, 1])
        assert refined["drift1"][g].tobytes() == o_ref[g, 2].tobytes()
        assert refined["sync1"][g].tobytes() == o_ref[g, 3].tobytes()
        assert refined["worth_a_try"][g] == int(o_ref[g, 4])
        if not refined["worth_a_try"][g]:
            assert not soft[g].any() and not jig["gate"][g].any()
            continue
        for t, call in enumerate(o_jigs[g]):
            assert jig["shift"][g, t] == call.shift_in
            assert jig["sync"][g, t].tobytes() == np.float32(call.sync_out).tobytes()
            assert np.array_equal(soft[g, t], np.frombuffer(bytes(call.symbols), np.uint8))
            y = soft[g, t].astype(np.float32) - 128.0
            rms = np.float32(np.sqrt(np.float64(np.float32((y * y).sum())) / 162.0))
            assert jig["rms"][g, t] == rms
            assert jig["gate"][g, t] == int(call.sync_out > np.float32(0.12) and rms > np.float32(40.625))


def fine_against_oracle(ctx, x, cands, cf):
    refined, jig, soft = ctx.fine(x.reshape(1, -1), np.array([len(cands)], np.int32), cands)
    assert_fine_rows(refined, jig, soft, x, cands, cf)
    return refined, jig, soft


def nonlinear_cands(freq, shift):
    """hand-made straight-line-model candidates (trajectories 0, 57, 124 of slm.cc's generator)"""
    c = np.zeros(3, ub.CAND_DTYPE)
    for g, k in enumerate([0, 57, 124]):
        c[g]["freq"], c[g]["sync"], c[g]["shift"], c[g]["m_type"] = freq, 0.5, shift, 1
        c[g]["V1"], c[g]["V2"], c[g]["p1"], c[g]["p2"] = ob.slm_trajectory(k)
    return c


# ---------------------------------------------------------------------------------------------------------------
# part 1: one context per row


def _cf_max():
    return dict(cf=last_accepted("cf", 3000, 128, maxdrift=2)[0], maxdrift=2)


def _maxdrift_max():
    return dict(maxdrift=last_accepted("maxdrift", 16, 1)[0])


def _halfbandwidth_max():
    return dict(halfbandwidth=last_accepted("halfbandwidth", 100, 16, maxfreqs=256)[0], maxfreqs=256)


def _differs_from_cf1500(info, t):
    base = tables(**dict(t["kw"], cf=1500))
    return info.n_unique == t["n_unique"] and t["seqs"] != base["seqs"]


# (id naming the path, parameters or a function finding them, the path reached, nonlinear candidates expected,
#  signals per window)
ROWS = [
    ("cf0-trajectories-collapse-to-drift0", dict(cf=0, maxdrift=2),
     lambda i, t: _differs_from_cf1500(i, t) and i.n_unique == i.n_lin, False, 3),
    ("cf0-threshold0-ratio-exactly-1", dict(cf=0, maxdrift=0, threshold=0),
     lambda i, t: _differs_from_cf1500(i, t) and i.n_unique == 1, True, 3),
    ("cf-1500-mirrored-offsets", dict(cf=-1500, maxdrift=2), _differs_from_cf1500, False, 3),
    ("cf501-offsets-other-than-cf1500", dict(cf=501, maxdrift=2), _differs_from_cf1500, False, 3),
    ("cf3000-wider-tile", dict(cf=3000, maxdrift=2), lambda i, t: _differs_from_cf1500(i, t) and t["tile_w"] > 17, False, 3),
    ("cf-largest-accepted-tile40", _cf_max, lambda i, t: _differs_from_cf1500(i, t) and t["tile_w"] == 40, False, 3),
    ("fs300-df0.586", dict(fs=300, halfbandwidth=10, maxdrift=2),
     lambda i, t: i.df == np.float32(300 / 512) and i.hpbm == 18 and i.n_unique == t["n_unique"], False, 3),
    ("fs750-df1.465", dict(fs=750, halfbandwidth=40, maxdrift=2),
     lambda i, t: i.df == np.float32(750 / 512) and i.hpbm == 28 and i.n_unique == t["n_unique"], False, 3),
    ("maxdrift16-nlin33-two-ballots", dict(maxdrift=16), lambda i, t: i.n_lin == 33, False, 3),
    ("maxdrift-largest-accepted-two-ballots", _maxdrift_max, lambda i, t: i.n_lin > 32 and t["tile_w"] == 40, False, 3),
    ("threshold0-no-group-skip", dict(threshold=0, maxdrift=2), lambda i, t: True, True, 3),
    ("threshold-5-no-group-skip", dict(threshold=-5, maxdrift=2), lambda i, t: True, True, 3),
    ("halfbandwidth1-maxcand1", dict(halfbandwidth=1), lambda i, t: i.max_cand_per_window == 1 and i.finpb == 4, False, 1),
    ("halfbandwidth-largest-accepted-maxcand-over-200", _halfbandwidth_max,
     lambda i, t: i.max_cand_per_window > 200, False, 16),
    ("maxfreqs1-maxcand1", dict(maxfreqs=1, maxdrift=1), lambda i, t: i.max_cand_per_window == 1, False, 3),
]


@pytest.mark.parametrize("row", ROWS, ids=[r[0] for r in ROWS])
def test_row_against_the_oracle(row):
    name, kw, reached, want_nonlinear, nsig = row
    kw = kw() if callable(kw) else dict(kw)
    full = dict(dict(fs=375, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10), **kw)
    t = tables(**full)
    assert isinstance(t, dict), t
    t["kw"] = full
    cf, nwin = full["cf"], 2
    # room for the three hand-made candidates below where maxcand is 1
    cap = nwin * t["maxcand"] + 3
    ctx = ub.Context(max_windows=nwin, max_candidates=cap, **kw)
    info = ctx.info
    assert info.n_unique == t["n_unique"] and info.n_lin == t["n_lin"] and info.max_cand_per_window == t["maxcand"]
    assert reached(info, t), name
    xs = np.stack([spread(100 * ROWS.index(row) + w, t["hpbm"], full["maxdrift"], nsig) for w in range(nwin)])
    ctx.set_debug(True)
    npk, cands, refined, jig, soft = ctx.coarse_fine(xs)
    base = np.concatenate([[0], np.cumsum(npk)])
    of = ob.OracleFDR(**{k: full[k] for k in ("fs", "maxdrift", "maxfreqs", "halfbandwidth", "cf", "threshold")})
    for w in range(nwin):
        want, *_ = oracle_on_gpu_ps(of, ctx, xs[w], w)
        assert npk[w] == len(want) <= info.max_cand_per_window
        assert cands_equal_exact(cands[base[w]:base[w + 1]], want), w
    assert npk.sum() >= 1
    nonlinear = int((cands["m_type"] == 1).sum())
    if want_nonlinear:
        assert nonlinear > 0
    print("%s: n_lin %d, n_unique %d (cf=1500: %d), tile_w %d, max_cand_per_window %d, df %.6f, candidates %s, "
          "nonlinear %d" % (name, info.n_lin, info.n_unique, tables(**dict(full, cf=1500))["n_unique"], t["tile_w"],
                            info.max_cand_per_window, info.df, list(npk), nonlinear))
    # refinement and soft symbols: up to 4 coarse candidates per window, then hand-made nonlinear ones
    for w in range(nwin):
        k = min(4, int(npk[w]))
        sl = slice(base[w], base[w] + k)
        assert_fine_rows(refined[sl], jig[sl], soft[sl], xs[w], cands[sl], cf)
    c0 = cands[0]
    hand = nonlinear_cands(c0["freq"], c0["shift"])
    fine_against_oracle(ctx, xs[0], hand, cf)
    ctx.close()
    ctx1 = ub.Context(max_windows=nwin, max_candidates=cap, nonlinear_intended_t=1, **kw)
    ob.lib().orc_set_nonlinear_intended_t(1)
    try:
        fine_against_oracle(ctx1, xs[0], hand, cf)
        for w in range(nwin):
            sub = cands[base[w]:base[w] + min(4, int(npk[w]))]
            if len(sub):
                fine_against_oracle(ctx1, xs[w], sub, cf)
    finally:
        ob.lib().orc_set_nonlinear_intended_t(0)
    ctx1.close()


def test_boundaries_are_where_the_table_rules_put_them():
    """the largest accepted cf (maxdrift 2), maxdrift (cf 1500) and halfbandwidth (maxfreqs 256), found by stepping
    up until create refuses, are the values build_tables' rules put the boundary at; values in between that create
    refuses are refused for bin-dependent offsets (H6), by the restated rules too"""
    for name, start, step, kw, rule in (("cf", 3000, 128, dict(maxdrift=2), R_TILE), ("maxdrift", 16, 1, {}, R_TILE),
                                        ("halfbandwidth", 100, 16, dict(maxfreqs=256), R_RANGE)):
        last, bad, why = last_accepted(name, start, step, **kw)
        print("%s: largest accepted %d, refused at %d: %s" % (name, last, bad, why))
        assert rule in why
        assert isinstance(tables(**{name: last}, **kw), dict)
        assert tables(**{name: bad}, **kw) == rule
        for v in range(last + 1, bad):
            assert tables(**{name: v}, **kw) == R_BIN
    assert last_accepted("maxdrift", 16, 1)[0] == 21
    assert last_accepted("halfbandwidth", 100, 16, maxfreqs=256)[0] == 181   # H3
    # the smallest halfbandwidth: 1 Hz gives 4 pass-band bins, 0 is refused before the tables are built
    assert refusal(halfbandwidth=0) is not None and tables(halfbandwidth=1)["maxcand"] == 1


@pytest.mark.parametrize("cf", [500, -1, 1581])
def test_offsets_that_depend_on_the_bin_are_refused(cf):
    """H6: at these centre frequencies the reference's truncated bin offset of some trajectory differs between bins
    of the search range; the coarse kernel keeps one offset sequence per hypothesis, so create refuses them"""
    why = refusal(cf=cf)
    assert why is not None and R_BIN in why
    assert tables(cf=cf) == R_BIN
    assert refusal(cf=cf + 1) is None or tables(cf=cf + 1) == R_BIN


# ---------------------------------------------------------------------------------------------------------------
# part 2: fine slices past 16 384 candidates


def busy(seed, nsig=32):
    """a window with many candidates at halfbandwidth 100: nsig signals over +-92 Hz"""
    rng = np.random.default_rng([7, seed])
    f0s = np.linspace(-92.0, 92.0, nsig) + rng.uniform(-1.5, 1.5, nsig)
    return window(1000 + seed, f0s, rng.uniform(-1.0, 1.0, nsig), snr_db=-8.0)


WIDE = dict(halfbandwidth=100, maxdrift=1)


@pytest.fixture(scope="module")
def distinct():
    """three busy windows, their results from one small call, checked against the oracle"""
    xs = np.stack([busy(s) for s in range(3)])
    ctx = ub.Context(max_windows=3, **WIDE)
    ctx.set_debug(True)
    res = ctx.coarse_fine(xs)
    npk, cands, refined, jig, soft = res
    base = np.concatenate([[0], np.cumsum(npk)])
    of = ob.OracleFDR(**WIDE)
    for w in range(3):
        want, *_ = oracle_on_gpu_ps(of, ctx, xs[w], w)
        assert cands_equal_exact(cands[base[w]:base[w + 1]], want), w
        sl = slice(base[w], base[w] + 6)
        assert_fine_rows(refined[sl], jig[sl], soft[sl], xs[w], cands[sl], 1500)
    assert refined["worth_a_try"].any()
    ctx.close()
    return xs, res


def assert_copies(got, small, reps):
    """got = coarse_fine on `reps` copies of the small call's windows: every copy's results equal the small call's"""
    npk, cands, refined, jig, soft = got
    s_npk, s_cands, s_refined, s_jig, s_soft = small
    T = len(s_cands)
    assert np.array_equal(npk, np.tile(s_npk, reps)) and len(cands) == reps * T
    for r in range(reps):
        sl = slice(r * T, (r + 1) * T)
        for a, b in ((cands, s_cands), (refined, s_refined), (jig, s_jig), (soft, s_soft)):
            assert a[sl].tobytes() == b.tobytes(), r
    # the candidates on both sides of the first two slice boundaries, explicitly
    for i in (SLICE - 1, SLICE, 2 * SLICE - 1, 2 * SLICE):
        j = i % T
        for a, b in ((cands, s_cands), (refined, s_refined), (jig, s_jig), (soft, s_soft)):
            assert a[i].tobytes() == b[j].tobytes(), i


def test_device_resident_chunk_of_three_slices(distinct):
    import torch
    xs, small = distinct
    T = len(small[1])
    reps = -(-int(2.5 * SLICE) // T) + 1
    nwin = reps * len(xs)
    assert reps * T > 2.5 * SLICE and nwin <= 16384     # one chunk (capi.cu: chunk_windows)
    dev = torch.from_numpy(xs.view(np.float32)).cuda().repeat(reps, 1).contiguous()
    ctx = ub.Context(max_windows=nwin, max_candidates=reps * T, **WIDE)
    got = ctx.coarse_fine((dev.data_ptr(), nwin * 45000), nwin=nwin, stride=45000)
    assert_copies(got, small, reps)
    ctx.close()


def host_chunk_windows(nwin, max_windows):
    """windows per host-fed chunk (capi.cu, run_impl: host_chunk, set_cap, cw)"""
    chunk_windows = min(max_windows, 16384)
    host_chunk = min(4096, max(1024, nwin // 16))
    set_cap = max(chunk_windows // 3, (nwin + 2) // 3) if nwin <= chunk_windows else chunk_windows // 3
    return max(1, min(host_chunk, set_cap))


def test_host_fed_chunks_of_several_slices_on_three_streams(distinct):
    """host-fed: chunk groups rotate over three buffer sets and compute streams, the last two groups are cut into
    pieces; with five or more groups the first three are whole and each holds more than a slice, one per stream"""
    xs, small = distinct
    s_npk = small[0]
    reps = -(-5 * 1024 // len(xs))
    nwin = reps * len(xs)
    cw = host_chunk_windows(nwin, nwin)
    assert -(-nwin // cw) >= 5 and cw * int(s_npk.min()) > SLICE
    ctx = ub.Context(max_windows=nwin, max_candidates=reps * int(s_npk.sum()), **WIDE)
    got = ctx.coarse_fine(np.tile(xs, (reps, 1)))
    assert_copies(got, small, reps)
    ctx.close()


def test_caller_list_longer_than_maxcand_past_one_slice(golden_windows):
    """fine() on one window with 2 slices + 17 candidates from the caller (a list the reference takes; this
    context's coarse search would keep at most 13 per window): every candidate is refined, each repeat equal to the
    first, and the first ones equal the oracle.  The slice loop is bounded by the caller's count, not by
    nwin * maxcand, which would stop after the first slice and return the rest unwritten."""
    x = golden_windows["mix_whales"]
    ctx = ub.Context(halfbandwidth=10, maxdrift=4, max_candidates=40000)
    npk, c = ctx.coarse(x.reshape(1, -1))
    assert 1 <= len(c) <= ctx.info.max_cand_per_window
    n = 2 * SLICE + 17
    rep = np.resize(c, n)
    # an earlier call of the same length leaves other bytes in the result buffers
    other = rep.copy()
    other["shift"] += 128
    before = ctx.fine(x.reshape(1, -1), np.array([n], np.int32), other)
    refined, jig, soft = ctx.fine(x.reshape(1, -1), np.array([n], np.int32), rep)
    k = len(c)
    for i in range(k, n, k):
        for a in (refined, jig, soft):
            if a[i:i + k].tobytes() != a[:len(a[i:i + k])].tobytes():
                stale = all(u[i:i + k].tobytes() == v[i:i + k].tobytes() for u, v in zip((refined, jig, soft), before))
                pytest.fail("candidate %d differs from its first copy%s" % (i, " (it holds the previous call's bytes)" if stale else ""))
    assert_fine_rows(refined[:k], jig[:k], soft[:k], x, c, 1500)
    ctx.close()


@pytest.mark.parametrize("n", [17, 31])
def test_lag_share_pairs_of_symbols_160_161(n):
    """k_fine_lagshare gives symbols 160 and 161 of 16 candidates to one warp-task: slices of 17 and 31 rotating
    (drifting) candidates leave a last task with 1 and 15 of them"""
    x = window(2024, [3.0], [1.5], snr_db=-6.0)
    rng = np.random.default_rng(n)
    cands = np.zeros(n, ub.CAND_DTYPE)
    for g in range(n):
        cands[g]["freq"] = np.float32(3.0 + rng.uniform(-0.7, 0.7))
        cands[g]["sync"] = 0.3
        cands[g]["shift"] = int(rng.integers(-4, 24)) * 64
        cands[g]["lin_drift"] = np.float32(rng.choice([-1.0, 1.0]) * rng.uniform(0.5, 3.0))
    ctx = ub.Context(maxdrift=4, max_candidates=n)
    refined, _, _ = fine_against_oracle(ctx, x, cands, 1500)
    assert refined["worth_a_try"].sum() >= 2          # stage D's lag search runs too
    ctx.close()
