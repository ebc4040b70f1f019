"""Synthetic WSPR workloads of SURVEY.md 8(d) / BASELINE.json configs[2..4], generated on the GPU.

torch is plumbing here (random numbers, device memory): the generators are not part of the measured
path.  Frames are made in batches of BATCH; batch b of stream `stream_id` depends only on
(SEED_BASE, stream_id, b), so a rank that holds a slice of a long stream generates exactly the samples
any other split would hold there, and the reference arm can regenerate a prefix of the GPU arm's batch.
Messages are encoded with the library's own transmit-side helpers (uwspr_b200.channel_symbols).
"""
import numpy as np

FL = 45000
FS = 375.0
SPS = 256
NSYM = 162
SEED_BASE = 20190222
BATCH = 500


def message_bytes(rng):
    """50 random payload bits packed MSB-first into 7 bytes (last 6 bits zero)"""
    b = np.zeros(56, np.uint8)
    b[:50] = rng.integers(0, 2, 50, dtype=np.uint8)
    return np.packbits(b)


def _frames_batch(stream_id, b, device, maxdrift=3.0, snr_lo=-30.0, snr_hi=0.0):
    """frames [b*BATCH, (b+1)*BATCH) of a stream: (x [BATCH, FL] complex64 on `device`, truth list).
    One frame per 45 000-sample slot: carrier offset U(-6, 6) Hz, linear drift U(-maxdrift, maxdrift) Hz,
    start sample 375 + U{0..2560}, SNR U(snr_lo, snr_hi) dB in 2500 Hz, complex AWGN."""
    import torch
    from .binding import channel_symbols
    rng = np.random.default_rng([SEED_BASE, stream_id, b])
    gen = torch.Generator(device=device)
    gen.manual_seed(SEED_BASE + 7919 * stream_id + 104729 * b)
    nb = BATCH
    df = FS / SPS
    k = torch.arange(NSYM * SPS, device=device)
    sym_idx = k // SPS
    msgs = [message_bytes(rng) for _ in range(nb)]
    syms = np.stack([channel_symbols(m) for m in msgs]).astype(np.float64)
    f0 = rng.uniform(-6, 6, nb)
    drift = rng.uniform(-maxdrift, maxdrift, nb)
    start = 375 + rng.integers(0, 2561, nb)
    snr = rng.uniform(snr_lo, snr_hi, nb)
    st = torch.from_numpy(syms).to(device)
    f = (torch.from_numpy(f0).to(device)[:, None] + (st[:, sym_idx] - 1.5) * df
         + (torch.from_numpy(drift).to(device)[:, None] / 2.0) * ((sym_idx[None, :].double() - 81.0) / 81.0))
    phase = 2 * np.pi * torch.cumsum(f, dim=1) / FS
    sig = torch.polar(torch.ones_like(phase), phase).to(torch.complex64)
    sigma = np.sqrt((FS / 2500.0) / 10 ** (snr / 10.0) / 2.0)
    noise = torch.randn((nb, FL, 2), generator=gen, device=device, dtype=torch.float32)
    x = torch.view_as_complex(noise) * torch.from_numpy(sigma.astype(np.float32)).to(device)[:, None]
    pos = torch.from_numpy(start).to(device)[:, None] + k[None, :]
    ok = pos < FL
    flat = (torch.arange(nb, device=device)[:, None] * FL + pos)[ok]
    torch.view_as_real(x).view(-1, 2).index_add_(0, flat, torch.view_as_real(sig)[ok])
    truth = [dict(msg=m, f0=a, drift=d, start=int(s), snr=q) for m, a, d, s, q in zip(msgs, f0, drift, start, snr)]
    return x, truth


def gen_frames(first, count, stream_id, device, **kw):
    """frames [first, first+count) of stream `stream_id` as a (count, FL) complex64 tensor + truth"""
    import torch
    out = torch.empty((count, FL), dtype=torch.complex64, device=device)
    truth = []
    b = first // BATCH
    while b * BATCH < first + count:
        x, t = _frames_batch(stream_id, b, device, **kw)
        lo, hi = max(first, b * BATCH), min(first + count, (b + 1) * BATCH)
        out[lo - first:hi - first] = x[lo - b * BATCH:hi - b * BATCH]
        truth += t[lo - b * BATCH:hi - b * BATCH]
        del x
        b += 1
    return out, truth


def gen_stream_span(w_lo, w_hi, stride, stream_id, device, **kw):
    """the samples windows [w_lo, w_hi) of a sliding-window stream read: stream[w_lo*stride, (w_hi-1)*stride + FL),
    where the stream is the frames of `stream_id` back to back (a frame every FL samples).
    Returns (1-D complex64 tensor, index of the first frame touched, truth of the frames touched)."""
    s0, s1 = w_lo * stride, (w_hi - 1) * stride + FL
    f_lo, f_hi = s0 // FL, (s1 + FL - 1) // FL
    frames, truth = gen_frames(f_lo, f_hi - f_lo, stream_id, device, **kw)
    span = frames.reshape(-1)[s0 - f_lo * FL:s1 - f_lo * FL].clone()
    del frames
    return span, f_lo, truth


def gen_array(chan_lo, chan_hi, nwin, whales, device, stream_id=64, snr_db=-21.0, whale_gain=1.0):
    """BASELINE.json configs[4]: channels [chan_lo, chan_hi) of a hydrophone array, `nwin` windows each.
    Window w carries one transmitted frame (the same on every channel) with per-channel delay U{0..64}
    samples and gain U(0.05, 0.2), independent AWGN at `snr_db` relative to a unit-amplitude frame scaled by
    the mean gain, plus the whale recording (375-sps complex, looped, per-channel circular offset) at
    `whale_gain` -- the x1 / x0.1 ratio of examples/WaveFilePlusNoiseDecode.grc:586,637.
    Returns (x [nchan, nwin, FL] complex64 tensor, truth per window); every (channel, window) depends only on
    (SEED_BASE, stream_id, channel, window), not on the slice asked for."""
    import torch
    from .binding import channel_symbols
    nch = chan_hi - chan_lo
    out = torch.empty((nch, nwin, FL), dtype=torch.complex64, device=device)
    wh = torch.from_numpy(np.ascontiguousarray(whales, dtype=np.complex64)).to(device)
    nwh = wh.numel()
    df = FS / SPS
    k = torch.arange(NSYM * SPS, device=device)
    sym_idx = k // SPS
    n = torch.arange(FL, device=device)
    truth = []
    sigma = float(np.sqrt((FS / 2500.0) / 10 ** (snr_db / 10.0) * 0.125 ** 2 / 2.0))
    for w in range(nwin):
        rng = np.random.default_rng([SEED_BASE, stream_id, w])
        msg = message_bytes(rng)
        syms = torch.from_numpy(channel_symbols(msg).astype(np.float64)).to(device)
        f0 = float(rng.uniform(-6, 6))
        start = int(375 + rng.integers(0, 2400))
        f = f0 + (syms[sym_idx] - 1.5) * df
        sig = torch.polar(torch.ones_like(f), 2 * np.pi * torch.cumsum(f, 0) / FS).to(torch.complex64)
        truth.append(dict(msg=msg, f0=f0, start=start))
        for c in range(chan_lo, chan_hi):
            crng = np.random.default_rng([SEED_BASE, stream_id, w, c])
            delay, gain, off = int(crng.integers(0, 65)), float(crng.uniform(0.05, 0.2)), int(crng.integers(0, nwh))
            gen = torch.Generator(device=device)
            gen.manual_seed(SEED_BASE + 31 * w + 1009 * c + 7919 * stream_id)
            x = torch.view_as_complex(torch.randn((FL, 2), generator=gen, device=device, dtype=torch.float32)) * sigma
            x += whale_gain * wh[(off + n) % nwh]
            p0 = start + delay
            m = min(NSYM * SPS, FL - p0)
            x[p0:p0 + m] += gain * sig[:m]
            out[c - chan_lo, w] = x
    return out, truth


def gen_plane_wave_audio(positions_m, direction, nchan, minutes, snr_db_per_channel, seed, message=("K1ABC", "FN42", 37),
                         f0=2.0, start_s=1.0, fs_in=12000.0, fc=1500.0, sound_speed=1500.0, noise_rms=0.2, fmt="int16"):
    """Audio of a hydrophone array hearing one WSPR transmitter as a plane wave, in independent noise per hydrophone.
    positions_m [nchan, 2 or 3] in metres; direction: unit vector from the array towards the source.  Hydrophone c hears
    the source at tau_c = -(p_c . u) / sound_speed (relative to the origin): its audio is cos(2 pi int_0^{t - tau_c} f),
    evaluated in float64 from the exact fractional delay (no integer shift at baseband), with f = fc + f0 +
    (symbol - 1.5) * 375/256 Hz for the 162 symbols of `message` from start_s on.  Each channel adds Gaussian noise of
    rms noise_rms (full scale 1) from its own generator, default_rng([seed, c]); snr_db_per_channel is the signal's
    power over the noise power in 2500 Hz, as WSPR states SNR.  fmt "int16" (PCM, x 32768, clipped) or "float32".
    Returns (audio [nchan, n], dict(msg=7 bytes, text, tau=[nchan] seconds, amplitude))."""
    from .binding import channel_symbols, pack_type1
    p = np.asarray(positions_m, dtype=np.float64)
    u = np.asarray(direction, dtype=np.float64)
    if p.shape != (nchan, u.size) or u.size not in (2, 3):
        raise ValueError("positions_m must be [nchan, 2 or 3] and direction of the same dimension")
    n = int(minutes * 60 * fs_in)
    tau = -(p @ u) / sound_speed
    msg = pack_type1(*message)
    sym = channel_symbols(msg).astype(np.float64)
    tsym = SPS / FS
    f = fc + f0 + (sym - 1.5) * FS / SPS                          # Hz, per symbol
    cyc0 = np.concatenate([[0.0], np.cumsum(f * tsym)])            # cycles at the start of each symbol
    amp = np.sqrt(2.0 * 10 ** (snr_db_per_channel / 10.0) * noise_rms ** 2 * 2500.0 / (fs_in / 2.0))
    t = np.arange(n, dtype=np.float64) / fs_in
    out = np.empty((nchan, n), np.int16 if fmt == "int16" else np.float32)
    for c in range(nchan):
        tp = t - tau[c] - start_s                                  # time since the first symbol, at this hydrophone
        k = np.floor(tp / tsym)
        on = (k >= 0) & (k < NSYM)
        ki = np.where(on, k, 0).astype(np.int64)
        cyc = cyc0[ki] + f[ki] * (tp - ki * tsym)
        a = np.where(on, amp * np.cos(2 * np.pi * (cyc - np.floor(cyc))), 0.0)
        a += np.random.default_rng([seed, c]).normal(0.0, noise_rms, n)
        out[c] = np.clip(np.round(a * 32768.0), -32768, 32767) if fmt == "int16" else a
    text = "%s %s %2d" % message
    return out, dict(msg=bytes(msg), text=text, tau=tau, amplitude=amp)
