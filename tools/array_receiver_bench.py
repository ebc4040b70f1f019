"""Throughput of the multi-channel receiver (uwspr_b200.ArrayReceiver) on 64 channels of int16 12 kHz audio.

Workload: 64 channels x `--minutes` of seeded audio (noise plus a few WSPR frames per channel at random frequencies
and times), the reference flowgraph's front-end (flowgraph_taps(), decim 32, delay 0) and sliding window (shift 9 s).
Reported:
  * rates of the whole receiver, audio on the host and on the device, for batch_windows 16 / 64 / 256:
    channel-windows per second and seconds of audio (all channels) per second of wall clock;
  * the time split between the front-end, coarse_fine and decode_device on the same audio, stage by stage (see
    stage_split for what each number times);
  * launches per batch;
  * the same audio through the composition available before the receiver (one-shot front-end, then one coarse_fine
    and one decode_device per channel), timed in the same run, with its messages checked equal to the receiver's.
Writes the JSON to --out (default profiles/r4_array_receiver_1gpu.json)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gr-uwspr_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import uwspr_b200 as ub  # noqa: E402

FS_IN, DECIM, SHIFT, FL = 12000.0, 32, 9, 45000
STRIDE = SHIFT * 375


def make_audio(nchan, minutes, seed):
    n = int(minutes * 60 * FS_IN) // DECIM * DECIM
    audio = np.empty((nchan, n), np.int16)
    for c in range(nchan):
        rng = np.random.default_rng(seed + c)
        a = rng.normal(0.0, 0.2 * 32768.0, n).astype(np.float32)
        for start in range(int(rng.integers(0, 60)) * int(FS_IN), n - 162 * 8192, int(240 * FS_IN)):
            msg = ub.pack_type1("K%dAB" % (c % 10), "FN%02d" % (c % 100), 30)
            sym = ub.channel_symbols(msg).astype(np.float64)
            f = 1500.0 + rng.uniform(-60.0, 60.0) + (np.repeat(sym, 8192) - 1.5) * 375.0 / 256.0
            a[start:start + 162 * 8192] += (0.1 * 32768.0 * np.cos(2 * np.pi * np.cumsum(f) / FS_IN)).astype(np.float32)
        audio[c] = np.clip(np.round(a), -32768, 32767).astype(np.int16)
    return audio


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = float(q.stdout.strip().splitlines()[0])
    except Exception:
        power = None
    return name, power


def run_receiver(audio, taps, batch, on_device):
    """(seconds, messages, windows per channel, launches per batch)"""
    import torch
    rx = ub.ArrayReceiver(audio.shape[0], shift=SHIFT, batch_windows=batch, input="int16", taps=taps, delay=0)
    if on_device:
        t = torch.from_numpy(audio).cuda()
        arg = (ctypes.c_void_p(t.data_ptr()), np.int16, audio.shape)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    msgs = rx.push(arg if on_device else audio, flush=True)
    dt = time.perf_counter() - t0
    nwin = rx.windows_done()
    nbatch = -(-nwin // batch)
    launches = rx.launch_count()
    rx.close()
    return dt, [(c, w, bytes(m)) for c, w, m, _ in msgs], nwin, launches / nbatch


def stage_split(audio, taps, batch):
    """per channel-window ms of the three stages, run one after the other on the same audio.
    Front-end: host clock around one synchronous push (it runs on the stream's own CUDA stream, so this includes its
    launches and the final synchronisation).  coarse_fine and decode_device: CUDA events on the stream the context
    runs its kernels on (set_stream), i.e. device time.  The coarse_fine windows are copied out as independent
    windows of fl samples (the receiver's ring is channel-major with a stride; the kernels' work is the same)."""
    import torch
    nchan, n = audio.shape
    m = n // DECIM
    a = torch.from_numpy(audio).cuda()
    x = torch.empty((nchan, m, 2), dtype=torch.float32, device="cuda")
    fs = ub.FrontendStream(nchan, taps=taps, delay=0, fmt=np.int16)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = fs.push((ctypes.c_void_p(a.data_ptr()), np.int16, audio.shape), out_device_ptr=x.data_ptr(), out_stride=m)
    fe_ms = 1e3 * (time.perf_counter() - t0)
    assert got == m
    nwin = 1 + (m - FL) // STRIDE
    ctx = ub.Context(maxdrift=0, max_windows=nchan * batch)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    cf_ms = dec_ms = 0.0
    wins = torch.empty((nchan, batch, FL, 2), dtype=torch.float32, device="cuda")
    nb = nwin // batch
    for b in range(nb):
        for k in range(batch):
            lo = (b * batch + k) * STRIDE
            wins[:, k] = x[:, lo:lo + FL]
        torch.cuda.synchronize()
        ev[0].record(stream)
        ctx.coarse_fine((wins.data_ptr(), nchan * batch * FL), nwin=nchan * batch, stride=FL, fetch=False)
        ev[1].record(stream)
        ctx.decode()
        ev[2].record(stream)
        stream.synchronize()
        cf_ms += ev[0].elapsed_time(ev[1])
        dec_ms += ev[1].elapsed_time(ev[2])
    ctx.set_stream(None)
    ctx.close()
    fs.close()
    # per channel-window: the front-end ran over every window's samples, the other two over nb whole batches
    return fe_ms / (nchan * nwin), cf_ms / (nchan * batch * nb), dec_ms / (nchan * batch * nb)


def baseline(audio, taps):
    """one-shot front-end, then one coarse_fine (17 jiggles, results left on the device) and decode_device per channel"""
    import torch
    nchan, n = audio.shape
    m = n // DECIM
    nwin = 1 + (m - FL) // STRIDE
    ctx = ub.Context(maxdrift=0, max_windows=nwin)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    x = ub.frontend(audio, taps=taps, delay=0)
    for c in range(nchan):
        ctx.coarse_fine(x[c], nwin=nwin, stride=STRIDE, fetch=False)
        ctx.decode()
    dt = time.perf_counter() - t0
    # its messages, in the receiver's (window, channel, candidate) order: an untimed pass that also fetches npk
    by_chan = []
    for c in range(nchan):
        npk = ctx.coarse_fine(x[c], nwin=nwin, stride=STRIDE)[0]
        win = np.repeat(np.arange(nwin), npk)
        by_chan.append([(int(win[g]), bytes(mm)) for g, mm, _ in ctx.decode()])
    ctx.close()
    msgs = []
    for k in range(nwin):
        for c in range(nchan):
            msgs += [(c, w, mm) for w, mm in by_chan[c] if w == k]
    return dt, nwin, msgs


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--minutes", type=float, default=20.0)
    ap.add_argument("--batches", default="16,64,256")
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_array_receiver_1gpu.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = gpu_info()
    t0 = time.perf_counter()
    audio = make_audio(a.channels, a.minutes, a.seed)
    gen_s = time.perf_counter() - t0
    taps = ub.flowgraph_taps()
    nchan, n = audio.shape
    audio_s = nchan * n / FS_IN
    # warm-up: every kernel and the allocator, on a short prefix
    run_receiver(audio[:, :FL * DECIM * 2], taps, 16, False)
    res = {"gpu": name, "power_limit_w": power, "workload": {
        "channels": nchan, "audio_samples_per_channel": n, "minutes_per_channel": n / FS_IN / 60, "fs_in": FS_IN,
        "format": "int16", "taps": "flowgraph_taps() (%d complex), delay 0" % len(taps), "decim": DECIM, "shift_s": SHIFT,
        "seed": a.seed, "generation_s": round(gen_s, 1)}}
    ref_msgs = None
    rows = []
    for batch in [int(b) for b in a.batches.split(",")]:
        for on_device in (False, True):
            dt, msgs, nwin, lpb = run_receiver(audio, taps, batch, on_device)
            if ref_msgs is None:
                ref_msgs = msgs
            rows.append({"batch_windows": batch, "audio": "device" if on_device else "host", "seconds": round(dt, 4),
                         "channel_windows": nwin * nchan, "channel_windows_per_s": round(nwin * nchan / dt, 1),
                         "audio_s_per_s": round(audio_s / dt, 1), "launches_per_batch": round(lpb, 2),
                         "messages": len(msgs), "messages_equal_first_run": msgs == ref_msgs})
            print(json.dumps(rows[-1]), flush=True)
    res["receiver"] = rows
    fe, cf, dec = stage_split(audio, taps, 64)
    tot = fe + cf + dec
    res["stage_split_batch64"] = {"frontend_us_per_channel_window": round(1e3 * fe, 2), "coarse_fine_us_per_channel_window": round(1e3 * cf, 2),
                                  "decode_device_us_per_channel_window": round(1e3 * dec, 2), "frontend_share": round(fe / tot, 3),
                                  "coarse_fine_share": round(cf / tot, 3), "decode_share": round(dec / tot, 3),
                                  "note": "stages run one after the other: the front-end stream over all the audio (host clock "
                                          "around one synchronous push), then whole batches of 64 windows x all channels as one "
                                          "coarse_fine each and decode_device on its results (CUDA events on the context's "
                                          "stream: device time); the coarse_fine windows are copied out as independent "
                                          "windows of fl samples"}
    print(json.dumps(res["stage_split_batch64"]), flush=True)
    # today's composition, and its messages against the receiver's
    dt, nwin, base_msgs = baseline(audio, taps)
    res["baseline"] = {"what": "one-shot uwspr_b200_frontend_ctaps over all channels, then per channel one coarse_fine "
                               "(all windows, 17 jiggles, results left on the device) and one decode_device",
                       "seconds": round(dt, 4), "channel_windows_per_s": round(nwin * nchan / dt, 1),
                       "audio_s_per_s": round(audio_s / dt, 1), "messages": len(base_msgs),
                       "messages_equal_receiver": base_msgs == ref_msgs}
    print(json.dumps(res["baseline"]), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
