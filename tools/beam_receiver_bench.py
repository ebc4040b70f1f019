"""The receiver on 64 delay-and-sum beams against the plain receiver on 64 hydrophones (uwspr_b200.ArrayReceiver with and
without beams=).

Workload: the shape of tools/array_receiver_bench.py -- 64 channels of int16 12 kHz audio, the reference flowgraph's
front-end (flowgraph_taps(), decim 32, delay 0), shift 9 s -- with the hydrophones at seeded random positions in a
200 m square and one WSPR transmitter arriving as a plane wave (synth.gen_plane_wave_audio: exact fractional delays in
the passband, independent noise per hydrophone) at a per-channel SNR below what one hydrophone decodes.  The beams are
a fan of 64 directions around the horizon (plane_wave_steering); the source arrives from beam SOURCE_BEAM's direction.
Reported:
  * k_beamform alone: kernel time per launch from torch.profiler over many one-shot launches, on the receiver's push
    piece (16 384 samples) and on the new samples of one 256-window batch (864 000), and the kernel time per batch of
    16 / 64 / 256 windows these give (the receiver launches once per piece of at most 16 384 samples); plus CUDA events
    around the same one-shot calls, which include their table upload;
  * rates of both receivers on the same audio (host-fed), alternated in one run, for batch_windows 16 / 64 / 256;
  * the messages each decodes (row, window, text);
  * launches per batch of each;
  * card name and power limit, read in the same run.
Writes the JSON to --out (default profiles/r6_beam_receiver_1gpu.json)."""
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
from uwspr_b200 import synth  # noqa: E402

FS_IN, DECIM, SHIFT, FL = 12000.0, 32, 9, 45000
STRIDE = SHIFT * 375
PIECE = 16384          # 375-sps samples per push piece of the receiver with beams (kRingPiece in csrc/receiver.cu)
SOURCE_BEAM = 10


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


def kernel_times(w, d, reps):
    """(profiler kernel ms per launch, event ms per one-shot call) at n = PIECE and n = 256 * STRIDE"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    nbeam, nchan = w.shape
    out = {}
    for n in (PIECE, 256 * STRIDE):
        x = torch.randn((nchan, n, 2), device="cuda")
        y = torch.empty((nbeam, n, 2), device="cuda")
        arg = (ctypes.c_void_p(x.data_ptr()), np.complex64, (nchan, n))
        for _ in range(3):
            ub.beamform(arg, w, d, out_device_ptr=y.data_ptr())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            ub.beamform(arg, w, d, out_device_ptr=y.data_ptr())
        e1.record()
        torch.cuda.synchronize()
        call_ms = e0.elapsed_time(e1) / reps
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                ub.beamform(arg, w, d, out_device_ptr=y.data_ptr())
            torch.cuda.synchronize()
        ks = [e for e in prof.events() if "k_beamform" in e.name]
        assert len(ks) == reps, len(ks)
        kern_ms = sum(e.device_time for e in ks) / 1e3 / reps
        out[n] = (kern_ms, call_ms)
        del x, y
    return out


def run(audio, taps, batch, beams):
    """(seconds, [(row, window, text)], windows, launches per batch)"""
    import torch
    rx = ub.ArrayReceiver(audio.shape[0], shift=SHIFT, batch_windows=batch, input="int16", taps=taps, delay=0, beams=beams)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    msgs = rx.push(audio, flush=True)
    dt = time.perf_counter() - t0
    nwin = rx.windows_done()
    launches = rx.launch_count()
    rx.close()
    u = ub.WSPR_unpacker()
    return dt, [(c, k, u.unpack(m)[1]) for c, k, m, _ in msgs], nwin, launches / -(-nwin // batch)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--beams", type=int, default=64)
    ap.add_argument("--minutes", type=float, default=6.0)
    ap.add_argument("--snr", type=float, default=-36.0, help="per-channel SNR of the source, dB in 2500 Hz")
    ap.add_argument("--batches", default="16,64,256")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--reps", type=int, default=50, help="launches per k_beamform timing")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_beam_receiver_1gpu.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = gpu_info()
    rng = np.random.default_rng(a.seed)
    pos = rng.uniform(0.0, 200.0, (a.channels, 2))
    ang = 2 * np.pi * np.arange(a.beams) / a.beams
    dirs = np.c_[np.cos(ang), np.sin(ang)]
    t0 = time.perf_counter()
    audio, truth = synth.gen_plane_wave_audio(pos, dirs[SOURCE_BEAM], a.channels, a.minutes, a.snr, seed=a.seed, f0=2.5,
                                              start_s=1.0)
    gen_s = time.perf_counter() - t0
    w, d = ub.plane_wave_steering(pos, dirs)
    taps = ub.flowgraph_taps()
    nchan, n = audio.shape
    res = {"gpu": name, "power_limit_w": power, "workload": {
        "channels": nchan, "beams": a.beams, "audio_samples_per_channel": n, "minutes_per_channel": n / FS_IN / 60,
        "fs_in": FS_IN, "format": "int16", "taps": "flowgraph_taps() (%d complex), delay 0" % len(taps), "decim": DECIM,
        "shift_s": SHIFT, "seed": a.seed, "positions": "uniform in a 200 m square", "largest_delay_samples": int(d.max()),
        "source": {"text": truth["text"], "beam": SOURCE_BEAM, "direction_deg": round(float(np.degrees(ang[SOURCE_BEAM])), 3),
                   "snr_db_per_channel_2500hz": a.snr, "start_s": 1.0, "f_hz": 1502.5},
        "generation_s": round(gen_s, 1)}}
    # k_beamform alone
    kt = kernel_times(w, d, a.reps)
    piece_ms = kt[PIECE][0]
    res["k_beamform"] = {
        "what": "torch.profiler device time of k_beamform per launch over %d one-shot launches (64 beams x 64 channels, "
                "device buffers); event_ms_per_call: CUDA events around the same uwspr_b200_beamform calls, which also "
                "upload the beam tables and synchronise" % a.reps,
        "piece_16384": {"kernel_ms": round(piece_ms, 4), "event_ms_per_call": round(kt[PIECE][1], 4)},
        "batch256_864000": {"kernel_ms": round(kt[256 * STRIDE][0], 4), "event_ms_per_call": round(kt[256 * STRIDE][1], 4),
                            "gflop": round(8 * a.beams * nchan * 256 * STRIDE / 1e9, 2),
                            "gflop_per_s": round(8 * a.beams * nchan * 256 * STRIDE / 1e6 / kt[256 * STRIDE][0], 1)},
        "receiver_ms_per_batch": {str(b): round(-(-b * STRIDE // PIECE) * piece_ms, 4) for b in (16, 64, 256)},
    }
    print(json.dumps(res["k_beamform"]), flush=True)
    # warm-up: every kernel and the allocator, on a short prefix
    for beams in (None, (w, d)):
        run(audio[:, :FL * DECIM * 2], taps, 16, beams)
    rows = []
    for rep in range(a.repeats):
        for batch in [int(b) for b in a.batches.split(",")]:
            for kind, beams in (("channels", None), ("beams", (w, d))):
                dt, msgs, nwin, lpb = run(audio, taps, batch, beams)
                rows.append({"repeat": rep, "batch_windows": batch, "receiver": kind, "seconds": round(dt, 4),
                             "row_windows": nwin * (nchan if beams is None else a.beams),
                             "audio_s_per_s": round(nchan * n / FS_IN / dt, 1), "launches_per_batch": round(lpb, 2),
                             "messages": msgs})
                print(json.dumps(rows[-1]), flush=True)
    res["runs"] = rows
    summary = {}
    for batch in [int(b) for b in a.batches.split(",")]:
        for kind in ("channels", "beams"):
            r = [x for x in rows if x["batch_windows"] == batch and x["receiver"] == kind]
            s = float(np.median([x["seconds"] for x in r]))
            summary["%s_batch%d" % (kind, batch)] = {
                "median_seconds": round(s, 4), "row_windows_per_s": round(r[0]["row_windows"] / s, 1),
                "audio_s_per_s": round(nchan * n / FS_IN / s, 1), "launches_per_batch": r[0]["launches_per_batch"],
                "messages": len(r[0]["messages"]), "source_heard_on": sorted({c for c, _, t in r[0]["messages"] if t == truth["text"]}),
                "same_messages_every_run": all(x["messages"] == r[0]["messages"] for x in r)}
    res["summary"] = summary
    print(json.dumps(summary, indent=1), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
