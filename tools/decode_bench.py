"""Decoder measurement on one GPU: the host Fano decoder (uwspr_b200_decode_batch on all host cores) against the
device decoder (uwspr_b200_decode_device) on the headline batch of bench.py (same generator, same PARAMS,
10 000 windows), and the whole receive chain with the decoder on the device.

  1. coarse_fine with all 17 jiggles (results fetched), then decode_batch on every host core and decode_device on
     the results the call left on the device; each timed from a device synchronise to a device synchronise, and
     the four outputs (decoded, message, idt_used, fano_cycles) asserted equal.
  2. coarse_fine without refinement / jiggle / soft-symbol outputs + decode_device, host-fed and device-resident,
     in windows per second.
  3. task count, decoder time-outs and the cycles of the longest decode (all derived from the per-candidate
     outputs: a gated jiggle before the decoding one, or any gated jiggle of a candidate that never decodes, is a
     time-out of 10000 x 81 + 2 cycles), device time of decode_device from CUDA events, GPU name and power limit.

    python tools/decode_bench.py [--windows 10000] [--steps 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gr-uwspr_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from bench import FL, PARAMS  # noqa: E402

TIMEOUT_CYCLES = 10000 * 81 + 2


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--windows", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=3, help="timed repetitions of every arm (mean reported)")
    ap.add_argument("--out", help="also write the JSON record to this file")
    args = ap.parse_args()

    import torch
    import uwspr_b200 as ub
    from uwspr_b200 import synth
    from uwspr_b200.binding import _p

    if not torch.cuda.is_available():
        raise SystemExit("decode_bench: no CUDA device")
    dev = torch.device("cuda:0")
    nwin, steps = args.windows, args.steps
    cores = len(os.sched_getaffinity(0))
    stream = torch.cuda.Stream(dev)
    ctx = ub.Context(device=0, max_windows=nwin, max_candidates=max(4 * nwin, 1024), **PARAMS)
    ctx.set_stream(stream.cuda_stream)
    L = ctx.L
    xs_dev, truth = synth.gen_frames(0, nwin, 0, dev)
    xs_host_t = torch.empty((nwin, FL), dtype=torch.complex64, pin_memory=True)
    xs_host_t.copy_(xs_dev)
    torch.cuda.synchronize(dev)
    xs_host = xs_host_t.numpy()
    dptr = (xs_dev.data_ptr(), nwin * FL)

    def sync():
        torch.cuda.synchronize(dev)

    # ---- 1. host decoder against device decoder on the same fine results ---------------------------------
    out = ctx.result_buffers(nwin)
    npk, cands, refined, jig, soft = ctx.coarse_fine(dptr, nwin=nwin, stride=FL, out=out)
    ncand = len(cands)

    def host_decode():
        r = (np.zeros(ncand, np.uint8), np.zeros((ncand, 7), np.int8), np.zeros(ncand, np.int32), np.zeros(ncand, np.uint32))
        got = L.uwspr_b200_decode_batch(_p(refined), _p(jig), _p(soft), ncand, ub.NJIG, 0, *(_p(a) for a in r))
        assert got >= 0
        return (got,) + r

    def device_decode():
        r = (np.zeros(ncand, np.uint8), np.zeros((ncand, 7), np.int8), np.zeros(ncand, np.int32), np.zeros(ncand, np.uint32))
        got = L.uwspr_b200_decode_device(ctx.h, None, None, None, 0, ncand, ub.NJIG, *(_p(a) for a in r))
        assert got >= 0, got
        return (got,) + r

    def timed(fn):
        sync()
        t0 = time.perf_counter()
        r = fn()
        sync()
        return time.perf_counter() - t0, r

    device_decode()   # first call allocates the decoder's workspaces
    t_host, t_dev, ev_ms = [], [], []
    for _ in range(steps):
        t, want = timed(host_decode)
        t_host.append(t)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t, got = timed(device_decode)
        e1.record(stream)
        e1.synchronize()
        t_dev.append(t)
        ev_ms.append(e0.elapsed_time(e1))
        assert got[0] == want[0]
        for a, b in zip(got[1:], want[1:]):
            assert np.array_equal(a, b)
    _, dec, msg, idt, cyc = want
    gated = (jig["gate"] != 0) & (refined["worth_a_try"] != 0)[:, None]
    ngated = gated.sum(axis=1)
    tasks = int(ngated.sum())
    before = np.array([gated[g, :max(idt[g], 0)].sum() for g in range(ncand)])
    timeouts = int(np.where(dec == 1, before, ngated).sum())
    win_cycles = cyc.astype(np.int64) - before * TIMEOUT_CYCLES
    longest = int(max(TIMEOUT_CYCLES if timeouts else 0, int(win_cycles[dec == 1].max()) if dec.any() else 0))
    never = int(((dec == 0) & (ngated > 0)).sum())

    # ---- 2. the receive chain with the decoder on the device ----------------------------------------------
    npk_b = np.zeros(nwin, np.int32)
    cands_b = np.zeros(ctx.info.max_candidates, ub.CAND_DTYPE)

    def chain(ptr, space):
        def run():
            total = C.c_int32(0)
            ctx._check(L.uwspr_b200_coarse_fine(ctx.h, ptr, space, FL, nwin, 0, ub.NJIG, _p(npk_b), _p(cands_b),
                                                ctx.info.max_candidates, C.byref(total), None, None, None))
            n = total.value
            r = (np.zeros(n, np.uint8), np.zeros((n, 7), np.int8))
            got = L.uwspr_b200_decode_device(ctx.h, None, None, None, 0, n, ub.NJIG, _p(r[0]), _p(r[1]), None, None)
            assert got >= 0, got
            return r
        return run

    rates = {}
    for name, ptr, space in (("host_fed", _p(xs_host.reshape(-1)), ub.binding.HOST),
                             ("device_resident", C.c_void_p(xs_dev.data_ptr()), ub.binding.DEVICE)):
        fn = chain(ptr, space)
        fn()
        ts = []
        for _ in range(steps):
            t, (d, m) = timed(fn)
            ts.append(t)
            assert np.array_equal(d, dec) and np.array_equal(m, msg)
        rates[name] = dict(windows_per_s=nwin / float(np.mean(ts)), seconds=float(np.mean(ts)))

    r2 = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_bench_1gpu.json")) as f:
            r2 = json.load(f)["receiver"]["value"]
    except Exception:
        pass
    rec = dict(
        gpu=torch.cuda.get_device_name(dev), power_limit=power_limit(), host_cores=cores, windows=nwin, steps=steps,
        params=PARAMS, candidates=ncand, decoded=int(want[0]), outputs_equal=True,
        tasks=tasks, timeouts=timeouts, candidates_never_decoded=never, longest_task_cycles=longest,
        decoder_seconds=dict(host_decode_batch=float(np.mean(t_host)), device_decode_device=float(np.mean(t_dev)),
                             device_events_ms=float(np.mean(ev_ms))),
        receive_chain=rates,
        round2_receiver_windows_per_s=r2,
        note="decoder seconds: from a device synchronise to a device synchronise, mean of the steps; device_events_ms: "
             "CUDA events around decode_device on the context's stream (task list, decoder, reduction, result copies); "
             "receive chain: coarse_fine without refinement/jiggle/soft outputs + decode_device on the results left on "
             "the device, all 17 jiggles of every candidate evaluated")
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
