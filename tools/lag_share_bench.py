"""A/B of the lag searches' shared-table kernel (k_fine_lagshare) on the headline workload of bench.py: 10 000
device-resident windows (3.6 GB, larger than L2) through coarse_fine, same generator and PARAMS.

Two contexts, one created with UWSPR_B200_NO_LAG_SHARE (the lag searches of stages A and D go through the
per-point kernel) and one without.  After a warm-up of each, the arms alternate --reps times, --steps calls each;
every call is timed from device synchronise to device synchronise, and the library's per-stage CUDA-event times
(last_timing) are averaged per arm.  The outputs of both arms (candidates, refined records, jiggles, soft symbols)
are compared byte for byte.  The record holds the GPU name and power limit, read in the same run.

--profile instead runs each arm once under torch.profiler and writes the per-kernel CUDA time.

    python tools/lag_share_bench.py [--windows 10000] [--steps 3] [--reps 3] [--out FILE] [--profile]
"""
import argparse
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

ARMS = ("share_off", "share_on")


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except Exception:
        return None


def make_ctx(ub, arm, nwin):
    if arm == "share_off":
        os.environ["UWSPR_B200_NO_LAG_SHARE"] = "1"
    else:
        os.environ.pop("UWSPR_B200_NO_LAG_SHARE", None)
    try:
        return ub.Context(device=0, max_windows=nwin, max_candidates=max(4 * nwin, 1024), **PARAMS)
    finally:
        os.environ.pop("UWSPR_B200_NO_LAG_SHARE", None)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--windows", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=3, help="timed calls per arm and repetition")
    ap.add_argument("--reps", type=int, default=3, help="alternations of the two arms")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON record to this file")
    ap.add_argument("--profile", action="store_true", help="per-kernel CUDA time of one call per arm (torch.profiler)")
    args = ap.parse_args()

    import torch
    import uwspr_b200 as ub
    from uwspr_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("lag_share_bench: no CUDA device")
    dev = torch.device("cuda:0")
    nwin = args.windows
    xs_dev, _ = synth.gen_frames(0, nwin, 0, dev)
    torch.cuda.synchronize(dev)
    dptr = (xs_dev.data_ptr(), nwin * FL)
    ctxs = {arm: make_ctx(ub, arm, nwin) for arm in ARMS}

    def call(arm):
        ctxs[arm].coarse_fine(dptr, nwin=nwin, stride=FL, fetch=False)

    for arm in ARMS:
        for _ in range(args.warmup):
            call(arm)
    torch.cuda.synchronize(dev)

    rec = dict(gpu=gpu_info(), windows=nwin, input_bytes=nwin * FL * 8, workload="bench.py headline: device-resident "
               "coarse_fine over %d synthetic windows (all 17 jiggles, results left on the device)" % nwin)
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for arm in ARMS:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(arm)
                torch.cuda.synchronize(dev)
            rows = {}
            for ev in prof.key_averages():
                t = getattr(ev, "device_time_total", None)
                if t is None:
                    t = ev.cuda_time_total
                if t > 0:
                    rows[ev.key] = dict(ms=t / 1e3, calls=ev.count)
            kern[arm] = dict(sorted(rows.items(), key=lambda kv: -kv[1]["ms"]))
        rec["kernels_one_call"] = kern
    else:
        step = {arm: [] for arm in ARMS}
        stages = {arm: [] for arm in ARMS}
        for _ in range(args.reps):
            for arm in ARMS:
                for _ in range(args.steps):
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    call(arm)
                    torch.cuda.synchronize(dev)
                    step[arm].append((time.perf_counter() - t0) * 1e3)
                    stages[arm].append(list(ctxs[arm].last_timing()))
        names = ("spectrogram_normalizer", "coarse_search", "fine_sync_demod", "call")
        arms = {}
        for arm in ARMS:
            s = np.array(stages[arm])
            arms[arm] = dict(step_ms=dict(mean=float(np.mean(step[arm])), std=float(np.std(step[arm])),
                                          min=float(np.min(step[arm])), max=float(np.max(step[arm]))),
                             stage_ms={n: dict(mean=float(s[:, k].mean()), std=float(s[:, k].std()),
                                               min=float(s[:, k].min()), max=float(s[:, k].max()))
                                       for k, n in enumerate(names)},
                             windows_per_s=float(nwin / (np.mean(step[arm]) / 1e3)))
        rec["arms"] = arms
        off, on = arms["share_off"], arms["share_on"]
        rec["fine_ms_saved"] = off["stage_ms"]["fine_sync_demod"]["mean"] - on["stage_ms"]["fine_sync_demod"]["mean"]
        rec["step_speedup"] = off["step_ms"]["mean"] / on["step_ms"]["mean"]
        rec["timing"] = "%d alternations x %d calls per arm after %d warm-up calls each; step = host clock between " \
                        "device synchronises; stages = the library's CUDA events" % (args.reps, args.steps, args.warmup)
        # the same bytes from both arms
        res = {}
        for arm in ARMS:
            res[arm] = ctxs[arm].coarse_fine(dptr, nwin=nwin, stride=FL)
        same = [np.asarray(u).tobytes() == np.asarray(v).tobytes() for u, v in zip(res["share_off"], res["share_on"])]
        rec["outputs_identical"] = dict(zip(("npk", "cands", "refined", "jig", "soft"), same))
        rec["candidates"] = int(np.asarray(res["share_on"][0]).sum())
        assert all(same), rec["outputs_identical"]
    for c in ctxs.values():
        c.close()
    line = json.dumps(rec, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
