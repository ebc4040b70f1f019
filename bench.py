#!/usr/bin/env python
"""bench.py -- WSPR windows/s through coarse search + fine sync + soft-symbol demodulation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--windows M] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[2], the largest single-GPU configuration): M = 10 000
independent synthetic WSPR windows per GPU (45 000 complex64 samples at 375 sps each, 3.6 GB,
far larger than L2), SNR ~ U(-30, 0) dB in 2500 Hz, carrier offset U(-6, 6) Hz, linear drift
U(-3, 3) Hz, random start; FDR(hbw=10, maxdrift=4, maxfreqs=200, thr=10).  One step = one pass
of the whole hot path over the batch: spectrogram + normalizer + peak pick, coarse search,
the refinement chain and the soft symbols of all 17 jiggled shifts of every gated candidate
(the decoder-independent upper bound of what the reference evaluates; Fano is excluded from
the metric on both sides).

  value  device-resident input, results left on the device (kernels only, CUDA events)
  e2e    the same step through the C ABI with pinned HOST buffers: host->device copy of the
         samples and device->host copy of every result inside the timed region

Sub-records of the same JSON line (each with its own value / e2e / decoded counts):

  overlap50  BASELINE.json configs[3]: ONE stream, a frame every 45 000 samples, windows every
             22 500 samples, --overlap-windows (100 000) windows in total; rank r of N takes a
             contiguous slice of the windows and ships the contiguous span of samples they read
             once (uwspr_b200.sharding.stream_span) -- strong scaling, no collective
  sliding9   the same stream geometry at the example flowgraphs' own setting (configs[1]): windows every 9 s =
             3 375 samples, --sliding-windows (40 000) windows in total; a sample belongs to 13 windows and
             crosses PCIe once, windows start on odd samples (no 16-byte alignment)
  array64    BASELINE.json configs[4]: 64 hydrophone channels x --array-windows windows with the whale
             recording mixed in (gain ratio of the example flowgraph), maxdrift 0 (the flowgraphs'
             own setting), channels split contiguously over the ranks (8 per GPU at N = 8)
  receiver   the headline batch through the staged receive chain a streaming caller would run:
             fine sync with the first jiggle only, host Fano decoder on all cores, the other 16
             jiggles only for gated candidates still undecoded, decoder again
  verify     (N = 1) every window of the headline batch, a slice of the overlapped stream and of the
             array through the reference chain on the host, on the same samples (oracle/verify.py)

With N > 1 (torchrun) each rank runs the headline workload on its own GPU (weak scaling, no data-path
collective); time is the max over ranks, value the sum of windows / that time.  The host-fed arms
at N > 1 deal the windows to the ranks in proportion to each rank's measured host-fed rate, because
the host links of one box are not equally fast when every GPU copies at once (--no-balance: equal).
The synthetic inputs are made with the library's own encoder (uwspr_b200.synth); oracle/ is used by
the reference arm, the cpu_baseline leg and the verify leg only, never inside a timed GPU region.
--impl reference times the reference's own CPU implementation (oracle/_ref, the unmodified
sources; the C restatement if it was not built) on all host cores, on a bounded sample that is a
prefix of the GPU arm's batch.

--steps K sets the number of timed steps of every arm.  --dump-outputs DIR writes the headline step's
results for rank 0's batch (dump_outputs) as DIR/<name>.npy, so that two builds can be compared output
for output: the inputs are seeded and the same on every run with the same arguments.  The timed steps
leave their results on the device, where the library offers no way to read them back, so after the
timed steps the same call runs once more on the same device samples with its results fetched; that
call is untimed, and its candidate count must equal the last timed step's.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "gr-uwspr_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

FL = 45000
try:
    _ALL_CPUS = set(os.sched_getaffinity(0))
except Exception:
    _ALL_CPUS = set(range(os.cpu_count() or 1))
PARAMS = dict(fs=375, fl=FL, spb=256, maxdrift=4, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10)
PARAMS_ARRAY = dict(PARAMS, maxdrift=0)
METRIC = "WSPR windows/sec (coarse+fine sync+demod)"
FLOP_SPEC, FLOP_POINT = 9.09e6, 1.327e6
FP32_NONFUSED_PEAK, FP32_FMA_PEAK = 37.2, 74.4     # T lane-op/s: 148 SM x 128 lanes x 1.965 GHz (x2 with FMA)


def flop_coarse(maxdrift):
    return 5 * 26 * (2 * maxdrift + 126) * 162 * 9.0


# ------------------------------------------------------------------ CPU reference arm
def _cpu_worker(args):
    path, lo, hi, use_ref, params = args
    sys.path.insert(0, ROOT)
    xs = np.load(path, mmap_mode="r")
    t_fano = 0.0
    ncand = 0
    if use_ref:
        from oracle import ref_binding as rb
        fdr = rb.RefFDR(**params)
        sd = rb.RefSD(params["fs"], params["fl"], params["spb"], params["maxdrift"], params["maxfreqs"], params["cf"], logdir="/tmp")
        rb.fano_stats(reset=True)
        t0 = time.perf_counter()
        for w in range(lo, hi):
            c, blobs, calls, fanos = rb.pipeline(fdr, sd, np.ascontiguousarray(xs[w]))
            ncand += len(c)
        dt = time.perf_counter() - t0
        t_fano = rb.fano_stats()[0]
    else:
        from oracle import port_binding as ob
        f = ob.OracleFDR(**params)
        t0 = time.perf_counter()
        for w in range(lo, hi):
            x = np.ascontiguousarray(xs[w])
            c = f.transform(x)
            ob.demodulate(x, c, cf=params["cf"], run_fano=True)
            ncand += len(c)
        dt = time.perf_counter() - t0
    return hi - lo, dt, t_fano, ncand


def cpu_reference_run(xs_host, n_sample, cores):
    """windows/s of the reference CPU path on `cores` processes over the first n_sample windows.
    Decoder (Fano) time is measured by interposition and subtracted (it is outside the metric)."""
    import multiprocessing as mp
    from oracle import ref_binding as rb
    use_ref = rb.available()
    n_sample = min(n_sample, len(xs_host))
    path = "/dev/shm/uwspr_bench_%d.npy" % os.getpid()
    np.save(path, xs_host[:n_sample])
    try:
        bounds = [(n_sample * i) // cores for i in range(cores + 1)]
        jobs = [(path, bounds[i], bounds[i + 1], use_ref, PARAMS) for i in range(cores) if bounds[i + 1] > bounds[i]]
        ctx = mp.get_context("spawn")
        t0 = time.perf_counter()
        with ctx.Pool(len(jobs)) as pool:
            res = pool.map(_cpu_worker, jobs)
        wall = time.perf_counter() - t0
    finally:
        os.unlink(path)
    busy = max(r[1] - r[2] for r in res)          # slowest worker, decoder time removed
    n = sum(r[0] for r in res)
    fano = sum(r[2] for r in res)
    return dict(value=n / busy, unit="windows/s", cores=len(jobs), kind="reference" if use_ref else "port",
                sample="the first %d windows of the GPU arm's batch (rank 0), %d per core; decoder (Fano) time %.2f s of %.2f core-s "
                       "subtracted; stub FFT/PMT (see oracle/stubs); wall %.1f s incl. process start"
                       % (n, n // len(jobs), fano, sum(r[1] for r in res), wall),
                per_core=n / sum(r[1] - r[2] for r in res), candidates=sum(r[3] for r in res))


# ------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """median SM clock and the throttle reasons seen between wall-clock times t0 and t1
        (the timed region); samples are stamped when read from nvidia-smi's 50 ms loop"""
        if self.proc:
            self.proc.terminate()
        rows = [r for t, r in self.rows if len(r) >= 8 and (t0 is None or t0 - 0.05 <= t <= t1 + 0.05)]
        if not rows:
            rows = [r for t, r in self.rows if len(r) >= 8]
        num = lambda v: float(v) if v.replace(".", "", 1).isdigit() else None  # noqa: E731
        sm = sorted(v for v in (num(r[1]) for r in rows) if v is not None)
        mx = [v for v in (num(r[2]) for r in rows) if v is not None]
        pw = [v for v in (num(r[3]) for r in rows) if v is not None]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(pw) if pw else None, reasons=sorted(reasons), samples=len(sm))


def recorded_traffic(nwin):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture
    (profiles/traffic.json, written from `ncu --set full` by tools/ncu_summary.py --traffic);
    only returned when the capture was taken at this workload size"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if int(t.get("windows", -1)) == int(nwin):
            return float(t["k_fine_dram_bytes"])
    except Exception:
        pass
    return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def whales_fixture():
    return np.load(os.path.join(ROOT, "tests", "golden", "whales_375sps.npy"))


DUMP_BYTES = 64 << 20
DUMP_WINDOWS, DUMP_CANDIDATES, DUMP_SOFT_CANDIDATES = 1 << 18, 1 << 15, 1 << 11


def _sample(n, k, seed):
    """all of range(n), or a fixed seeded sample of k of them in increasing order"""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(path, npk, cands, refined, jig, soft):
    """writes the arrays coarse_fine returns (npk, cands, refined, jig, soft) as path/<name>.npy, one file per
    field, in float32 (float fields, soft symbols) or float64 (integer fields, indices).  Where there are more
    windows or candidates than DUMP_BYTES holds, a fixed seeded sample of them is written; *_index.npy says which.
    Union fields are written where they are defined (lin_drift for linear candidates, V1, V2, p1, p2 for
    nonlinear ones) and are 0 elsewhere; candidate_t.drift is never written by the reference and is left out."""
    wi = _sample(len(npk), DUMP_WINDOWS, 1)
    ci = _sample(len(cands), DUMP_CANDIDATES, 2)
    si = _sample(len(cands), DUMP_SOFT_CANDIDATES, 3)
    c, r, j = cands[ci], refined[ci], jig[ci]
    lin, nonlin = c["m_type"] == 0, c["m_type"] == 1
    f32, f64 = (lambda a: np.asarray(a, np.float32)), (lambda a: np.asarray(a, np.float64))
    out = dict(counts=f64([len(npk), len(cands)]), window_index=f64(wi), npk=f64(npk[wi]), cand_index=f64(ci),
               cand_freq=f32(c["freq"]), cand_snr=f32(c["snr"]), cand_sync=f32(c["sync"]), cand_shift=f64(c["shift"]),
               cand_m_type=f64(c["m_type"]), cand_lin_drift=f32(np.where(lin, c["lin_drift"], 0)),
               cand_V1=f64(np.where(nonlin, c["V1"], 0)), cand_V2=f64(np.where(nonlin, c["V2"], 0)),
               cand_p1=f64(np.where(nonlin, c["p1"], 0)), cand_p2=f64(np.where(nonlin, c["p2"], 0)),
               refined_f1=f32(r["f1"]), refined_shift1=f64(r["shift1"]), refined_drift1=f32(r["drift1"]),
               refined_sync1=f32(r["sync1"]), refined_worth_a_try=f64(r["worth_a_try"]),
               jig_sync=f32(j["sync"]), jig_rms=f32(j["rms"]), jig_shift=f64(j["shift"]), jig_gate=f64(j["gate"]),
               soft_index=f64(si), soft=f32(soft[si]))
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_BYTES, total
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)
    return total


# ------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(_ALL_CPUS) or os.cpu_count() or 1
    n = min(args.windows, max(cores, args.ref_windows))
    # the sample is the prefix of the GPU arm's batch (same generator, same keys); the generator needs torch,
    # on the GPU when there is one (bit-identical to the GPU arm's data), else on the CPU (same distribution)
    import torch
    from uwspr_b200 import synth
    dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    xs_t, _ = synth.gen_frames(0, n, 0, dev)
    xs = xs_t.cpu().numpy()
    del xs_t
    vals = []
    for step in range(args.warmup + args.steps):
        r = cpu_reference_run(xs, n, cores)
        if step >= args.warmup:
            vals.append(r)
    v = float(np.mean([r["value"] for r in vals]))
    line = dict(metric=METRIC, value=v, unit="windows/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * n / v, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload="the first %d windows of the GPU arm's batch (10k synthetic WSPR windows, SNR U(-30,0) dB, drift U(-3,3) Hz), "
                                     "FDR hbw=10 maxdrift=4 thr=10; generated on %s" % (n, dev.type),
                            windows=n, **{k: PARAMS[k] for k in ("maxdrift", "halfbandwidth", "threshold", "maxfreqs")}),
                cpu_baseline=dict(vals[-1], value=v),
                e2e=dict(value=v, unit="windows/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------ our arm
class Harness:
    """timing plumbing shared by the workloads: barriers, CUDA events on the context's stream, max over ranks"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            # NCCL writes its version / debug lines to stdout by default; stdout carries the one JSON line
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.stream = torch.cuda.current_stream(self.dev)
        self.args = args
        self.group = dist if self.world > 1 else None

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def timed(self, fn, steps):
        """ms for `steps` calls of fn, max over ranks"""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def sum_ints(self, v):
        from uwspr_b200.sharding import gather_counts
        return sum(gather_counts(int(v), self.group))

    def pinned(self, t):
        """pinned host copy of a device tensor"""
        h = self.torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        self.torch.cuda.synchronize(self.dev)
        return h


def window_of_candidates(npk):
    return np.repeat(np.arange(len(npk)), npk)


def score_decodes(ub, npk, refined, jig, soft, truth_of_window, limit_windows=None):
    """host decoder over fetched results; (messages published, messages equal to the transmitted payload,
    windows with their payload recovered, windows scored).  truth_of_window(w) -> 7 bytes or None."""
    nw = len(npk) if limit_windows is None else min(len(npk), limit_windows)
    ncand = int(np.sum(npk[:nw]))
    dec = ub.decode_candidates(refined[:ncand], jig[:ncand], soft[:ncand])
    win = window_of_candidates(npk[:nw])
    good, heard = 0, set()
    for g, m, _ in dec:
        w = int(win[g])
        t = truth_of_window(w)
        ts = [] if t is None else (list(t) if isinstance(t, (list, tuple)) else [t])
        if any(bytes(m) == bytes(x) for x in ts):
            good += 1
            heard.add(w)
    return dict(messages=len(dec), correct=good, windows_heard=len(heard), windows=nw), dec


def run_ours(args):
    H = Harness(args)
    torch, dist = H.torch, H.dist
    import uwspr_b200 as ub
    from uwspr_b200 import synth
    from uwspr_b200.sharding import balanced_counts, gather_counts, gather_floats
    world, rank, dev = H.world, H.rank, H.dev
    steps, warmup = args.steps, args.warmup
    skip = set(s for s in args.skip.split(",") if s)

    sampler = ClockSampler(H.local)
    if rank == 0:
        sampler.start()

    # ======================================================================== headline: configs[2]
    nwin = args.windows
    balance = world > 1 and not args.no_balance
    nmax = int(1.5 * nwin) if balance else nwin
    ctx = ub.Context(device=H.local, max_windows=nmax, max_candidates=max(4 * nmax, 1024), **PARAMS)
    ctx.set_stream(H.stream.cuda_stream)
    xs_dev, truth = synth.gen_frames(0, nwin, rank, dev)
    dptr = (xs_dev.data_ptr(), nwin * FL)
    xs_host_t = torch.empty((nmax, FL), dtype=torch.complex64, pin_memory=True)
    xs_host_t[:nwin].copy_(xs_dev)
    if nmax > nwin:
        extra, truth_extra = synth.gen_frames(nwin, nmax - nwin, rank, dev)
        xs_host_t[nwin:].copy_(extra)
        truth = list(truth) + list(truth_extra)
        del extra
    torch.cuda.synchronize(dev)
    xs_host = xs_host_t.numpy()
    out_bufs = ctx.result_buffers(nmax)   # pinned, allocated once (as a streaming caller would)

    stage_ms = np.zeros(4)
    totals = []

    def step_dev():
        totals.append(ctx.coarse_fine(dptr, nwin=nwin, stride=FL, fetch=False))
        stage_ms[:] += ctx.last_timing()

    n_e2e = [nwin]
    e2e_out = {}

    def step_e2e():
        e2e_out["r"] = ctx.coarse_fine(xs_host.reshape(-1), nwin=n_e2e[0], stride=FL, out=out_bufs)

    for _ in range(warmup):
        step_dev()
    stage_ms[:] = 0
    l0 = ctx.launch_count()
    t_w0 = time.time()
    ms = H.timed(step_dev, steps)
    t_w1 = time.time()
    launches = ctx.launch_count() - l0
    st = stage_ms / steps
    ncand_dev = totals[-1]
    if args.dump_outputs and rank == 0:
        # a recompute: the timed calls leave their results on the device, and the library has no call to read them
        # back; the same call on the same device samples, untimed and with results fetched, returns them
        res = ctx.coarse_fine(dptr, nwin=nwin, stride=FL, out=out_bufs)
        assert len(res[1]) == ncand_dev, (len(res[1]), ncand_dev)
        dump_outputs(args.dump_outputs, *res)
    for _ in range(min(warmup, 1) or 1):
        step_e2e()
    e2e_counts = [nwin] * world
    rates = [1.0] * world
    if balance:
        # three rounds: the rates seen under an equal split are already those of full contention for the
        # fast links; the later rounds correct the slow ones (they sped up once the fast ranks had finished)
        for _ in range(3):
            H.barrier()
            t0 = time.perf_counter()
            step_e2e()
            torch.cuda.synchronize(dev)
            rates = gather_floats(n_e2e[0] / (time.perf_counter() - t0), dist)
            e2e_counts = balanced_counts(world * nwin, rates, lo=max(1, nwin // 4), hi=nmax)
            n_e2e[0] = e2e_counts[rank]
    ms_e2e = H.timed(step_e2e, steps)
    clocks = sampler.stop(t_w0, t_w1) if rank == 0 else None
    h2d = nwin * FL * 8
    # context for the end-to-end number: the plain pinned-host -> device copy rate of this box
    scratch = torch.empty_like(xs_dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch.copy_(xs_host_t[:nwin], non_blocking=True)
    H.barrier()   # every rank copies at the same time, as in the host-fed steps
    ev0.record(H.stream)
    scratch.copy_(xs_host_t[:nwin], non_blocking=True)
    ev1.record(H.stream)
    torch.cuda.synchronize(dev)
    pcie_gbs = h2d / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
    pcie_all = gather_floats(pcie_gbs, H.group)
    del scratch
    # statistics and correctness come from the DEVICE arm's own batch (this rank's first nwin windows):
    # one more untimed host-fed pass over exactly those windows
    npk, cands, refined, jig, soft = [np.array(a, copy=True) for a in
                                      ctx.coarse_fine(xs_host.reshape(-1), nwin=nwin, stride=FL, out=out_bufs)]
    d2h_main = npk.nbytes + cands.nbytes + refined.nbytes + jig.nbytes + soft.nbytes
    ncand = len(cands)
    gated = int(refined["worth_a_try"].sum())
    nonlin = int((cands["m_type"] == 1).sum())
    evals = 12 * ncand - 2 * nonlin + (10 + 17) * gated     # sync_and_demodulate() points of the reference
    tot_windows = sum(gather_counts(nwin, H.group))
    tot_cand, tot_gated, tot_evals = H.sum_ints(ncand), H.sum_ints(gated), H.sum_ints(evals)
    value = tot_windows * steps / (ms / 1e3)
    e2e_value = tot_windows * steps / (ms_e2e / 1e3)
    decoded_main, dec_main = score_decodes(ub, npk, refined, jig, soft, lambda w: truth[w]["msg"])

    # ======================================================================== receiver: staged jiggles + host decoder
    receiver = None
    if "receiver" not in skip:
        receiver = bench_receiver(H, ub, ctx, xs_host, nwin, out_bufs, truth, dec_main, steps)

    verify_jobs = []
    do_verify = (world == 1 and not args.no_verify) or args.verify
    if do_verify and rank == 0:
        nv = min(nwin, args.verify_windows)
        base = np.concatenate([[0], np.cumsum(npk)])
        msgs_of = [[] for _ in range(nv)]
        win = window_of_candidates(npk)
        for g, m, _ in dec_main:
            if win[g] < nv:
                msgs_of[int(win[g])].append(bytes(m))
        k = int(base[nv])
        verify_jobs.append(("headline", dict(stream=np.array(xs_host[:nv], copy=True).reshape(-1), stride=FL, nwin=nv, params=PARAMS,
                                              npk=npk[:nv], cands=cands[:k], refined=refined[:k], jig=jig[:k], soft=soft[:k],
                                              gpu_messages=msgs_of, full=min(nv, args.verify_full_jiggle))))

    main_stats = dict(stage_ms=st, fine_ms=float(st[2]), ncand=ncand_dev)
    ctx.close()
    del ctx, out_bufs, xs_dev, xs_host_t, xs_host
    torch.cuda.empty_cache()

    # ======================================================================== overlap50: configs[3]
    overlap = None
    if "overlap50" not in skip:
        overlap = bench_stream(H, ub, synth, rates if balance else None, verify_jobs if do_verify else None, "overlap50",
                               args.overlap_windows, FL // 2, args.verify_overlap_windows)
    sliding = None
    if "sliding9" not in skip:
        sliding = bench_stream(H, ub, synth, rates if balance else None, verify_jobs if do_verify else None, "sliding9",
                               args.sliding_windows, 9 * 375, args.verify_sliding_windows)
    # ======================================================================== array64: configs[4]
    array = None
    if "array64" not in skip:
        array = bench_array64(H, ub, synth, verify_jobs if do_verify else None)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ======================================================================== verification against the reference chain
    verify = None
    if verify_jobs:
        from oracle import verify as vf
        try:
            os.sched_setaffinity(0, _ALL_CPUS)
        except Exception:
            pass
        verify = {}
        for name, job in verify_jobs:
            prm = job["params"]

            def dbg(n, prm=prm):
                c = ub.Context(device=H.local, max_windows=max(n, 1), **prm)
                c.set_debug(True)
                return c
            verify[name] = vf.verify(job["stream"], job["stride"], job["nwin"], prm, job["npk"], job["cands"], job["refined"],
                                     job["jig"], job["soft"], job["gpu_messages"], cores=len(_ALL_CPUS),
                                     full_jiggle_windows=job["full"], make_debug_context=dbg)

    # ======================================================================== CPU baseline (rank 0, N = 1)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cores = len(_ALL_CPUS) or os.cpu_count() or 1
        xs_cpu, _ = synth.gen_frames(0, min(nwin, max(cores, args.ref_windows)), rank, dev)
        cpu = cpu_reference_run(xs_cpu.cpu().numpy(), len(xs_cpu), cores)
        del xs_cpu

    peaks = measured_peaks()
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    fine_ms, spec_ms, coarse_ms = float(st[2]), float(st[0]), float(st[1])
    alg_bytes = 360000.0 * nwin + 2818.0 * ncand
    alg_flops = tot_windows * FLOP_SPEC + tot_cand * flop_coarse(PARAMS["maxdrift"]) + tot_evals * FLOP_POINT
    info_nbp = 44
    fine_alg_t = evals * FLOP_POINT / (fine_ms * 1e-3) / 1e12
    # executed fp32 lane-operations of the fine path per candidate: the chain evaluates 19 new points with
    # routine R1 (14 mul/add per tone-sample: 8 for the two correlations, 6 for the table rotation) and 16 jiggles
    # with R2 (8 per lag + 6 per lag group of 4, 4 groups; jiggle 0 is the refined point itself and is taken from the
    # stage that evaluated it); the packed forms carry two of them per instruction
    fine_exec = gated * (19 * 14 + (16 * 8 + 4 * 6)) * 162 * 4 * 256 + (ncand - gated) * 11 * 14 * 162 * 4 * 256
    fine_exec_t = fine_exec / (fine_ms * 1e-3) / 1e12
    coarse_alg_t = ncand * flop_coarse(PARAMS["maxdrift"]) / (coarse_ms * 1e-3) / 1e12
    spec_bytes = nwin * (360000.0 + 348 * info_nbp * 4)
    rooflines = [
        dict(kernel="fine path: k_fine_points (stages A-D) + k_fine_lags (stage E) + k_fine_step / k_fine_finish", ms=fine_ms,
             bound="fp32 pipe, non-fused (separately rounded mul and add, as the reference's sums require)",
             algorithmic=dict(achieved=fine_alg_t, unit="TFLOP/s", frac_of_fma_peak=fine_alg_t / FP32_FMA_PEAK, frac_of_nonfused_peak=fine_alg_t / FP32_NONFUSED_PEAK,
                              note="reference operation count: 162 x 4 x 256 x 8 flop per evaluated point (SURVEY 8(d))"),
             executed=dict(achieved=fine_exec_t, unit="T lane-op/s", frac_of_nonfused_peak=fine_exec_t / FP32_NONFUSED_PEAK,
                           frac_of_measured_nonfused=fine_exec_t / 35.1,
                           note="model count of the mul/add lane-operations the generic routines issue (table rotation included); an upper "
                                "bound: constant-frequency points run 8 instead of 14 per tone-sample. Measured non-fused rate 35.1 T/s "
                                "from tools/fp32_pipes.cu (profiles/r2_fp32_pipes.txt)")),
        dict(kernel="k_spectrogram", ms=spec_ms, bound="hbm (nominal; in practice shared-memory exchange + issue, see DESIGN.md 4.1)",
             achieved=spec_bytes / (spec_ms * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s", frac=spec_bytes / (spec_ms * 1e-3) / 1e9 / hbm_peak),
        dict(kernel="k_coarse", ms=coarse_ms, bound="fp32 adds + shared loads",
             achieved=coarse_alg_t, unit="TFLOP/s", frac_of_fma_peak=coarse_alg_t / FP32_FMA_PEAK,
             note="reference operation count (all 125 trajectories); only the distinct offset sequences are evaluated, so the "
                  "algorithmic rate may exceed what the pipes execute"),
    ]
    line = dict(
        metric=METRIC, value=value, unit="windows/s", n_gpus=world, steps=steps, warmup=warmup,
        ms_per_step=ms / steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
        config=dict(workload="10k synthetic WSPR windows swept over SNR -30..0 dB with random drift, 1 B200 (BASELINE.json configs[2]); per GPU",
                    windows_per_gpu=nwin, input_bytes_per_gpu=h2d, l2="inputs larger than L2 (3.6 GB vs 126 MB)",
                    jiggles="all 17 per gated candidate", candidates=tot_cand, gated=tot_gated, sync_evaluations=tot_evals,
                    counts="candidates / gated / sync_evaluations are summed over the ranks' device-arm batches",
                    **{k: PARAMS[k] for k in ("maxdrift", "halfbandwidth", "threshold", "maxfreqs")}),
        e2e=dict(value=e2e_value, unit="windows/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=int(d2h_main), ms_per_step=ms_e2e / steps,
                 pcie_h2d_gbs=pcie_gbs, pcie_h2d_gbs_per_rank=[round(v, 2) for v in pcie_all],
                 pcie_bound_windows_per_s=sum(pcie_all) * 1e9 / (h2d / nwin),
                 windows_per_rank=e2e_counts,
                 split=("windows split over the ranks in proportion to each rank's measured host-fed rate "
                        "(uwspr_b200.sharding.balanced_counts); same total as the equal split" if balance else "equal")),
        gpu_launches=int(launches),
        stage_ms=dict(spectrogram_normalizer=spec_ms, coarse_search=coarse_ms, fine_sync_demod=fine_ms, call=float(st[3])),
        roofline=dict(bound="hbm", kernel="fine path (k_fine_points + k_fine_lags: fine sync + soft symbols)", achieved=alg_bytes / (fine_ms * 1e-3) / 1e9, peak=hbm_peak,
                      unit="GB/s", frac=alg_bytes / (fine_ms * 1e-3) / 1e9 / hbm_peak, traffic=recorded_traffic(nwin),
                      launches_per_step="the fine path is a sequence of launches per slice of candidates; `achieved` uses their summed device time",
                      peak_source="MEASURED_PEAKS.json (measured copy)" if peaks else "fallback 6650 GB/s",
                      note="the dominant kernel is FP32-pipe bound, not HBM bound: see rooflines[0]"),
        rooflines=rooflines,
        roofline_fp32=dict(bound="fp32 (non-fused)", achieved=alg_flops / (ms / steps * 1e-3) / 1e12, peak=FP32_NONFUSED_PEAK, unit="TFLOP/s",
                           frac=alg_flops / (ms / steps * 1e-3) / 1e12 / FP32_NONFUSED_PEAK, peak_fma=FP32_FMA_PEAK,
                           note="whole step, all ranks: algorithmic flops of the reference operation count / step time; per-kernel figures in `rooflines`"),
        decoded=dict(decoded_main, frames=nwin),
        overlap50=overlap, sliding9=sliding, array64=array, receiver=receiver, verify=verify,
        clocks=clocks, cpu_baseline=cpu,
    )
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_receiver(H, ub, ctx, xs_host, nwin, out_bufs, truth, dec_full, steps):
    """The receive chain a streaming caller runs on the headline batch (host-fed): coarse + refinement + the first
    jiggle, host decoder, then jiggles 1..16 only for gated candidates still undecoded, decoder again
    (sync_and_demodulate_impl.cc:457-490 stops at the first decode too).  Everything, host decoder included, is inside
    the timed region (wall clock: the decoder runs on the host cores)."""
    torch = H.torch
    cores = max(1, len(_ALL_CPUS) // max(1, H.world))
    stats = {}
    bufs1 = ctx.result_buffers(nwin, jig_count=1)   # pinned result buffers of the one-jiggle pass

    def one():
        t0 = time.perf_counter()
        npk, cands, refined, jig, soft = ctx.coarse_fine(xs_host.reshape(-1), nwin=nwin, stride=FL, jig_first=0, jig_count=1, out=bufs1)
        t1 = time.perf_counter()
        dec1 = ub.decode_candidates(refined, jig, soft, nthreads=cores)
        t2 = time.perf_counter()
        done = np.zeros(len(cands), bool)
        done[[g for g, _, _ in dec1]] = True
        retry = np.flatnonzero(~done & (refined["worth_a_try"] != 0))
        msgs = {g: bytes(m) for g, m, _ in dec1}
        t3 = t4 = t2
        if len(retry):
            win = window_of_candidates(npk)
            npk2 = np.bincount(win[retry], minlength=nwin).astype(np.int32)
            r2, j2, s2 = ctx.fine(xs_host.reshape(-1), npk2, cands[retry], nwin=nwin, stride=FL, jig_first=1, jig_count=16)
            t3 = time.perf_counter()
            dec2 = ub.decode_candidates(r2, j2, s2, nthreads=cores)
            t4 = time.perf_counter()
            for k, m, _ in dec2:
                msgs[int(retry[k])] = bytes(m)
        stats.update(device_1=t1 - t0, decode_1=t2 - t1, device_2=t3 - t2, decode_2=t4 - t3, retry=len(retry), cands=len(cands), msgs=msgs)
        return t4 - t0

    one()
    H.barrier()
    t = [one() for _ in range(steps)]
    sec = float(np.mean(t))
    tt = torch.tensor([sec], device=H.dev)
    if H.world > 1:
        H.dist.all_reduce(tt, op=H.dist.ReduceOp.MAX)
    full = {g: bytes(m) for g, m, _ in dec_full}
    return dict(value=H.world * nwin / float(tt.item()), unit="windows/s", steps=steps, host_threads=cores,
                seconds=dict(device_first_jiggle=stats["device_1"], host_decode_first=stats["decode_1"],
                             device_other_jiggles=stats["device_2"], host_decode_rest=stats["decode_2"]),
                candidates=stats["cands"], retried=stats["retry"], messages=len(stats["msgs"]),
                same_messages_as_full_evaluation=bool(stats["msgs"] == full),
                note="rank 0's breakdown; host-fed, host Fano decoder included (outside the headline metric); a gated candidate that never "
                     "decodes costs 17 decoder time-outs of 10000 x 81 cycles, the reference's own limit")


def bench_stream(H, ub, synth, rates, verify_jobs, name, W, stride, nverify):
    """one synthetic stream (a frame every 45 000 samples), W windows every `stride` samples, contiguous slices per rank"""
    from uwspr_b200.sharding import balanced_counts, gather_floats, shard_range
    args, world, rank, dev = H.args, H.world, H.rank, H.dev
    steps = args.steps
    # device-resident arm: equal contiguous slices
    lo, hi = shard_range(W, rank, world)
    # host-fed arm: contiguous slices in proportion to the host-link rates measured by the headline arm
    if rates is not None:
        counts = balanced_counts(W, rates, lo=max(1, W // (4 * world)), hi=min(W, int(1.6 * W / world) + 1))
    else:
        counts = [shard_range(W, r, world)[1] - shard_range(W, r, world)[0] for r in range(world)]
    elo = sum(counts[:rank])
    ehi = elo + counts[rank]
    nmaxw = max(hi - lo, ehi - elo)
    ctx = ub.Context(device=H.local, max_windows=nmaxw, max_candidates=max(3 * nmaxw, 1024), **PARAMS)
    ctx.set_stream(H.stream.cuda_stream)
    span, f_lo, truth = synth.gen_stream_span(lo, hi, stride, 777, dev)
    nw = hi - lo
    dptr = (span.data_ptr(), span.numel())
    if (elo, ehi) == (lo, hi):
        host_t = H.pinned(span)
        e_flo, e_truth = f_lo, truth
    else:
        espan, e_flo, e_truth = synth.gen_stream_span(elo, ehi, stride, 777, dev)
        host_t = H.pinned(espan)
        del espan
    host = host_t.numpy()
    enw = ehi - elo
    out_bufs = ctx.result_buffers(enw)
    totals = []

    def step_dev():
        totals.append(ctx.coarse_fine(dptr, nwin=nw, stride=stride, fetch=False))

    res = {}

    def step_e2e():
        res["r"] = ctx.coarse_fine(host, nwin=enw, stride=stride, out=out_bufs)

    for _ in range(min(args.warmup, 2)):
        step_dev()
    ms = H.timed(step_dev, steps)
    step_e2e()
    ms_e2e = H.timed(step_e2e, steps)
    npk, cands, refined, jig, soft = res["r"]
    d2h = npk.nbytes + cands.nbytes + refined.nbytes + jig.nbytes + soft.nbytes
    h2d = host.nbytes
    link = gather_floats(h2d * steps / (ms_e2e * 1e-3) / 1e9, H.group)

    # correctness on a bounded prefix of this rank's host-fed slice: a published message must be the payload of a
    # frame the window overlaps (a window whose start falls a little after a frame's start can still decode it);
    # `windows_holding_a_frame` counts the windows with a frame start inside the first 3 328 samples, the range the
    # coarse search looks at
    def frames_of(w):
        s0 = (elo + w) * stride
        return [f for f in (s0 // FL, s0 // FL + 1) if 0 <= f - e_flo < len(e_truth)]

    def truth_of(w):
        return [e_truth[f - e_flo]["msg"] for f in frames_of(w)]

    def holds_frame(w):
        s0 = (elo + w) * stride
        return any(0 <= f * FL + e_truth[f - e_flo]["start"] - s0 < 3328 for f in frames_of(w))
    nscore = min(enw, args.decode_limit)
    decoded, dec = score_decodes(ub, npk, refined, jig, soft, truth_of, limit_windows=nscore)
    frames_scored = sum(1 for w in range(nscore) if holds_frame(w))
    if verify_jobs is not None and rank == 0:
        nv = min(enw, nverify)
        base = np.concatenate([[0], np.cumsum(npk)])
        msgs_of = [[] for _ in range(nv)]
        win = window_of_candidates(npk[:nscore])
        for g, m, _ in dec:
            if win[g] < nv:
                msgs_of[int(win[g])].append(bytes(m))
        k = int(base[nv])
        verify_jobs.append((name, dict(stream=np.array(host[:(nv - 1) * stride + FL], copy=True), stride=stride, nwin=nv, params=PARAMS,
                                              npk=np.array(npk[:nv]), cands=np.array(cands[:k]), refined=np.array(refined[:k]),
                                              jig=np.array(jig[:k]), soft=np.array(soft[:k]), gpu_messages=msgs_of, full=0)))
    ncand = H.sum_ints(totals[-1])
    out = dict(workload="one synthetic stream, a frame every 45 000 samples, windows every %d samples (%s); "
                        "%d windows in total, contiguous slices per rank, each rank's span shipped once"
                        % (stride, "50 % overlap, BASELINE.json configs[3]" if stride == FL // 2 else
                           "shift = %g s as in the example flowgraphs' sliding_window_stream_to_pdu" % (stride / 375.0), W),
               scaling="strong", windows=W, steps=steps, value=W * steps / (ms / 1e3), unit="windows/s", ms_per_step=ms / steps,
               e2e=dict(value=W * steps / (ms_e2e / 1e3), unit="windows/s", ms_per_step=ms_e2e / steps,
                        h2d_bytes_per_step_rank0=int(h2d), d2h_bytes_per_step_rank0=int(d2h), windows_per_rank=counts,
                        link_gbs_per_rank=[round(v, 2) for v in link],
                        split="equal" if rates is None else "contiguous slices in proportion to the host-link rates of the headline arm"),
               candidates=ncand, decoded=dict(decoded, windows_holding_a_frame=frames_scored,
                            note="rank 0, first %d windows of its slice; `correct` counts published messages equal to the payload of "
                                 "a frame the window overlaps, `messages` everything published" % nscore))
    ctx.close()
    return out


def bench_array64(H, ub, synth, verify_jobs):
    from uwspr_b200.sharding import shard_range
    args, world, rank, dev = H.args, H.world, H.rank, H.dev
    nchan, nwin_c = args.array_channels, args.array_windows
    c_lo, c_hi = shard_range(nchan, rank, world)
    nch = c_hi - c_lo
    whales = whales_fixture()
    x, truth = synth.gen_array(c_lo, c_hi, nwin_c, whales, dev)     # [nch, nwin_c, FL]
    nw = nch * nwin_c                                               # flattened (channel, window), contiguous per channel
    ctx = ub.Context(device=H.local, max_windows=max(nw, 1), max_candidates=max(8 * nw, 1024), **PARAMS_ARRAY)
    ctx.set_stream(H.stream.cuda_stream)
    dptr = (x.data_ptr(), x.numel())
    host_t = H.pinned(x)
    host = host_t.numpy().reshape(-1)
    out_bufs = ctx.result_buffers(max(nw, 1))
    totals, res, st = [], {}, np.zeros(4)

    def step_dev():
        totals.append(ctx.coarse_fine(dptr, nwin=nw, stride=FL, fetch=False))
        st[:] += ctx.last_timing()

    def step_e2e():
        res["r"] = ctx.coarse_fine(host, nwin=nw, stride=FL, out=out_bufs)

    for _ in range(min(args.warmup, 2)):
        step_dev()
    st[:] = 0
    ms = H.timed(step_dev, args.steps)
    st /= args.steps
    step_e2e()
    ms_e2e = H.timed(step_e2e, args.steps)
    npk, cands, refined, jig, soft = res["r"]
    d2h = npk.nbytes + cands.nbytes + refined.nbytes + jig.nbytes + soft.nbytes
    decoded, dec = score_decodes(ub, npk, refined, jig, soft, lambda i: truth[i % nwin_c]["msg"])
    if verify_jobs is not None and rank == 0:
        # the first windows of every local channel: (channel, window) pairs of a small slice
        wv = min(nwin_c, args.verify_array_windows)
        idx = np.array([c * nwin_c + w for c in range(nch) for w in range(wv)])
        base = np.concatenate([[0], np.cumsum(npk)])
        sel = np.concatenate([np.arange(base[i], base[i + 1]) for i in idx]) if len(idx) else np.zeros(0, int)
        win = window_of_candidates(npk)
        msgs_all = {}
        for g, m, _ in dec:
            msgs_all.setdefault(int(win[g]), []).append(bytes(m))
        hx = host_t.numpy().reshape(nch * nwin_c, FL)
        verify_jobs.append(("array64", dict(stream=np.ascontiguousarray(hx[idx]).reshape(-1), stride=FL, nwin=len(idx), params=PARAMS_ARRAY,
                                            npk=np.array(npk[idx]), cands=np.array(cands[sel]), refined=np.array(refined[sel]),
                                            jig=np.array(jig[sel]), soft=np.array(soft[sel]),
                                            gpu_messages=[msgs_all.get(int(i), []) for i in idx], full=len(idx))))
    W = nchan * nwin_c
    out = dict(workload="%d-channel synthetic hydrophone array x %d windows, whale recording mixed in at gain 1.0 against signal gains U(0.05, 0.2) "
                        "(BASELINE.json configs[4]); maxdrift 0 (the example flowgraphs' setting); channels split contiguously over the ranks" % (nchan, nwin_c),
               scaling="strong", channels=nchan, channels_per_rank=[shard_range(nchan, r, world)[1] - shard_range(nchan, r, world)[0] for r in range(world)],
               windows=W, value=W * args.steps / (ms / 1e3), unit="windows/s", ms_per_step=ms / args.steps,
               e2e=dict(value=W * args.steps / (ms_e2e / 1e3), unit="windows/s", ms_per_step=ms_e2e / args.steps,
                        h2d_bytes_per_step_rank0=int(host.nbytes), d2h_bytes_per_step_rank0=int(d2h)),
               stage_ms_rank0=dict(spectrogram_normalizer=float(st[0]), coarse_search=float(st[1]), fine_sync_demod=float(st[2])),
               candidates=H.sum_ints(totals[-1]), gated_rank0=int(refined["worth_a_try"].sum()),
               decoded=dict(decoded, note="rank 0's channels; windows_heard counts (channel, window) pairs whose payload was recovered"))
    ctx.close()
    return out


def main():
    # stdout carries exactly one JSON line.  Libraries (NCCL prints its version with printf) write to
    # file descriptor 1, so fd 1 is pointed at stderr and Python's sys.stdout keeps the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--windows", type=int, default=10000, help="headline windows per GPU")
    ap.add_argument("--overlap-windows", type=int, default=100000, help="overlap50: windows of the one stream, all ranks together")
    ap.add_argument("--sliding-windows", type=int, default=40000, help="sliding9: windows of the one stream (shift 9 s), all ranks together")
    ap.add_argument("--verify-sliding-windows", type=int, default=1000)
    ap.add_argument("--array-channels", type=int, default=64)
    ap.add_argument("--array-windows", type=int, default=156, help="array64: windows per channel")
    ap.add_argument("--decode-limit", type=int, default=20000, help="overlap50: windows of rank 0's slice scored with the host decoder")
    ap.add_argument("--ref-windows", type=int, default=1024, help="windows of the CPU reference sample")
    ap.add_argument("--verify-windows", type=int, default=10000)
    ap.add_argument("--verify-full-jiggle", type=int, default=1000, help="headline windows whose 17 jiggles are all compared")
    ap.add_argument("--verify-overlap-windows", type=int, default=2000)
    ap.add_argument("--verify-array-windows", type=int, default=4, help="windows per channel compared in the array64 slice")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--verify", action="store_true", help="run the verification leg at N > 1 as well (rank 0)")
    ap.add_argument("--skip", default="", help="comma list of sub-records to leave out: overlap50,sliding9,array64,receiver")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-balance", action="store_true", help="host-fed arms at N > 1: equal split instead of link-rate balanced")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, recompute the headline step once with results fetched and write them "
                                                           "(rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's results; the reference arm has none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
