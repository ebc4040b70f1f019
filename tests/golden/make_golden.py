#!/usr/bin/env python
"""Generates tests/golden/*.npy|*.npz from the UNMODIFIED reference (oracle/_ref).

Needs /root/reference and `make -C oracle ref`; run from the repo root:

    python tests/golden/make_golden.py

Outputs (committed; the GPU box has no /root/reference):
  win_<name>.npy   four 375-sps complex64 windows derived from the reference fixtures
                   (examples/VE3EMB.c2 conjugated as lib/c2file_source_impl.cc:91 does;
                   the wavs through oracle.testdata.frontend)
  whales_375sps.npy  channel 0 of examples/whales_12000sps.wav through the same front-end
  golden.npz       per case: reference candidates, the per-call refinement trace, the
                   decoder records, the published 7-byte blobs, spectrogram probes;
                   plus known-answer vectors for the SLM model, the encoder, the
                   deinterleaver and the decoder.
Cases = the four fixture windows (FDR hbw=10, maxdrift=0, thr=10, as in
examples/WaveFilePlusNoiseDecode.grc) + seeded synthetic windows at maxdrift 0 and 4.

    python tests/golden/make_golden.py --reference-cases [--from-repository]

writes only recorded_cases.npz: the reference's side of every case in tests/golden/reference_cases.py (what the
comparisons with the reference compare against where oracle/_ref is not built).  It needs oracle/_ref; with
--from-repository the answers come from this repository's side of the same cases instead, and the file's
`source` entry says so.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gr-uwspr_b200"))
from oracle import ref_binding as rb  # noqa: E402
from oracle import testdata as td  # noqa: E402

EX = "/root/reference/examples/"
OUT = os.path.join(ROOT, "tests", "golden")

SYNTH_CASES = [
    # (name, stream, window, snr_db, maxdrift)
    ("syn_m0_w0", 0, 0, -10.0, 0), ("syn_m0_w1", 0, 1, -20.0, 0), ("syn_m0_w2", 0, 2, -24.0, 0),
    ("syn_m0_w3", 0, 3, -27.0, 0), ("syn_m0_w4", 0, 4, -29.0, 0), ("syn_m0_w5", 0, 5, -31.0, 0),
    ("syn_m4_w0", 0, 0, -10.0, 4), ("syn_m4_w3", 0, 3, -27.0, 4), ("syn_m4_w6", 0, 6, -18.0, 4),
    ("syn_m4_w7", 0, 7, -23.0, 4),
]


def calls_array(calls):
    return np.frombuffer(b"".join(bytes(c) for c in calls), dtype=np.uint8).reshape(len(calls), -1) if calls else np.zeros((0, 216), np.uint8)


def fanos_array(fanos):
    a = np.frombuffer(b"".join(bytes(f) for f in fanos), dtype=np.uint8).reshape(len(fanos), -1).copy() if fanos else np.zeros((0, 192), np.uint8)
    if len(a):
        a[:, 172] = 0  # data[10] is never written by the reference decoder (Fano.cc:243-247)
    return a


def write_whales():
    """channel 0 of examples/whales_12000sps.wav at 375 sps (the interference of BASELINE.json configs[4];
    oracle.testdata.synth_array loops it)"""
    w, _ = td.read_wav(EX + "whales_12000sps.wav")
    y = td.frontend(w[:, 0]).astype(np.complex64)
    np.save(os.path.join(OUT, "whales_375sps.npy"), y)
    print("whales_375sps", y.shape, float(np.sqrt((np.abs(y) ** 2).mean())))


def write_reference_cases(ref):
    from tests.golden import reference_cases as rc
    if ref and not rb.available():
        raise SystemExit("oracle/_ref is not built (make -C oracle ref); --from-repository records this repository's side")
    golden = np.load(os.path.join(OUT, "golden.npz"))
    windows = {n: np.load(os.path.join(OUT, "win_%s.npy" % n)) for n in ("ve3emb_c2", "mix_whales")}
    out = dict(source=np.array("oracle/_ref (the unmodified upstream sources)" if ref else
                               "this repository: the oracle's C restatement; the library's unpacker and message-log formatter"))
    for name in rc.CASES:
        for k, v in rc.compute(name, ref, golden, windows).items():
            out[name + "/" + k] = v
    np.savez_compressed(rc.RECORDED, **out)
    print("wrote", rc.RECORDED, os.path.getsize(rc.RECORDED), "bytes, source:", out["source"])


def main():
    if "--reference-cases" in sys.argv:
        write_reference_cases(ref="--from-repository" not in sys.argv)
        return
    write_whales()
    if "--whales-only" in sys.argv:
        return
    wins = {}
    wins["ve3emb_c2"] = td.load_c2(EX + "VE3EMB.c2")
    a, _ = td.read_wav(EX + "test_1500_Hz.wav")
    b, _ = td.read_wav(EX + "150613_1920.wav")
    w, _ = td.read_wav(EX + "whales_12000sps.wav")
    wins["test_1500"] = td.frontend(a[:, 0])[:45000]
    wins["rec_150613"] = td.frontend(b[:, 0])[:45000]
    wl = np.resize(w[:, 0], len(a))
    wins["mix_whales"] = td.frontend(0.1 * a[:, 0] + 1.0 * wl)[:45000]
    for k, v in wins.items():
        np.save(os.path.join(OUT, "win_%s.npy" % k), v.astype(np.complex64))

    out = {}
    cases = [(k, v, 0) for k, v in wins.items()]
    for name, stream, window, snr, md in SYNTH_CASES:
        x, meta = td.synth_window(stream, window, snr_db=snr)
        cases.append((name, x, md))
        out[name + "/msg"] = meta["msg"]
    out["case_names"] = np.array([c[0] for c in cases])
    out["case_maxdrift"] = np.array([c[2] for c in cases])
    fdrs, sds = {}, {}
    for name, x, md in cases:
        if md not in fdrs:
            fdrs[md] = rb.RefFDR(maxdrift=md)
            sds[md] = rb.RefSD(maxdrift=md)
        cands, ps, psavg = fdrs[md].transform(x, want_ps=True)
        c2, blobs, calls, fanos = rb.pipeline(fdrs[md], sds[md], x)
        cands = td.canon_cands(cands)  # drop never-written / stale bytes
        assert td.canon_cands(c2).tobytes() == cands.tobytes()
        out[name + "/cands"] = cands.view(np.uint8).reshape(len(cands), 48)  # raw candidate_t records
        out[name + "/blobs"] = blobs
        out[name + "/calls"] = calls_array(calls)
        out[name + "/fanos"] = fanos_array(fanos)
        out[name + "/psavg"] = psavg
        out[name + "/ps_rows"] = ps[[0, 1, 100, 347], :]
        out[name + "/ps_sum"] = np.array([ps.astype(np.float64).sum()])
        print(name, "npk", len(cands), "blobs", blobs.tobytes().hex(), "calls", len(calls), "fanos", len(fanos))

    # known-answer vectors
    out["kat/slm_qa"] = np.array([rb.slm_frequency_drift(1, -2.0, 0, 50, 1500.0, float(i)) for i in range(120)], np.float32)
    traj = rb.slm_generate()
    out["kat/slm_traj"] = traj
    out["kat/slm_table"] = np.array(
        [[rb.slm_frequency_drift(t[0], t[1], int(t[2]), int(t[3]), 1500.0, float(k * 111 // 162)) for k in range(162)] for t in traj], np.float32)
    msg = np.array([0xD4, 0x2C, 0x73, 0xEB, 0x3A, 0x77, 0x80, 0, 0, 0, 0], np.uint8)
    out["kat/encode_in"] = msg
    out["kat/encode_out"] = rb.fano_encode(msg)
    sd = sds[0]
    out["kat/deinterleave_of_iota"] = sd.deinterleave(np.arange(162, dtype=np.uint8))
    out["kat/pr3"] = rb.pr3()
    out["kat/mettab"] = rb.fano_mettab()
    np.savez_compressed(os.path.join(OUT, "golden.npz"), **out)
    print("wrote", os.path.join(OUT, "golden.npz"))


if __name__ == "__main__":
    main()
