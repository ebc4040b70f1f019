"""bench.py --dump-outputs: float32 / float64 files within 64 MB, the same on every call, and equal to what the
library returns for the benchmark's own seeded batch."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import uwspr_b200 as ub

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_sampled_within_budget_and_repeatable(tmp_path):
    """more windows and candidates than the budget holds: seeded samples, every value taken from the input"""
    rng = np.random.default_rng(0)
    nwin, ncand = bench.DUMP_WINDOWS + 1000, bench.DUMP_CANDIDATES + 5000
    npk = rng.integers(0, 4, nwin).astype(np.int32)
    cands = np.zeros(ncand, ub.CAND_DTYPE)
    cands["freq"], cands["sync"], cands["shift"] = rng.standard_normal(ncand), rng.random(ncand), rng.integers(-500, 4000, ncand)
    cands["m_type"] = rng.random(ncand) < 0.3
    lin = cands["m_type"] == 0
    cands["lin_drift"][lin] = rng.standard_normal(lin.sum())
    cands["V2"][~lin], cands["p2"][~lin] = rng.standard_normal((~lin).sum()), rng.integers(0, 120, (~lin).sum())
    refined = np.zeros(ncand, ub.REFINED_DTYPE)
    refined["f1"], refined["shift1"], refined["worth_a_try"] = rng.standard_normal(ncand), rng.integers(0, 9, ncand), 1
    jig = np.zeros((ncand, ub.NJIG), ub.JIG_DTYPE)
    jig["sync"], jig["gate"] = rng.random((ncand, ub.NJIG)), rng.random((ncand, ub.NJIG)) < 0.5
    # a view, not 100 MB: each candidate's symbols are one value that identifies it
    soft = np.broadcast_to((np.arange(ncand) % 251).astype(np.uint8)[:, None, None], (ncand, ub.NJIG, ub.NSYM))
    total = bench.dump_outputs(str(tmp_path / "a"), npk, cands, refined, jig, soft)
    bench.dump_outputs(str(tmp_path / "b"), npk, cands, refined, jig, soft)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert sorted(a) == sorted(b)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert a[k].tobytes() == b[k].tobytes(), k
    assert total == sum(v.nbytes for v in a.values()) <= 64 << 20
    assert list(a["counts"]) == [nwin, ncand]
    wi, ci, si = (a[k].astype(np.int64) for k in ("window_index", "cand_index", "soft_index"))
    assert len(wi) == bench.DUMP_WINDOWS and len(ci) == bench.DUMP_CANDIDATES and len(si) == bench.DUMP_SOFT_CANDIDATES
    assert np.all(np.diff(wi) > 0) and np.all(np.diff(ci) > 0) and np.all(np.diff(si) > 0)
    assert np.array_equal(a["npk"], npk[wi])
    assert np.array_equal(a["cand_freq"], cands["freq"][ci]) and np.array_equal(a["cand_shift"], cands["shift"][ci])
    assert np.array_equal(a["cand_lin_drift"], np.where(lin[ci], cands["lin_drift"][ci], 0))
    assert np.array_equal(a["cand_V2"], np.where(lin[ci], 0, cands["V2"][ci]))
    assert np.array_equal(a["refined_shift1"], refined["shift1"][ci]) and np.array_equal(a["jig_gate"], jig["gate"][ci])
    assert np.array_equal(a["soft"], soft[si])


def test_small_dump_keeps_everything(tmp_path):
    npk = np.array([2, 0, 1], np.int32)
    cands = np.zeros(3, ub.CAND_DTYPE)
    cands["freq"] = [1.5, -2.25, 0.5]
    soft = np.arange(3 * ub.NJIG * ub.NSYM).reshape(3, ub.NJIG, ub.NSYM).astype(np.uint8)
    bench.dump_outputs(str(tmp_path), npk, cands, np.zeros(3, ub.REFINED_DTYPE), np.zeros((3, ub.NJIG), ub.JIG_DTYPE), soft)
    a = _load(str(tmp_path))
    assert list(a["npk"]) == [2, 0, 1] and list(a["cand_freq"]) == [1.5, -2.25, 0.5]
    assert np.array_equal(a["soft"], soft) and list(a["soft_index"]) == [0, 1, 2]


@pytest.mark.gpu
def test_bench_dump_equals_the_library_on_its_batch(tmp_path):
    """a short bench run: every arm times --steps steps (the overlapped stream at 50 000 windows and the receiver
    included), and the dump is what coarse_fine returns for the benchmark's seeded windows"""
    import torch
    from uwspr_b200 import synth
    nwin, steps = 48, 4
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--windows", str(nwin), "--overlap-windows", "50000", "--decode-limit", "64", "--no-verify",
                          "--no-cpu-baseline", "--skip", "sliding9,array64", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == line["overlap50"]["steps"] == line["receiver"]["steps"] == steps
    d = _load(str(tmp_path / "dump"))
    assert int(d["counts"][1]) == line["config"]["candidates"]
    xs, _ = synth.gen_frames(0, nwin, 0, torch.device("cuda", 0))
    ctx = ub.Context(max_windows=nwin, max_candidates=max(4 * nwin, 1024), **bench.PARAMS)
    npk, cands, refined, jig, soft = ctx.coarse_fine((xs.data_ptr(), nwin * bench.FL), nwin=nwin, stride=bench.FL)
    ctx.close()
    bench.dump_outputs(str(tmp_path / "direct"), npk, cands, refined, jig, soft)
    want = _load(str(tmp_path / "direct"))
    assert sorted(d) == sorted(want)
    for k in want:
        assert d[k].tobytes() == want[k].tobytes(), k
