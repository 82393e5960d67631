"""bench.py --dump-outputs: the results of the last timed step as DIR/<field>.npy (float32 / float64, 64 MB at most), the same
from run to run, through the writer, the CPU arm (--impl reference) and, on a GPU, the C2 batch and --workload c5."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_fit_records_are_written_as_float_arrays_under_the_size_cap(tmp_path, monkeypatch):
    from ransac_b200 import capi
    rec = np.zeros(1000, dtype=np.dtype(capi.FitResult))
    rec["model"] = np.arange(9000, dtype=np.float32).reshape(1000, 9)
    rec["evals"] = np.arange(1000, dtype=np.uint64) * 10**10
    bench.dump_outputs(str(tmp_path / "all"), bench.record_fields(rec))
    out = load(tmp_path / "all")
    assert set(out) == set(rec.dtype.names)
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert np.array_equal(out["model"], rec["model"]) and np.array_equal(out["evals"], rec["evals"].astype(np.float64))
    monkeypatch.setattr(bench, "DUMP_LIMIT", 20000)
    bench.dump_outputs(str(tmp_path / "cut"), bench.record_fields(rec))
    cut = load(tmp_path / "cut")
    assert sum(os.path.getsize(tmp_path / "cut" / f) for f in os.listdir(tmp_path / "cut")) <= 20000
    rows = cut["rows"].astype(np.int64)
    assert 0 < len(rows) < 1000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(cut["model"], rec["model"][rows]) and np.array_equal(cut["evals"], rec["evals"][rows].astype(np.float64))


def test_cpu_arm_dumps_the_same_outputs_every_run(tmp_path):
    runs = []
    for name in ("a", "b"):
        d = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                            "--ref-problems", "1", "--dump-outputs", str(d)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        runs.append(load(d))
    a, b = runs
    assert {"model", "inliers", "iterations"} <= set(a) and a.keys() == b.keys()
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert a["model"].shape[1] == 9 and (a["inliers"] > 0).all()


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode != 0 and "--steps" in r.stderr


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_gpu_arms_dump_the_last_timed_step(tmp_path, golden_dir):
    """The C2 batch writes one row per image pair, each the oracle's fit of that pair, and --steps reaches every timed leg;
    --workload c5 writes the one record of the 1M-point fit (tests/golden/c5_n1_oracle.json)."""
    from oracle import oracle as O
    line = run_bench("--steps", "2", "--warmup", "1", "--no-cpu", "--problems", "64", "--dump-outputs", str(tmp_path / "c2"))
    assert line["steps"] == line["config"]["c5"]["steps"] == line["roofline_f"]["steps"] == line["roofline_e"]["steps"] == 2
    out = load(tmp_path / "c2")
    assert out["model"].shape == (64, 9) and all(len(a) == 64 for a in out.values())
    for i, pts in enumerate(bench.make_problems(4, 1000)):
        ref = O.ransac(pts, O.EST_HOMOGRAPHY, rng=O.RNG_PHILOX, threshold=bench.THR, confidence=bench.CONF, max_iterations=bench.MAX_IT, seed=1)
        assert (out["inliers"][i], out["iterations"][i], out["best_hyp"][i]) == (ref["inliers"], ref["iterations"], ref["best_hyp"])
        assert np.array_equal(out["model"][i].view(np.uint32), ref["model"].view(np.uint32))
    run_bench("--workload", "c5", "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path / "c5"))
    c5 = load(tmp_path / "c5")
    gold = json.load(open(os.path.join(golden_dir, "c5_n1_oracle.json")))
    assert len(c5["inliers"]) == 1 and (c5["inliers"][0], c5["iterations"][0], c5["best_hyp"][0]) == (gold["inliers"], gold["iterations"], gold["best_hyp"])
