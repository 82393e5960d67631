#!/usr/bin/env python
"""Randomised sweep through the C++ plug-in layer (ransac_b200/usac/usac_harness --both): the fused Ransac::run(), the
one-hypothesis-at-a-time run_sequential() over the virtual plug-in classes (Sampler, Estimator, Quality / SPRT, TerminationCriteria,
LocalOptimization) and the CPU oracle + refit must agree: iterations, inliers, inlier list, model bits. run_sequential() is held to the
oracle's sequential loop (batch = 0: the reference's semantics); the fused run() to the oracle's rounds of K (batch = K = --round): without
SPRT the two are the same loop, with SPRT a round freezes the test and starts model q at pool offset cursor + 32 q (SURVEY hard part 3),
which differs from the sequential walk (next model starts where the last one stopped) even for K = 1 - about one SPRT fit in ten ends
with another iteration count or model.
usage: stress_harness.py [cases=40] [seed=0] [round=1] [napsac]"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from ransac_b200 import generator as gen  # noqa: E402

HARNESS = os.path.join(ROOT, "ransac_b200", "usac", "usac_harness")
CASES = int(sys.argv[1]) if len(sys.argv) > 1 else 40
g = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
ROUND = int(sys.argv[3]) if len(sys.argv) > 3 else 1
NAPSAC = len(sys.argv) > 4 and sys.argv[4] == "napsac"          # homography cases also draw NAPSAC (grid / kNN) samplers
NAMES = {1: "line2d", 2: "homography", 3: "fundamental", 4: "essential"}
EST = {1: O.EST_LINE2D, 2: O.EST_HOMOGRAPHY, 3: O.EST_FUNDAMENTAL, 4: O.EST_ESSENTIAL}


def fnv(ids):
    h = 1469598103934665603
    for i in ids:
        h = ((h ^ int(i)) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return f"{h:016x}"


def parse(out):
    res = {}
    for line in out.splitlines():
        if not line.startswith(("fused", "sequential")):
            continue
        tag, *kv = line.split()
        d = dict(x.split("=") for x in kv)
        res[tag] = {"iterations": int(d["iterations"]), "inliers": int(d["inliers"]), "hash": d["inlier_hash"],
                    "model": np.array([int(x, 16) for x in d["model_bits"].split(",")], np.uint32)}
    return res


bad = []
differ = 0      # SPRT fits where the oracle's rounds of K and its sequential loop end differently
with tempfile.TemporaryDirectory() as tmp:
    for case in range(CASES):
        cfg = int(g.choice([1, 2, 2, 3, 4]))
        est = EST[cfg]
        n = int(g.integers(300, 2500))
        ratio = float(g.choice([0.3, 0.5, 0.7]))
        thr = 8.0 if cfg == 1 else (2.5e-3 if cfg == 4 else 2.0)
        seed, max_it = int(g.integers(1, 500)), int(g.choice([100, 400]))
        sampler = "uniform" if cfg == 1 else str(g.choice(["uniform", "uniform", "prosac"]))
        knn = 0
        if NAPSAC and cfg == 2 and g.random() < 0.6:                     # NAPSAC over the cell grid (cell 50) or the k nearest neighbours
            sampler, knn = "napsac", int(g.choice([0, 0, 5, 8]))
        pts = gen.make(cfg, seed_offset=7000 + case, n=n, inlier_ratio=ratio, **({"clustered": True} if sampler == "napsac" else {}))[0]
        n = len(pts)
        sprt = bool(g.random() < 0.5)
        lo = int(g.choice([0, 0, 1, 2]))
        path = os.path.join(tmp, "p.txt")
        with open(path, "w") as fh:
            fh.write(f"{n}\n")
            for row in pts:
                fh.write(" ".join(f"{v:.9g}" for v in row) + "\n")
        cmd = [HARNESS, path, NAMES[cfg], sampler, repr(thr), "0.95", str(seed), "--both", "--round", str(ROUND), "--max-iter", str(max_it)]
        if sprt:
            cmd.append("--sprt")
        if lo:
            cmd += ["--lo", str(lo)]
        if knn:
            cmd += ["--knn", str(knn)]
        tag = f"case {case}: {' '.join(cmd[2:])} n {n}"
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        if r.returncode != 0:
            bad.append((tag, "exit code", r.returncode, r.stderr[-300:]))
            continue
        got = parse(r.stdout)
        f, s = got["fused"], got["sequential"]
        wants = {}
        for name, batch in (("sequential", 0), ("fused", ROUND)):
            kw = {"sampler": O.SAMPLER_PROSAC if sampler == "prosac" else O.SAMPLER_UNIFORM}
            if sampler == "napsac":
                kw = {"sampler": O.SAMPLER_NAPSAC, "neighbors": O.NEIGH_KNN, "knn_table": O.knn_build(pts, knn)} if knn else \
                     {"sampler": O.SAMPLER_NAPSAC, "neighbors": O.NEIGH_GRID, "cell_size": 50}
            ref = O.ransac(pts, est, rng=O.RNG_PHILOX, threshold=thr, confidence=0.95, max_iterations=max_it, seed=seed, sprt=sprt, lo=lo,
                           batch=batch, **kw)
            fin = O.refit(est, pts, ref["model"], ref["inliers"], thr)
            wants[name] = {"iterations": ref["iterations"], "inliers": fin["inliers"], "hash": fnv(fin["ids"][:fin["inliers"]]),
                           "model": np.asarray(fin["model"], np.float32).view(np.uint32)}
            differ += name == "fused" and (wants["fused"]["iterations"] != wants["sequential"]["iterations"]
                                           or not np.array_equal(wants["fused"]["model"], wants["sequential"]["model"]))
        for name, x in (("fused", f), ("sequential", s)):
            want = wants[name]
            d = [k for k in ("iterations", "inliers", "hash") if x[k] != want[k]]
            if not np.array_equal(x["model"][:len(want["model"])], want["model"]):
                d.append("model")
            if d:
                bad.append((tag, name, d, {k: (x[k], want[k]) for k in d if k != "model"}))
print(f"stress_harness: {CASES} runs of usac_harness --both (fused, sequential) against the oracle, {len(bad)} mismatches "
      f"({differ} SPRT fits where rounds of {ROUND} and the sequential loop end differently - each side matched its own oracle form)")
for b in bad:
    print("MISMATCH", b)
sys.exit(1 if bad else 0)
