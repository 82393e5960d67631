#!/usr/bin/env python
"""C1 (line2d, N = 1000, 50 % inliers, threshold 8, confidence 0.99, 10 000 iterations) with local optimisation off (0),
InItLORsc (1) and InItFLORsc (2). Per case and seed: ms per fit as the median of repeated fits after a warm-up fit, from device
events (last_timing) and from a host clock around the call (it returns after a device synchronise), inliers against the true
inliers, LO counters, and whether the result equals the CPU oracle's. One JSON line per case, the card's name and power limit,
read in the same run, in each."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402
from ransac_b200 import GpuContext  # noqa: E402
from ransac_b200 import generator as gen  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception:   # noqa: BLE001
        return "unknown", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--seeds", type=int, nargs="+", default=[1, 2, 3])
    ap.add_argument("--round", type=int, default=0, help="round size (0 = automatic)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    name, power = card()
    pts, _, mask = gen.make(1)
    thr, conf = gen.CONFIGS[1]["threshold"], gen.CONFIGS[1]["confidence"]
    ctx = GpuContext(0)
    ctx.set_points(O.EST_LINE2D, pts)
    lines = []
    for seed in args.seeds:
        for lo in (0, 1, 2):
            kw = dict(seed=seed, round_size=args.round, lo=lo)
            ctx.fit(thr, conf, 10000, **kw)                                     # warm-up: modules, buffers, tables
            dev, host = [], []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                r = ctx.fit(thr, conf, 10000, **kw)[0]
                host.append((time.perf_counter() - t0) * 1e3)
                dev.append(ctx.last_timing()["total_ms"])
            ref = O.ransac(pts, O.EST_LINE2D, rng=O.RNG_PHILOX, threshold=thr, confidence=conf, max_iterations=10000, seed=seed, lo=lo)
            parity = all(r[k] == ref[k] for k in ("inliers", "iterations", "best_hyp", "lo_inner", "lo_iterative")) and \
                np.array_equal(np.asarray(r["model"], np.float32).view(np.uint32), np.asarray(ref["model"], np.float32).view(np.uint32))
            line = {"case": "c1", "lo": lo, "seed": seed, "round_size": args.round, "device_ms_median": float(np.median(dev)),
                    "device_ms_min": float(np.min(dev)), "host_ms_median": float(np.median(host)), "host_ms_min": float(np.min(host)),
                    "reps": args.reps, "iterations": int(r["iterations"]), "inliers": int(r["inliers"]), "true_inliers": int(mask.sum()),
                    "lo_inner": int(r["lo_inner"]), "lo_iterative": int(r["lo_iterative"]), "oracle_parity": bool(parity),
                    "card": name, "power_limit": power}
            print(json.dumps(line), flush=True)
            lines.append(line)
    ctx.close()
    if args.out:
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
