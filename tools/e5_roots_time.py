#!/usr/bin/env python
"""C4 at full size (essential 5-pt, N = 20 000, 20 % inliers, 10 000 iterations, seed 1) with the reference's first-valid-root rule
and with every valid root (usac_fit_cfg::essential_roots), each without and with SPRT. Per case: ms per fit from device events
(last_timing) and from a host clock around the call (it returns after a device synchronise), evals, inliers against the true
inliers, and whether the result equals the CPU oracle's. One JSON line per case, the card's name and power limit in each."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import e5_roots_oracle as E  # noqa: E402
from oracle import oracle as O  # noqa: E402
from ransac_b200 import GpuContext, capi  # noqa: E402
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--round", type=int, default=512)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    name, power = card()
    pts, _, mask = gen.make(4)
    thr, conf = gen.CONFIGS[4]["threshold"], gen.CONFIGS[4]["confidence"]
    true = int(mask.sum())
    ctx = GpuContext(0)
    ctx.set_points(capi.EST_ESSENTIAL, pts)
    ctx.set_sprt_pool(0, O.sprt_pool(1, len(pts)))
    lines = []
    for sprt in (False, True):
        for roots in (capi.E5_ROOTS_FIRST_VALID, capi.E5_ROOTS_ALL_VALID):
            kw = dict(seed=1, round_size=args.round, sprt=sprt, essential_roots=roots)
            ctx.fit(thr, conf, 10000, **kw)                                     # warm-up: modules, buffers, tables
            dev, host = [], []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                r = ctx.fit(thr, conf, 10000, **kw)[0]
                host.append((time.perf_counter() - t0) * 1e3)
                dev.append(ctx.last_timing()["total_ms"])
            oracle_fit = E.ransac if roots == capi.E5_ROOTS_ALL_VALID else O.ransac
            ref = oracle_fit(pts, O.EST_ESSENTIAL, rng=O.RNG_PHILOX, threshold=thr, confidence=conf, max_iterations=10000, seed=1,
                             sprt=sprt, batch=args.round if sprt else 0)
            parity = all(r[k] == ref[k] for k in ("inliers", "iterations", "best_hyp", "best_model_idx")) and \
                np.array_equal(np.asarray(r["model"], np.float32).view(np.uint32), np.asarray(ref["model"], np.float32).view(np.uint32))
            line = {"case": "c4", "essential_roots": "all_valid" if roots else "first_valid", "sprt": sprt, "round_size": args.round,
                    "device_ms_median": float(np.median(dev)), "device_ms_min": float(np.min(dev)), "host_ms_median": float(np.median(host)),
                    "host_ms_min": float(np.min(host)), "reps": args.reps, "evals": int(r["evals"]), "useful_evals": int(r["useful_evals"]),
                    "iterations": int(r["iterations"]), "inliers": int(r["inliers"]), "true_inliers": true,
                    "best_model_idx": int(r["best_model_idx"]), "oracle_parity": bool(parity), "card": name, "power_limit": power}
            print(json.dumps(line), flush=True)
            lines.append(line)
    ctx.close()
    if args.out:
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
