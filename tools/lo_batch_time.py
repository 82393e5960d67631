#!/usr/bin/env python
"""Batched LO-RANSAC against the same problems fitted one at a time. Cases: C2 (homography, N = 4000, 30 % inliers) + LO 1 / 2 at
P = 2, 8, 64, 512, 2368; C1 lines + LO at P = 512; E (N = 5000, 30 % inliers) + SPRT + LO at P = 64. Per case: device-event ms
(last_timing) and host ms (a host clock around the call, which returns after a device synchronise) of the batched fit, and the
total of the P single-problem fits; the batch's LO calls and LO steps (USAC_GPU_TRACE line of the fit); whether every batched record
equals its single-problem record byte for byte; whether problem 0 agrees with the CPU oracle; the card's name and power limit, read
in the same run. --seq runs with USAC_GPU_LO_SEQ=1 (one CTA per LO call, no waves). One JSON line per case."""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--cases", nargs="+", default=None, help="subset of case names")
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--seq", action="store_true")
ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
args = ap.parse_args()
os.environ["USAC_GPU_TRACE"] = "1"
if args.seq:
    os.environ["USAC_GPU_LO_SEQ"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402
from ransac_b200 import GpuContext  # noqa: E402
from ransac_b200 import generator as gen  # noqa: E402
from lo_line_time import card  # noqa: E402

CASES = [(f"c2_lo{lo}_P{P}", 2, P, lo, False) for lo in (1, 2) for P in (2, 8, 64, 512, 2368)] + \
        [("c1_lo1_P512", 1, 512, 1, False), ("e_sprt_lo1_P64", 4, 64, 1, True)]


def problems(cfg, P):
    if cfg == 4:
        return [gen.essential(n=5000, inlier_ratio=0.3, seed=1000 + i)[0] for i in range(P)]
    return [gen.make(cfg, seed_offset=i)[0] for i in range(P)]


class Stderr:
    """the C library's stderr (fd 2) of one call, for its USAC_GPU_TRACE line"""
    def __enter__(self):
        self.f = tempfile.TemporaryFile(mode="w+")
        sys.stderr.flush()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def main():
    name, power = card()
    batch, solo = GpuContext(0), GpuContext(0)
    lines = []
    for case, cfg, P, lo, sprt in CASES:
        if args.cases and case not in args.cases:
            continue
        est = {1: O.EST_LINE2D, 2: O.EST_HOMOGRAPHY, 4: O.EST_ESSENTIAL}[cfg]
        thr, conf = gen.CONFIGS[cfg]["threshold"], gen.CONFIGS[cfg]["confidence"]
        K = 512
        sets = problems(cfg, P)
        kw = dict(seed=1, round_size=K, lo=lo, sprt=sprt)
        batch.set_points(est, np.concatenate(sets), [len(s) for s in sets])
        if sprt:
            for p, s in enumerate(sets):
                batch.set_sprt_pool(p, O.sprt_pool(1, len(s)))
        batch.fit_records(thr, conf, 10000, **kw)                                  # warm-up
        dev, host = [], []
        for _ in range(args.reps):
            with Stderr() as err:
                t0 = time.perf_counter()
                rec = batch.fit_records(thr, conf, 10000, **kw)
                host.append((time.perf_counter() - t0) * 1e3)
            dev.append(batch.last_timing()["total_ms"])
        trace = [l for l in err.text.splitlines() if l.startswith("usac_gpu_fit[batch replay]")]
        calls = steps = wave_steps = -1
        if trace:
            t = trace[-1]
            calls = int(t.split("LO ")[1].split(" calls")[0])
            steps = int(t.split(" calls in ")[1].split(" steps")[0])
            wave_steps = int(t.split(" steps (")[1].split(" with waves")[0])
        # the same problems one at a time
        single_dev, single_host, equal = 0.0, 0.0, True
        for p, s in enumerate(sets):
            solo.set_points(est, s)
            if sprt:
                solo.set_sprt_pool(0, O.sprt_pool(1, len(s)))
            if p == 0:
                solo.fit_records(thr, conf, 10000, **kw)                            # warm-up
            t0 = time.perf_counter()
            one = solo.fit_records(thr, conf, 10000, **kw)
            single_host += (time.perf_counter() - t0) * 1e3
            single_dev += solo.last_timing()["total_ms"]
            equal = equal and one[0].tobytes() == rec[p].tobytes()
        ref = O.ransac(sets[0], est, rng=O.RNG_PHILOX, threshold=thr, confidence=conf, max_iterations=10000, seed=1, sprt=sprt,
                       batch=K, lo=lo)
        r0 = batch.fit(thr, conf, 10000, **kw)[0]
        w = 3 if est == O.EST_LINE2D else 9
        oracle = all(r0[k] == ref[k] for k in ("inliers", "iterations", "best_hyp", "lo_inner", "lo_iterative")) and \
            np.array_equal(np.asarray(r0["model"], np.float32).view(np.uint32), np.asarray(ref["model"], np.float32)[:w].view(np.uint32))
        line = {"case": case, "P": P, "lo": lo, "sprt": sprt, "round_size": K, "lo_seq": args.seq,
                "batch_device_ms_median": float(np.median(dev)), "batch_device_ms_min": float(np.min(dev)),
                "batch_host_ms_median": float(np.median(host)), "batch_host_ms_min": float(np.min(host)), "reps": args.reps,
                "single_device_ms_total": single_dev, "single_host_ms_total": single_host,
                "speedup_host": single_host / float(np.median(host)),
                "lo_calls": calls, "lo_steps": steps, "lo_wave_steps": wave_steps,
                "records_equal_single": bool(equal), "oracle_spot_check": bool(oracle), "card": name, "power_limit": power}
        print(json.dumps(line), flush=True)
        lines.append(line)
    batch.close()
    solo.close()
    if args.out:
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
