#!/usr/bin/env python
"""C5 at full size (homography, N = 1 000 000, 10 % clustered inliers, 10 000 iterations, seed 1) with four samplers:
NAPSAC over the grid (cell 50, the bench's arm), NAPSAC over the device-built kNN table, Progressive NAPSAC with the default
length (20 N local samples) and with 1000 local samples, each without and with LO (InItLORsc); the kNN arms at k = 8 and k = 31.
Per arm: ms per fit from device events (last_timing, median of --reps), the sampler kernels' share of the fit's device time (from
a second process with USAC_GPU_TRACE=2, whose per-kernel events would perturb the timed fits), inliers, the share of true inliers
among them and the share of the true inliers found; per k the device kNN build time on its own. One JSON line per arm, the card's
name and power limit in each."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ransac_b200 import GpuContext, capi  # noqa: E402
from ransac_b200 import generator as gen  # noqa: E402

THR, CONF, MAX_IT, SEED = 2.0, 0.95, 10000, 1
ARMS = [("napsac_grid50", capi.SAMPLER_NAPSAC, capi.NEIGH_GRID, 0), ("napsac_knn", capi.SAMPLER_NAPSAC, capi.NEIGH_KNN, 0),
        ("pnapsac_default", capi.SAMPLER_PROGRESSIVE_NAPSAC, capi.NEIGH_KNN, 0),
        ("pnapsac_L1000", capi.SAMPLER_PROGRESSIVE_NAPSAC, capi.NEIGH_KNN, 1000)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception:   # noqa: BLE001
        return "unknown", "unknown"


def cases(ks):
    """(arm, k, lo): the grid arm does not depend on k and runs once"""
    out = []
    for k in ks:
        for arm in ARMS:
            if arm[2] == capi.NEIGH_GRID and k != ks[0]:
                continue
            for lo in (0, 1):
                out.append((arm, k, lo))
    return out


def prepare(ctx, arm, k):
    """install the arm's neighbourhood and length -> build time in ms (host clock around a call that ends in a device sync)"""
    import torch
    name, sampler, neighbors, length = arm
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if neighbors == capi.NEIGH_GRID:
        ctx.set_neighbors_grid(0, 50)
    else:
        ctx.build_neighbors_knn(0, k)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    ctx.set_pnapsac_length(0, length)
    return ms


def fit_kw(arm, lo, round_size):
    return dict(threshold=THR, confidence=CONF, max_iterations=MAX_IT, seed=SEED, round_size=round_size, sampler=arm[1],
                neighbors=arm[2], lo=lo)


def shares(args):
    """child process (USAC_GPU_TRACE=2): per case, the sampler kernels' part of the device time between the fit's launches"""
    pts = gen.make(5)[0]
    ctx = GpuContext(0)
    ctx.set_points(capi.EST_HOMOGRAPHY, pts)
    out = {}
    for arm, k, lo in cases(args.k):
        prepare(ctx, arm, k)
        kw = fit_kw(arm, lo, args.round)
        ctx.fit(**kw)
        saved = os.dup(2)
        with tempfile.TemporaryFile() as tmp:
            os.dup2(tmp.fileno(), 2)
            try:
                ctx.fit(**kw)
            finally:
                os.dup2(saved, 2)
                os.close(saved)
            tmp.seek(0)
            text = tmp.read().decode(errors="replace")
        line = [ln for ln in text.splitlines() if "kernels (us" in ln][-1]
        us = {m.group(1): float(m.group(2)) for m in re.finditer(r" ([a-z0-9_+]+)=([0-9.]+)", line.split(":", 1)[1])}
        sampler_us = us.get("sampler", 0.0) + us.get("sample", 0.0)      # fused rounds / the host-replay path of LO
        out[f"{arm[0]}|{k}|{lo}"] = {"sampler_us": sampler_us, "traced_us": sum(us.values())}
    ctx.close()
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--round", type=int, default=5000, help="samples per round (bench.py's C5 leg uses 5000)")
    ap.add_argument("--k", type=int, nargs="+", default=[8, 31])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--shares", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.shares:
        return shares(args)
    name, power = card()
    env = dict(os.environ, USAC_GPU_TRACE="2")
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--shares", "--round", str(args.round), "--k"] + [str(k) for k in args.k],
                           stdout=subprocess.PIPE, env=env, text=True, check=True)
    share = json.loads(child.stdout.strip().splitlines()[-1])
    pts, _, mask = gen.make(5)
    true = int(mask.sum())
    ctx = GpuContext(0)
    ctx.set_points(capi.EST_HOMOGRAPHY, pts)
    lines = []
    for arm, k, lo in cases(args.k):
        build_ms = min(prepare(ctx, arm, k) for _ in range(2))
        kw = fit_kw(arm, lo, args.round)
        ctx.fit(**kw)                                                            # warm-up: modules, buffers, tables
        dev = []
        for _ in range(args.reps):
            r = ctx.fit(**kw)[0]
            dev.append(ctx.last_timing()["total_ms"])
        ids = ctx.get_inliers(r["model"], THR)
        s = share[f"{arm[0]}|{k}|{lo}"]
        line = {"case": "c5", "arm": arm[0], "neighbors": "grid50" if arm[2] == capi.NEIGH_GRID else f"knn{k}",
                "pnapsac_local_samples": (arm[3] or 20 * len(pts)) if arm[1] == capi.SAMPLER_PROGRESSIVE_NAPSAC else None,
                "lo": lo, "round_size": args.round, "max_iterations": MAX_IT, "seed": SEED,
                "device_ms_median": float(np.median(dev)), "device_ms_min": float(np.min(dev)), "reps": args.reps,
                "neighbourhood_build_ms": build_ms,
                "sampler_share": s["sampler_us"] / s["traced_us"] if s["traced_us"] > 0 else None,
                "sampler_us_traced": s["sampler_us"], "traced_fit_us": s["traced_us"],
                "iterations": int(r["iterations"]), "evals": int(r["evals"]), "inliers": int(r["inliers"]),
                "true_inliers_among_inliers": float(mask[ids].mean()) if len(ids) else 0.0,
                "true_inliers_found": float(mask[ids].sum()) / true, "true_inliers": true, "card": name, "power_limit": power}
        print(json.dumps(line), flush=True)
        lines.append(line)
    ctx.close()
    if args.out:
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
