#!/usr/bin/env python
"""Randomised parity sweep against the CPU oracle (test infrastructure, like tests/): estimators x samplers x SPRT / LO x odd
problem sizes x seeds x round sizes, every fit compared field by field (inliers, iterations, winning sample, model bits, and
under SPRT samples drawn / evaluations). Also get_inliers and the refit loop at sizes on both sides of the multi-launch switch.
usage: stress_parity.py [cases=120] [seed=0]   -> prints the number of cases and every mismatch; exit code 1 on any mismatch."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402
from ransac_b200 import GpuContext, capi  # noqa: E402
from ransac_b200 import generator as gen  # noqa: E402

CASES = int(sys.argv[1]) if len(sys.argv) > 1 else 120
g = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
EST = {1: O.EST_LINE2D, 2: O.EST_HOMOGRAPHY, 3: O.EST_FUNDAMENTAL, 4: O.EST_ESSENTIAL}


def bits(a):
    a = np.ascontiguousarray(a, dtype=np.float32).copy()
    a[np.isnan(a)] = np.float32(np.nan)
    return a.view(np.uint32)


ONLY = set(int(x) for x in os.environ.get("STRESS_ONLY_CASES", "").split(",") if x)   # re-run single cases of a sweep (same random stream)
ctx = GpuContext(0)
bad, ties, t0 = [], [], time.time()
for case in range(CASES):
    cfg = int(g.choice([1, 2, 2, 3, 3, 4]))
    est = EST[cfg]
    n = int(g.integers(200, 6000)) | 1
    if case % 10 == 9:                                     # tiny problems: down to the minimal sample itself
        n = int(O.SAMPLE_SIZE[est] + g.choice([0, 1, 2, 5, 11, 30, 57, 70]))
    ratio = float(g.choice([0.15, 0.3, 0.5, 0.7]))
    pts = gen.make(cfg, seed_offset=1000 + case, n=n, inlier_ratio=ratio)[0]
    if len(pts) != n:
        n = len(pts)
    thr, conf = gen.CONFIGS[cfg]["threshold"], gen.CONFIGS[cfg]["confidence"]
    seed = int(g.integers(1, 1000))
    K = int(g.choice([1, 7, 32, 100, 256, 512]))
    max_it = int(g.choice([50, 300, 1000]))
    sprt = bool(g.random() < 0.5)
    lo = int(g.choice([0, 0, 1, 2]))
    sampler = str(g.choice(["uniform", "uniform", "prosac", "napsac"])) if cfg != 1 else "uniform"
    kw = dict(threshold=thr, confidence=conf, max_iterations=max_it, seed=seed, round_size=K)
    okw = dict(threshold=thr, confidence=conf, max_iterations=max_it, seed=seed, rng=O.RNG_PHILOX)
    ctx.set_points(est, pts)
    if sampler == "prosac":
        kw["sampler"] = capi.SAMPLER_PROSAC; okw["sampler"] = O.SAMPLER_PROSAC
    elif sampler == "napsac":
        if g.random() < 0.5:
            ctx.set_neighbors_grid(0, 50)
            kw.update(sampler=capi.SAMPLER_NAPSAC, neighbors=capi.NEIGH_GRID); okw.update(sampler=O.SAMPLER_NAPSAC, neighbors=O.NEIGH_GRID, cell_size=50)
        else:
            kk = min(7, n - 1)
            if kk < O.SAMPLE_SIZE[est] - 1:
                sampler = "uniform"
            else:
                ctx.build_neighbors_knn(0, kk)
                kw.update(sampler=capi.SAMPLER_NAPSAC, neighbors=capi.NEIGH_KNN); okw.update(sampler=O.SAMPLER_NAPSAC, neighbors=O.NEIGH_KNN, knn_table=O.knn_build(pts, kk))
    if sprt:
        ctx.set_sprt_pool(0, O.sprt_pool(seed, n))
        kw["sprt"] = True; okw["sprt"] = True
    if lo:
        kw["lo"] = lo; okw["lo"] = lo
    if sprt or sampler == "prosac" or lo:
        okw["batch"] = min(K, max_it)          # usac_gpu_fit never draws more than max_iterations samples per round
    tag = f"case {case}: cfg {cfg} n {n} ratio {ratio} {sampler} sprt {sprt} lo {lo} K {K} max_it {max_it} seed {seed}"
    if ONLY and case not in ONLY:
        continue
    try:
        r = ctx.fit(**kw)[0]
        ref = O.ransac(pts, est, **okw)
        keys = ["inliers", "iterations", "best_hyp", "best_model_idx"] + (["samples_drawn", "evals"] if sprt else [])
        diff = [k for k in keys if r[k] != ref[k]]
        if not np.array_equal(bits(r["model"]), bits(ref["model"])):
            diff.append("model")
        if diff and set(diff) <= {"best_hyp", "best_model_idx", "model"} and not sprt and not lo:
            # Score::bigger breaks ties between equal inlier counts by the error SUM, which the device accumulates in another order than
            # the host restatement (1e-4 relative, BASELINE.json): two hypotheses whose sums agree to rounding noise (the same points drawn
            # twice, a tiny problem) may swap. Accepted when the device's winner, scored by the oracle, has the oracle's count and its sum.
            oc = O.score(est, pts, r["model"], thr)
            if oc[0] == ref["inliers"] and abs(oc[1] - ref["score"]) <= 1e-4 * abs(ref["score"]) + 1e-4 * thr:
                ties.append(tag)
                diff = []
        if diff:
            bad.append((tag, diff, {k: (r[k], ref[k]) for k in diff if k != "model"}))
            if os.environ.get("STRESS_DEBUG"):
                kw2 = {k: v for k, v in kw.items() if k not in ("lo", "sprt")}
                okw2 = {k: v for k, v in okw.items() if k not in ("lo", "sprt", "batch")}
                r2, ref2 = ctx.fit(**kw2)[0], O.ransac(pts, est, **okw2)
                print("DEBUG", tag, "neighbors", kw.get("neighbors"), "| with flags: gpu", {k: r[k] for k in ("inliers", "iterations", "best_hyp", "rounds", "samples_drawn")},
                      "oracle", {k: ref[k] for k in ("inliers", "iterations", "best_hyp")}, "| plain fit: gpu", {k: r2[k] for k in ("inliers", "iterations", "best_hyp")},
                      "oracle", {k: ref2[k] for k in ("inliers", "iterations", "best_hyp")})
                for K2 in (1, 16, 512):
                    r3 = ctx.fit(**dict(kw, round_size=K2))[0]
                    print("DEBUG   same flags, round size", K2, {k: r3[k] for k in ("inliers", "iterations", "best_hyp", "rounds")})
        # Quality::getInliers and the refit loop on the result
        if r["inliers"] > 0 and cfg != 1:
            ids = ctx.get_inliers(r["model"], thr)
            oc = O.score(est, pts, r["model"], thr, want_inliers=True)
            if len(ids) != oc[0] or not np.array_equal(ids, oc[3][:oc[0]]):
                bad.append((tag, ["get_inliers"], {}))
            rf = ctx.refit(r["model"], r["inliers"], thr)
            orf = O.refit(est, pts, r["model"], r["inliers"], thr)
            if rf["inliers"] != orf["inliers"] or not np.array_equal(bits(rf["model"]), bits(np.asarray(orf["model"], np.float32))):
                bad.append((tag, ["refit"], {"inliers": (rf["inliers"], orf["inliers"])}))
    except Exception as e:   # noqa: BLE001
        bad.append((tag, ["exception"], {"error": repr(e)}))

# the plug-in entry points one by one: minimal solvers (model bits), Quality counts, per-point errors (bits), sampler tables, non-minimal fits
N_API = 0 if ONLY else max(6, CASES // 10)
for case in range(N_API):
    cfg = int(g.choice([1, 2, 3, 4]))
    est = EST[cfg]
    n = int(g.integers(50, 5000)) | 1
    pts, _, mask = gen.make(cfg, seed_offset=9000 + case, n=n, inlier_ratio=float(g.choice([0.2, 0.5, 0.8])))
    n = len(pts)
    thr = gen.CONFIGS[cfg]["threshold"]
    m = O.SAMPLE_SIZE[est]
    tag = f"api {case}: cfg {cfg} n {n}"
    try:
        ctx.set_points(est, pts)
        inl = np.where(mask)[0]
        samples = np.stack([(g.choice(inl, m, replace=False) if (i % 2 == 0 and len(inl) >= m) else g.choice(n, m, replace=False)) for i in range(40)]).astype(np.int32)
        models, nm = ctx.estimate(samples)
        w = 3 if cfg == 1 else 9
        allm = []
        for i, smp in enumerate(samples):
            ref = O.solve_minimal(est, pts, smp)
            if nm[i] != len(ref) or not np.array_equal(bits(models[i, :nm[i], :w]), bits(ref[:, :w])):
                bad.append((tag, ["estimate"], {"sample": i, "count": (int(nm[i]), len(ref))}))
                break
            allm.extend(ref[:, :w])
        if allm:
            allm = np.stack(allm)
            cnt, sm = ctx.score(allm, thr)
            for i, mod in enumerate(allm):
                oc = O.score(est, pts, mod, thr)
                # counts exact; the MSAC cost sum + (n - inliers) thr within 1e-4 relative (BASELINE.json). The raw sum of a model that fits only
                # its own sample is rounding noise of the evaluator (~1e-3 px per point at coordinates ~1000) and is not compared.
                msac_g, msac_o = sm[i] + (n - cnt[i]) * thr, oc[1] + (n - oc[0]) * thr
                if cnt[i] != oc[0] or abs(msac_g - msac_o) > 1e-4 * abs(msac_o):
                    bad.append((tag, ["score"], {"model": i, "count": (int(cnt[i]), int(oc[0])), "sum": (float(sm[i]), float(oc[1]))}))
                    break
            e = ctx.errors(allm[0])
            if not np.array_equal(bits(e), bits(O.errors(est, pts, allm[0]))):
                bad.append((tag, ["errors"], {}))
        if cfg != 1 and len(inl) >= 30:
            ids = np.sort(g.choice(inl, int(g.integers(8, min(len(inl), 2000))), replace=False)).astype(np.int32)
            got, ref = ctx.estimate_nonminimal(ids), O.nonminimal(est, pts, ids)
            if (got is None) != (ref is None) or (got is not None and not np.array_equal(bits(got), bits(np.asarray(ref, np.float32)))):
                bad.append((tag, ["estimate_nonminimal"], {"count": len(ids)}))
        # sampler tables: PROSAC, and NAPSAC over a grid (with the switch to uniform on sparse data), in chunks of random size
        for kind in ("prosac", "napsac"):
            if cfg == 1:
                continue
            seed = int(g.integers(1, 1000))
            T = 600
            if kind == "prosac":
                ref = O.Sampler(O.SAMPLER_PROSAC, O.RNG_PHILOX, n, m, seed).table(T)
                skw = dict(sampler=capi.SAMPLER_PROSAC)
            else:
                ctx.set_neighbors_grid(0, 50)
                ref = O.Sampler(O.SAMPLER_NAPSAC, O.RNG_PHILOX, n, m, seed, points=pts, cell_size=50).table(T)
                skw = dict(sampler=capi.SAMPLER_NAPSAC, neighbors=capi.NEIGH_GRID)
            if kind == "prosac":
                got = ctx.sample(T, seed=seed, **skw)              # the PROSAC state is a function of the counter: one call
            else:
                chunk, parts, h = int(g.choice([1, 37, 600])), [], 0
                while h < (T if chunk > 1 else 120):
                    k = min(chunk, T - h)
                    parts.append(ctx.sample(k, seed=seed, first_hyp=h, **skw))
                    h += k
                got = np.concatenate(parts)
            if not np.array_equal(got, ref[:len(got)]):
                bad.append((tag, ["sample " + kind], {"first difference": int(np.argmax((got != ref[:len(got)]).any(axis=1)))}))
    except Exception as e:   # noqa: BLE001
        bad.append((tag, ["exception"], {"error": repr(e)}))

# batches of ragged problems in flight: the plain path (device-side select) and the SPRT batch path (host replay per problem)
for case in range(max(4, CASES // 15)):
    cfg = int(g.choice([1, 2, 3, 4]))
    est = EST[cfg]
    B = int(g.integers(2, 9))
    sizes = [int(g.integers(100, 3000)) for _ in range(B)]
    sets = [gen.make(cfg, seed_offset=5000 + 31 * case + i, n=sizes[i], inlier_ratio=float(g.choice([0.05, 0.3, 0.6])))[0] for i in range(B)]
    sizes = [len(x) for x in sets]
    thr, conf = gen.CONFIGS[cfg]["threshold"], gen.CONFIGS[cfg]["confidence"]
    seed, K, max_it = int(g.integers(1, 1000)), int(g.choice([16, 100, 256])), int(g.choice([300, 1000]))
    sprt = bool(g.random() < 0.6)
    ctx.set_points(est, np.concatenate(sets), sizes)
    kw = dict(threshold=thr, confidence=conf, max_iterations=max_it, seed=seed, round_size=K)
    okw = dict(threshold=thr, confidence=conf, max_iterations=max_it, seed=seed, rng=O.RNG_PHILOX)
    if sprt:
        for p_ in range(B):
            ctx.set_sprt_pool(p_, O.sprt_pool(seed, sizes[p_]))
        kw["sprt"] = True; okw.update(sprt=True, batch=min(K, max_it))
    tag = f"batch {case}: cfg {cfg} sizes {sizes} sprt {sprt} K {K} max_it {max_it} seed {seed}"
    try:
        res = ctx.fit(**kw)
        for p_ in range(B):
            ref = O.ransac(sets[p_], est, **okw)
            keys = ["inliers", "iterations", "best_hyp", "best_model_idx"] + (["samples_drawn", "evals"] if sprt else [])
            diff = [k for k in keys if res[p_][k] != ref[k]]
            if not np.array_equal(bits(res[p_]["model"]), bits(ref["model"])):
                diff.append("model")
            if diff:
                bad.append((tag + f" problem {p_}", diff, {k: (res[p_][k], ref[k]) for k in diff if k != "model"}))
    except Exception as e:   # noqa: BLE001
        bad.append((tag, ["exception"], {"error": repr(e)}))

# the ordered inlier list across the multi-launch switch (32768 points) and at sizes that are not multiples of 1024
for n in (32767, 32768, 40001, 131073):
    pts, H, mask = gen.homography(n=n, inlier_ratio=0.3, seed=n)
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    ids = ctx.get_inliers(np.asarray(H, np.float32), 2.0)
    oc = O.score(O.EST_HOMOGRAPHY, pts, np.asarray(H, np.float32), 2.0, want_inliers=True)
    if len(ids) != oc[0] or not np.array_equal(ids, oc[3][:oc[0]]):
        bad.append((f"get_inliers n={n}", ["ids"], {"count": (len(ids), oc[0])}))
    rf = ctx.refit(np.asarray(H, np.float32), int(oc[0]), 2.0)
    orf = O.refit(O.EST_HOMOGRAPHY, pts, np.asarray(H, np.float32), int(oc[0]), 2.0)
    if rf["inliers"] != orf["inliers"] or not np.array_equal(bits(rf["model"]), bits(np.asarray(orf["model"], np.float32))):
        bad.append((f"refit n={n}", ["refit"], {"inliers": (rf["inliers"], orf["inliers"])}))
ctx.close()
print(f"stress_parity: {CASES} fits + {N_API} API sweeps + {max(4, CASES // 15)} ragged batches + 4 large inlier lists in {time.time() - t0:.1f} s, {len(bad)} mismatches ({len(ties)} tie(s) between equal counts broken by sums that agree to rounding noise)")
for b in bad:
    print("MISMATCH", b)
sys.exit(1 if bad else 0)
