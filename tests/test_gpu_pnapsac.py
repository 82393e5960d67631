"""Progressive NAPSAC (DESIGN.md section 4.8) on the GPU against the sequential reference (pnapsac_oracle): samples index-exact,
whole fits bit-exact (the oracle's loop replaying the reference sampler's stream), through the C ABI and the C++ plug-in layer."""
import os
import re
import subprocess
import threading

import numpy as np
import pytest

import pnapsac_oracle as PN
from oracle import oracle as O
from ransac_b200 import generator as gen

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
USAC = os.path.join(ROOT, "ransac_b200", "usac")


@pytest.fixture(scope="module")
def ctx():
    from ransac_b200 import GpuContext
    c = GpuContext(0)
    yield c
    c.close()


def bits(a):
    a = np.ascontiguousarray(a, dtype=np.float32).copy()
    a[np.isnan(a)] = np.float32(np.nan)
    return a.view(np.uint32)


def assert_fit_equal(r, ref, keys=("inliers", "iterations", "best_hyp", "best_model_idx")):
    for key in keys:
        assert r[key] == ref[key], (key, r[key], ref[key])
    assert np.array_equal(bits(r["model"]), bits(ref["model"]))
    assert abs(r["score"] - ref["score"]) <= 1e-4 * ref["score"] + 1e-3


SPRT_KEYS = ("inliers", "iterations", "best_hyp", "best_model_idx", "samples_drawn", "evals")


def problem(est, n, seed):
    if est == O.EST_LINE2D:
        return gen.line2d(n=n, seed=seed)[0]
    if est == O.EST_FUNDAMENTAL:
        return gen.make(3, n=n, seed_offset=seed)[0]
    return gen.homography(n=n, inlier_ratio=0.2, clustered=True, seed=seed)[0]


def pn_kw():
    from ransac_b200.api import NEIGH_KNN, SAMPLER_PROGRESSIVE_NAPSAC
    return dict(sampler=SAMPLER_PROGRESSIVE_NAPSAC, neighbors=NEIGH_KNN)


# ---- the sampler -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("est,k", [(O.EST_HOMOGRAPHY, 7), (O.EST_FUNDAMENTAL, 31), (O.EST_LINE2D, 12)])
def test_sample_matches_reference(ctx, est, k):
    """One call, and the same stream in chunks of several sizes (first_hyp > 0 continues the use counts)."""
    pts = problem(est, 500, 7)
    m = O.SAMPLE_SIZE[est]
    ctx.set_points(est, pts)
    ctx.build_neighbors_knn(0, k)
    table = ctx.get_neighbors_knn(0)
    ref = PN.table(9, table, m, 4000)
    assert np.array_equal(ctx.sample(4000, seed=9, **pn_kw()), ref)
    got, h = [], 0
    for K in (1, 130, 999, 7, 2863):
        got.append(ctx.sample(K, seed=9, first_hyp=h, **pn_kw()))
        h += K
    assert np.array_equal(np.concatenate(got), ref)


def test_sample_reuses_centres_within_one_round(ctx):
    """60 points, 3000 samples in one call: every centre is drawn ~40 times in the round (the search over earlier uses), and the
    neighbourhoods reach k; then a length that ends the local phase inside the table, and its reset by a new point upload."""
    pts = problem(O.EST_HOMOGRAPHY, 60, 2)
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    ctx.build_neighbors_knn(0, 9)
    table = ctx.get_neighbors_knn(0)
    ref = PN.table(4, table, 4, 3000)                             # default length 20 n = 1200: global from there on
    assert np.bincount(ref[:1200, 0]).max() > 2
    assert np.array_equal(ctx.sample(3000, seed=4, **pn_kw()), ref)
    ctx.set_pnapsac_length(0, 777)
    ref777 = PN.table(4, table, 4, 3000, length=777)
    assert np.array_equal(ctx.sample(3000, seed=4, **pn_kw()), ref777)
    assert np.array_equal(np.concatenate([ctx.sample(500, seed=4, **pn_kw()), ctx.sample(2500, seed=4, first_hyp=500, **pn_kw())]), ref777)
    ctx.set_points(O.EST_HOMOGRAPHY, pts)                         # new points: default length again
    ctx.build_neighbors_knn(0, 9)
    assert np.array_equal(ctx.sample(3000, seed=4, **pn_kw()), ref)


# ---- whole fits ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def clustered():
    pts, _, mask = gen.homography(n=6000, inlier_ratio=0.15, clustered=True, seed=41)
    return pts, mask


@pytest.mark.parametrize("round_size", [128, 1024])
def test_fit_matches_reference(ctx, clustered, round_size):
    pts, _ = clustered
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    ctx.build_neighbors_knn(0, 8)
    table = ctx.get_neighbors_knn(0)
    for seed in (1, 2):
        r = ctx.fit(2.0, 0.95, 3000, seed=seed, round_size=round_size, **pn_kw())[0]
        ref = PN.ransac(pts, O.EST_HOMOGRAPHY, table, seed=seed, threshold=2.0, confidence=0.95, max_iterations=3000)
        assert_fit_equal(r, ref)
        assert r["useful_evals"] == ref["evals"]


def test_fit_crosses_into_the_global_phase(ctx, clustered):
    pts, _ = clustered
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    ctx.build_neighbors_knn(0, 8)
    table = ctx.get_neighbors_knn(0)
    ctx.set_pnapsac_length(0, 300)
    r = ctx.fit(2.0, 0.95, 2000, seed=5, round_size=256, **pn_kw())[0]
    ref = PN.ransac(pts, O.EST_HOMOGRAPHY, table, length=300, seed=5, threshold=2.0, confidence=0.95, max_iterations=2000)
    assert ref["iterations"] > 300
    assert_fit_equal(r, ref)


@pytest.mark.parametrize("K", [64, 512])
def test_fit_sprt_matches_reference(ctx, clustered, K):
    pts, _ = clustered
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    ctx.build_neighbors_knn(0, 8)
    table = ctx.get_neighbors_knn(0)
    for seed in (1, 3):
        ctx.set_sprt_pool(0, O.sprt_pool(seed, len(pts)))
        r = ctx.fit(2.0, 0.95, 3000, seed=seed, round_size=K, sprt=True, **pn_kw())[0]
        ref = PN.ransac(pts, O.EST_HOMOGRAPHY, table, seed=seed, threshold=2.0, confidence=0.95, max_iterations=3000, sprt=True, batch=K)
        assert_fit_equal(r, ref, SPRT_KEYS)


@pytest.mark.parametrize("est,sprt", [(O.EST_HOMOGRAPHY, False), (O.EST_FUNDAMENTAL, True)])
def test_fit_with_local_optimisation_matches_reference(ctx, est, sprt):
    pts = gen.homography(n=4000, inlier_ratio=0.2, clustered=True, seed=8)[0] if est == O.EST_HOMOGRAPHY else gen.make(3, n=4000)[0]
    thr = 2.0 if est == O.EST_HOMOGRAPHY else gen.CONFIGS[3]["threshold"]
    ctx.set_points(est, pts)
    ctx.build_neighbors_knn(0, 8)
    table = ctx.get_neighbors_knn(0)
    K = 256
    if sprt:
        ctx.set_sprt_pool(0, O.sprt_pool(2, len(pts)))
    r = ctx.fit(thr, 0.95, 2000, seed=2, round_size=K, sprt=sprt, lo=1, **pn_kw())[0]
    ref = PN.ransac(pts, est, table, seed=2, threshold=thr, confidence=0.95, max_iterations=2000, sprt=sprt, batch=K if sprt else 0, lo=1)
    assert_fit_equal(r, ref, ("inliers", "iterations", "best_hyp", "best_model_idx", "lo_inner", "lo_iterative"))
    assert r["score"] == ref["score"] and r["lo_inner"] > 0


def test_fit_sprt_batch_of_ragged_problems(ctx):
    """Several problems under SPRT (one set of launches per round for all of them): each has its own kNN table, length and use
    counts, and ends where its one-problem reference ends."""
    sizes, lengths = [1500, 700, 2200, 64, 1500], [0, 500, 0, 100, 2000]
    sets = [gen.homography(n=n, inlier_ratio=[0.4, 0.3, 0.15, 0.6, 0.1][i], clustered=True, seed=70 + i)[0] for i, n in enumerate(sizes)]
    ctx.set_points(O.EST_HOMOGRAPHY, np.concatenate(sets), sizes)
    tables = []
    for p, n in enumerate(sizes):
        ctx.build_neighbors_knn(p, 6)
        tables.append(ctx.get_neighbors_knn(p))
        ctx.set_pnapsac_length(p, lengths[p])
        ctx.set_sprt_pool(p, O.sprt_pool(3, n))
    res = ctx.fit(2.0, 0.95, 1200, seed=3, round_size=64, sprt=True, **pn_kw())
    for p, pts in enumerate(sets):
        ref = PN.ransac(pts, O.EST_HOMOGRAPHY, tables[p], length=lengths[p], seed=3, threshold=2.0, confidence=0.95, max_iterations=1200,
                        sprt=True, batch=64)
        assert_fit_equal(res[p], ref, SPRT_KEYS)


@pytest.mark.parametrize("exchange", ["peer", "hook"])
def test_two_emulated_ranks(clustered, exchange):
    """Hypotheses of every round split over two ranks (two contexts on one GPU, one host thread each): every rank draws the
    centres and use counts of all samples and solves its own."""
    from ransac_b200 import GpuContext
    pts, _ = clustered
    world = 2
    ctxs = [GpuContext(0) for _ in range(world)]
    if exchange == "peer":
        wins = [c.peer_window() for c in ctxs]
    else:
        from test_gpu_multirank import HostExchange
        ex = HostExchange(world)
    for r, c in enumerate(ctxs):
        c.set_points(O.EST_HOMOGRAPHY, pts)
        c.build_neighbors_knn(0, 8)
        c.set_pnapsac_length(0, 1500)
        if exchange == "peer":
            c.peer_attach_ptrs(wins, r, world)
        else:
            c._check(c.L.usac_gpu_set_allgather(c.h, ex.fns[r], None), "set_allgather")
    table = ctxs[0].get_neighbors_knn(0)
    results, errors = [None] * world, []

    def run(rank):
        try:
            results[rank] = ctxs[rank].fit(2.0, 0.95, 3000, seed=6, round_size=128, rank=rank, nranks=world, **pn_kw())[0]
        except Exception as e:   # noqa: BLE001
            errors.append(e)
            if exchange == "hook":
                ex.barrier.abort()
    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(120)
    for c in ctxs:
        c.close()
    assert not errors, errors
    ref = PN.ransac(pts, O.EST_HOMOGRAPHY, table, length=1500, seed=6, threshold=2.0, confidence=0.95, max_iterations=3000)
    for r in results:
        assert_fit_equal(r, ref)
    assert sum(r["useful_evals"] for r in results) == ref["evals"]


def test_config5_full_size(ctx):
    """C5 (homography, N = 1 000 000, 10 % clustered inliers) over the device-built kNN table, which the reference is given too.
    The reference's iterations are capped at 2560 as in the NAPSAC grid test of C5."""
    pts, _, mask = gen.make(5)
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    ctx.build_neighbors_knn(0, 8)
    table = ctx.get_neighbors_knn(0)
    r = ctx.fit(2.0, 0.95, 2560, round_size=512, seed=1, **pn_kw())[0]
    ref = PN.ransac(pts, O.EST_HOMOGRAPHY, table, seed=1, threshold=2.0, confidence=0.95, max_iterations=2560)
    assert_fit_equal(r, ref)
    assert r["useful_evals"] == ref["evals"]
    ids = ctx.get_inliers(r["model"], 2.0)
    assert len(ids) == r["inliers"] > 0


# ---- argument checks -------------------------------------------------------------------------------------------------------------
def test_rejects_grid_and_missing_neighbourhoods(ctx):
    from ransac_b200 import UsacGpuError, capi
    from ransac_b200.api import NEIGH_GRID, NEIGH_KNN, NEIGH_NONE, SAMPLER_PROGRESSIVE_NAPSAC as PNS

    def rc_of(fn):
        with pytest.raises(UsacGpuError) as e:
            fn()
        return int(re.search(r"failed \((\d+)\)", str(e.value)).group(1))
    pts = problem(O.EST_HOMOGRAPHY, 300, 1)
    ctx.set_points(O.EST_HOMOGRAPHY, pts)
    for neighbors in (NEIGH_NONE, NEIGH_GRID):
        assert rc_of(lambda: ctx.fit(2.0, 0.95, 100, sampler=PNS, neighbors=neighbors)) == capi.ERR_ARG
        assert rc_of(lambda: ctx.sample(16, sampler=PNS, neighbors=neighbors)) == capi.ERR_ARG
    ctx.set_neighbors_grid(0, 50)
    assert rc_of(lambda: ctx.fit(2.0, 0.95, 100, sampler=PNS, neighbors=NEIGH_GRID)) == capi.ERR_ARG
    assert rc_of(lambda: ctx.fit(2.0, 0.95, 100, sampler=PNS, neighbors=NEIGH_KNN)) == capi.ERR_STATE   # no kNN table
    assert rc_of(lambda: ctx.sample(16, sampler=PNS, neighbors=NEIGH_KNN)) == capi.ERR_STATE
    for bad in (-1, 1):
        assert rc_of(lambda: ctx.set_pnapsac_length(bad, 10)) == capi.ERR_ARG
    ctx.build_neighbors_knn(0, 5)
    assert ctx.fit(2.0, 0.95, 200, sampler=PNS, neighbors=NEIGH_KNN)[0]["iterations"] > 0   # usable after the failures


# ---- the C++ plug-in layer -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def harness():
    from ransac_b200 import build
    build.build()
    subprocess.check_call(["make", "-s", "-C", USAC])
    return os.path.join(USAC, "usac_harness")


def parse(out):
    res = {}
    for line in out.splitlines():
        if line.startswith(("fused", "sequential")):
            tag, *kv = line.split()
            d = dict(x.split("=") for x in kv)
            res[tag] = {"iterations": int(d["iterations"]), "inliers": int(d["inliers"]), "hash": d["inlier_hash"],
                        "model": np.array([int(x, 16) for x in d["model_bits"].split(",")], np.uint32)}
    return res


def fnv(ids):
    h = 1469598103934665603
    for i in ids:
        h = ((h ^ int(i)) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return f"{h:016x}"


@pytest.mark.parametrize("length", [0, 400])
def test_harness_fused_equals_sequential_equals_reference(harness, tmp_path, length):
    """`pnapsac --knn 8 --both`: Ransac::run (rounds on the device) == run_sequential (one usac_gpu_sample per block, the use counts
    carried across calls) == the reference's loop + the refit loop (ransac.cpp:157-207)."""
    pts = gen.homography(n=1500, inlier_ratio=0.3, clustered=True, seed=17)[0]
    p = tmp_path / "p.txt"
    with open(p, "w") as fh:
        fh.write(f"{len(pts)}\n")
        for row in pts:
            fh.write(" ".join(f"{v:.9g}" for v in row) + "\n")
    extra = ["--pn-length", str(length)] if length else []
    r = subprocess.run([harness, str(p), "homography", "pnapsac", "2.0", "0.95", "5", "--knn", "8", "--both"] + extra,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    got = parse(r.stdout)
    f, s = got["fused"], got["sequential"]
    assert f["iterations"] == s["iterations"] and f["inliers"] == s["inliers"] and f["hash"] == s["hash"]
    assert np.array_equal(f["model"], s["model"])
    ref = PN.ransac(pts, O.EST_HOMOGRAPHY, O.knn_build(pts, 8), length=length, seed=5, threshold=2.0, confidence=0.95)
    fin = O.refit(O.EST_HOMOGRAPHY, pts, ref["model"], ref["inliers"], 2.0)
    assert f["iterations"] == ref["iterations"] and f["inliers"] == fin["inliers"]
    assert np.array_equal(f["model"], np.asarray(fin["model"], np.float32).view(np.uint32))
    assert f["hash"] == fnv(fin["ids"][:fin["inliers"]])
