"""LO-RANSAC (InItLORsc = 1, InItFLORsc = 2) for 2-D lines on the device against the CPU oracle, whose LO is estimator-generic
(orc_lo_*, the PCA non-minimal fit for lines): every fit record field bit for bit - model, inliers, score, iterations, winning
sample, LO counters - through the fused fit, the one-CTA LO kernel, the plug-in entry point usac_gpu_lo_model_score and the C++
layer. Line error sums of the MAIN loop agree with the oracle only to 1e-4 (DESIGN.md section 4.1, "Ties"): the seeds here have no
tie between equal counts, which the equal winning sample ids state; and a winner that LO did not improve keeps its main-loop
score (the reference's GetModelScore leaves the score alone then), so only that score is compared to 1e-4 (assert_score)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
from ransac_b200 import capi
from ransac_b200 import generator as gen

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
USAC = os.path.join(ROOT, "ransac_b200", "usac")
THR, CONF = gen.CONFIGS[1]["threshold"], gen.CONFIGS[1]["confidence"]
LO_KEYS = ("inliers", "iterations", "best_hyp", "best_model_idx", "lo_inner", "lo_iterative")


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


def lane_sum(pts, model):
    """The error sum of LO's scoring (cta_score, the oracle's lo_score): 1024 lanes in point order, then the fixed tree."""
    e = O.errors(O.EST_LINE2D, pts, model).astype(np.float32)
    part = np.zeros(1024, np.float32)
    for i in np.where(e < np.float32(THR))[0]:
        part[i % 1024] = np.float32(part[i % 1024] + e[i])
    s = 1024
    while s > 1:
        s //= 2
        part[:s] = part[:s] + part[s:2 * s]
    return part[0]


def assert_score(pts, r, ref, tag):
    """Scores that LO produced are bit-identical. A score that is not: the fit ended on a main-loop winner that LO did not improve
    (both sides made the same decisions: every other field is equal), so the oracle's score is its main-loop sum of that model, the
    device's is not LO's lane sum, and the two agree to the main loop's 1e-4 (DESIGN.md section 4.1)."""
    g, o = np.float32(r["score"]), np.float32(ref["score"])
    if bits(g) == bits(o):
        return
    model = np.asarray(ref["model"], np.float32)
    assert bits(o) == bits(np.float32(O.score(O.EST_LINE2D, pts, model, THR)[1])), (tag, "oracle score is not a main-loop sum", g, o)
    assert bits(g) != bits(lane_sum(pts, model)), (tag, "device score is an LO sum", g, o)
    assert abs(float(g) - float(o)) <= 1e-4 * abs(float(o)), (tag, g, o)


def assert_fit_equal(r, ref, keys=LO_KEYS, tag="", pts=None):
    for key in keys:
        assert r[key] == ref[key], (tag, key, r[key], ref[key])
    assert np.array_equal(bits(r["model"]), bits(ref["model"])), (tag, r["model"], ref["model"])
    if pts is None:                                                   # two device results: the same arithmetic
        assert bits(np.float32(r["score"])) == bits(np.float32(ref["score"])), (tag, r["score"], ref["score"])
    else:
        assert_score(pts, r, ref, tag)


def fit_pair(ctx, pts, lo, seed, K=256, max_it=10000, sprt=False, gpu_kw=None, ref_kw=None):
    """GPU fit of problem 0 and the oracle's fit of the same inputs (rounds of K: the SPRT / PROSAC host replay)."""
    if sprt:
        ctx.set_sprt_pool(0, O.sprt_pool(seed, len(pts)))
    r = ctx.fit(THR, CONF, max_it, seed=seed, round_size=K, sprt=sprt, lo=lo, **(gpu_kw or {}))[0]
    ref = O.ransac(pts, O.EST_LINE2D, rng=O.RNG_PHILOX, threshold=THR, confidence=CONF, max_iterations=max_it, seed=seed, sprt=sprt,
                   batch=min(K, max_it), lo=lo, **(ref_kw or {}))
    return r, ref


# ---- 1. C1 at full size ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lo", [1, 2])
def test_config1_full_size(ctx, lo):
    pts, line, mask = gen.make(1)
    assert len(pts) == 1000
    ctx.set_points(O.EST_LINE2D, pts)
    for seed in (1, 2, 3):
        r, ref = fit_pair(ctx, pts, lo, seed)
        assert_fit_equal(r, ref, tag=seed, pts=pts)
        assert r["lo_inner"] > 0 and r["inliers"] >= 0.95 * mask.sum()


@pytest.mark.parametrize("ratio", [0.15, 0.3, 0.7])
@pytest.mark.parametrize("lo", [1, 2])
def test_config1_inlier_ratios(ctx, ratio, lo):
    pts = gen.make(1, inlier_ratio=ratio)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    for seed in (4, 5):
        r, ref = fit_pair(ctx, pts, lo, seed)
        assert_fit_equal(r, ref, tag=(ratio, seed), pts=pts)


# ---- 2. line LO with the other parts of the loop -----------------------------------------------------------------------------------
@pytest.mark.parametrize("lo", [1, 2])
def test_with_sprt(ctx, lo):
    pts = gen.make(1, seed_offset=11, inlier_ratio=0.3)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    for seed in (1, 7):
        r, ref = fit_pair(ctx, pts, lo, seed, K=256, sprt=True)
        assert_fit_equal(r, ref, LO_KEYS + ("samples_drawn", "evals"), tag=seed, pts=pts)


def test_with_prosac(ctx):
    from ransac_b200.api import SAMPLER_PROSAC
    pts = gen.make(1, seed_offset=12, inlier_ratio=0.3)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    for lo, sprt in ((1, False), (2, True)):
        r, ref = fit_pair(ctx, pts, lo, 3, K=128, sprt=sprt, gpu_kw=dict(sampler=SAMPLER_PROSAC), ref_kw=dict(sampler=O.SAMPLER_PROSAC))
        assert_fit_equal(r, ref, tag=(lo, sprt), pts=pts)


def test_with_napsac_knn(ctx):
    from ransac_b200.api import NEIGH_KNN, SAMPLER_NAPSAC
    pts = gen.make(1, seed_offset=13, inlier_ratio=0.5)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    ctx.build_neighbors_knn(0, 7)
    for lo in (1, 2):
        r, ref = fit_pair(ctx, pts, lo, 5, K=256, gpu_kw=dict(sampler=SAMPLER_NAPSAC, neighbors=NEIGH_KNN),
                          ref_kw=dict(sampler=O.SAMPLER_NAPSAC, neighbors=O.NEIGH_KNN, knn_table=O.knn_build(pts, 7)))
        assert_fit_equal(r, ref, tag=lo, pts=pts)


def test_with_progressive_napsac(ctx):
    import pnapsac_oracle as PN
    from ransac_b200.api import NEIGH_KNN, SAMPLER_PROGRESSIVE_NAPSAC
    pts = gen.make(1, seed_offset=14, inlier_ratio=0.5)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    ctx.build_neighbors_knn(0, 12)
    table = ctx.get_neighbors_knn(0)
    for lo, sprt in ((1, False), (2, True)):
        if sprt:
            ctx.set_sprt_pool(0, O.sprt_pool(6, len(pts)))
        r = ctx.fit(THR, CONF, 2000, seed=6, round_size=256, sprt=sprt, lo=lo, sampler=SAMPLER_PROGRESSIVE_NAPSAC, neighbors=NEIGH_KNN)[0]
        ref = PN.ransac(pts, O.EST_LINE2D, table, seed=6, threshold=THR, confidence=CONF, max_iterations=2000, sprt=sprt, batch=256, lo=lo)
        assert_fit_equal(r, ref, tag=(lo, sprt), pts=pts)


@pytest.mark.parametrize("K", [1, 32, 512])
def test_round_sizes(ctx, K):
    pts = gen.make(1, seed_offset=15, inlier_ratio=0.3)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    for lo in (1, 2):
        r, ref = fit_pair(ctx, pts, lo, 8, K=K, max_it=3000)
        assert_fit_equal(r, ref, tag=(K, lo), pts=pts)


def test_ragged_batch(ctx):
    """LO fits of a batch run problem by problem: each result equals the fit of its problem alone, and the oracle's."""
    sizes = [1000, 37, 2500, 400, 12]
    ratios = [0.5, 0.7, 0.2, 0.3, 0.9]
    sets = [gen.make(1, seed_offset=40 + i, n=n, inlier_ratio=ratios[i])[0] for i, n in enumerate(sizes)]
    sizes = [len(s) for s in sets]
    ctx.set_points(O.EST_LINE2D, np.concatenate(sets), sizes)
    for lo in (1, 2):
        res = ctx.fit(THR, CONF, 3000, seed=9, round_size=128, lo=lo)
        assert len(res) == len(sets)
        for p, pts in enumerate(sets):
            ref = O.ransac(pts, O.EST_LINE2D, rng=O.RNG_PHILOX, threshold=THR, confidence=CONF, max_iterations=3000, seed=9, batch=128, lo=lo)
            assert_fit_equal(res[p], ref, tag=(lo, p), pts=pts)
    for lo in (1, 2):
        single = []
        for pts in sets:
            ctx.set_points(O.EST_LINE2D, pts)
            single.append(ctx.fit(THR, CONF, 3000, seed=9, round_size=128, lo=lo)[0])
        ctx.set_points(O.EST_LINE2D, np.concatenate(sets), sizes)
        batch = ctx.fit(THR, CONF, 3000, seed=9, round_size=128, lo=lo)
        for p in range(len(sets)):
            assert_fit_equal(batch[p], single[p], LO_KEYS + ("samples_drawn", "rounds"), tag=(lo, p))


# ---- 3. the one-CTA LO kernel (USAC_GPU_LO_SEQ=1) gives the speculative waves' records --------------------------------------------
SEQ_SCRIPT = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from oracle import oracle as O
from ransac_b200 import GpuContext
from ransac_b200 import generator as gen
ctx = GpuContext(0)
out = []
for off, ratio in ((0, 0.5), (21, 0.15), (22, 0.7)):
    pts = gen.make(1, seed_offset=off, inlier_ratio=ratio)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    for lo in (1, 2):
        for seed in (1, 2):
            r = ctx.fit(8.0, 0.99, 10000, seed=seed, round_size=256, lo=lo)[0]
            r["model"] = [int(x) for x in r["model"].view("uint32")]
            r["score"] = int(__import__("numpy").float32(r["score"]).view("uint32"))
            out.append(r)
ctx.close()
print(json.dumps(out))
"""


def run_fits(seq):
    env = dict(os.environ)
    env.pop("USAC_GPU_LO_SEQ", None)
    if seq:
        env["USAC_GPU_LO_SEQ"] = "1"
    r = subprocess.run([sys.executable, "-c", SEQ_SCRIPT, ROOT], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_one_cta_kernel_equals_the_waves():
    waves, seq = run_fits(False), run_fits(True)
    assert len(waves) == len(seq) == 12
    for a, b in zip(waves, seq):
        assert a == b
    assert all(r["lo_inner"] > 0 for r in waves)


# ---- 4. usac_gpu_lo_model_score against orc_lo_get_model_score over a chain of calls -----------------------------------------------
class OracleLo:
    """orc_lo_* of the oracle library. Its LO state is one LoState (oracle/usac_oracle_refit.cpp): the ints est, n, m, kind,
    sample_limit, ..., then the point pointer and the floats theta, lo_thr, step. orc_lo_new fixes sample_limit at the reference
    default 14; other sizes are set in the state after its layout has been checked against the values orc_lo_new wrote."""

    def __init__(self, pts, theta, kind, seed, sample_limit):
        L = O.lib()
        L.orc_lo_new.restype = C.c_void_p
        L.orc_lo_new.argtypes = [C.c_int, C.POINTER(C.c_float), C.c_int, C.c_float, C.c_int, C.c_uint64]
        L.orc_lo_free.argtypes = [C.c_void_p]
        L.orc_lo_counters.argtypes = [C.c_void_p, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_ulonglong)]
        L.orc_lo_get_model_score.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_float)]
        self.L, self.pts = L, np.ascontiguousarray(pts, np.float32)
        self.h = L.orc_lo_new(O.EST_LINE2D, self.pts.ctypes.data_as(C.POINTER(C.c_float)), len(self.pts), theta, kind, seed)
        ints, floats = C.cast(self.h, C.POINTER(C.c_int)), C.cast(self.h, C.POINTER(C.c_float))
        assert [ints[i] for i in range(8)] == [O.EST_LINE2D, len(self.pts), 2, kind, 14, 20, 4, 10]
        assert floats[10] == np.float32(theta) and floats[11] == np.float32(theta)
        ints[4] = sample_limit
        self.floats = floats

    def lo_threshold(self):
        return self.floats[11]

    def call(self, model, inliers, score):
        m = np.zeros(9, np.float32)
        m[:3] = model
        i, s = C.c_int(inliers), C.c_float(score)
        self.L.orc_lo_get_model_score(self.h, m.ctypes.data_as(C.POINTER(C.c_float)), C.byref(i), C.byref(s))
        return m[:3].copy(), i.value, s.value

    def counters(self):
        a, b, c = C.c_uint(), C.c_uint(), C.c_ulonglong()
        self.L.orc_lo_counters(self.h, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def close(self):
        self.L.orc_lo_free(self.h)


def gpu_lo_cfg(kind, seed, sample_size):
    cfg = capi.FitCfg()
    cfg.sampler = capi.SamplerCfg(capi.SAMPLER_UNIFORM, capi.RNG_PHILOX, seed, capi.NEIGH_NONE, 0, 0)
    cfg.threshold, cfg.confidence, cfg.max_iterations = THR, CONF, 10000
    cfg.lo, cfg.lo_sample_size = kind, sample_size
    return cfg


def gpu_lo_call(ctx, cfg, state, model, inliers, score):
    m = np.zeros(9, np.float32)
    m[:3] = model
    i, s = C.c_int(inliers), C.c_float(score)
    rc = ctx.L.usac_gpu_lo_model_score(ctx.h, 0, C.byref(cfg), C.byref(state["calls"]), C.byref(state["thr"]), m.ctypes.data_as(C.POINTER(C.c_float)),
                                       C.byref(i), C.byref(s), C.byref(state["inner"]), C.byref(state["iter"]))
    assert rc == capi.OK, ctx.L.usac_gpu_last_error(ctx.h).decode()
    return m[:3].copy(), i.value, s.value


@pytest.mark.parametrize("sample_size", [3, 14, 16])
@pytest.mark.parametrize("kind", [1, 2])
def test_lo_model_score_chain_matches_oracle(ctx, kind, sample_size):
    pts, line, mask = gen.make(1, seed_offset=30, inlier_ratio=0.4)
    ctx.set_points(O.EST_LINE2D, pts)
    g = np.random.default_rng(100 + 10 * kind + sample_size)
    inl, seed = np.where(mask)[0], 77
    orc = OracleLo(pts, THR, kind, seed, sample_size)
    cfg = gpu_lo_cfg(kind, seed, sample_size)
    state = {"calls": C.c_uint64(0), "thr": C.c_float(0.0), "inner": C.c_uint(0), "iter": C.c_uint(0)}
    try:
        pools = {"below": 0, "above": 0}
        for call in range(12):
            # minimal models of inlier pairs and of random pairs; a claimed inlier count below the model's support makes the
            # pool (min(claimed, support) ids) smaller than the subset size on every third call
            smp = g.choice(inl, 2, replace=False) if call % 2 == 0 else g.choice(len(pts), 2, replace=False)
            models = O.solve_minimal(O.EST_LINE2D, pts, smp.astype(np.int32))
            if not len(models):
                continue
            model = np.asarray(models[0][:3], np.float32)
            cnt, ssum = O.score(O.EST_LINE2D, pts, model, THR)[:2]
            claimed = min(int(cnt), 12 + call % 2) if call % 3 == 0 else int(cnt)
            pools["below" if min(claimed, int(cnt)) <= sample_size else "above"] += claimed >= 12
            got = gpu_lo_call(ctx, cfg, state, model, claimed, np.float32(ssum))
            ref = orc.call(model, claimed, np.float32(ssum))
            assert np.array_equal(bits(got[0]), bits(ref[0])), (call, got, ref)
            assert got[1] == ref[1] and bits(np.float32(got[2])) == bits(np.float32(ref[2])), (call, got, ref)
            assert (state["inner"].value, state["iter"].value, state["calls"].value) == orc.counters(), call
            assert bits(np.float32(state["thr"].value)) == bits(np.float32(orc.lo_threshold())), call
        assert state["inner"].value > 0 and pools["above"] > 0
        if sample_size >= 14:
            assert pools["below"] > 0
    finally:
        orc.close()


# ---- 5. argument checks ------------------------------------------------------------------------------------------------------------
def test_lo_sample_size_is_checked_by_both_entry_points(ctx):
    pts = gen.make(1, n=300)[0]
    ctx.set_points(O.EST_LINE2D, pts)
    model = np.asarray(gen.make(1, n=300)[1], np.float32).ravel()[:3]
    for bad in (2, 17):
        res = (capi.FitResult * 1)()
        cfg = gpu_lo_cfg(1, 1, bad)
        assert ctx.L.usac_gpu_fit(ctx.h, C.byref(cfg), res) == capi.ERR_ARG
        state = {"calls": C.c_uint64(0), "thr": C.c_float(0.0), "inner": C.c_uint(0), "iter": C.c_uint(0)}
        m = np.zeros(9, np.float32)
        m[:3] = model
        i, s = C.c_int(200), C.c_float(100.0)
        assert ctx.L.usac_gpu_lo_model_score(ctx.h, 0, C.byref(cfg), C.byref(state["calls"]), C.byref(state["thr"]), m.ctypes.data_as(C.POINTER(C.c_float)),
                                             C.byref(i), C.byref(s), None, None) == capi.ERR_ARG
    for good in (0, 3, 16):                                           # the bounds themselves are valid
        assert ctx.fit(THR, CONF, 200, seed=1, lo=1, lo_params=(good, 0, 0, 0))[0]["inliers"] > 0
    # a homography with lo_sample_size 17: refused by lo_model_score too (lo_subset draws at most 16 positions)
    hp, H, _ = gen.homography(n=500, seed=3)
    ctx.set_points(O.EST_HOMOGRAPHY, hp)
    cfg = gpu_lo_cfg(1, 1, 17)
    m = np.asarray(H, np.float32).ravel().copy()
    calls, thr, i, s = C.c_uint64(0), C.c_float(0.0), C.c_int(400), C.c_float(100.0)
    assert ctx.L.usac_gpu_lo_model_score(ctx.h, 0, C.byref(cfg), C.byref(calls), C.byref(thr), m.ctypes.data_as(C.POINTER(C.c_float)),
                                         C.byref(i), C.byref(s), None, None) == capi.ERR_ARG
    assert ctx.fit(2.0, 0.95, 200, seed=1, lo=1)[0]["inliers"] > 0   # the context is still usable


# ---- 6. the C++ layer: fused Ransac::run() and run_sequential() with LO on lines ---------------------------------------------------
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


@pytest.mark.parametrize("lo,flags", [(1, []), (2, []), (1, ["--sprt"])])
def test_plugin_layer_fused_and_sequential(tmp_path, lo, flags):
    from ransac_b200 import build
    build.build()
    subprocess.check_call(["make", "-s", "-C", USAC])
    pts = gen.make(1, seed_offset=50, inlier_ratio=0.4)[0]
    p = tmp_path / "p.txt"
    with open(p, "w") as fh:
        fh.write(f"{len(pts)}\n")
        for row in pts:
            fh.write(" ".join(f"{v:.9g}" for v in row) + "\n")
    max_it = 400
    r = subprocess.run([os.path.join(USAC, "usac_harness"), str(p), "line2d", "uniform", repr(THR), "0.95", "7", "--both", "--round", "1",
                        "--max-iter", str(max_it), "--lo", str(lo)] + flags, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    got = parse(r.stdout)
    sprt = "--sprt" in flags
    for name, batch in (("sequential", 0), ("fused", 1)):
        ref = O.ransac(pts, O.EST_LINE2D, rng=O.RNG_PHILOX, threshold=THR, confidence=0.95, max_iterations=max_it, seed=7, sprt=sprt, lo=lo, batch=batch)
        assert ref["lo_inner"] > 0
        fin = O.refit(O.EST_LINE2D, pts, ref["model"], ref["inliers"], THR)
        f = got[name]
        assert f["iterations"] == ref["iterations"] and f["inliers"] == fin["inliers"], name
        assert np.array_equal(f["model"], np.asarray(fin["model"], np.float32).view(np.uint32)), name
        assert f["hash"] == fnv(fin["ids"][:fin["inliers"]]), name
