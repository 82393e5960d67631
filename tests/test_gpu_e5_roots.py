"""Essential fits with every cheirality-valid five-point root as a model (usac_fit_cfg::essential_roots = USAC_E5_ROOTS_ALL_VALID),
against the all-roots CPU oracle (e5_roots_oracle.py: the oracle's fit loop with every valid root a model). Thresholds on C4
come from that oracle's own fits of the same data (profiles/e5_roots_oracle_c4.txt)."""
import subprocess
import threading

import numpy as np
import pytest

import e5_roots_oracle as E
from oracle import oracle as O
from ransac_b200 import generator as gen

pytestmark = pytest.mark.gpu
ALL = 1


@pytest.fixture(scope="module")
def ctx():
    from ransac_b200 import GpuContext
    c = GpuContext(0)
    yield c
    c.close()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_same(r, ref, sprt, drawn=None):
    """drawn: compare samples_drawn too (rounds of the same size on both sides; default: with SPRT)"""
    keys = ("inliers", "iterations", "best_hyp", "best_model_idx") + (("samples_drawn",) if (sprt if drawn is None else drawn) else ()) \
        + (("evals",) if sprt else ())
    for k in keys:
        assert r[k] == ref[k], (k, r[k], ref[k])
    assert np.array_equal(bits(r["model"]), bits(ref["model"]))
    if sprt:
        assert r["score"] == ref["score"]
    else:
        assert abs(r["score"] - ref["score"]) <= 1e-4 * ref["score"] + 1e-3


@pytest.fixture(scope="module")
def small():
    """A reduced essential problem on which several roots of one sample compete (asserted below)."""
    pts, _, _ = gen.essential(n=2000, inlier_ratio=0.35, seed=41)
    return pts, 2.5e-3


def test_estimate_essential_roots_matches_oracle(ctx):
    pts, _, _ = gen.make(4)
    ctx.set_points(O.EST_ESSENTIAL, pts)
    g = np.random.default_rng(12)
    samples = np.stack([g.choice(len(pts), 5, replace=False) for _ in range(2000)]).astype(np.int32)
    models, nm = ctx.estimate_essential_roots(samples)
    assert models.shape == (2000, 10, 9)
    first, n1 = ctx.estimate(samples)
    for j, s in enumerate(samples):
        ref = E.all_roots(pts, s)
        assert nm[j] == len(ref), j
        assert np.array_equal(bits(models[j, :nm[j]]), bits(ref)), j
        assert not models[j, nm[j]:].any()
        assert n1[j] == min(1, nm[j]) and (nm[j] == 0 or np.array_equal(bits(first[j, 0]), bits(ref[0])))
    assert (nm > 1).sum() > 0


@pytest.mark.parametrize("sprt,lo", [(False, 0), (True, 0), (True, 1)])
def test_fit_uniform_matches_oracle(ctx, small, sprt, lo):
    pts, thr = small
    ctx.set_points(O.EST_ESSENTIAL, pts)
    idx = []
    for seed in (1, 2, 3):
        if sprt:
            ctx.set_sprt_pool(0, O.sprt_pool(seed, len(pts)))
        r = ctx.fit(thr, 0.95, 1500, seed=seed, round_size=256, sprt=sprt, lo=lo, essential_roots=ALL)[0]
        ref = E.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_PHILOX, threshold=thr, confidence=0.95, max_iterations=1500, seed=seed,
                       sprt=sprt, batch=256 if sprt or lo else 0, lo=lo)
        assert_same(r, ref, sprt, drawn=sprt or lo)
        idx.append(r["best_model_idx"])
    if not sprt:
        assert max(idx) > 0                                          # a root after the first one won at least once


def test_fit_prosac_matches_oracle(ctx, small):
    from ransac_b200.api import SAMPLER_PROSAC
    pts, thr = small
    ctx.set_points(O.EST_ESSENTIAL, pts)
    for seed in (1, 4):
        r = ctx.fit(thr, 0.95, 1500, sampler=SAMPLER_PROSAC, seed=seed, round_size=128, essential_roots=ALL)[0]
        ref = E.ransac(pts, O.EST_ESSENTIAL, sampler=O.SAMPLER_PROSAC, rng=O.RNG_PHILOX, threshold=thr, confidence=0.95,
                       max_iterations=1500, seed=seed, batch=128)
        assert_same(r, ref, False, drawn=True)


@pytest.mark.parametrize("sprt", [False, True])
def test_fit_batch_of_problems_matches_oracle(ctx, sprt):
    """P > 1: the fused fit without SPRT, fit_sprt_batch with it."""
    sizes, ratios = [1500, 900, 2000], [0.5, 0.3, 0.2]
    sets = [gen.essential(n=n, inlier_ratio=ratios[i], seed=70 + i)[0] for i, n in enumerate(sizes)]
    ctx.set_points(O.EST_ESSENTIAL, np.concatenate(sets), sizes)
    if sprt:
        for p, n in enumerate(sizes):
            ctx.set_sprt_pool(p, O.sprt_pool(3, n))
    res = ctx.fit(2.5e-3, 0.95, 600, seed=3, round_size=64, sprt=sprt, essential_roots=ALL)
    for p, pts in enumerate(sets):
        ref = E.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_PHILOX, threshold=2.5e-3, confidence=0.95, max_iterations=600, seed=3,
                       sprt=sprt, batch=64 if sprt else 0)
        assert_same(res[p], ref, sprt)


def test_two_ranks_in_one_process_match_oracle(small):
    """Hypothesis sharding over two emulated ranks: the winner kernel re-solves the other rank's samples with all roots."""
    from test_gpu_multirank import HostExchange
    from ransac_b200 import GpuContext
    pts, thr = small
    ex = HostExchange(2)
    results, errors = [None, None], []

    def run(rank):
        try:
            c = GpuContext(0)
            c.set_points(O.EST_ESSENTIAL, pts)
            c._check(c.L.usac_gpu_set_allgather(c.h, ex.fns[rank], None), "set_allgather")
            results[rank] = c.fit(thr, 0.95, 1500, seed=5, round_size=128, rank=rank, nranks=2, essential_roots=ALL)[0]
            c.close()
        except Exception as e:   # noqa: BLE001
            errors.append(e)
            ex.barrier.abort()
    threads = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(120)
    assert not errors, errors
    ref = E.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_PHILOX, threshold=thr, confidence=0.95, max_iterations=1500, seed=5)
    assert ref["best_hyp"] % 2 == 1 and ref["best_model_idx"] > 0      # rank 1's sample, root 2: rank 0 re-solves it
    for r in results:
        assert_same(r, ref, False)


@pytest.fixture(scope="module")
def c4():
    pts, _, mask = gen.make(4)
    return pts, mask, gen.CONFIGS[4]["threshold"], gen.CONFIGS[4]["confidence"]


def test_c4_full_size_all_roots(ctx, c4):
    """C4 as stated (N = 20 000, 20 % inliers, 10 000 iterations). Oracle, seed 1: 2227 inliers without SPRT (the first rule: 1186),
    1528 with SPRT, 4037 with SPRT + LO; the refit after the plain fit reaches 3981 (3929 of them true)."""
    pts, mask, thr, conf = c4
    true = int(mask.sum())
    ctx.set_points(O.EST_ESSENTIAL, pts)
    kw = dict(rng=O.RNG_PHILOX, threshold=thr, confidence=conf, max_iterations=10000, seed=1)
    r = ctx.fit(thr, conf, 10000, seed=1, round_size=512, essential_roots=ALL)[0]
    ref = E.ransac(pts, O.EST_ESSENTIAL, **kw)
    assert_same(r, ref, False)
    assert r["inliers"] >= 0.5 * true, (r["inliers"], true)
    rf = ctx.refit(r["model"], r["inliers"], thr)
    ref_rf = O.refit(O.EST_ESSENTIAL, pts, ref["model"], ref["inliers"], thr)
    assert rf["inliers"] == ref_rf["inliers"] and np.array_equal(bits(rf["model"]), bits(ref_rf["model"]))
    ids = ctx.get_inliers(rf["model"], thr)
    assert mask[ids].sum() >= 0.9 * true, (int(mask[ids].sum()), true)
    ctx.set_sprt_pool(0, O.sprt_pool(1, len(pts)))
    for lo in (0, 1):
        r = ctx.fit(thr, conf, 10000, seed=1, round_size=512, sprt=True, lo=lo, essential_roots=ALL)[0]
        ref = E.ransac(pts, O.EST_ESSENTIAL, sprt=True, batch=512, lo=lo, **kw)
        assert_same(r, ref, True)
        assert (r["lo_inner"], r["lo_iterative"]) == (ref["lo_inner"], ref["lo_iterative"])
        if lo:
            assert r["inliers"] >= 0.5 * true, (r["inliers"], true)


def test_c4_default_rule_unchanged(ctx, c4):
    pts, mask, thr, conf = c4
    ctx.set_points(O.EST_ESSENTIAL, pts)
    r = ctx.fit(thr, conf, 10000, seed=1, round_size=512, essential_roots=0)[0]
    ref = O.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_PHILOX, threshold=thr, confidence=conf, max_iterations=10000, seed=1)
    assert_same(r, ref, False)
    assert r["best_model_idx"] == 0


def test_rejects_bad_essential_roots(ctx):
    from ransac_b200 import UsacGpuError, capi
    pts, _, _ = gen.essential(n=300, seed=3)
    ctx.set_points(O.EST_ESSENTIAL, pts)
    with pytest.raises(UsacGpuError, match=r"\(2\)"):
        ctx.fit(2.5e-3, 0.95, 100, essential_roots=2)
    with pytest.raises(UsacGpuError, match=r"\(2\)"):
        ctx.fit(2.5e-3, 0.95, 100, essential_roots=-1)
    hp, _, _ = gen.homography(n=300, seed=1)
    ctx.set_points(O.EST_HOMOGRAPHY, hp)
    with pytest.raises(UsacGpuError, match=r"\(2\)"):
        ctx.fit(2.0, 0.95, 100, essential_roots=1)
    with pytest.raises(UsacGpuError, match=r"\(2\)"):
        ctx.estimate_essential_roots(np.arange(5, dtype=np.int32).reshape(1, 5))
    assert ctx.fit(2.0, 0.95, 100, essential_roots=0)[0]["inliers"] > 0
    assert capi.ERR_ARG == 2


def test_harness_fused_equals_sequential_all_roots(small, tmp_path):
    from test_host_layer import USAC, HARNESS, parse, write_points, fnv
    from ransac_b200 import build
    build.build()
    subprocess.check_call(["make", "-s", "-C", USAC])
    pts, thr = small
    p = tmp_path / "p.txt"
    write_points(p, pts)
    r = subprocess.run([HARNESS, str(p), "essential", "uniform", repr(thr), "0.95", "5", "--both", "--all-roots", "--max-iter", "1500"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    got = parse(r.stdout)
    f, s = got["fused"], got["sequential"]
    assert f["iterations"] == s["iterations"] and f["inliers"] == s["inliers"] and f["hash"] == s["hash"]
    assert np.array_equal(f["model"], s["model"])
    ref = E.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_PHILOX, threshold=thr, confidence=0.95, max_iterations=1500, seed=5)
    assert ref["best_model_idx"] > 0
    fin = O.refit(O.EST_ESSENTIAL, pts, ref["model"], ref["inliers"], thr)
    assert f["iterations"] == ref["iterations"] and f["inliers"] == fin["inliers"]
    assert np.array_equal(f["model"], bits(fin["model"]))
    assert f["hash"] == fnv(fin["ids"][:fin["inliers"]])
