"""Batched LO-RANSAC (usac_gpu_fit with P > 1 and lo = 1 / 2, with or without SPRT): every problem of a ragged batch against the same
points fitted alone. The batch pauses each problem at a new best that LO works on, runs the paused problems' LO calls as one device
step and resumes; rounds stay K. So every fit record must equal, byte for byte, the record of the problem fitted alone (P = 1, the
same round size), and the key fields and model bits must equal the CPU oracle's.

Every batch holds a problem whose best never reaches 12 inliers (no LO call), one that ends in its first round, one that runs to
max_iterations and problems that need several LO calls in one round."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
from ransac_b200 import generator as gen
from ransac_b200.api import E5_ROOTS_ALL_VALID, NEIGH_KNN, SAMPLER_NAPSAC, SAMPLER_PROGRESSIVE_NAPSAC, SAMPLER_PROSAC

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("inliers", "iterations", "samples_drawn", "best_hyp", "best_model_idx", "lo_inner", "lo_iterative")
THR = {O.EST_LINE2D: 8.0, O.EST_HOMOGRAPHY: 2.0, O.EST_FUNDAMENTAL: 2.0, O.EST_ESSENTIAL: 2.5e-3}
MAX_IT = 1500


@pytest.fixture(scope="module")
def ctxs():
    from ransac_b200 import GpuContext
    batch, solo = GpuContext(0), GpuContext(0)
    yield batch, solo
    batch.close()
    solo.close()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def problems(est, seed=0):
    """(points, label) of a ragged batch: no LO call / ends in round 1 / runs to max_iterations / several LO calls per round."""
    g = np.random.default_rng(1234 + seed)
    if est == O.EST_LINE2D:
        make = lambda n, r, s: gen.line2d(n=n, inlier_ratio=r, seed=s)[0]
        noise = g.uniform(0, 1000, (40, 2)).astype(np.float32)
    elif est == O.EST_HOMOGRAPHY:
        make = lambda n, r, s: gen.homography(n=n, inlier_ratio=r, seed=s)[0]
        noise = g.uniform(0, 1000, (40, 4)).astype(np.float32)
    elif est == O.EST_FUNDAMENTAL:
        make = lambda n, r, s: gen.fundamental(n=n, inlier_ratio=r, seed=s)[0]
        noise = g.uniform(0, 1000, (40, 4)).astype(np.float32)
    else:
        make = lambda n, r, s: gen.essential(n=n, inlier_ratio=r, seed=s)[0]
        noise = g.uniform(-0.6, 0.6, (40, 4)).astype(np.float32)
    low = 0.02 if est == O.EST_LINE2D else 0.08                         # a two-point sample finds 8 % inliers within MAX_IT
    return [(noise, "no LO"), (make(600, 0.8, 50 + seed), "first round"), (make(1500, low, 60 + seed), "max_iterations"),
            (make(1200, 0.35, 70 + seed), "several LO calls"), (make(2000, 0.5, 80 + seed), "several LO calls")]


def upload(ctx, est, sets, ids, kw, sprt, seed, knn):
    ctx.set_points(est, np.concatenate([sets[i] for i in ids]), [len(sets[i]) for i in ids])
    for p, i in enumerate(ids):
        if knn:
            ctx.build_neighbors_knn(p, knn)
        if sprt:
            ctx.set_sprt_pool(p, O.sprt_pool(seed, len(sets[i])))


def batch_vs_solo(ctxs, est, lo, sprt, K, seed=3, kw=None, knn=0, sets=None):
    """Fit records of the batch and of every problem alone: byte for byte equal. Returns (sets, batch records as dicts)."""
    batch, solo = ctxs
    kw = dict(kw or {})
    sets = sets if sets is not None else [s for s, _ in problems(est)]
    fit_kw = dict(seed=seed, round_size=K, sprt=sprt, lo=lo, **kw)
    upload(batch, est, sets, range(len(sets)), kw, sprt, seed, knn)
    rec = batch.fit_records(THR[est], 0.95, MAX_IT, **fit_kw)
    dicts = batch.fit(THR[est], 0.95, MAX_IT, **fit_kw)
    for p, pts in enumerate(sets):
        upload(solo, est, sets, [p], kw, sprt, seed, knn)
        one = solo.fit_records(THR[est], 0.95, MAX_IT, **fit_kw)
        assert rec[p].tobytes() == one[0].tobytes(), (p, rec[p], one[0])
    return sets, dicts


def assert_oracle(est, sets, res, lo, sprt, K, seed=3, ref_fn=None, **ref_kw):
    ref_fn = ref_fn or O.ransac
    for p, pts in enumerate(sets):
        ref = ref_fn(pts, est, rng=O.RNG_PHILOX, threshold=THR[est], confidence=0.95, max_iterations=MAX_IT, seed=seed, sprt=sprt,
                     batch=K, lo=lo, **ref_kw)
        for k in KEYS:
            assert res[p][k] == ref[k], (p, k, res[p][k], ref[k])
        w = 3 if est == O.EST_LINE2D else 9
        assert np.array_equal(bits(res[p]["model"]), bits(np.asarray(ref["model"], np.float32)[:w])), (p, res[p]["model"], ref["model"])
        if est == O.EST_LINE2D:
            from test_gpu_lo_line import assert_score        # lines: a main-loop score agrees to 1e-4 only (DESIGN 4.1)
            assert_score(pts, res[p], ref, p)
        else:
            assert bits(np.float32(res[p]["score"])) == bits(np.float32(ref["score"])), (p, res[p]["score"], ref["score"])


ESTS = [O.EST_LINE2D, O.EST_HOMOGRAPHY, O.EST_FUNDAMENTAL, O.EST_ESSENTIAL]


@pytest.mark.parametrize("sprt", [False, True])
@pytest.mark.parametrize("lo", [1, 2])
@pytest.mark.parametrize("est", ESTS)
def test_batch_equals_single_and_oracle(ctxs, est, lo, sprt):
    sets, res = batch_vs_solo(ctxs, est, lo, sprt, K=128)
    assert res[0]["lo_inner"] == 0 and res[0]["inliers"] < 12                      # no LO call
    assert res[1]["rounds"] == 1                                                   # ends in its first round
    assert any(r["iterations"] >= MAX_IT for r in res)                             # runs to max_iterations
    assert res[3]["lo_inner"] > 0 and res[4]["lo_inner"] > 0
    assert_oracle(est, sets, res, lo, sprt, 128)


@pytest.mark.parametrize("K", [32, 512])
@pytest.mark.parametrize("sprt", [False, True])
def test_round_sizes(ctxs, K, sprt):
    sets, res = batch_vs_solo(ctxs, O.EST_HOMOGRAPHY, 1, sprt, K=K, seed=5)
    assert_oracle(O.EST_HOMOGRAPHY, sets, res, 1, sprt, K, seed=5)


@pytest.mark.parametrize("sprt", [False, True])
def test_essential_all_roots(ctxs, sprt):
    import e5_roots_oracle as E
    sets, res = batch_vs_solo(ctxs, O.EST_ESSENTIAL, 2, sprt, K=128, kw=dict(essential_roots=E5_ROOTS_ALL_VALID))
    assert_oracle(O.EST_ESSENTIAL, sets, res, 2, sprt, 128, ref_fn=E.ransac)


@pytest.mark.parametrize("sampler", [SAMPLER_NAPSAC, SAMPLER_PROGRESSIVE_NAPSAC])
@pytest.mark.parametrize("sprt", [False, True])
def test_knn_samplers(ctxs, sampler, sprt):
    sets = [gen.homography(n=n, inlier_ratio=r, clustered=True, seed=90 + i)[0] for i, (n, r) in enumerate([(900, 0.4), (1500, 0.2), (400, 0.6)])]
    _, res = batch_vs_solo(ctxs, O.EST_HOMOGRAPHY, 1, sprt, K=64, kw=dict(sampler=sampler, neighbors=NEIGH_KNN), knn=8, sets=sets)
    import pnapsac_oracle as PN
    batch, _ = ctxs
    for p, pts in enumerate(sets):
        table = batch.get_neighbors_knn(p)
        kw = dict(threshold=2.0, confidence=0.95, max_iterations=MAX_IT, seed=3, sprt=sprt, batch=64, lo=1)
        if sampler == SAMPLER_NAPSAC:
            ref = O.ransac(pts, O.EST_HOMOGRAPHY, sampler=O.SAMPLER_NAPSAC, rng=O.RNG_PHILOX, neighbors=O.NEIGH_KNN, knn_table=table, **kw)
        else:
            ref = PN.ransac(pts, O.EST_HOMOGRAPHY, table, **kw)
        for k in KEYS:
            assert res[p][k] == ref[k], (p, k, res[p][k], ref[k])
        assert np.array_equal(bits(res[p]["model"]), bits(np.asarray(ref["model"], np.float32))), p


def test_prosac_batch_stays_on_the_one_problem_path(ctxs):
    """PROSAC + LO with P > 1 runs problem by problem (fit_host_replay): each equals the oracle."""
    batch, _ = ctxs
    sets = [s for s, _ in problems(O.EST_HOMOGRAPHY)][1:4]
    batch.set_points(O.EST_HOMOGRAPHY, np.concatenate(sets), [len(s) for s in sets])
    res = batch.fit(2.0, 0.95, MAX_IT, seed=3, round_size=128, lo=1, sampler=SAMPLER_PROSAC)
    for p, pts in enumerate(sets):
        ref = O.ransac(pts, O.EST_HOMOGRAPHY, sampler=O.SAMPLER_PROSAC, rng=O.RNG_PHILOX, threshold=2.0, confidence=0.95,
                       max_iterations=MAX_IT, seed=3, batch=128, lo=1)
        for k in KEYS:
            assert res[p][k] == ref[k], (p, k)
        assert np.array_equal(bits(res[p]["model"]), bits(np.asarray(ref["model"], np.float32)))


def _trace(code):
    env = dict(os.environ, USAC_GPU_TRACE="1", PYTHONPATH=ROOT + os.pathsep + os.path.join(ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    return [l for l in out.stderr.splitlines() if l.startswith("usac_gpu_fit[batch replay]")]


def test_both_device_forms_run():
    """A small batch keeps its LO steps under the pending-call threshold (speculative waves); a large one goes over it (one CTA per
    call). Both give each problem's single-fit record."""
    code = r'''
import numpy as np
import test_gpu_lo_batch as T
from oracle import oracle as O
from ransac_b200 import GpuContext, generator as gen
ctxs = (GpuContext(0), GpuContext(0))
for P in (2, 24):
    sets = [gen.homography(n=800, inlier_ratio=0.4, seed=300 + i)[0] for i in range(P)]
    T.batch_vs_solo(ctxs, O.EST_HOMOGRAPHY, 1, True, K=128, sets=sets)
    print("ok", P, flush=True)
'''
    lines = _trace(code)
    steps = [l for l in lines if "P=2 " in l or "P=24 " in l]
    small = [l for l in steps if "P=2 " in l]
    large = [l for l in steps if "P=24 " in l]
    assert small and large, lines
    waves = lambda l: int(l.split("(")[1].split(" with waves")[0])
    lo_steps = lambda l: int(l.split(" steps")[0].split(" in ")[-1])
    assert all(waves(l) == lo_steps(l) > 0 for l in small), small             # every step with <= 4 calls: waves
    assert any(waves(l) < lo_steps(l) for l in large), large                  # a step above the threshold: one CTA per call


def test_second_context_after_another_contexts_lo_fit():
    """LO fits, batched and alone, on contexts created after another context's LO fit and after that context is gone. The
    shared-memory opt-in is set when a context is created; on one GPU every context shares the device's primary context, so this
    shows that creating and destroying contexts leaves LO working, not that a second device gets the opt-in."""
    from ransac_b200 import GpuContext
    sets = [s for s, _ in problems(O.EST_HOMOGRAPHY, seed=1)][1:]
    first = GpuContext(0)
    first.set_points(O.EST_HOMOGRAPHY, sets[0])
    r0 = first.fit(2.0, 0.95, MAX_IT, seed=3, round_size=128, lo=2)[0]
    first.close()
    ctxs = (GpuContext(0), GpuContext(0))
    try:
        _, res = batch_vs_solo(ctxs, O.EST_HOMOGRAPHY, 2, False, K=128, sets=sets)
        assert res[0]["inliers"] == r0["inliers"] and np.array_equal(bits(res[0]["model"]), bits(r0["model"]))
    finally:
        for c in ctxs:
            c.close()
