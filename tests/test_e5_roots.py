"""The all-roots five-point oracle (e5_roots_oracle.cpp / .py): every cheirality-valid root of a sample is a model, handled like
the seven-point solver's roots. It is the reference the GPU tests of usac_fit_cfg::essential_roots compare against."""
import numpy as np
import pytest

import e5_roots_oracle as E
from oracle import oracle as O
from ransac_b200 import generator as gen

# C4, seed 1: hypothesis 3930 is the first all-inlier sample; its three valid roots have 100, 141 and 2227 inliers and the
# reference's rule keeps the first one
C4_HYP = 3930


def test_all_roots_solve_is_the_valid_candidates_in_order():
    pts, _, _ = gen.make(4)
    g = np.random.default_rng(5)
    multi = 0
    for _ in range(300):
        s = g.choice(len(pts), 5, replace=False).astype(np.int32)
        Es, valid = O.essential5_candidates(pts, s)
        got = E.all_roots(pts, s)
        want = Es[valid].reshape(-1, 9).astype(np.float32)
        assert got.shape == want.shape
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
        first = O.solve_minimal(O.EST_ESSENTIAL, pts, s)
        assert np.array_equal(first.view(np.uint32), got[:1].view(np.uint32))      # the reference's rule = the first of them
        multi += len(got) > 1
    assert multi > 0


def test_c4_all_roots_fit_finds_half_the_true_inliers():
    pts, _, mask = gen.make(4)
    thr, conf = gen.CONFIGS[4]["threshold"], gen.CONFIGS[4]["confidence"]
    kw = dict(rng=O.RNG_PHILOX, threshold=thr, confidence=conf, max_iterations=4000, seed=1)    # the cap keeps hypothesis 3930
    first = O.ransac(pts, O.EST_ESSENTIAL, **kw)
    allr = E.ransac(pts, O.EST_ESSENTIAL, **kw)
    assert allr["inliers"] >= 0.5 * mask.sum(), (allr["inliers"], int(mask.sum()))
    assert first["inliers"] < 0.5 * mask.sum()
    assert allr["best_hyp"] == C4_HYP and allr["best_model_idx"] == 2
    assert allr["models_scored"] > first["models_scored"]
    assert allr["samples_drawn"] == allr["iterations"] == 4000          # iterations count samples, not models


def test_all_roots_fit_reports_the_winning_root():
    pts, _, _ = gen.make(4)
    thr = gen.CONFIGS[4]["threshold"]
    table = O.philox_unique(1, C4_HYP, 0, len(pts), 5).reshape(1, 5)
    roots = E.all_roots(pts, table[0])
    counts = [O.score(O.EST_ESSENTIAL, pts, m, thr)[0] for m in roots]
    r = E.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_TABLE, sample_table=table, threshold=thr, max_iterations=1)
    assert len(roots) > 1 and r["best_model_idx"] == int(np.argmax(counts)) > 0
    assert r["inliers"] == max(counts) and r["iterations"] == 1 and r["models_scored"] == len(roots)
    assert np.array_equal(r["model"].view(np.uint32), roots[r["best_model_idx"]].view(np.uint32))
    r0 = O.ransac(pts, O.EST_ESSENTIAL, rng=O.RNG_TABLE, sample_table=table, threshold=thr, max_iterations=1)
    assert r0["best_model_idx"] == 0 and r0["inliers"] == counts[0]


@pytest.mark.parametrize("cfg,kw", [(3, dict(max_iterations=500)), (3, dict(max_iterations=800, sprt=True, batch=64)),
                                    (2, dict(max_iterations=2000, lo=1, batch=128)), (3, dict(sampler=O.SAMPLER_PROSAC, max_iterations=800, batch=64))])
def test_all_roots_loop_is_the_oracle_loop_for_other_estimators(cfg, kw):
    """The all-roots loop is the oracle's loop with another essential solve: on the other estimators it returns the oracle's result."""
    est = {2: O.EST_HOMOGRAPHY, 3: O.EST_FUNDAMENTAL}[cfg]
    pts, _, _ = gen.make(cfg, n=1500)
    kw = dict(kw, rng=O.RNG_PHILOX, threshold=gen.CONFIGS[cfg]["threshold"], confidence=0.95, seed=2)
    a, b = O.ransac(pts, est, **kw), E.ransac(pts, est, **kw)
    assert np.array_equal(a.pop("model"), b.pop("model")) and a == b
