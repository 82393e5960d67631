"""The oracle restatement against the REFERENCE'S OWN code: oracle/_ref/libusac_ref.so is the reference's usac/ tree compiled
where it lies under /root/reference (oracle/Makefile.ref; OpenCV / Eigen / nanoflann answered by oracle/ref_shim/). CPU only.

What this pins (bit for bit unless a tolerance is written): the four GetError metrics and Quality::getNumberInliers; the
UniformSampler stream under srand(seed); StandardTerminationCriteria; the PROSAC growth function and subset-size schedule;
SPRT - pool shuffle, sequential accept/reject decisions, inlier counts, pool cursor, the (epsilon, delta, A, k) test history
and getUpperBoundIterations; ProsacTerminationCriteria; the grid / kNN neighbourhoods; the line solver; and Ransac::run as a
whole for line fitting (iterations, inliers). What stays outside (and why) is asserted too: the reference's 4-point DLT does
not interpolate its own sample (thin-SVD row, dlt.cpp:43-48), its 7-point / 5-point / non-minimal solvers agree with the oracle's
to the accuracy float32 + a different null-space basis allow.
"""
import numpy as np
import pytest

from oracle import oracle as O
from oracle import ref as R
from ransac_b200 import generator as gen

# every test but the two that hold the stand-in numerics (oracle/libref_shim.so, built with the oracle) against OpenCV fixtures
needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref/libusac_ref.so is not built: the reference's sources are not part of this repository")

EST_OF_CFG = {1: O.EST_LINE2D, 2: O.EST_HOMOGRAPHY, 3: O.EST_FUNDAMENTAL, 4: O.EST_ESSENTIAL}


def bits(a):
    a = np.ascontiguousarray(a, dtype=np.float32).copy()
    a[np.isnan(a)] = np.float32(np.nan)
    return a.view(np.uint32)


def unit(m):
    m = np.asarray(m, np.float64).ravel()
    m = m / np.linalg.norm(m)
    return m if m[np.argmax(np.abs(m))] > 0 else -m


def data(cfg, n=3000):
    return gen.make(cfg) if cfg == 1 else gen.make(cfg, n=n)


def some_models(est, pts, mask, count, g, every=3):
    m, out, inl = O.SAMPLE_SIZE[est], [], np.where(mask)[0]
    while len(out) < count:
        s = g.choice(inl, m, replace=False) if len(out) % every == 0 else g.choice(len(pts), m, replace=False)
        out.extend(O.solve_minimal(est, pts, s.astype(np.int32)))
    return out[:count]


@needs_ref
@pytest.mark.parametrize("cfg", [1, 2, 3, 4])
def test_errors_and_scores_bit_exact(cfg):
    """Estimator::GetError (all four metrics) and Quality::getNumberInliers: every error value, the count, the float32 error sum
    in point order and the inlier list are identical. Includes degenerate models (zero / singular -> NaN, inf)."""
    est, thr = EST_OF_CFG[cfg], gen.CONFIGS[cfg]["threshold"]
    pts, gt, mask = data(cfg)
    g = np.random.default_rng(cfg)
    w = 3 if cfg == 1 else 9
    models = some_models(est, pts, mask, 40, g) + [np.asarray(gt, np.float32).ravel()[:w], np.zeros(w, np.float32), np.ones(w, np.float32)]
    for mod in models:
        assert np.array_equal(bits(O.errors(est, pts, mod)), bits(R.errors(est, pts, mod)))
        c_o, s_o, _, ids_o = O.score(est, pts, mod, thr, want_inliers=True)
        c_r, s_r, ids_r = R.score(est, pts, mod, thr, want_inliers=True)
        assert c_o == c_r and np.array_equal(bits([s_o]), bits([s_r])) and np.array_equal(ids_o, ids_r)


@needs_ref
def test_uniform_sampler_stream_and_termination_values():
    for seed, n, m in ((1, 4000, 4), (7, 1000, 2), (12345, 10000, 7), (3, 11, 5)):      # n = 11: the pool wraps (uniform_sampler.hpp:43-45)
        assert np.array_equal(O.Sampler(O.SAMPLER_UNIFORM, O.RNG_GLIBC, n, m, seed).table(2500), R.uniform_samples(seed, n, m, 2500))
    for n, m, conf in ((4000, 4, 0.95), (1000, 2, 0.99), (10000, 7, 0.95), (20000, 5, 0.95)):
        for inl in list(range(0, n + 1, 13)) + [n]:
            assert O.standard_termination(inl, n, m, conf, 10000) == R.standard_termination(inl, n, m, conf, 10000)


@needs_ref
def test_prosac_growth_function_and_schedule():
    """ProsacSampler: T'_n table, and for every sample the subset size n, the counter t and the forced last point u_n
    (prosac_sampler.hpp:147-168). The m-1 random points come from mt19937 in the reference and from Philox in the oracle."""
    for n, m in ((5000, 7), (4000, 4), (300, 5)):
        r = R.prosac_samples(1, n, m, 4000)
        S = O.Sampler(O.SAMPLER_PROSAC, O.RNG_PHILOX, n, m, 1)
        assert np.array_equal(S.growth(n), r["growth"])
        tab = S.table(4000)
        assert np.array_equal(tab[:, -1], r["samples"][:, -1])
        assert np.array_equal(r["subset"], r["samples"][:, -1] + 1) and np.array_equal(r["hyp"], np.arange(2, 4002))
        assert (tab[:, :-1] < tab[:, -1:]).all() and (r["samples"][:, :-1] < r["samples"][:, -1:]).all()
    # termination-length mode (prosac_sampler.hpp:141-144): once the pool has outgrown the stopping length everything freezes
    # and m points come from the closed range [0, termination_length]
    r = R.prosac_samples(2, 5000, 7, 3000, termination_length=40)
    S = O.Sampler(O.SAMPLER_PROSAC, O.RNG_PHILOX, 5000, 7, 2)
    S.set_termination_length(40)
    tab = S.table(3000)
    frozen = np.where(r["subset"] > 40)[0][0]
    assert np.array_equal(tab[:frozen + 1, -1], r["samples"][:frozen + 1, -1])
    assert (r["subset"][frozen:] == r["subset"][frozen]).all() and (r["hyp"][frozen:] == r["hyp"][frozen]).all()
    assert tab[frozen + 1:].max() <= 40 and r["samples"][frozen + 1:].max() <= 40


@needs_ref
@pytest.mark.parametrize("cfg", [1, 2, 3, 4])
def test_sprt_sequences_identical(cfg):
    """SPRT::SPRT pool shuffle (srand(seed)), then SPRT::verifyModelAndGetModelScore over 400 models in sequence with the
    running best as `maximum_score`: decisions, inlier counts (tested, and completed for the first 20 hypotheses), the pool
    cursor after every model, the test history (epsilon, delta, A as IEEE doubles, k) and SPRT::getUpperBoundIterations on
    every improvement."""
    est, thr = EST_OF_CFG[cfg], gen.CONFIGS[cfg]["threshold"]
    pts, gt, mask = data(cfg)
    g = np.random.default_rng(10 + cfg)
    models = some_models(est, pts, mask, 400, g, every=5)
    hyp = np.arange(len(models)) // (3 if est == O.EST_FUNDAMENTAL else 1)
    for seed in (1, 5):
        a = R._sequence(O.lib().orc_sprt_sequence, est, pts, thr, seed, 10000, models, hyp)
        b = R.sprt_sequence(est, pts, thr, seed, 10000, models, hyp)
        assert np.array_equal(a["pool"], b["pool"]) and np.array_equal(a["pool"], O.sprt_pool(seed, len(pts)))
        for k in ("good", "inliers", "pool_idx", "bound"):
            assert np.array_equal(a[k], b[k]), k
        assert a["history"].shape == b["history"].shape and np.array_equal(a["history"].view(np.uint64), b["history"].view(np.uint64))
        assert len(a["history"]) > 5 and 0 < a["good"].sum() < len(models)          # the sequence exercised accepts, rejects and re-designs


@needs_ref
def test_prosac_termination_sequence_identical():
    pts, gt, mask = gen.make(3, n=5000)
    g = np.random.default_rng(4)
    models = []
    while len(models) < 40:
        s = g.choice(np.where(mask)[0][:600], 7, replace=False) if len(models) % 2 == 0 else g.choice(len(pts), 7, replace=False)
        models.extend(O.solve_minimal(O.EST_FUNDAMENTAL, pts, s.astype(np.int32)))
    hc = np.sort(g.integers(1, 3000, len(models))).astype(np.uint32)
    lg = np.minimum(5000, 7 + hc // 3).astype(np.uint32)
    a = R.prosac_termination_sequence(O.EST_FUNDAMENTAL, pts, 2.0, 0.95, 10000, models, hc, lg, fn=O.lib().orc_prosac_termination_sequence)
    b = R.prosac_termination_sequence(O.EST_FUNDAMENTAL, pts, 2.0, 0.95, 10000, models, hc, lg)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert a[1].min() < 5000 and a[0].min() < 10000                                  # the criterion did shorten the run


@needs_ref
def test_neighbourhoods():
    pts = gen.homography(n=3000, inlier_ratio=0.2, clustered=True, seed=3)[0]
    nb = R.grid_neighbors(pts, 50)
    cell, members, start = O.grid_cells(pts, 50)
    for i in range(len(pts)):
        mem = members[start[cell[i]]:start[cell[i] + 1]]
        assert np.array_equal(nb[i], mem[mem != i])          # same members, same (ascending) order: the NAPSAC cursor walks this list
    assert np.array_equal(R.knn(pts, 6), O.knn_build(pts, 6))


@needs_ref
def test_line_solver_and_whole_run():
    """Line2DEstimator::EstimateModel bit for bit, and the whole driver - Ransac::Ransac + Ransac::run over UniformSampler on the
    glibc stream, with and without SPRT: iteration counts equal the oracle's main loop, inlier counts equal after the refit."""
    pts, gt, mask = gen.make(1)
    g = np.random.default_rng(2)
    for _ in range(200):
        s = g.choice(len(pts), 2, replace=False).astype(np.int32)
        assert np.array_equal(bits(O.solve_minimal(O.EST_LINE2D, pts, s)), bits(R.solve_minimal(O.EST_LINE2D, pts, s)))
    for sprt in (False, True):
        for seed in (1, 2, 3, 4, 5):
            a = R.ransac_run(O.EST_LINE2D, pts, 8.0, conf=0.99, max_it=10000, sprt=sprt, seed=seed)
            b = O.ransac(pts, O.EST_LINE2D, rng=O.RNG_GLIBC, threshold=8.0, confidence=0.99, max_iterations=10000, seed=seed, sprt=sprt)
            assert a["iterations"] == b["iterations"]
            assert a["inliers"] == O.refit(O.EST_LINE2D, pts, b["model"], b["inliers"], 8.0)["inliers"]


@needs_ref
def test_reference_four_point_dlt_is_not_a_minimal_solver():
    """SURVEY finding 5, now shown with the reference's own code: DLT4p takes the last row of a THIN SVD of the 8 x 9 system
    (dlt.cpp:43-48), i.e. the 8th singular vector instead of the null vector - its model does not pass through its own four
    points. The oracle / GPU use the true null vector of the normalised DLT (what BASELINE.json names), which does."""
    pts, H, mask = gen.make(2)
    g = np.random.default_rng(3)
    inl = np.where(mask)[0]
    ref_err, orc_err = [], []
    for _ in range(40):
        s = g.choice(inl, 4, replace=False).astype(np.int32)
        r, o = R.solve_minimal(O.EST_HOMOGRAPHY, pts, s), O.solve_minimal(O.EST_HOMOGRAPHY, pts, s)
        if len(r) and len(o):
            ref_err.append(R.errors(O.EST_HOMOGRAPHY, pts, r[0])[s].max())
            orc_err.append(O.errors(O.EST_HOMOGRAPHY, pts, o[0])[s].max())
    assert np.median(orc_err) < 1e-2 and np.median(ref_err) > 0.5
    # the consequence at the level of the whole driver: the termination criterion never fires for the reference
    a = R.ransac_run(O.EST_HOMOGRAPHY, pts, 2.0, conf=0.95, max_it=3000, seed=1)
    b = O.ransac(pts, O.EST_HOMOGRAPHY, rng=O.RNG_GLIBC, threshold=2.0, confidence=0.95, max_iterations=3000, seed=1)
    assert a["iterations"] == 3000 and b["iterations"] < 1500


@needs_ref
def test_reference_four_point_dlt_against_opencv_and_the_oracle_switch(golden_dir):
    """The same solver three ways (SURVEY Appendix B quirk 1): (i) the compiled reference's DLt::DLT4p on the stand-in SVD of
    oracle/ref_shim (which, like cv::SVD, orthogonalises the ROWS of a wide matrix), (ii) the oracle's documented switch
    orc_solve_homography_dlt4p_thin, (iii) the real OpenCV on the same float32 system (tests/golden/dlt4p_cv.npz). All three agree
    to float32 conditioning (sigma_8 / sigma_1 ~ 1e-7), and a whole fit with the switch behaves like the compiled reference's
    Ransac::run: every iteration spent, the same inlier set after the non-minimal refit."""
    import os
    d = np.load(os.path.join(golden_dir, "dlt4p_cv.npz"))
    s = np.arange(4, dtype=np.int32)
    ref_cv, ref_orc = [], []
    for pts, H in zip(d["pts"], d["H"]):
        r, o = R.solve_minimal(O.EST_HOMOGRAPHY, pts, s), O.solve_homography_dlt4p_thin(pts, s)
        assert len(r) == 1 and len(o) == 1
        ref_cv.append(np.abs(r[0] - H).max() / np.abs(H).max())
        ref_orc.append(np.abs(r[0] - o[0]).max() / np.abs(H).max())
    for rel in (np.array(ref_cv), np.array(ref_orc)):
        assert np.median(rel) < 1e-4 and np.quantile(rel, 0.9) < 1e-3 and rel.max() < 2e-2
    pts, H, mask = gen.make(2)
    for seed in (1, 2):
        a = R.ransac_run(O.EST_HOMOGRAPHY, pts, 2.0, conf=0.95, max_it=3000, seed=seed)
        b = O.ransac(pts, O.EST_HOMOGRAPHY, rng=O.RNG_GLIBC, threshold=2.0, confidence=0.95, max_iterations=3000, seed=seed, ref_thin_svd=True)
        fin = O.refit(O.EST_HOMOGRAPHY, pts, b["model"], b["inliers"], 2.0)
        assert a["iterations"] == b["iterations"] == 3000 and a["inliers"] == fin["inliers"]


@needs_ref
def test_nonminimal_solvers_agree():
    """Normalised DLT / 8-point on >= 20 points (2N x 9 resp. N x 9 with at least 9 rows: the thin SVD's last row IS the null
    vector there): unit-norm models agree to 1e-4 (BASELINE.json's model tolerance); the oracle uses an eigen-solve of A'A."""
    g = np.random.default_rng(5)
    for cfg in (2, 3, 4):
        pts, gt, mask = data(cfg, n=4000)
        inl = np.where(mask)[0]
        for cnt in (20, 100, len(inl)):
            ids = g.choice(inl, cnt, replace=False).astype(np.int32)
            a, b = O.nonminimal(EST_OF_CFG[cfg], pts, ids), R.nonminimal(EST_OF_CFG[cfg], pts, ids)
            assert a is not None and b is not None and np.abs(unit(a) - unit(b)).max() < 1e-4


@needs_ref
def test_seven_point_and_five_point_solvers_agree():
    """7-point: float32 SVD null space + solveCubic in the reference vs float64 elimination + bracketing in the oracle: the same
    number of models for >= 85 % of the samples, matched models within 1e-3 for >= 90 % (float32 conditioning, SURVEY hard part 4).
    5-point: the reference returns ONE essential matrix - the first root (Jenkins-Traub order, in a basis of the null space that
    depends on the SVD implementation) whose decomposition puts all five points in front of both cameras; it must be one of
    the oracle's candidates for that sample, and one the oracle also marks cheirality-valid."""
    pts, F, mask = gen.make(3, n=4000)
    g = np.random.default_rng(6)
    inl = np.where(mask)[0]
    same, diffs = 0, []
    for t in range(120):
        s = (g.choice(inl, 7, replace=False) if t % 2 else g.choice(len(pts), 7, replace=False)).astype(np.int32)
        a, b = O.solve_minimal(O.EST_FUNDAMENTAL, pts, s), R.solve_minimal(O.EST_FUNDAMENTAL, pts, s)
        if len(a) == len(b):
            same += 1
            diffs += [min(np.abs(unit(x) - unit(y)).max() for y in b) for x in a]
    assert same >= 0.85 * 120 and np.mean(np.asarray(diffs) < 1e-3) >= 0.9
    pts, E, mask = gen.make(4, n=4000)
    inl = np.where(mask)[0]
    returned = member = 0
    for t in range(80):
        s = (g.choice(inl, 5, replace=False) if t % 2 else g.choice(len(pts), 5, replace=False)).astype(np.int32)
        b = R.solve_minimal(O.EST_ESSENTIAL, pts, s)
        if len(b):
            returned += 1
            cands, valid = O.essential5_candidates(pts, s)
            d = [np.abs(unit(b[0]) - unit(c)).max() for c in cands]
            member += bool(len(d) and min(d) < 1e-4 and valid[int(np.argmin(d))])
    assert returned >= 20 and member >= 0.9 * returned


@needs_ref
def test_jenkins_traub_real_roots():
    """essential/rpoly.cpp on degree-10 polynomials with known roots (the degree of the five-point determinant)."""
    g = np.random.default_rng(7)
    for _ in range(100):
        real = g.uniform(-3, 3, 4)
        cplx = g.uniform(-2, 2, 3) + 1j * g.uniform(0.1, 2, 3)
        c = np.real(np.poly(np.concatenate([real, cplx, np.conj(cplx)])))
        zr, zi = R.rpoly(c)
        assert np.allclose(np.sort(zr[zi == 0]), np.sort(real), atol=1e-6)


def test_stand_in_svd_against_opencv(golden_dir):
    """The compiled reference runs on a stand-in cv::SVD (oracle/ref_shim/cvshim.hpp). tests/golden/svd_cv.npz holds what the REAL
    OpenCV returns for 220 matrices of the kinds the reference's estimators decompose (make_svd_golden.py: 7 x 9 float32 FULL_UV of the
    7-point solver, 5 x 9 float64 FULL_UV of the 5-point solver, the 8 x 9 thin system of DLT4p, 2N x 9 / N x 9 thin systems of the
    non-minimal solvers, 4 x 4 and 3 x 3 double). Same shapes of w / vt, singular values to working precision, the same null SPACE
    (compared as a projector - the basis inside it is the implementation's choice) and the same last row of a thin vt up to sign."""
    import os
    d = np.load(os.path.join(golden_dir, "svd_cv.npz"))
    worst = {}
    for i in range(len(d["kind"])):
        kind, depth, fl = int(d["kind"][i]), int(d["depth"][i]), int(d["flags"][i])
        r, c, vr, vc = (int(x) for x in d["shape"][i])
        A = d["A"][i][:r, :c]
        w_cv, vt_cv = d["w"][i][:min(r, c)], d["vt"][i][:vr, :vc]
        w, u, vt = R.shim_svd(A, depth == 64, fl)
        assert vt.shape == (vr, vc) and len(w) == min(r, c)
        e_w = np.abs(w - w_cv).max() / w_cv.max()
        if kind in (0, 1):                                   # FULL_UV of a wide matrix: rows r.. of vt span the null space
            e_v = np.abs(vt[r:].T @ vt[r:] - vt_cv[r:].T @ vt_cv[r:]).max()
        elif kind == 6:
            e_v = 0.0
        else:
            e_v = min(np.abs(vt[-1] - vt_cv[-1]).max(), np.abs(vt[-1] + vt_cv[-1]).max())
        e_rec = np.abs((u[:, :len(w)] * w) @ vt[:len(w)] - A).max() / np.abs(A).max()
        tol = 1e-10 if depth == 64 else 2e-6
        assert e_w < tol and e_rec < 10 * tol, (kind, i, e_w, e_rec)
        worst.setdefault(kind, []).append(e_v)
    for kind, errs in worst.items():
        errs = np.array(errs)
        if kind == 2:                                        # DLT4p's 8th singular vector: sigma_8 / sigma_1 ~ 1e-7 in float32
            assert np.median(errs) < 1e-5 and errs.max() < 2e-2
        else:
            assert errs.max() < (1e-10 if kind in (1, 5, 6) else 1e-4), (kind, errs.max())


def test_stand_in_eigen_cubic_inverse_against_opencv(golden_dir):
    """The other stand-in routines on the path, against cv2 fixtures: cv::eigen on the 2 x 2 float32 scatter matrix of the non-minimal
    line fit (eig_cv.npz: values and vectors to float32 rounding), cv::solveCubic of the 7-point solver (cv_primitives.npz: the same
    root COUNT and ORDER for all 512 cubics - which needs OpenCV's expanded discriminant - and the same values to 1e-9 except where
    the trigonometric formula itself is ill-conditioned, <= 1e-5), Mat::inv of a float 3 x 3 (bit-identical, singular -> zeros)."""
    import os
    d = np.load(os.path.join(golden_dir, "eig_cv.npz"))
    for A, vals, vecs in zip(d["A"], d["vals"], d["vecs"]):
        e, v = R.shim_eigen(A, False)
        assert np.abs(e - vals).max() <= 4e-7 * np.abs(vals).max()
        for i in range(2):
            assert min(np.abs(v[i] - vecs[i]).max(), np.abs(v[i] + vecs[i]).max()) < 1e-6
    c = np.load(os.path.join(golden_dir, "cv_primitives.npz"))
    loose = 0
    for co, ref, n in zip(c["cubic_in"], c["cubic_out"], c["cubic_n"]):
        k, r = R.shim_cubic(co)
        assert k == n, co
        for a, b in zip(r[:k], ref[:n]):
            err = abs(a - b) / max(1.0, abs(b))
            assert err < 1e-5, (co, a, b)
            loose += err > 1e-9
    assert loose <= 8
    for m, ref in zip(c["inv_in"], c["inv_out"]):
        assert np.array_equal(R.shim_inv3(m).view(np.uint32), ref.view(np.uint32))


@needs_ref
def test_reference_runs_past_max_iterations():
    """`max_iterations` is the INITIAL bound of `while (iters < max_iters)` (ransac.cpp:58), not a cap: the standard criterion answers
    it only while w^m < 0.0005 and an uncapped value otherwise (standard_termination_criteria.hpp:52-62), so the compiled reference's
    Ransac::run ends line fits with max_iterations 3 / 5 / 10 after 15 - 46 iterations - and so does the oracle, identically. (The GPU
    side of this: test_fit_runs_past_max_iterations_like_the_reference.)"""
    pts = gen.make(1)[0]
    for conf in (0.99, 0.999999):
        for max_it in (3, 5, 10):
            for seed in (1, 4):
                a = R.ransac_run(O.EST_LINE2D, pts, 8.0, conf=conf, max_it=max_it, seed=seed)
                b = O.ransac(pts, O.EST_LINE2D, rng=O.RNG_GLIBC, threshold=8.0, confidence=conf, max_iterations=max_it, seed=seed)
                assert a["iterations"] == b["iterations"] > max_it
                assert a["inliers"] == O.refit(O.EST_LINE2D, pts, b["model"], b["inliers"], 8.0)["inliers"]
