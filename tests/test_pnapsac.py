"""Progressive NAPSAC (DESIGN.md section 4.8), CPU part: the sequential reference sampler (pnapsac_oracle.cpp) against an
independent restatement of its four steps, and the properties the definition promises."""
import math

import numpy as np
import pytest

import pnapsac_oracle as PN
from oracle import oracle as O
from ransac_b200 import generator as gen


def restated(seed, knn, m, count, length):
    """Steps 1-4 of the definition, one hypothesis at a time -> (samples, centre, s) with centre -1 in the global phase."""
    n, k = knn.shape
    uses = np.zeros(n, np.int64)
    rows, centres, sizes = [], [], []
    for h in range(count):
        if h >= length:
            rows.append(O.philox_unique(seed, h, 0, n, m)); centres.append(-1); sizes.append(0)
            continue
        p = int(O.philox_unique(seed, h, 5, n, 1)[0])
        uses[p] += 1
        s = next((c for c in range(m - 1, k + 1) if math.comb(c, m - 1) >= uses[p]), k)
        j = O.philox_unique(seed, h, 6, s - 1, m - 2) if m > 2 else np.zeros(0, np.int32)
        rows.append(np.concatenate([[p], knn[p, j], [knn[p, s - 1]]]).astype(np.int32)); centres.append(p); sizes.append(s)
    return np.stack(rows), np.array(centres), np.array(sizes)


def problem(est, n, seed):
    if est == O.EST_LINE2D:
        return gen.line2d(n=n, seed=seed)[0]
    if est == O.EST_FUNDAMENTAL:
        return gen.make(3, n=n, seed_offset=seed)[0]
    return gen.homography(n=n, inlier_ratio=0.3, clustered=True, seed=seed)[0]


@pytest.mark.parametrize("est", [O.EST_HOMOGRAPHY, O.EST_FUNDAMENTAL, O.EST_LINE2D])
@pytest.mark.parametrize("k", [7, 31])
def test_reference_table_matches_the_definition(est, k):
    m = O.SAMPLE_SIZE[est]
    pts = problem(est, 400, 3 + k)
    knn = O.knn_build(pts, k)
    count, length = 3000, 2600                       # ~7 uses per centre, and the switch to global sampling inside the table
    got = PN.table(11, knn, m, count, length)
    want, centres, sizes = restated(11, knn, m, count, length)
    assert np.array_equal(got, want)
    local = centres >= 0
    assert local.sum() == length
    for h in np.where(local)[0]:
        p, s, row = centres[h], sizes[h], got[h]
        assert row[0] == p                                        # contains its centre
        assert set(row[1:]) <= set(knn[p, :s])                    # draws only from the centre's s(t) nearest
        assert row[-1] == knn[p, s - 1]                           # includes the s(t)-th nearest
        assert len(set(row)) == m
    for h in np.where(~local)[0]:
        assert np.array_equal(got[h], O.philox_unique(11, h, 0, len(pts), m))
    assert sizes[local].max() > m - 1 and sizes.max() <= k        # neighbourhoods grow past the first m - 1 nearest, up to k


def test_first_use_of_a_centre_is_its_nearest_neighbours():
    """t = 1: s = m - 1, so the sample is the centre and its m - 1 nearest - the set NAPSAC-kNN draws first."""
    pts = problem(O.EST_HOMOGRAPHY, 2000, 5)
    knn = O.knn_build(pts, 8)
    got = PN.table(2, knn, 4, 500)
    seen = set()
    for row in got:
        p = row[0]
        if p not in seen:
            assert set(row[1:]) == set(knn[p, :3])
            seen.add(p)
    assert len(seen) > 400


def test_default_length_is_twenty_n():
    pts = problem(O.EST_LINE2D, 30, 1)
    knn = O.knn_build(pts, 5)
    got = PN.table(4, knn, 2, 700)
    want, centres, _ = restated(4, knn, 2, 700, 600)
    assert np.array_equal(got, want) and (centres[:600] >= 0).all() and (centres[600:] < 0).all()


def test_fit_with_the_sampler_draws_its_stream():
    """PN.ransac is the oracle's loop replaying the sampler's stream: its winning sample is the stream's sample of best_hyp."""
    pts, _, mask = gen.homography(n=3000, inlier_ratio=0.2, clustered=True, seed=12)
    knn = O.knn_build(pts, 8)
    r = PN.ransac(pts, O.EST_HOMOGRAPHY, knn, seed=3, threshold=2.0, confidence=0.95, max_iterations=2000)
    assert r["rc"] == 0 and 0 <= r["best_hyp"] < r["samples_drawn"]
    smp = PN.table(3, knn, 4, r["best_hyp"] + 1)[-1]
    model = O.solve_minimal(O.EST_HOMOGRAPHY, pts, smp)[0]
    assert np.array_equal(model.view(np.uint32), np.asarray(r["model"], np.float32).view(np.uint32))
    assert O.score(O.EST_HOMOGRAPHY, pts, model, 2.0)[0] == r["inliers"]
