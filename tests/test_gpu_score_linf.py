"""Inlier counts of the survivor-queue scoring kernel (score_sq.cuh) for homographies, against the oracle.

`GpuContext.score` normally runs the loop kernel (score.cuh: caller-supplied models are mostly good ones), so the queue kernel's
rejection test - FastModel<HOMOGRAPHY>::reject, which runs in every fit - is exercised here in a subprocess with
USAC_GPU_SCORE_LEGACY=2 (read once per process), which sends every launch to the queue kernel. Two model sets:
  - the random-sample, all-inlier and perturbed ground-truth models of test_score_counts_exact_stress;
  - hand-built points around a scaling model whose inlier boundary lies just inside the rejection bound (the backward
    distance is 1/256 of the forward one): points on the axes and diagonals just inside and outside the threshold and the
    bound, points in the corners of the max-norm square outside the disc (outliers that must be drained), and, around a
    projective model, points with nz exactly 0, nz near 0, and NaN coordinates.
Every count must equal the oracle's; a rejection test that claims an inlier as an outlier lowers a count."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THRS = (0.5, 2.0, 20.0)


def stress_models(seed):
    """The homography models of test_score_counts_exact_stress (tests/test_gpu_parity.py) for one seed."""
    from oracle import oracle as O
    from ransac_b200 import generator as gen
    g = np.random.default_rng(seed)
    pts, H, mask = gen.homography(n=4000, seed=200 + seed)
    inl = np.where(mask)[0]
    models = []
    while len(models) < 1500:
        models.extend(O.solve_minimal(O.EST_HOMOGRAPHY, pts, g.choice(4000, 4, replace=False).astype(np.int32)))
    while len(models) < 1800:
        models.extend(O.solve_minimal(O.EST_HOMOGRAPHY, pts, g.choice(inl, 4, replace=False).astype(np.int32)))
    for _ in range(248):
        P = H.astype(np.float64) * (1 + g.normal(0, 10 ** g.uniform(-7, -2), (3, 3)))
        P[:2, 2] += g.normal(0, 10 ** g.uniform(-3, 0.5), 2)
        models.append((P / P[2, 2]).astype(np.float32).ravel())
    return pts, np.stack(models[:2048]).astype(np.float32)


def project(H, p1):
    q = np.c_[p1.astype(np.float64), np.ones(len(p1))] @ H.astype(np.float64).T
    return q[:, :2] / q[:, 2:3]


def boundary_set(thr, seed=5):
    """Points around S = scale 256 (+ a small rotation in a second model): offsets of the forward projection at distances that put
    the reference's error just below / above thr (d1 = 2 thr 256/257) and at the rejection bound (d1 = 2 thr), along the axes, the
    diagonals and random directions, plus max-norm corners (a, a) with 2 thr / sqrt 2 < a < 2 thr. Odd count: a padded last pair."""
    g = np.random.default_rng(seed)
    s = 256.0
    S = np.array([[s, 0, 3], [0, s, -2], [0, 0, 1]], np.float32)
    c, sn = np.cos(0.3), np.sin(0.3)
    R = np.array([[s * c, -s * sn, 5], [s * sn, s * c, 1], [0, 0, 1]], np.float32)
    T2 = 2.0 * thr
    inner = s / (s + 1)                                          # reference error = thr at d1 = 2 thr s / (s + 1) for S
    fr = np.r_[inner * (1 + np.array([-1e-3, -1e-4, -1e-5, -1e-6, 0, 1e-6, 1e-5, 1e-4, 1e-3])),
               1 + np.array([-1e-3, -1e-4, -1e-5, -1e-6, 0, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2]), [0.5, 0.9, 1.1, 1.5]]
    ang = np.r_[np.arange(8) * np.pi / 4, g.uniform(0, 2 * np.pi, 8)]
    offs = [T2 * f * np.array([np.cos(a), np.sin(a)]) for f in fr for a in ang]
    for a in (0.71, 0.72, 0.8, 0.9, 0.99, 0.999):                  # corners of the square outside the disc
        offs += [T2 * a * np.array([sx, sy]) for sx in (-1, 1) for sy in (-1, 1)]
    offs = np.array(offs)
    pts = []
    for M in (S, R):
        p1 = g.uniform(0, 4, (len(offs), 2)).astype(np.float32)
        pts.append(np.c_[p1, project(M, p1) + offs])
    pts = np.concatenate(pts).astype(np.float32)
    if len(pts) % 2 == 0:
        pts = pts[:-1]
    rest = [S.ravel(), R.ravel(), np.eye(3, dtype=np.float32).ravel()]
    for _ in range(61):                                          # S and R perturbed by up to the band's scale
        M = (S if _ % 2 else R).astype(np.float64) * (1 + g.normal(0, 10 ** g.uniform(-8, -4), (3, 3)))
        M[2, 2] = 1
        rest.append(M.astype(np.float32).ravel())
    return pts, np.stack(rest).astype(np.float32)


def degenerate_set(thr, seed=6):
    """Around P (h31 = 1/512, h32 = -1/1024): points with nz = h31 x1 + h32 y1 + 1 exactly 0 (x1 = -512, y1 = 0; also with y1 on
    the line y1 = 2 x1 + 1024), nz within a few ulps of 0, ordinary points, and points with a NaN coordinate (x1, y1, x2 or y2 alone:
    a NaN in one coordinate of the forward residual)."""
    g = np.random.default_rng(seed)
    P = np.array([[1.1, 0.05, 10], [-0.03, 0.95, -4], [1 / 512, -1 / 1024, 1]], np.float32)
    p1 = [[-512.0, 0.0], [0.0, 1024.0], [-256.0, 512.0], [-128.0, 768.0]]
    for e in (2.0 ** -k for k in (4, 8, 12, 16, 20)):
        p1 += [[-512.0 + e, 0.0], [-512.0 - e, 0.0], [0.0, 1024.0 + e], [0.0, 1024.0 - e]]
    p1 = np.array(p1, np.float32)
    p2 = np.r_[g.uniform(-800, 800, (len(p1) - 4, 2)), [[0.0, 0.0], [1e3, -1e3], [3.0, 4.0], [-7.0, 2.0]]]
    q1 = g.uniform(-400, 400, (200, 2)).astype(np.float32)
    q2 = project(P, q1) + g.normal(0, thr, (200, 2))
    pts = np.r_[np.c_[p1, p2], np.c_[q1, q2]].astype(np.float32)
    pts = np.clip(pts, -2000, 2000)                              # the far projections of nz ~ 0 stay in the problem's range
    nan = pts[:8].copy()
    for k in range(4):
        nan[2 * k, k] = np.nan                                   # NaN in one coordinate, its pair partner finite
    pts = np.r_[pts[:40], nan, pts[40:]].astype(np.float32)
    models = [P.ravel(), np.eye(3, dtype=np.float32).ravel()]
    for _ in range(30):
        M = P.astype(np.float64) * (1 + g.normal(0, 10 ** g.uniform(-7, -2), (3, 3)))
        models.append((M / M[2, 2]).astype(np.float32).ravel())
    return pts, np.stack(models).astype(np.float32)


def cases():
    out = []
    for seed in (11, 12):
        pts, models = stress_models(seed)
        out += [(f"stress{seed}", thr, pts, models) for thr in THRS]
    for thr in THRS:
        out.append((f"boundary@{thr}", thr) + boundary_set(thr))
        out.append((f"degenerate@{thr}", thr) + degenerate_set(thr))
    return out


def device_counts(path_in, path_out):
    """Subprocess side: every case through ctx.score with the queue kernel."""
    from ransac_b200 import GpuContext, capi
    d = np.load(path_in)
    ctx = GpuContext(0)
    res = {}
    for k in range(int(d["n"])):
        ctx.set_points(capi.EST_HOMOGRAPHY, d[f"pts{k}"])
        res[f"cnt{k}"], _ = ctx.score(d[f"models{k}"], float(d[f"thr{k}"]))
    ctx.close()
    np.savez(path_out, **res)


@pytest.mark.gpu
def test_queue_kernel_homography_counts_exact(tmp_path):
    from oracle import oracle as O
    cs = cases()
    fin, fout = tmp_path / "cases.npz", tmp_path / "counts.npz"
    arrays = {"n": len(cs)}
    for k, (_, thr, pts, models) in enumerate(cs):
        arrays.update({f"pts{k}": pts, f"models{k}": models, f"thr{k}": thr})
    np.savez(fin, **arrays)
    env = dict(os.environ, USAC_GPU_SCORE_LEGACY="2")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(fin), str(fout)], cwd=ROOT, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:]
    got = np.load(fout)
    for k, (name, thr, pts, models) in enumerate(cs):
        ref = np.array([O.score(O.EST_HOMOGRAPHY, pts, m, thr)[0] for m in models])
        cnt = got[f"cnt{k}"]
        bad = np.where(cnt != ref)[0]
        assert len(bad) == 0, (name, bad[:10], cnt[bad[:10]], ref[bad[:10]])
        if name.startswith("boundary"):
            assert 0 < ref[0] < len(pts), (name, ref[0])         # S has inliers and near-inlier outliers in the set


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    device_counts(sys.argv[1], sys.argv[2])
