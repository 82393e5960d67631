"""ctypes binding of the CPU oracle (oracle/libusac_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs. The product package (ransac_b200) must never import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libusac_oracle.so")
SHIM_LIB = os.path.join(_HERE, "libref_shim.so")      # the stand-in OpenCV numerics of ref_shim/ (ref_shim_entry.cpp), for oracle/ref.py

EST_LINE2D, EST_HOMOGRAPHY, EST_FUNDAMENTAL, EST_ESSENTIAL = 1, 2, 3, 4
SAMPLER_UNIFORM, SAMPLER_PROGRESSIVE_NAPSAC, SAMPLER_NAPSAC, SAMPLER_PROSAC = 1, 2, 3, 4
NEIGH_NONE, NEIGH_KNN, NEIGH_GRID = 0, 1, 2
RNG_GLIBC, RNG_PHILOX, RNG_TABLE = 0, 1, 2
SAMPLE_SIZE = {EST_LINE2D: 2, EST_HOMOGRAPHY: 4, EST_FUNDAMENTAL: 7, EST_ESSENTIAL: 5}
MAX_MODELS = {EST_LINE2D: 1, EST_HOMOGRAPHY: 1, EST_FUNDAMENTAL: 3, EST_ESSENTIAL: 1}


def build(force=False):
    """Compile the oracle with its Makefile (g++). Building the checker is not using it."""
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".h"))]
    libs = (_LIB, SHIM_LIB)
    if force or not all(os.path.exists(lib) for lib in libs) or any(os.path.getmtime(s) > os.path.getmtime(lib) for s in srcs for lib in libs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB


class Config(C.Structure):
    _fields_ = [("estimator", C.c_int), ("sampler", C.c_int), ("rng", C.c_int), ("threshold", C.c_float),
                ("confidence", C.c_float), ("max_iterations", C.c_uint), ("sprt", C.c_int), ("batch", C.c_int),
                ("neighbors", C.c_int), ("knn", C.c_int), ("cell_size", C.c_int), ("seed", C.c_uint64),
                ("sample_table", C.POINTER(C.c_int)), ("sample_table_rows", C.c_uint),
                ("knn_table", C.POINTER(C.c_int)), ("lo", C.c_int), ("ref_thin_svd", C.c_int)]


class Result(C.Structure):
    _fields_ = [("model", C.c_float * 9), ("inliers", C.c_int), ("score", C.c_float), ("iterations", C.c_uint),
                ("samples_drawn", C.c_uint), ("best_hyp", C.c_longlong), ("best_model_idx", C.c_int),
                ("evals", C.c_ulonglong), ("models_scored", C.c_uint), ("lo_inner", C.c_uint), ("lo_iterative", C.c_uint)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        fp, ip, dp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)
        L.orc_glibc_rand_new.restype = C.c_void_p
        L.orc_glibc_rand_new.argtypes = [C.c_uint]
        L.orc_glibc_rand_free.argtypes = [C.c_void_p]
        L.orc_glibc_rand_next.restype = C.c_int32
        L.orc_glibc_rand_next.argtypes = [C.c_void_p]
        L.orc_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.orc_errors.argtypes = [C.c_int, fp, C.c_int, fp, fp]
        L.orc_score.argtypes = [C.c_int, fp, C.c_int, fp, C.c_float, ip, fp, ip, C.c_double, ip]
        L.orc_inv3x3.argtypes = [fp, fp]
        L.orc_inv3x3.restype = C.c_int
        L.orc_solve_minimal.argtypes = [C.c_int, fp, ip, fp]
        L.orc_solve_minimal.restype = C.c_int
        L.orc_solve_homography_dlt4p_thin.argtypes = [fp, ip, fp]
        L.orc_solve_homography_dlt4p_thin.restype = C.c_int
        L.orc_solve_cubic.argtypes = [dp, dp]
        L.orc_solve_cubic.restype = C.c_int
        L.orc_fundamental_is_valid.argtypes = [fp, fp, ip]
        L.orc_fundamental_is_valid.restype = C.c_int
        L.orc_null_space.argtypes = [dp, C.c_int, dp]
        L.orc_null_space.restype = C.c_int
        L.orc_sampler_new.restype = C.c_void_p
        L.orc_sampler_new.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64]
        L.orc_sampler_free.argtypes = [C.c_void_p]
        L.orc_sampler_set_knn.argtypes = [C.c_void_p, ip, C.c_int]
        L.orc_sampler_set_grid.argtypes = [C.c_void_p, fp, C.c_int]
        L.orc_sampler_set_termination_length.argtypes = [C.c_void_p, C.c_uint]
        L.orc_sampler_largest_sample_size.argtypes = [C.c_void_p]
        L.orc_sampler_largest_sample_size.restype = C.c_uint
        L.orc_sampler_growth_function.argtypes = [C.c_void_p]
        L.orc_sampler_growth_function.restype = C.POINTER(C.c_uint)
        L.orc_sampler_generate.argtypes = [C.c_void_p, C.c_uint64, ip]
        L.orc_philox_unique.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, ip]
        L.orc_standard_termination.argtypes = [C.c_uint, C.c_uint, C.c_int, C.c_float, C.c_uint]
        L.orc_standard_termination.restype = C.c_uint
        L.orc_grid_cells.argtypes = [fp, C.c_int, C.c_int, ip, ip, ip, ip]
        L.orc_knn_build.argtypes = [fp, C.c_int, C.c_int, C.c_int, ip]
        L.orc_knn_build.restype = C.c_int
        L.orc_ransac.argtypes = [C.POINTER(Config), fp, C.c_int, C.POINTER(Result)]
        L.orc_ransac.restype = C.c_int
        L.orc_essential5_candidates.argtypes = [fp, ip, dp, ip]
        L.orc_essential5_candidates.restype = C.c_int
        L.orc_nonminimal.argtypes = [C.c_int, fp, ip, C.c_int, fp]
        L.orc_nonminimal.restype = C.c_int
        L.orc_refit.argtypes = [C.c_int, fp, C.c_int, C.c_float, fp, C.c_int, ip, ip]
        L.orc_refit.restype = C.c_int
        L.orc_sprt_pool.argtypes = [C.c_uint64, C.c_int, ip]
        L.orc_sprt_pool.restype = None
        up = C.POINTER(C.c_uint)
        L.orc_sprt_sequence.argtypes = [C.c_int, fp, C.c_int, C.c_float, C.c_uint64, C.c_uint, fp, C.c_int, ip, ip, ip, up, up, dp, ip, ip]
        L.orc_prosac_termination_sequence.argtypes = [C.c_int, fp, C.c_int, C.c_float, C.c_float, C.c_uint, fp, C.c_int, up, up, up, up]
        _lib = L
    return _lib


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _pts(points):
    p = np.ascontiguousarray(points, dtype=np.float32)
    return p, p.shape[0]


def glibc_random(seed, count):
    L = lib()
    g = L.orc_glibc_rand_new(seed)
    out = [L.orc_glibc_rand_next(g) for _ in range(count)]
    L.orc_glibc_rand_free(g)
    return out


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return list(o)


def errors(est, points, model):
    p, n = _pts(points)
    m = np.ascontiguousarray(model, dtype=np.float32).ravel()
    out = np.empty(n, np.float32)
    lib().orc_errors(est, _f(p), n, _f(m), _f(out))
    return out


def score(est, points, model, thr, band_rel=1e-6, want_inliers=False):
    """-> (count, sum, flagged[, inlier ids])"""
    p, n = _pts(points)
    m = np.ascontiguousarray(model, dtype=np.float32).ravel()
    cnt, flg, s = C.c_int(), C.c_int(), C.c_float()
    ids = np.empty(n, np.int32) if want_inliers else None
    lib().orc_score(est, _f(p), n, _f(m), thr, C.byref(cnt), C.byref(s), _i(ids) if want_inliers else None, band_rel, C.byref(flg))
    if want_inliers:
        return cnt.value, s.value, flg.value, ids[:cnt.value].copy()
    return cnt.value, s.value, flg.value


def inv3x3(m):
    a = np.ascontiguousarray(m, dtype=np.float32).ravel()
    out = np.empty(9, np.float32)
    ok = lib().orc_inv3x3(_f(a), _f(out))
    return out.reshape(3, 3), ok


def solve_minimal(est, points, sample):
    """-> array (k, 9) (line: (k, 3)) of the k models of this sample"""
    p, _ = _pts(points)
    s = np.ascontiguousarray(sample, dtype=np.int32)
    out = np.zeros(27, np.float32)
    k = lib().orc_solve_minimal(est, _f(p), _i(s), _f(out))
    w = 3 if est == EST_LINE2D else 9
    return out[:k * w].reshape(k, w).copy() if est != EST_LINE2D else out[:3 * k].reshape(k, 3).copy()


def solve_homography_dlt4p_thin(points, sample):
    """SURVEY Appendix B quirk 1: the reference's DLt::DLT4p (8th singular vector of the raw 8 x 9 system) -> (k, 9), k in {0, 1}"""
    p, _ = _pts(points)
    s = np.ascontiguousarray(sample, dtype=np.int32)
    out = np.zeros(9, np.float32)
    k = lib().orc_solve_homography_dlt4p_thin(_f(p), _i(s), _f(out))
    return out.reshape(1, 9)[:k].copy()


def essential5_candidates(points, sample):
    """-> (E [k,3,3] float64, valid [k] bool) in the solver's visiting order"""
    p, _ = _pts(points)
    s = np.ascontiguousarray(sample, dtype=np.int32)
    Es = np.zeros(90, np.float64)
    valid = np.zeros(10, np.int32)
    k = lib().orc_essential5_candidates(_f(p), _i(s), Es.ctypes.data_as(C.POINTER(C.c_double)), _i(valid))
    return Es[:9 * k].reshape(k, 3, 3).copy(), valid[:k].astype(bool)


def solve_cubic(c):
    cc = (C.c_double * 4)(*c)
    r = (C.c_double * 3)()
    n = lib().orc_solve_cubic(cc, r)
    return n, list(r)


def null_space(A):
    a = np.array(A, dtype=np.float64, order="C")
    rows = a.shape[0]
    out = np.zeros((9 - rows, 9), np.float64)
    ok = lib().orc_null_space(a.ctypes.data_as(C.POINTER(C.c_double)), rows, out.ctypes.data_as(C.POINTER(C.c_double)))
    return out if ok else None


def philox_unique(seed, hyp, stream, n, m):
    out = np.empty(m, np.int32)
    lib().orc_philox_unique(seed, hyp, stream, n, m, _i(out))
    return out


def standard_termination(inliers, n, m, conf, max_it):
    return lib().orc_standard_termination(inliers, n, m, conf, max_it)


def grid_cells(points, cell_size):
    p, n = _pts(points)
    cell = np.empty(n, np.int32)
    members = np.empty(n, np.int32)
    start = np.empty(n + 1, np.int32)
    nc = C.c_int()
    lib().orc_grid_cells(_f(p), n, cell_size, _i(cell), _i(members), _i(start), C.byref(nc))
    return cell, members, start[:nc.value + 1].copy()


def knn_build(points, k):
    """n x k table of nearest_neighbors.cpp:69-128 (brute force; ties by ascending index)."""
    p, n = _pts(points)
    out = np.empty((n, k), np.int32)
    if lib().orc_knn_build(_f(p), n, p.shape[1], k, _i(out)) != 0:
        raise ValueError("knn_build: needs n >= k + 1")
    return out


class Sampler:
    def __init__(self, kind, rng, n, m, seed, points=None, cell_size=50, knn_table=None):
        self.L = lib()
        self.m = m
        self.h = self.L.orc_sampler_new(kind, rng, n, m, seed)
        if kind == SAMPLER_NAPSAC:
            if knn_table is not None:
                t = np.ascontiguousarray(knn_table, dtype=np.int32)
                self.L.orc_sampler_set_knn(self.h, _i(t), t.shape[1])
            else:
                p, _ = _pts(points)
                self.L.orc_sampler_set_grid(self.h, _f(p), cell_size)

    def generate(self, hyp_id=0):
        out = np.empty(self.m, np.int32)
        self.L.orc_sampler_generate(self.h, hyp_id, _i(out))
        return out

    def table(self, count, first_hyp=0):
        return np.stack([self.generate(first_hyp + i) for i in range(count)])

    def set_termination_length(self, v):
        self.L.orc_sampler_set_termination_length(self.h, v)

    def growth(self, n):
        g = self.L.orc_sampler_growth_function(self.h)
        return np.array([g[i] for i in range(n)], np.uint32)

    def __del__(self):
        try:
            self.L.orc_sampler_free(self.h)
        except Exception:
            pass


def nonminimal(est, points, ids):
    """EstimateModelNonMinimalSample on point ids -> model or None"""
    p, _ = _pts(points)
    t = np.ascontiguousarray(ids, dtype=np.int32)
    out = np.zeros(9, np.float32)
    ok = lib().orc_nonminimal(est, _f(p), _i(t), len(t), _f(out))
    return out[:3 if est == EST_LINE2D else 9].copy() if ok else None


def refit(est, points, model, best_inliers, thr):
    """ransac.cpp:157-207 -> dict(model, inliers, accepted, ids)"""
    p, n = _pts(points)
    m = np.zeros(9, np.float32)
    w = 3 if est == EST_LINE2D else 9
    m[:w] = np.asarray(model, np.float32).ravel()[:w]
    ids = np.zeros(n + 1, np.int32)
    acc = C.c_int()
    best = lib().orc_refit(est, _f(p), n, thr, _f(m), int(best_inliers), _i(ids), C.byref(acc))
    cnt = score(est, points, m[:w], thr)[0]
    return {"model": m[:w].copy(), "inliers": best, "accepted": acc.value, "ids": ids[:cnt].copy()}


def sprt_pool(seed, n):
    out = np.empty(n, np.int32)
    lib().orc_sprt_pool(seed, n, _i(out))
    return out


def ransac(points, est, sampler=SAMPLER_UNIFORM, rng=RNG_PHILOX, threshold=2.0, confidence=0.95, max_iterations=10000,
           sprt=False, batch=0, seed=1, neighbors=NEIGH_NONE, knn=5, cell_size=50, sample_table=None, knn_table=None, lo=0,
           ref_thin_svd=False):
    p, n = _pts(points)
    cfg = Config()
    cfg.estimator, cfg.sampler, cfg.rng = est, sampler, rng
    cfg.threshold, cfg.confidence, cfg.max_iterations = threshold, confidence, max_iterations
    cfg.sprt, cfg.batch, cfg.neighbors, cfg.knn, cfg.cell_size, cfg.seed = int(sprt), batch, neighbors, knn, cell_size, seed
    cfg.lo = lo
    cfg.ref_thin_svd = int(ref_thin_svd)     # SURVEY Appendix B quirk 1: the reference's DLT4p instead of the normalised DLT
    keep = []
    if sample_table is not None:
        t = np.ascontiguousarray(sample_table, dtype=np.int32)
        keep.append(t)
        cfg.sample_table, cfg.sample_table_rows = _i(t), t.shape[0]
    if knn_table is not None:
        t = np.ascontiguousarray(knn_table, dtype=np.int32)
        keep.append(t)
        cfg.knn_table, cfg.knn = _i(t), t.shape[1]
    res = Result()
    rc = lib().orc_ransac(C.byref(cfg), _f(p), n, C.byref(res))
    w = 3 if est == EST_LINE2D else 9
    return {"rc": rc, "model": np.array(res.model[:w], np.float32), "inliers": res.inliers, "score": res.score,
            "iterations": res.iterations, "samples_drawn": res.samples_drawn, "best_hyp": res.best_hyp,
            "best_model_idx": res.best_model_idx, "evals": res.evals, "models_scored": res.models_scored,
            "lo_inner": res.lo_inner, "lo_iterative": res.lo_iterative}
