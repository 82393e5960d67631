"""ctypes binding of oracle/_ref/libusac_ref.so: the REFERENCE'S OWN usac/ sources compiled where they lie under
/root/reference (oracle/Makefile.ref), OpenCV / Eigen / nanoflann answered by the stand-ins in oracle/ref_shim/.

TEST INFRASTRUCTURE ONLY (same contract as oracle.py). The library is built in the development container (where
/root/reference exists) and travels to the GPU box as a prebuilt file; `available()` is False when neither is present.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_ref", "libusac_ref.so")
REFERENCE = os.environ.get("USAC_REFERENCE", "/root/reference")


def build(force=False):
    """Compile the reference (only possible where its sources are); returns the library path or None."""
    if not os.path.isdir(os.path.join(REFERENCE, "usac")):
        return _LIB if os.path.exists(_LIB) else None
    subprocess.check_call(["make", "-C", _HERE, "-f", "Makefile.ref", "-s", "-j8", f"REF={REFERENCE}"] + (["-B"] if force else []))
    return _LIB


def available():
    return os.path.exists(_LIB) or os.path.isdir(os.path.join(REFERENCE, "usac"))


class RunResult(C.Structure):
    _fields_ = [("model", C.c_float * 9), ("inliers", C.c_int), ("iterations", C.c_uint), ("lo_inner", C.c_uint), ("lo_iterative", C.c_uint),
                ("time_us", C.c_longlong)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if build() is None:
            raise RuntimeError("oracle/_ref/libusac_ref.so is missing and the reference sources are not here to build it")
        L = C.CDLL(_LIB)
        fp, ip, up, dp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_uint), C.POINTER(C.c_double)
        L.ref_errors.argtypes = [C.c_int, fp, C.c_int, fp, fp]
        L.ref_score.argtypes = [C.c_int, fp, C.c_int, fp, C.c_float, ip, fp, ip]
        L.ref_solve_minimal.argtypes = [C.c_int, fp, C.c_int, ip, fp]
        L.ref_nonminimal.argtypes = [C.c_int, fp, C.c_int, ip, C.c_int, fp]
        L.ref_standard_termination.argtypes = [C.c_uint, C.c_uint, C.c_int, C.c_float, C.c_uint]
        L.ref_standard_termination.restype = C.c_uint
        L.ref_uniform_samples.argtypes = [C.c_uint, C.c_int, C.c_int, C.c_int, ip]
        L.ref_uniform_samples.restype = None
        L.ref_prosac_samples.argtypes = [C.c_uint, C.c_int, C.c_int, C.c_int, C.c_uint, ip, up, up, up, up]
        L.ref_prosac_samples.restype = None
        L.ref_sprt_sequence.argtypes = [C.c_int, fp, C.c_int, C.c_float, C.c_uint, C.c_uint, fp, C.c_int, ip, ip, ip, up, up, dp, ip, ip]
        L.ref_prosac_termination_sequence.argtypes = [C.c_int, fp, C.c_int, C.c_float, C.c_float, C.c_uint, fp, C.c_int, up, up, up, up]
        L.ref_grid_neighbors.argtypes = [fp, C.c_int, C.c_int, ip, C.c_longlong, C.POINTER(C.c_longlong)]
        L.ref_knn.argtypes = [fp, C.c_int, C.c_int, C.c_int, ip]
        L.ref_rpoly.argtypes = [dp, C.c_int, dp, dp]
        L.ref_ransac_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, fp, C.c_int, C.c_float, C.c_float, C.c_uint, C.c_uint, C.c_int,
                                     C.c_uint, C.c_uint, C.POINTER(RunResult), ip]
        _lib = L
    return _lib


_shim = None


def shim_lib():
    """oracle/libref_shim.so: the stand-in OpenCV numerics alone (ref_shim_entry.cpp), built with the oracle - needs no reference."""
    global _shim
    if _shim is None:
        from oracle import oracle as O
        O.build()
        _shim = C.CDLL(O.SHIM_LIB)
    return _shim


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _u(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint))


def _pts(points):
    p = np.ascontiguousarray(points, dtype=np.float32)
    return p, p.shape[0]


def _model(m):
    out = np.zeros(9, np.float32)
    v = np.asarray(m, np.float32).ravel()
    out[:len(v)] = v
    return out


def errors(est, points, model):
    p, n = _pts(points)
    out = np.empty(n, np.float32)
    lib().ref_errors(est, _f(p), n, _f(_model(model)), _f(out))
    return out


def score(est, points, model, thr, want_inliers=False):
    p, n = _pts(points)
    cnt, s = C.c_int(), C.c_float()
    ids = np.empty(n, np.int32) if want_inliers else None
    lib().ref_score(est, _f(p), n, _f(_model(model)), thr, C.byref(cnt), C.byref(s), _i(ids) if want_inliers else None)
    return (cnt.value, s.value, ids[:cnt.value].copy()) if want_inliers else (cnt.value, s.value)


def solve_minimal(est, points, sample):
    p, n = _pts(points)
    s = np.ascontiguousarray(sample, dtype=np.int32)
    out = np.zeros(90, np.float32)
    k = lib().ref_solve_minimal(est, _f(p), n, _i(s), _f(out))
    w = 3 if est == 1 else 9
    return out.reshape(10, 9)[:k, :w].copy()


def nonminimal(est, points, ids):
    p, n = _pts(points)
    t = np.ascontiguousarray(ids, dtype=np.int32)
    out = np.zeros(9, np.float32)
    ok = lib().ref_nonminimal(est, _f(p), n, _i(t), len(t), _f(out))
    return out[:3 if est == 1 else 9].copy() if ok else None


def standard_termination(inliers, n, m, conf, max_it):
    return lib().ref_standard_termination(inliers, n, m, conf, max_it)


def uniform_samples(seed, n, m, K):
    out = np.empty((K, m), np.int32)
    lib().ref_uniform_samples(seed, n, m, K, _i(out))
    return out


def prosac_samples(rd_seed, n, m, K, termination_length=0):
    out = np.empty((K, m), np.int32)
    growth, subset, hyp, largest = (np.empty(n, np.uint32), np.empty(K, np.uint32), np.empty(K, np.uint32), np.empty(K, np.uint32))
    lib().ref_prosac_samples(rd_seed, n, m, K, termination_length, _i(out), _u(growth), _u(subset), _u(hyp), _u(largest))
    return {"samples": out, "growth": growth, "subset": subset, "hyp": hyp, "largest": largest}


def _sequence(fn, est, points, thr, seed, max_it, models, hyp):
    p, n = _pts(points)
    mods = np.zeros((len(models), 9), np.float32)
    for q, m in enumerate(models):
        mods[q] = _model(m)
    M = len(mods)
    h = np.ascontiguousarray(hyp, dtype=np.int32)
    good, inl, pool = np.empty(M, np.int32), np.empty(M, np.int32), np.empty(n, np.int32)
    idx, bound = np.empty(M, np.uint32), np.empty(M, np.uint32)
    hist = np.zeros((4096, 4), np.float64)
    nh = C.c_int()
    fn(est, _f(p), n, thr, seed, max_it, _f(mods), M, _i(h), _i(good), _i(inl), _u(idx), _u(bound),
       hist.ctypes.data_as(C.POINTER(C.c_double)), C.byref(nh), _i(pool))
    return {"good": good, "inliers": inl, "pool_idx": idx, "bound": bound, "history": hist[:nh.value].copy(), "pool": pool}


def sprt_sequence(est, points, thr, seed, max_it, models, hyp):
    return _sequence(lib().ref_sprt_sequence, est, points, thr, seed, max_it, models, hyp)


def prosac_termination_sequence(est, points, thr, conf, max_it, models, hyp_count, largest, fn=None):
    p, n = _pts(points)
    mods = np.stack([_model(m) for m in models])
    M = len(mods)
    hc, lg = np.ascontiguousarray(hyp_count, dtype=np.uint32), np.ascontiguousarray(largest, dtype=np.uint32)
    ms, tl = np.empty(M, np.uint32), np.empty(M, np.uint32)
    (fn or lib().ref_prosac_termination_sequence)(est, _f(p), n, thr, conf, max_it, _f(mods), M, _u(hc), _u(lg), _u(ms), _u(tl))
    return ms, tl


def grid_neighbors(points, cell):
    p, n = _pts(points)
    offs = np.empty(n + 1, np.int64)
    cap = 1 << 22
    while True:
        flat = np.empty(cap, np.int32)
        if lib().ref_grid_neighbors(_f(p), n, cell, _i(flat), cap, offs.ctypes.data_as(C.POINTER(C.c_longlong))) == 0:
            return [flat[offs[i]:offs[i + 1]].copy() for i in range(n)]
        cap = int(offs[n]) + 1


def knn(points, k):
    p, n = _pts(points)
    out = np.empty((n, k), np.int32)
    lib().ref_knn(_f(p), n, p.shape[1], k, _i(out))
    return out


def shim_svd(A, depth64=False, flags=0):
    """cv::SVD::compute of the stand-in OpenCV (oracle/ref_shim/cvshim.hpp) -> (w, u, vt) as float64 arrays"""
    A = np.ascontiguousarray(A, dtype=np.float64)
    r, c = A.shape
    w, u, vt, dims = np.zeros(max(r, c)), np.zeros(max(r, c) ** 2), np.zeros(max(r, c) ** 2), np.zeros(5, np.int32)
    dp = C.POINTER(C.c_double)
    fn = shim_lib().ref_shim_svd
    fn.argtypes = [dp, C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, dp, C.POINTER(C.c_int)]
    fn(A.ctypes.data_as(dp), r, c, int(depth64), int(flags), w.ctypes.data_as(dp), u.ctypes.data_as(dp), vt.ctypes.data_as(dp), _i(dims))
    return w[:dims[0]].copy(), u[:dims[1] * dims[2]].reshape(dims[1], dims[2]).copy(), vt[:dims[3] * dims[4]].reshape(dims[3], dims[4]).copy()


def shim_eigen(A, depth64=False):
    """cv::eigen of the stand-in OpenCV on a symmetric matrix -> (eigenvalues descending, eigenvectors as rows)"""
    A = np.ascontiguousarray(A, dtype=np.float64)
    n = A.shape[0]
    ev, vec = np.zeros(n), np.zeros((n, n))
    dp = C.POINTER(C.c_double)
    fn = shim_lib().ref_shim_eigen
    fn.argtypes = [dp, C.c_int, C.c_int, dp, dp]
    ok = fn(A.ctypes.data_as(dp), n, int(depth64), ev.ctypes.data_as(dp), vec.ctypes.data_as(dp))
    return (ev, vec) if ok else None


def shim_cubic(coeffs4):
    c = np.ascontiguousarray(coeffs4, dtype=np.float64)
    r = np.zeros(3)
    dp = C.POINTER(C.c_double)
    fn = shim_lib().ref_shim_cubic
    fn.argtypes = [dp, dp]
    n = fn(c.ctypes.data_as(dp), r.ctypes.data_as(dp))
    return n, r


def shim_inv3(m):
    a = np.ascontiguousarray(m, dtype=np.float32).reshape(9)
    out = np.zeros(9, np.float32)
    fn = shim_lib().ref_shim_inv3
    fn.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float)]
    fn(_f(a), _f(out))
    return out.reshape(3, 3)


def rpoly(coeffs_high_first):
    c = np.ascontiguousarray(coeffs_high_first, dtype=np.float64)
    deg = len(c) - 1
    zr, zi = np.zeros(deg + 1), np.zeros(deg + 1)
    d = lib().ref_rpoly(c.ctypes.data_as(C.POINTER(C.c_double)), deg, zr.ctypes.data_as(C.POINTER(C.c_double)), zi.ctypes.data_as(C.POINTER(C.c_double)))
    return zr[:d].copy(), zi[:d].copy()


def ransac_run(est, points, thr, conf=0.95, max_it=10000, sampler=1, neighbors=0, sprt=False, lo=0, knn=5, cell=50, seed=1, rd_seed=5489):
    """Ransac::Ransac + Ransac::run + RansacOutput (the reference's whole driver, refit loop included)."""
    p, n = _pts(points)
    r = RunResult()
    ids = np.empty(n, np.int32)
    lib().ref_ransac_run(est, sampler, neighbors, int(sprt), lo, _f(p), n, thr, conf, max_it, knn, cell, seed, rd_seed, C.byref(r), _i(ids))
    w = 3 if est == 1 else 9
    return {"model": np.array(r.model[:w], np.float32), "inliers": r.inliers, "iterations": r.iterations, "lo_inner": r.lo_inner,
            "lo_iterative": r.lo_iterative, "time_us": r.time_us, "ids": ids[:r.inliers].copy()}
