"""The all-roots five-point oracle (e5_roots_oracle.cpp): the CPU oracle's fit loop with every cheirality-valid root of an essential
sample as a model. TEST INFRASTRUCTURE ONLY. Compiled on first use, with the oracle's flags and its unmodified sources, into the
temporary directory (the tree may be read-only), keyed by the hash of the sources."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRCS = [os.path.join(_HERE, "e5_roots_oracle.cpp")] + [os.path.join(_ORACLE, f) for f in
                                                         ("usac_oracle.cpp", "usac_oracle_essential.cpp", "usac_oracle_refit.cpp")]
_DEPS = _SRCS + [os.path.join(_ORACLE, f) for f in ("usac_oracle_ransac.cpp", "usac_oracle.h", "oracle_internal.h")]
# oracle/Makefile's flags: one rounding per operator, as in the oracle the GPU is compared with everywhere else
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-w", "-shared"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in _DEPS:
            h.update(open(f, "rb").read())
        h.update(" ".join(_FLAGS).encode())
        path = os.path.join(tempfile.gettempdir(), f"e5_roots_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CXX", "g++")] + _FLAGS + ["-o", tmp] + _SRCS + ["-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.orc_ransac_e5_all_roots.argtypes = [C.POINTER(O.Config), C.POINTER(C.c_float), C.c_int, C.POINTER(O.Result)]
        L.orc_ransac_e5_all_roots.restype = C.c_int
        L.essential5_all_roots.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_float)]
        L.essential5_all_roots.restype = C.c_int
        _lib = L
    return _lib


def all_roots(points, sample):
    """-> float32 (k, 9): every cheirality-valid five-point root of the sample in visiting order"""
    p = np.ascontiguousarray(points, dtype=np.float32)
    s = np.ascontiguousarray(sample, dtype=np.int32)
    out = np.zeros(90, np.float32)
    k = lib().essential5_all_roots(O._f(p), O._i(s), O._f(out))
    return out[:9 * k].reshape(k, 9).copy()


def ransac(points, est, sampler=O.SAMPLER_UNIFORM, rng=O.RNG_PHILOX, threshold=2.0, confidence=0.95, max_iterations=10000,
           sprt=False, batch=0, seed=1, sample_table=None, lo=0):
    """O.ransac with every valid root of an essential sample as a model (other estimators: O.ransac's result)."""
    p = np.ascontiguousarray(points, dtype=np.float32)
    cfg = O.Config()
    cfg.estimator, cfg.sampler, cfg.rng = est, sampler, rng
    cfg.threshold, cfg.confidence, cfg.max_iterations = threshold, confidence, max_iterations
    cfg.sprt, cfg.batch, cfg.seed, cfg.lo = int(sprt), batch, seed, lo
    keep = None
    if sample_table is not None:
        keep = np.ascontiguousarray(sample_table, dtype=np.int32)
        cfg.sample_table, cfg.sample_table_rows = O._i(keep), keep.shape[0]
    res = O.Result()
    rc = lib().orc_ransac_e5_all_roots(C.byref(cfg), O._f(p), p.shape[0], C.byref(res))
    w = 3 if est == O.EST_LINE2D else 9
    return {"rc": rc, "model": np.array(res.model[:w], np.float32), "inliers": res.inliers, "score": res.score,
            "iterations": res.iterations, "samples_drawn": res.samples_drawn, "best_hyp": res.best_hyp,
            "best_model_idx": res.best_model_idx, "evals": res.evals, "models_scored": res.models_scored,
            "lo_inner": res.lo_inner, "lo_iterative": res.lo_iterative}
