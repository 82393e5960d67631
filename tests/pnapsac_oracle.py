"""The Progressive NAPSAC reference (pnapsac_oracle.cpp): the sequential sampler of DESIGN.md section 4.8, and whole oracle fits
that draw from it. TEST INFRASTRUCTURE ONLY. Compiled on first use, with the oracle's flags and its unmodified sources, into the
temporary directory (the tree may be read-only), keyed by the hash of the sources.

A fit with this sampler is the oracle's own loop (O.ransac) replaying the sampler's stream as a sample table: the sampler's output
depends on the hypothesis id and the earlier samples only, never on the fit, so the table is the sampler."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRCS = [os.path.join(_HERE, "pnapsac_oracle.cpp")] + [os.path.join(_ORACLE, f) for f in
                                                        ("usac_oracle.cpp", "usac_oracle_ransac.cpp", "usac_oracle_essential.cpp",
                                                         "usac_oracle_refit.cpp")]
_DEPS = _SRCS + [os.path.join(_ORACLE, f) for f in ("usac_oracle.h", "oracle_internal.h")]
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-w", "-shared"]   # oracle/Makefile's
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in _DEPS:
            h.update(open(f, "rb").read())
        h.update(" ".join(_FLAGS).encode())
        path = os.path.join(tempfile.gettempdir(), f"pnapsac_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CXX", "g++")] + _FLAGS + ["-o", tmp] + _SRCS + ["-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.pnapsac_table.argtypes = [C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int, C.c_ulonglong, C.c_int, C.POINTER(C.c_int)]
        L.pnapsac_table.restype = None
        _lib = L
    return _lib


def default_length(n):
    return 20 * n


def table(seed, knn_table, m, count, length=0):
    """Samples of hypotheses 0 .. count-1 of one stream -> int32 (count, m). length 0 = the default, 20 n."""
    t = np.ascontiguousarray(knn_table, dtype=np.int32)
    n, k = t.shape
    out = np.empty((count, m), np.int32)
    lib().pnapsac_table(seed, n, m, O._i(t), k, length or default_length(n), count, O._i(out))
    return out


def ransac(points, est, knn_table, length=0, seed=1, max_iterations=10000, batch=0, **kw):
    """O.ransac with the Progressive NAPSAC sampler over knn_table. The table holds more samples than the loop can draw (the
    uncapped termination bound stays below 8192 at the confidences used here); running past it would be a silent change of
    sampler, so that is an error."""
    m = O.SAMPLE_SIZE[est]
    rows = max_iterations + 8192 + max(batch, 0)
    smp = table(seed, knn_table, m, rows, length)
    r = O.ransac(points, est, rng=O.RNG_TABLE, sample_table=smp, seed=seed, max_iterations=max_iterations, batch=batch, **kw)
    assert r["samples_drawn"] <= rows, (r["samples_drawn"], rows)
    return r
