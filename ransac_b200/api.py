"""Thin Python host layer over the C ABI: device context, Quality/Sampler/Estimator calls and the fused fit.

This mirrors what the C++ plugin classes in ransac_b200/usac/ do (GpuQuality, GpuEstimator, GpuSampler, GpuRansac);
tests and bench.py drive the library through it. numpy arrays are host buffers; torch tensors (CPU, ideally pinned)
are accepted through their data_ptr.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import (E5_MAX_ROOTS, E5_ROOTS_ALL_VALID, E5_ROOTS_FIRST_VALID, EST_ESSENTIAL, EST_FUNDAMENTAL,  # noqa: F401
                   EST_HOMOGRAPHY, EST_LINE2D, MAX_MODELS, NEIGH_GRID, NEIGH_KNN, NEIGH_NONE, RNG_PHILOX, RNG_TABLE, SAMPLE_SIZE,
                   SAMPLER_NAPSAC, SAMPLER_PROGRESSIVE_NAPSAC, SAMPLER_PROSAC, SAMPLER_UNIFORM)


class UsacGpuError(RuntimeError):
    pass


def _ptr(a, ctype):
    if hasattr(a, "data_ptr"):          # torch tensor
        return C.cast(a.data_ptr(), C.POINTER(ctype))
    return a.ctypes.data_as(C.POINTER(ctype))


class GpuContext:
    def __init__(self, device=0):
        self.L = capi.load()
        h = C.c_void_p()
        rc = self.L.usac_gpu_create(C.byref(h), device)
        if rc != capi.OK:
            raise UsacGpuError(f"usac_gpu_create failed ({rc}): {self.L.usac_gpu_last_error(None).decode()}")
        self.h = h
        self.est = None
        self.n = None

    def close(self):
        if getattr(self, "h", None):
            self.L.usac_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != capi.OK:
            raise UsacGpuError(f"{what} failed ({rc}): {self.L.usac_gpu_last_error(self.h).decode()}")

    def device_info(self):
        info = (C.c_int * 4)()
        self._check(self.L.usac_gpu_device_info(self.h, C.byref(info)), "device_info")
        return {"sm_count": info[0], "sm_clock_khz": info[1], "cc": info[2], "l2_bytes": info[3]}

    def set_stream(self, cuda_stream):
        """cuda_stream: integer cudaStream_t handle (e.g. torch.cuda.Stream().cuda_stream); the caller keeps it alive."""
        self._check(self.L.usac_gpu_set_stream(self.h, C.c_void_p(cuda_stream)), "set_stream")

    # ---- data ----
    def set_points(self, est, points, n_per_problem=None):
        """points: [sum(n), dim] float32 host array (numpy or CPU torch tensor); n_per_problem: list of row counts."""
        dim = 2 if est == EST_LINE2D else 4
        if not hasattr(points, "data_ptr"):
            points = np.ascontiguousarray(points, dtype=np.float32)
            assert points.ndim == 2 and points.shape[1] == dim
        total = points.shape[0]
        if n_per_problem is None:
            n_per_problem = [total]
        ns = np.ascontiguousarray(n_per_problem, dtype=np.int32)
        assert int(ns.sum()) == total
        self._keep = points
        self.est, self.n = est, ns.copy()
        self._check(self.L.usac_gpu_set_points(self.h, est, C.cast(_ptr(points, C.c_float), C.c_void_p), _ptr(ns, C.c_int), len(ns)), "set_points")

    def set_neighbors_grid(self, problem, cell_size):
        self._check(self.L.usac_gpu_set_neighbors_grid(self.h, problem, cell_size), "set_neighbors_grid")

    def set_neighbors_knn(self, problem, table):
        t = np.ascontiguousarray(table, dtype=np.int32)
        self._check(self.L.usac_gpu_set_neighbors_knn(self.h, problem, _ptr(t, C.c_int), t.shape[1]), "set_neighbors_knn")

    def build_neighbors_knn(self, problem, k):
        """nearest_neighbors.cpp:69-128 on the device; installs the table and returns nothing (see get_neighbors_knn)."""
        self._check(self.L.usac_gpu_build_neighbors_knn(self.h, problem, int(k)), "build_neighbors_knn")
        self._knn_k = getattr(self, "_knn_k", {})
        self._knn_k[problem] = int(k)

    def get_neighbors_knn(self, problem, k_max=31):
        out = np.empty((int(self.n[problem]), k_max), np.int32)
        k = C.c_int()
        self._check(self.L.usac_gpu_get_neighbors_knn(self.h, problem, _ptr(out, C.c_int), C.byref(k)), "get_neighbors_knn")
        return out.reshape(-1)[:int(self.n[problem]) * k.value].reshape(int(self.n[problem]), k.value).copy()

    def set_pnapsac_length(self, problem, local_samples):
        """Progressive NAPSAC: hypotheses from local_samples on are sampled uniformly (0 = the default, 20 n)."""
        self._check(self.L.usac_gpu_set_pnapsac_length(self.h, problem, int(local_samples)), "set_pnapsac_length")

    def set_sprt_pool(self, problem, pool):
        t = np.ascontiguousarray(pool, dtype=np.int32)
        assert t.shape[0] == self.n[problem]
        self._check(self.L.usac_gpu_set_sprt_pool(self.h, problem, _ptr(t, C.c_int)), "set_sprt_pool")

    # ---- Quality ----
    def score(self, models, threshold, problem=0):
        w = 3 if self.est == EST_LINE2D else 9
        m = np.ascontiguousarray(models, dtype=np.float32).reshape(-1, w)
        M = m.shape[0]
        cnt = np.zeros(M, np.int32)
        s = np.zeros(M, np.float32)
        self._check(self.L.usac_gpu_score(self.h, problem, _ptr(m, C.c_float), M, threshold, _ptr(cnt, C.c_int), _ptr(s, C.c_float)), "score")
        return cnt, s

    def errors(self, model, problem=0):
        m = np.ascontiguousarray(model, dtype=np.float32).ravel()
        out = np.empty(int(self.n[problem]), np.float32)
        self._check(self.L.usac_gpu_errors(self.h, problem, _ptr(m, C.c_float), _ptr(out, C.c_float)), "errors")
        return out

    def get_inliers(self, model, threshold, problem=0):
        m = np.ascontiguousarray(model, dtype=np.float32).ravel()
        ids = np.empty(int(self.n[problem]), np.int32)
        k = C.c_int()
        self._check(self.L.usac_gpu_get_inliers(self.h, problem, _ptr(m, C.c_float), threshold, _ptr(ids, C.c_int), C.byref(k)), "get_inliers")
        return ids[:k.value].copy()

    # ---- Sampler / Estimator ----
    def sample(self, K, sampler=SAMPLER_UNIFORM, seed=1, first_hyp=0, problem=0, neighbors=NEIGH_NONE,
               prosac_termination_length=0, prosac_hyp_count=0):
        cfg = capi.SamplerCfg(sampler, RNG_PHILOX, seed, neighbors, prosac_termination_length, prosac_hyp_count)
        out = np.empty((K, SAMPLE_SIZE[self.est]), np.int32)
        self._check(self.L.usac_gpu_sample(self.h, problem, C.byref(cfg), first_hyp, K, _ptr(out, C.c_int)), "sample")
        return out

    def estimate(self, samples, problem=0):
        s = np.ascontiguousarray(samples, dtype=np.int32).reshape(-1, SAMPLE_SIZE[self.est])
        K, S = s.shape[0], MAX_MODELS[self.est]
        models = np.zeros((K, S, 9), np.float32)
        nm = np.zeros(K, np.int32)
        self._check(self.L.usac_gpu_estimate(self.h, problem, _ptr(s, C.c_int), K, _ptr(models, C.c_float), _ptr(nm, C.c_int)), "estimate")
        return models, nm

    def estimate_essential_roots(self, samples, problem=0):
        """Five-point solve keeping every cheirality-valid root -> (models [K, 10, 9], nmodels [K]); models in visiting order."""
        s = np.ascontiguousarray(samples, dtype=np.int32).reshape(-1, SAMPLE_SIZE[EST_ESSENTIAL])
        K = s.shape[0]
        models = np.zeros((K, E5_MAX_ROOTS, 9), np.float32)
        nm = np.zeros(K, np.int32)
        self._check(self.L.usac_gpu_estimate_essential_roots(self.h, problem, _ptr(s, C.c_int), K, _ptr(models, C.c_float), _ptr(nm, C.c_int)),
                    "estimate_essential_roots")
        return models, nm

    # ---- fused fit ----
    def fit_records(self, threshold, confidence=0.95, max_iterations=10000, sampler=SAMPLER_UNIFORM, rng=RNG_PHILOX, seed=1,
                    sprt=False, round_size=0, neighbors=NEIGH_NONE, sample_table=None, rank=0, nranks=1, lo=0, lo_params=None,
                    max_hypothesis_test_before_sprt=0, essential_roots=E5_ROOTS_FIRST_VALID):
        """One robust fit per uploaded problem; returns a numpy record array laid out as usac_fit_result (no per-problem
        Python work: this is what a batched caller uses). lo=1 (InItLORsc) / 2 (InItFLORsc): local optimisation of every new
        best model, for every estimator (lines refit with the PCA fit); with several problems (and no PROSAC / sample table) the LO
        calls of all problems run side by side on the device, each record that of the problem fitted alone; lo_params = (lo_sample_size, lo_inner_iterations,
        lo_iterative_iterations, lo_threshold_multiplier), 0 = default. essential_roots=E5_ROOTS_ALL_VALID (essential only): every
        cheirality-valid five-point root is a model, so best_model_idx ranges over 0..9."""
        cfg = capi.FitCfg()
        cfg.sampler = capi.SamplerCfg(sampler, rng, seed, neighbors, 0, 0)
        cfg.threshold, cfg.confidence, cfg.max_iterations = threshold, confidence, max_iterations
        cfg.sprt, cfg.round_size, cfg.rank, cfg.nranks, cfg.lo = int(sprt), round_size, rank, nranks, int(lo)
        if lo_params is not None:     # (lo_sample_size, lo_inner_iterations, lo_iterative_iterations, lo_threshold_multiplier), model.hpp:26-29
            cfg.lo_sample_size, cfg.lo_inner_iterations, cfg.lo_iterative_iterations, cfg.lo_threshold_multiplier = [int(v) for v in lo_params]
        cfg.max_hypothesis_test_before_sprt = int(max_hypothesis_test_before_sprt)
        cfg.essential_roots = int(essential_roots)
        if sample_table is not None:
            t = np.ascontiguousarray(sample_table, dtype=np.int32)
            self._table = t
            cfg.sample_table, cfg.sample_table_rows = _ptr(t, C.c_int), t.shape[0]
        P = len(self.n)
        res = (capi.FitResult * P)()
        self._check(self.L.usac_gpu_fit(self.h, C.byref(cfg), res), "fit")
        return np.frombuffer(res, dtype=np.dtype(capi.FitResult), count=P)

    def fit(self, *args, **kw):
        """fit_records as a list of dicts (model as float32 array of 9, or 3 for lines)."""
        rec = self.fit_records(*args, **kw)
        w = 3 if self.est == EST_LINE2D else 9
        return [{"model": np.array(r["model"][:w], np.float32), "inliers": int(r["inliers"]), "score": float(r["score"]),
                 "iterations": int(r["iterations"]), "samples_drawn": int(r["samples_drawn"]), "best_hyp": int(r["best_hyp"]),
                 "best_model_idx": int(r["best_model_idx"]), "rounds": int(r["rounds"]), "evals": int(r["evals"]),
                 "useful_evals": int(r["useful_evals"]), "lo_inner": int(r["lo_inner_iters"]), "lo_iterative": int(r["lo_iterative_iters"]), "msac": float(r["msac"])} for r in rec]

    def estimate_nonminimal(self, ids, problem=0):
        """Estimator::EstimateModelNonMinimalSample on a list of point ids -> model (9 or 3 floats) or None."""
        t = np.ascontiguousarray(ids, dtype=np.int32)
        w = 3 if self.est == EST_LINE2D else 9
        m = np.zeros(9, np.float32)
        ok = C.c_int()
        self._check(self.L.usac_gpu_estimate_nonminimal(self.h, problem, _ptr(t, C.c_int), len(t), _ptr(m, C.c_float), C.byref(ok)), "estimate_nonminimal")
        return m[:w].copy() if ok.value else None

    def refit(self, model, best_inliers, threshold, problem=0):
        """The final refit loop of Ransac::run (ransac.cpp:157-207)."""
        m = np.ascontiguousarray(model, dtype=np.float32).ravel()
        r = capi.RefitResult()
        self._check(self.L.usac_gpu_refit(self.h, problem, _ptr(m, C.c_float), int(best_inliers), threshold, C.byref(r)), "refit")
        w = 3 if self.est == EST_LINE2D else 9
        return {"model": np.array(r.model[:w], np.float32), "inliers": r.inliers, "accepted": r.accepted}

    def last_timing(self):
        t, s = C.c_float(), C.c_float()
        n, ns = C.c_int(), C.c_int()
        self._check(self.L.usac_gpu_last_timing(self.h, C.byref(t), C.byref(s), C.byref(n), C.byref(ns)), "last_timing")
        return {"total_ms": t.value, "score_ms": s.value, "launches": n.value, "score_launches": ns.value}

    def measure_fp32_peak(self):
        v = C.c_double()
        self._check(self.L.usac_gpu_measure_fp32_peak(self.h, C.byref(v)), "measure_fp32_peak")
        return v.value

    # ---- multi-GPU ----
    def nccl_init(self, unique_id, rank, nranks):
        self._check(self.L.usac_gpu_nccl_init(self.h, unique_id, rank, nranks), "nccl_init")

    PEER_HANDLE_BYTES = 64

    def peer_export(self):
        """-> the CUDA IPC handle (bytes) of this rank's exchange window; all-gather the handles and call peer_attach."""
        buf = C.create_string_buffer(self.PEER_HANDLE_BYTES)
        self._check(self.L.usac_gpu_peer_export(self.h, buf), "peer_export")
        return buf.raw

    def peer_attach(self, handles, rank, nranks):
        """handles: the nranks IPC handles in rank order (bytes objects or one concatenated bytes)."""
        blob = handles if isinstance(handles, (bytes, bytearray)) else b"".join(handles)
        assert len(blob) == nranks * self.PEER_HANDLE_BYTES
        self._check(self.L.usac_gpu_peer_attach(self.h, bytes(blob), rank, nranks), "peer_attach")

    def peer_detach(self):
        self._check(self.L.usac_gpu_peer_detach(self.h), "peer_detach")

    def peer_window(self):
        p = C.c_void_p()
        self._check(self.L.usac_gpu_peer_window(self.h, C.byref(p)), "peer_window")
        return p.value

    def peer_attach_ptrs(self, windows, rank, nranks):
        arr = (C.c_void_p * nranks)(*windows)
        self._check(self.L.usac_gpu_peer_attach_ptrs(self.h, arr, rank, nranks), "peer_attach_ptrs")


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    rc = capi.load().usac_gpu_nccl_unique_id(buf)
    if rc != capi.OK:
        raise UsacGpuError("usac_gpu_nccl_unique_id failed")
    return buf.raw
