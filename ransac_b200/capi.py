"""ctypes binding of libusac_gpu.so (the C ABI declared in include/usac_gpu.h).

There is no CPU fallback: loading fails loudly when the shared library has not been built, and every call fails
with USAC_ERR_CUDA when no sm_100 device is present.
"""
import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("USAC_GPU_LIB", os.path.join(_HERE, "libusac_gpu.so"))   # env override: tuning variants only
HEADER_PATH = os.path.join(_HERE, "..", "include", "usac_gpu.h")

EST_LINE2D, EST_HOMOGRAPHY, EST_FUNDAMENTAL, EST_ESSENTIAL = 1, 2, 3, 4
SAMPLER_UNIFORM, SAMPLER_PROGRESSIVE_NAPSAC, SAMPLER_NAPSAC, SAMPLER_PROSAC = 1, 2, 3, 4
NEIGH_NONE, NEIGH_KNN, NEIGH_GRID = 0, 1, 2
RNG_PHILOX, RNG_TABLE = 1, 2
OK, ERR_CUDA, ERR_ARG, ERR_STATE, ERR_NCCL = 0, 1, 2, 3, 4
SAMPLE_SIZE = {EST_LINE2D: 2, EST_HOMOGRAPHY: 4, EST_FUNDAMENTAL: 7, EST_ESSENTIAL: 5}
MAX_MODELS = {EST_LINE2D: 1, EST_HOMOGRAPHY: 1, EST_FUNDAMENTAL: 3, EST_ESSENTIAL: 1}
E5_MAX_ROOTS = 10
E5_ROOTS_FIRST_VALID, E5_ROOTS_ALL_VALID = 0, 1


class SamplerCfg(C.Structure):
    _fields_ = [("sampler", C.c_int), ("rng", C.c_int), ("seed", C.c_uint64), ("neighbors", C.c_int),
                ("prosac_termination_length", C.c_uint), ("prosac_hyp_count", C.c_uint)]


class FitCfg(C.Structure):
    _fields_ = [("sampler", SamplerCfg), ("threshold", C.c_float), ("confidence", C.c_float), ("max_iterations", C.c_uint),
                ("sprt", C.c_int), ("round_size", C.c_int), ("sample_table", C.POINTER(C.c_int)),
                ("sample_table_rows", C.c_uint), ("rank", C.c_int), ("nranks", C.c_int), ("lo", C.c_int),
                ("lo_sample_size", C.c_uint), ("lo_inner_iterations", C.c_uint), ("lo_iterative_iterations", C.c_uint),
                ("lo_threshold_multiplier", C.c_uint), ("max_hypothesis_test_before_sprt", C.c_uint), ("essential_roots", C.c_int)]


class FitResult(C.Structure):
    _fields_ = [("model", C.c_float * 9), ("inliers", C.c_int), ("score", C.c_float), ("iterations", C.c_uint),
                ("samples_drawn", C.c_uint), ("best_hyp", C.c_longlong), ("best_model_idx", C.c_int), ("rounds", C.c_uint),
                ("evals", C.c_ulonglong), ("useful_evals", C.c_ulonglong), ("lo_inner_iters", C.c_uint), ("lo_iterative_iters", C.c_uint),
                ("msac", C.c_float)]


class SprtResult(C.Structure):
    _fields_ = [("good", C.c_int), ("tested_inliers", C.c_int), ("tested_points", C.c_int), ("inliers", C.c_int)]


class RefitResult(C.Structure):
    _fields_ = [("model", C.c_float * 9), ("inliers", C.c_int), ("accepted", C.c_int)]


ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p)


def declared_symbols():
    """Every function the header declares (used by the symbol-export test)."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(usac_(?:gpu|prosac)_[a-z0-9_]+)\s*\(", text)) - {"usac_gpu_ctx"})


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m ransac_b200.build` (nvcc, sm_100a). "
                           "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, fp, ip = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)
    L.usac_gpu_create.argtypes = [C.POINTER(vp), C.c_int]
    L.usac_gpu_destroy.argtypes = [vp]
    L.usac_gpu_destroy.restype = None
    L.usac_gpu_last_error.argtypes = [vp]
    L.usac_gpu_last_error.restype = C.c_char_p
    L.usac_gpu_device_info.argtypes = [vp, C.POINTER(C.c_int * 4)]
    L.usac_gpu_set_stream.argtypes = [vp, vp]
    L.usac_gpu_set_points.argtypes = [vp, C.c_int, vp, ip, C.c_int]
    L.usac_gpu_set_neighbors_grid.argtypes = [vp, C.c_int, C.c_int]
    L.usac_gpu_set_neighbors_knn.argtypes = [vp, C.c_int, ip, C.c_int]
    L.usac_gpu_build_neighbors_knn.argtypes = [vp, C.c_int, C.c_int]
    L.usac_gpu_get_neighbors_knn.argtypes = [vp, C.c_int, ip, ip]
    L.usac_gpu_set_pnapsac_length.argtypes = [vp, C.c_int, C.c_ulonglong]
    L.usac_gpu_set_sprt_pool.argtypes = [vp, C.c_int, ip]
    L.usac_gpu_score.argtypes = [vp, C.c_int, fp, C.c_int, C.c_float, ip, fp]
    L.usac_gpu_errors.argtypes = [vp, C.c_int, fp, fp]
    L.usac_gpu_get_inliers.argtypes = [vp, C.c_int, fp, C.c_float, ip, ip]
    L.usac_gpu_sample.argtypes = [vp, C.c_int, C.POINTER(SamplerCfg), C.c_uint64, C.c_int, ip]
    L.usac_gpu_estimate.argtypes = [vp, C.c_int, ip, C.c_int, fp, ip]
    L.usac_gpu_estimate_essential_roots.argtypes = [vp, C.c_int, ip, C.c_int, fp, ip]
    L.usac_gpu_fit.argtypes = [vp, C.POINTER(FitCfg), C.POINTER(FitResult)]
    L.usac_gpu_estimate_nonminimal.argtypes = [vp, C.c_int, ip, C.c_int, fp, ip]
    L.usac_gpu_refit.argtypes = [vp, C.c_int, fp, C.c_int, C.c_float, C.POINTER(RefitResult)]
    L.usac_gpu_sprt_verify.argtypes = [vp, C.c_int, fp, C.c_int, C.c_float, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_uint), ip, C.POINTER(SprtResult)]
    L.usac_gpu_lo_model_score.argtypes = [vp, C.c_int, C.POINTER(FitCfg), C.POINTER(C.c_uint64), fp, fp, ip, fp, C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
    L.usac_prosac_growth_function.argtypes = [C.c_uint, C.c_uint, C.POINTER(C.c_uint)]
    L.usac_prosac_growth_function.restype = None
    L.usac_gpu_set_allgather.argtypes = [vp, ALLGATHER_FN, vp]
    L.usac_gpu_nccl_unique_id.argtypes = [C.c_char_p]
    L.usac_gpu_nccl_init.argtypes = [vp, C.c_char_p, C.c_int, C.c_int]
    L.usac_gpu_peer_export.argtypes = [vp, C.c_char_p]
    L.usac_gpu_peer_attach.argtypes = [vp, C.c_char_p, C.c_int, C.c_int]
    L.usac_gpu_peer_detach.argtypes = [vp]
    L.usac_gpu_peer_window.argtypes = [vp, C.POINTER(C.c_void_p)]
    L.usac_gpu_peer_attach_ptrs.argtypes = [vp, C.POINTER(C.c_void_p), C.c_int, C.c_int]
    L.usac_gpu_last_timing.argtypes = [vp, fp, fp, ip, ip]
    L.usac_gpu_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_double)]
    for name in declared_symbols():
        fn = getattr(L, name)
        if name not in ("usac_gpu_destroy", "usac_gpu_last_error", "usac_prosac_growth_function"):
            fn.restype = C.c_int
    _lib = L
    return L
