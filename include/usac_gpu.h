/*
 * usac_gpu.h - C ABI of libusac_gpu.so: the B200 (sm_100a) hypothesize-and-verify engine behind the USAC plugin
 * surface of MathsionYang/Ransac.
 *
 * Every entry point names the reference interface it replaces (paths relative to the reference tree, file:line).
 * Conventions: plain C, opaque handle, int status (0 = USAC_OK), never throws, never exit()s (the reference prints and
 * exit(111)s, init.cpp:17-19, ransac.cpp:143-147). All pointers are HOST pointers unless the name starts with `d_`.
 * A handle owns one CUDA stream and is thread-compatible (one handle per host thread). There is no CPU fallback:
 * every call fails with USAC_ERR_CUDA when no sm_100 device is present.
 *
 * Point sets: `points` is the reference's layout - row-major float32, N x 4 `x1 y1 x2 y2` (homography_estimator.hpp:
 * 22-27) or N x 2 `x y` for lines (line2d_estimator.hpp:17-22). The reference borrows the pointer for the lifetime of
 * the estimator (ransac.hpp:41); this library COPIES the points to HBM in usac_gpu_set_points (pair-interleaved SoA
 * for the scoring kernel + the original AoS for the solvers' gathers).
 */
#ifndef USAC_GPU_H
#define USAC_GPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* enums mirror usac/model.hpp:10-13 */
enum { USAC_EST_LINE2D = 1, USAC_EST_HOMOGRAPHY = 2, USAC_EST_FUNDAMENTAL = 3, USAC_EST_ESSENTIAL = 4 };
enum { USAC_SAMPLER_UNIFORM = 1, USAC_SAMPLER_PROGRESSIVE_NAPSAC = 2, USAC_SAMPLER_NAPSAC = 3, USAC_SAMPLER_PROSAC = 4 };
enum { USAC_NEIGH_NONE = 0, USAC_NEIGH_KNN = 1, USAC_NEIGH_GRID = 2 };
enum { USAC_RNG_PHILOX = 1 /* counter based, keyed by (seed, hypothesis id) */,
       USAC_RNG_TABLE = 2  /* replay a host-supplied K x m index table (e.g. the reference's glibc random() stream) */ };
enum { USAC_OK = 0, USAC_ERR_CUDA = 1, USAC_ERR_ARG = 2, USAC_ERR_STATE = 3, USAC_ERR_NCCL = 4 };

#define USAC_MAX_MODELS_PER_SAMPLE 3   /* seven-point cubic: up to 3 roots (ransac.cpp:24-28) */
#define USAC_E5_MAX_ROOTS 10           /* five-point solver: up to 10 real roots, every cheirality-valid one a model (usac_fit_cfg::essential_roots) */
/* usac_fit_cfg::essential_roots: which roots of a five-point sample become models */
enum { USAC_E5_ROOTS_FIRST_VALID = 0 /* the reference's rule (default): the first root, in visiting order, that passes the
                                        cheirality vote (five_points.cpp:217-262) */,
       USAC_E5_ROOTS_ALL_VALID = 1   /* every root that passes it, up to USAC_E5_MAX_ROOTS, in visiting order; the fit treats
                                        them as it treats the seven-point solver's roots (ransac.cpp:24-28) */ };

typedef struct usac_gpu_ctx usac_gpu_ctx;

/* ---- lifetime ------------------------------------------------------------------------------------------------ */
int usac_gpu_create(usac_gpu_ctx** out, int device);
void usac_gpu_destroy(usac_gpu_ctx* ctx);
const char* usac_gpu_last_error(const usac_gpu_ctx* ctx);   /* ctx may be NULL: error of the failed create */
/* {sm_count, sm_clock_khz, cc_major*10+cc_minor, l2_bytes} of the bound device */
int usac_gpu_device_info(const usac_gpu_ctx* ctx, int info[4]);
/* Run every later call on the caller's CUDA stream (a cudaStream_t passed as void*; the caller keeps ownership) instead
 * of the handle's own non-blocking stream - lets a host time several calls with its own events on that stream. */
int usac_gpu_set_stream(usac_gpu_ctx* ctx, void* cuda_stream);

/* ---- data: replaces `Ransac::Ransac(Model*, cv::InputArray points)` (ransac.hpp:41-55) + initEstimator (init.cpp:3) */
/* One call uploads `num_problems` independent point sets (image pairs) of one estimator type; problem p owns rows
 * [sum(n[0..p)), sum(n[0..p+1))) of `points`. num_problems == 1 is the reference's single-fit case. */
int usac_gpu_set_points(usac_gpu_ctx* ctx, int estimator, const float* points, const int* n_per_problem, int num_problems);
/* PROSAC assumes rows sorted by descending quality (prosac_sampler.hpp:75); nothing to upload. NAPSAC neighbourhoods: */
int usac_gpu_set_neighbors_grid(usac_gpu_ctx* ctx, int problem, int cell_size);              /* nearest_neighbors.cpp:160-201 */
int usac_gpu_set_neighbors_knn(usac_gpu_ctx* ctx, int problem, const int* neighbors, int k); /* nearest_neighbors.cpp:69-128 output */
/* NearestNeighbors::getNearestNeighbors_nanoflann (nearest_neighbors.cpp:69-128) on the device: exact k nearest neighbours
 * of every point (squared L2 over all columns, ascending, the query itself dropped; equidistant points in ascending index
 * order), installed as the problem's kNN table. 1 <= k <= 31, n >= k + 1. */
int usac_gpu_build_neighbors_knn(usac_gpu_ctx* ctx, int problem, int k);
/* copy the installed kNN table (n x k) back to the host; k_out receives k */
int usac_gpu_get_neighbors_knn(usac_gpu_ctx* ctx, int problem, int* neighbors_out, int* k_out);
/* Progressive NAPSAC: hypotheses 0 .. local_samples-1 of a fit or sample stream are local (DESIGN.md section 4.8), later ones are
 * the uniform sampler's. 0 = the default, 20 n. Reset by usac_gpu_set_points, like the neighbourhoods. */
int usac_gpu_set_pnapsac_length(usac_gpu_ctx* ctx, int problem, unsigned long long local_samples);
/* SPRT's shuffled point pool (sprt.hpp:93-107); host-generated so that it can replay the reference's random() stream */
int usac_gpu_set_sprt_pool(usac_gpu_ctx* ctx, int problem, const int* pool);

/* ---- Quality: replaces Quality::getNumberInliers / getInliers (quality.hpp:60-101, 108-121) --------------------- */
/* M models (row-major 9 floats each; line: 3 floats each, stride 3) against problem `problem`. threshold <= 0 is
 * invalid. inliers_out[M], sumerr_out[M] (sum of errors of the inliers, quality.hpp:85-100). Inlier counts are
 * bit-exact w.r.t. the reference's float32 arithmetic (fast path + strict re-evaluation inside a guard band). */
int usac_gpu_score(usac_gpu_ctx* ctx, int problem, const float* models, int M, float threshold, int* inliers_out, float* sumerr_out);
/* same arithmetic as the reference for every point (slow, for parity tests): err_out[n] */
int usac_gpu_errors(usac_gpu_ctx* ctx, int problem, const float* model, float* err_out);
/* ids in ascending point order, *n_out of them; ids_out must hold n entries */
int usac_gpu_get_inliers(usac_gpu_ctx* ctx, int problem, const float* model, float threshold, int* ids_out, int* n_out);

/* ---- Sampler: replaces Sampler::generateSample x K (sampler.hpp:21; uniform/prosac/napsac_sampler.hpp) ---------- */
typedef struct {
    int sampler;                 /* USAC_SAMPLER_* */
    int rng;                     /* USAC_RNG_* */
    uint64_t seed;
    int neighbors;               /* NAPSAC: USAC_NEIGH_* (set with usac_gpu_set_neighbors_*); Progressive NAPSAC: USAC_NEIGH_KNN */
    unsigned prosac_termination_length;   /* PROSAC: frozen for the call; 0 = n */
    unsigned prosac_hyp_count;            /* PROSAC: t of the first sample of this call (starts at 1) */
} usac_sampler_cfg;
/* samples_out: K x m int32 (m = 2/4/7/5), hypothesis ids first_hyp .. first_hyp+K-1. Samplers other than UNIFORM / NAPSAC /
 * PROSAC / PROGRESSIVE_NAPSAC (Evsac / ProsacNapsac are not wired in init.cpp:23-50) and rng values other than USAC_RNG_* are
 * rejected with USAC_ERR_ARG. PROGRESSIVE_NAPSAC is this library's definition (DESIGN.md section 4.8; the reference's
 * progressive_sampler.hpp:149-172 is an unfinished stub): a centre point per hypothesis, drawn from a neighbourhood of its kNN
 * list that grows with the centre's uses, then uniform sampling from hypothesis usac_gpu_set_pnapsac_length on. It needs
 * neighbors = USAC_NEIGH_KNN (else USAC_ERR_ARG) and an installed kNN table (else USAC_ERR_STATE). NAPSAC and Progressive NAPSAC
 * are stateful: a call with first_hyp == 0 starts the stream afresh, a later call continues it. */
int usac_gpu_sample(usac_gpu_ctx* ctx, int problem, const usac_sampler_cfg* cfg, uint64_t first_hyp, int K, int* samples_out);

/* ---- Estimator: replaces Estimator::EstimateModel x K (estimator.hpp:19; line2d/homography/fundamental/essential) */
/* samples: K x m. models_out: K x S x 9 floats (S = 3 for fundamental, else 1; line models use the first 3 floats of
 * their 9-float slot), nmodels_out[K] = number of valid models of each sample (0 = degenerate). */
int usac_gpu_estimate(usac_gpu_ctx* ctx, int problem, const int* samples, int K, float* models_out, int* nmodels_out);
/* the five-point solver with USAC_E5_ROOTS_ALL_VALID (essential problems only): models_out K x USAC_E5_MAX_ROOTS x 9 floats, every
 * cheirality-valid root of sample k in visiting order (ascending |z|), unused slots zero; nmodels_out[K] = how many (0..10) */
int usac_gpu_estimate_essential_roots(usac_gpu_ctx* ctx, int problem, const int* samples, int K, float* models_out, int* nmodels_out);

/* ---- fused robust fit: replaces the loop of Ransac::run (ransac.cpp:58-139) for every uploaded problem ---------- */
typedef struct {
    usac_sampler_cfg sampler;
    float threshold;             /* model.hpp:17 */
    float confidence;            /* model.hpp:18 desired_prob */
    unsigned max_iterations;     /* model.hpp:22. The initial bound of `while (iters < max_iters)` (ransac.cpp:58) and the value the standard
                                  * criterion answers while w^m < 0.0005 - NOT a hard cap: as in the reference, a better model may answer a larger,
                                  * uncapped bound (up to 5990 at confidence 0.95) and the fit then runs past max_iterations
                                  * (standard_termination_criteria.hpp:52-62); usac_fit_result::iterations reports what was done */
    int sprt;                    /* model.hpp:38 */
    int round_size;              /* K: samples per round and problem; 0 = automatic */
    const int* sample_table;     /* rng == USAC_RNG_TABLE: rows of m indices, used by problem 0 */
    unsigned sample_table_rows;
    /* multi-GPU hypothesis sharding (one process per GPU): this rank scores samples j with j % nranks == rank of
     * every round and the per-sample scores are exchanged with one all-gather per round */
    int rank, nranks;
    /* model.hpp:13,25: LocOpt - 0 NullLO, 1 InItLORsc (inner + iterative LO), 2 InItFLORsc (limited samples); runs on every new
     * best model (ransac.cpp:108-110; local_optimization/inner_local_optimization.hpp:74-133, iterative_local_optimization.hpp), for
     * every estimator: lines refit with the PCA non-minimal fit (line2d_estimator.hpp:59-106) */
    int lo;
    /* model.hpp:26-29 (Model::setLOParametres): 0 = the reference defaults 14 / 20 / 4 / 10. lo_sample_size must be 0 or lie in
     * [m + 1, 16] (m = the minimal sample: 2 lines, 4 homography, 7 fundamental, 5 essential), else USAC_ERR_ARG */
    unsigned lo_sample_size, lo_inner_iterations, lo_iterative_iterations, lo_threshold_multiplier;
    /* model.hpp:39: SPRT-rejected models of the first this-many hypotheses still get a full inlier count (sprt.hpp:243-257)
     * and do not burn an iteration (ransac.cpp:77-85). 0 = the reference default 20. */
    unsigned max_hypothesis_test_before_sprt;
    /* USAC_E5_ROOTS_*: essential fits only (any other value, or a non-zero value for another estimator, is USAC_ERR_ARG).
     * ALL_VALID needs fewer than 2^28 points per problem. 0 (a zero-initialised config) = the reference's rule. */
    int essential_roots;
} usac_fit_cfg;

typedef struct {
    float model[9];
    int inliers;                 /* Score::inlier_number */
    float score;                 /* Score::score = sum of inlier errors (inlier count under SPRT, sprt.hpp:240-241) */
    unsigned iterations;         /* `iters` when the loop ended (RansacOutput::number_iterations) */
    unsigned samples_drawn;
    long long best_hyp;          /* sample id of the best model, -1 if none */
    int best_model_idx;          /* which model of that sample: 0..2 for fundamental, 0..9 for essential with USAC_E5_ROOTS_ALL_VALID, else 0 */
    unsigned rounds;
    unsigned long long evals;    /* hypothesis x point evaluations executed on this GPU (whole rounds) */
    unsigned long long useful_evals; /* the part of `evals` the sequential loop of ransac.cpp:58-139 would also have
                                        executed: models of the samples up to the one that ended the loop */
    unsigned lo_inner_iters, lo_iterative_iters;   /* RansacOutput::getLOInnerIters / getLOIterativeIters */
    float msac;                  /* MSAC truncated cost sum_i min(err_i, threshold) = score + (n - inliers) * threshold, from the two
                                    quantities of Score (quality.hpp:85-100); NaN under SPRT, where `score` is an inlier count */
} usac_fit_result;

/* the same derivation for the Quality API: MSAC truncated cost of a model from usac_gpu_score's outputs */
static inline float usac_msac_cost(int n_points, int inliers, float sum_err, float threshold) {
    return sum_err + (float)(n_points - inliers) * threshold;
}

int usac_gpu_fit(usac_gpu_ctx* ctx, const usac_fit_cfg* cfg, usac_fit_result* results /* [num_problems] */);

/* ---- non-minimal estimation and the final refit ------------------------------------------------------------------ */
/* replaces Estimator::EstimateModelNonMinimalSample(sample, sample_size, model) (estimator.hpp:22; homography_estimator.hpp:
 * 67-75 -> dlt/normalized_dlt.cpp:7-23, fundamental/essential -> fundamental/eight_points.cpp:4-100, line2d_estimator.hpp:59-106):
 * one model from `count` point ids; *ok_out = 0 when the estimation failed. model_out: 9 floats (line: 3). */
int usac_gpu_estimate_nonminimal(usac_gpu_ctx* ctx, int problem, const int* ids, int count, float* model_out, int* ok_out);
/* replaces the refit loop that follows the main loop of Ransac::run (ransac.cpp:157-207): up to four rounds of "estimate from
 * the first `inliers` inliers of the current model, re-score, keep unless it lost more than 20 % or did not improve". */
typedef struct {
    float model[9];
    int inliers;      /* best_score->inlier_number after the loop */
    int accepted;     /* refits that replaced the model (0..4) */
} usac_refit_result;
int usac_gpu_refit(usac_gpu_ctx* ctx, int problem, const float* model_in, int best_inliers, float threshold, usac_refit_result* out);

/* ---- plugin-granularity entry points for SPRT, PROSAC and local optimisation --------------------------------------------------- */
/* replaces the point walk of SPRT::verifyModelAndGetModelScore (sprt.hpp:191-257) for M models: model q walks the shuffled pool
 * (usac_gpu_set_sprt_pool) from position start[q] under the test (epsilon, delta, A), lambda in double exactly as sprt.hpp:205-234;
 * count_all[q] != 0 (the first max_hypothesis_test_before_sprt hypotheses): a rejected model still gets its full inlier count
 * (sprt.hpp:243-257). The test history / re-design (sprt.hpp:259-311) is host arithmetic and stays with the caller (usac/sprt.hpp). */
typedef struct { int good, tested_inliers, tested_points, inliers; } usac_sprt_result;
int usac_gpu_sprt_verify(usac_gpu_ctx* ctx, int problem, const float* models, int M, float threshold, double epsilon, double delta, double A,
                         const unsigned* start, const int* count_all, usac_sprt_result* out);
/* replaces LocalOptimization::GetModelScore (local_optimization.hpp:19) for InItLORsc (1) / InItFLORsc (2): inner + iterative local
 * optimisation of one so-far-the-best model (inner_local_optimization.hpp:74-133, iterative_local_optimization.hpp:61-135), for every
 * estimator (model: 9 floats, a line's 3 in the first three).
 * One kernel launch per call (the whole inner / iterative loop runs on the device). model / inliers / score are updated in place when
 * LO finds a bigger Score; *call_counter keys the random 14-point subsets (Philox, seed) and advances; *lo_threshold carries
 * IterativeLocalOptimization's running threshold between calls (a member in the reference; NULL or <= 0 = start from the model
 * threshold); *inner_iters / *iterative_iters accumulate. Parameters as in usac_fit_cfg (0 = defaults), checked as usac_gpu_fit checks
 * them (cfg->lo 1 or 2, lo_sample_size 0 or in [m + 1, 16]: USAC_ERR_ARG otherwise). */
int usac_gpu_lo_model_score(usac_gpu_ctx* ctx, int problem, const usac_fit_cfg* cfg, uint64_t* call_counter, float* lo_threshold, float* model, int* inliers,
                            float* score, unsigned* inner_iters, unsigned* iterative_iters);
/* ProsacSampler::initProsacSampler growth function T'_n (prosac_sampler.hpp:62-114); pure host arithmetic, out[n] */
void usac_prosac_growth_function(unsigned n, unsigned sample_size, unsigned* out);

/* Exchange hook for nranks > 1: called once per round with this rank's packed per-sample scores; must fill `all`
 * with the nranks contributions in rank order (an all-gather). `d_` pointers are device memory on ctx's stream.
 * libusac_gpu's own NCCL binding (usac_gpu_nccl_*) installs one; tests install a host emulation. */
typedef int (*usac_allgather_fn)(void* user, const void* d_send, void* d_recv_all, size_t bytes_per_rank, void* cuda_stream);
int usac_gpu_set_allgather(usac_gpu_ctx* ctx, usac_allgather_fn fn, void* user);
/* NCCL over NVLink: id is ncclUniqueId (128 bytes) created on rank 0 and distributed by the caller */
int usac_gpu_nccl_unique_id(char id_out[128]);
int usac_gpu_nccl_init(usac_gpu_ctx* ctx, const char id[128], int rank, int nranks);

/* Exchange over peer memory (NVLink), the default of the hypothesis-sharded fit when attached: every rank owns an exchange
 * window in its HBM; the kernel that reduces a round's scores stores this rank's part straight into every rank's window and
 * raises a flag there, and the kernel that applies the round (best update + termination, ransac.cpp:103-137) waits for all
 * flags - no collective call and no extra launch. One process per GPU: usac_gpu_peer_export on every rank, all-gather the
 * USAC_PEER_HANDLE_BYTES handles with the launcher (rank order), usac_gpu_peer_attach on every rank. Ranks inside one process
 * (one thread per GPU, or tests): usac_gpu_peer_window + usac_gpu_peer_attach_ptrs. Rounds larger than a window (131072
 * samples x problems) fall back to the all-gather hook above. A rank that does not arrive within 2 s makes the others
 * return USAC_ERR_NCCL instead of waiting for ever. */
#define USAC_PEER_HANDLE_BYTES 64
int usac_gpu_peer_export(usac_gpu_ctx* ctx, char handle_out[USAC_PEER_HANDLE_BYTES]);
int usac_gpu_peer_attach(usac_gpu_ctx* ctx, const char* handles /* nranks x USAC_PEER_HANDLE_BYTES */, int rank, int nranks);
int usac_gpu_peer_window(usac_gpu_ctx* ctx, void** window_out);
int usac_gpu_peer_attach_ptrs(usac_gpu_ctx* ctx, void* const* windows /* [nranks], windows[rank] = own */, int rank, int nranks);
/* back to the all-gather hook (every rank must do the same before the next fit, e.g. when the attach failed on one of them) */
int usac_gpu_peer_detach(usac_gpu_ctx* ctx);

/* ---- measurement helpers --------------------------------------------------------------------------------------- */
/* device time (ms, CUDA events on ctx's stream) and launch count of the kernels of the last usac_gpu_fit/score call */
int usac_gpu_last_timing(const usac_gpu_ctx* ctx, float* total_ms, float* score_kernel_ms, int* launches, int* score_launches);
/* achieved FP32 FMA rate of a register-resident FFMA loop on this device (TFLOP/s): the roofline denominator */
int usac_gpu_measure_fp32_peak(usac_gpu_ctx* ctx, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif
