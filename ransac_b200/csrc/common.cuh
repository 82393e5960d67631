// common.cuh - shared definitions of libusac_gpu (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/usac_gpu.h"

#define USAC_REC_STRIDE 32          // floats per prepared-model record (128 B)
#define USAC_TILE_PAIRS 128         // point pairs per shared-memory tile (256 points)
#ifndef USAC_WARP_STAGES
#define USAC_WARP_STAGES 2          // bulk-copy pipeline depth of each warp of the scoring kernel
#endif
#define USAC_SCORE_THREADS 128      // models per scoring CTA
#ifndef USAC_SCORE_MIN_CTAS
#define USAC_SCORE_MIN_CTAS 4        // resident scoring CTAs per SM (4 -> 118 registers, no spills; 16 warps/SM sustain the same rate as 20
                                     // and leave room for the small kernels of other streams: measured best, profiles/README.md)
#endif
#ifndef USAC_SCORE_GRID_CTAS
#define USAC_SCORE_GRID_CTAS USAC_SCORE_MIN_CTAS   // scoring CTAs launched per SM (<= USAC_SCORE_MIN_CTAS; fewer leaves room for other streams' kernels)
#endif
#ifndef USAC_SQ_MIN_CTAS
#define USAC_SQ_MIN_CTAS 5           // resident CTAs per SM of the survivor-queue scoring kernel (score_sq.cuh): 96 registers, a few bytes of
                                     // spill in the drain; one-box A/B (profiles/README.md): 5 beats 4 by 4 % on the bench and 6 - 9 % on the
                                     // epipolar kernels, 6 is slower (spills)
#endif
#ifndef USAC_PPI
#define USAC_PPI 4                  // point pairs per trip of the scoring loop (independent instruction streams)
#endif

// Prepared-model record (one per valid model, written by prepare_kernel, read by the scoring kernels):
//   [0..8]   model, row-major (line: a b c in [0..2])
//   [9..17]  inverse homography (cv::Mat::inv() semantics, homography_estimator.hpp:35)
//   [18..21] guard-band constants of the fast path (estimator specific, see score.cuh)
//   [22]     threshold the record was prepared for
enum { REC_MODEL = 0, REC_HINV = 9, REC_BAND = 18, REC_THR = 22 };

// Per-problem descriptor, resident in HBM.
struct ProblemDesc {
    int n;                 // points
    int n_pairs;           // ceil(n/2)
    long long aos_off;     // first row of this problem in the AoS point array
    long long pair_off;    // first pair of this problem in the pair-interleaved array
    float mx1, my1, mx2, my2;   // max |coordinate| per column (guard-band analysis); line: mx1, my1 only
    // NAPSAC neighbourhoods
    int neigh_type, knn;
    long long knn_off;     // into d_knn
    long long grid_off;    // into d_cell_of_point / d_members / d_rank (n entries each)
    long long cell_start_off;   // into d_cell_start (n+1 entries)
    // PROSAC growth function / termination table / SPRT pool offsets (n or n+1 entries each, -1 = absent)
    long long growth_off, term_off, pool_off;
    long long cursor_off;  // NAPSAC per-point use counters (n entries)
    unsigned long long pn_len;   // Progressive NAPSAC: local samples before the sampler turns global (usac_gpu_set_pnapsac_length); 0 = 20 n
};

// Progressive NAPSAC (DESIGN.md section 4.8): the hypothesis id at which sampling turns uniform
__host__ __device__ __forceinline__ unsigned long long pnapsac_length(const ProblemDesc& pd) {
    return pd.pn_len ? pd.pn_len : 20ull * (unsigned long long)pd.n;
}

// Evolving state of one robust fit (Ransac::run locals, ransac.cpp:17-56), resident in HBM between rounds.
struct FitState {
    float best_model[9];
    int best_cnt;
    float best_sum;
    long long best_hyp;
    int best_midx;
    unsigned iters, max_iters, samples_drawn, rounds;
    int done;
    int round_pending;     // select_kernel processed a round that winner_kernel has not finished yet (rounds may be enqueued ahead of the host's knowledge)
    unsigned long long evals, useful_evals;
    // PROSAC sampler state (prosac_sampler.hpp:19-31)
    unsigned prosac_t, prosac_n, prosac_largest, prosac_term_len;
    unsigned prosac_t_next, prosac_n_next, prosac_largest_next;   // written by the sampler, committed at round end
    // SPRT state (sprt.hpp:66-82): current test, pool cursor, history bookkeeping
    double sprt_eps, sprt_delta, sprt_A;
    unsigned sprt_cursor;
    int sprt_last_update, sprt_ntests;
};

#define CUDA_TRY(ctx, expr)                                                                         \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) { (ctx)->set_error(#expr, cudaGetErrorString(_e)); return USAC_ERR_CUDA; } \
    } while (0)

__host__ __device__ __forceinline__ int usac_sample_size(int est) {
    return est == USAC_EST_LINE2D ? 2 : est == USAC_EST_HOMOGRAPHY ? 4 : est == USAC_EST_FUNDAMENTAL ? 7 : 5;
}
__host__ __device__ __forceinline__ int usac_models_per_sample(int est) { return est == USAC_EST_FUNDAMENTAL ? 3 : 1; }
__host__ __device__ __forceinline__ int usac_point_dim(int est) { return est == USAC_EST_LINE2D ? 2 : 4; }

// Philox4x32-10 (Salmon et al. SC'11), the counter-based stream of the Philox sampler mode.
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// m distinct indices in [0,n): draw i picks the j-th smallest unused index, j = mulhi(word_i, n-i).
__host__ __device__ __forceinline__ void philox_unique(uint64_t seed, uint64_t hyp, uint32_t stream, int n, int m, int* out) {
    uint32_t w[8];
    for (int blk = 0; blk * 4 < m; blk++)
        philox4x32_10((uint32_t)hyp, (uint32_t)(hyp >> 32), (uint32_t)blk, stream, (uint32_t)seed, (uint32_t)(seed >> 32), w + 4 * blk);
    int sorted[8];
    for (int i = 0; i < m; i++) {
        int j = (int)(((uint64_t)w[i] * (uint64_t)(uint32_t)(n - i)) >> 32);
        int pos = 0;
        while (pos < i && j >= sorted[pos]) { j++; pos++; }
        for (int q = i; q > pos; q--) sorted[q] = sorted[q - 1];
        sorted[pos] = j;
        out[i] = j;
    }
}

// Orderable key of Score (quality.hpp:16-31): inliers first, then the larger error sum.
__device__ __forceinline__ unsigned long long score_key(int cnt, float sum) {
    // sums are >= 0 (NaN and -0 map to 0): the IEEE bit pattern of a positive float is monotone
    const unsigned s = (sum > 0.f) ? __float_as_uint(sum) : 0u;
    return ((unsigned long long)(unsigned)cnt << 32) | s;
}
