// lo.cuh - LO-RANSAC as ONE device-side loop: InnerLocalOptimization::GetModelScore with its IterativeLocalOptimization
// (usac/local_optimization/inner_local_optimization.hpp:74-133, iterative_local_optimization.hpp:61-135) for a so-far-the-best
// model, one launch of one CTA of 1024 threads per call. In round 1 the control flow was host code between device calls
// (~100 stream synchronisations per LO call, 27 ms for a homography fit with LO); here the host uploads the model and reads
// the result back - one synchronisation.
//
// The arithmetic is that of refit.cuh / score.cuh, order included, so the results stay bit-identical to the CPU restatement the parity tests use:
//  * non-minimal estimation (cta_nonminimal): lanes = the first 256 threads; every sum over the points is thread t adding
//    elements t, t + 256, ... in order, then the fixed binary tree stride 128 ... 1 over the 256 partials. The 45 entries of A'A
//    are accumulated in ONE pass over the points (each entry still sees its addends in the same order) and go through the tree
//    together: 5 CTA barriers per fit instead of 45 x 9.
//  * scoring with the ordered inlier list (cta_score): lanes = all 1024 threads, errors in the reference's arithmetic
//    (strict_error), error sum = lane sums + fixed tree stride 512 ... 1.
#pragma once
#include <type_traits>
#include "pipeline.cuh"
#include "refit.cuh"
#include "score.cuh"

#define LO_THREADS 1024

struct LoIO {                    // in/out record of one LO call (global memory)
    float model[9];
    int inliers;
    float score;
    float lo_thr;                // IterativeLocalOptimization's running threshold (a member in the reference: it survives calls)
    unsigned long long calls;    // keys the random inlier subsets
    unsigned inner_done, iterative_done;
};

struct LoArgs {
    const float* aos;            // points of the problem
    const ProblemDesc* prob;
    int problem, n, m, kind, sample_limit, inner_iters, iter_iters, mult;
    float theta, step;
    unsigned long long seed;
    LoIO* io;
    int* A;                      // inliers of the best model (n entries)
    int* B;                      // inliers of the candidate (n entries)
};

struct LoShared {
    double tree[45 * REFIT_THREADS];     // A'A partials of the 256 lanes (also used for the float trees)
    double S[81], V[81], h[9];
    float part[LO_THREADS];              // error-sum partials of the 1024 scoring lanes
    float rec[USAC_REC_STRIDE];
    float model[9], best_model[9], stats[8];
    int warp_tot[2][32];                 // inliers per warp of the current / previous block of 1024 points
    int sample[16];
    int ok, cnt;
    float sum;
};

// fixed binary tree over 256 float / double partials of `count` quantities laid out tree[q * 256 + t]; result q in tree[q * 256].
// Pairing and order are those of refit_tree_f / refit_tree_d (sm[t] += sm[t + s], s = 128 ... 1).
template <class T>
__device__ __forceinline__ void lo_tree256(T* tree, int count) {
    const int t = threadIdx.x;
    __syncthreads();
    for (int s = REFIT_THREADS / 2; s >= 32; s >>= 1) {               // partners live in different warps
        for (int i = t; i < count * s; i += LO_THREADS) {
            const int q = i / s, l = i % s;
            if (sizeof(T) == 8) tree[q * REFIT_THREADS + l] = (T)__dadd_rn((double)tree[q * REFIT_THREADS + l], (double)tree[q * REFIT_THREADS + l + s]);
            else tree[q * REFIT_THREADS + l] = (T)__fadd_rn((float)tree[q * REFIT_THREADS + l], (float)tree[q * REFIT_THREADS + l + s]);
        }
        __syncthreads();
    }
    // s = 16 ... 1: one warp per quantity, partners in the same warp
    const int warp = t >> 5, lane = t & 31;
    for (int q = warp; q < count; q += LO_THREADS / 32) {
        for (int s = 16; s > 0; s >>= 1) {
            if (lane < s) {
                if (sizeof(T) == 8) tree[q * REFIT_THREADS + lane] = (T)__dadd_rn((double)tree[q * REFIT_THREADS + lane], (double)tree[q * REFIT_THREADS + lane + s]);
                else tree[q * REFIT_THREADS + lane] = (T)__fadd_rn((float)tree[q * REFIT_THREADS + lane], (float)tree[q * REFIT_THREADS + lane + s]);
            }
            __syncwarp();
        }
    }
    __syncthreads();
}

// one point of estimator EST as loaded from the problem's rows: float2 (x, y) for lines, float4 (x1, y1, x2, y2) for two views
template <int EST>
using LoPoint = typename std::conditional<usac_point_dim(EST) == 2, float2, float4>::type;

// The points of virtual lane l (ids[l], ids[l + 256], ...) in order, four gathers in flight: f(point) is called once per point.
template <int EST, class F>
__device__ __forceinline__ void lo_lane_points(const float* __restrict__ pts, const int* ids, int n, int l, F f) {
    using P = LoPoint<EST>;
    for (int k = l; k < n; k += 4 * REFIT_THREADS) {
        P p[4];
        // lines: defined on every path, or ptxas keeps the float2 array in local memory inside this loop (lo_kernel<LINE2D>)
        if constexpr (usac_point_dim(EST) == 2) {
#pragma unroll
            for (int u = 0; u < 4; u++) p[u] = P{0.f, 0.f};
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = k + u * REFIT_THREADS;
            if (i < n) p[u] = reinterpret_cast<const P*>(pts)[ids[i]];
        }
#pragma unroll
        for (int u = 0; u < 4; u++) if (k + u * REFIT_THREADS < n) f(p[u]);
    }
}

// entry e = 0..44 of the upper triangle of the 9 x 9 matrix A'A, row-major: (i, j)
__host__ __device__ constexpr int aat_row(int e) { int i = 0; while (e >= 9 - i) { e -= 9 - i; i++; } return i; }
__host__ __device__ constexpr int aat_col(int e) { int i = 0; while (e >= 9 - i) { e -= 9 - i; i++; } return i + e; }

template <int NROWS, int G, int C, int CNT>
struct LoAatAcc {                                                      // acc[C] += term of entry G + 4 C, indices known at compile time
    static __device__ __forceinline__ void run(double* acc, const float (&r)[2][9]) {
        constexpr int I = aat_row(G + 4 * C), J = aat_col(G + 4 * C);
        double a2 = 0.0;
#pragma unroll
        for (int q = 0; q < NROWS; q++) a2 = __dadd_rn(a2, __dmul_rn((double)r[q][I], (double)r[q][J]));
        acc[C] = __dadd_rn(acc[C], a2);
        LoAatAcc<NROWS, G, C + 1, CNT>::run(acc, r);
    }
};
template <int NROWS, int G, int CNT>
struct LoAatAcc<NROWS, G, CNT, CNT> { static __device__ __forceinline__ void run(double*, const float (&)[2][9]) {} };

// A'A partials of virtual lane l for the entries e = G, G + 4, ... (thread group G of four): every entry still adds its terms
// point by point in the lane's order, as one thread holding all 45 accumulators would - but 12 accumulators fit in registers.
template <int EST, int G>
__device__ __forceinline__ void lo_aat_group(const float* __restrict__ pts, const int* ids, int n, int l, float s1, float t1x, float t1y,
                                             float s2, float t2x, float t2y, double* tree) {
    constexpr int NROWS = (EST == USAC_EST_HOMOGRAPHY) ? 2 : 1;
    constexpr int CNT = (45 - G + 3) / 4;
    double acc[CNT];
#pragma unroll
    for (int c = 0; c < CNT; c++) acc[c] = 0.0;
    lo_lane_points<EST>(pts, ids, n, l, [&](const float4& p) {
        const float x1 = (sf(s1) * sf(p.x) + sf(t1x)).v, y1 = (sf(s1) * sf(p.y) + sf(t1y)).v;
        const float x2 = (sf(s2) * sf(p.z) + sf(t2x)).v, y2 = (sf(s2) * sf(p.w) + sf(t2y)).v;
        float r[2][9];
        if (EST == USAC_EST_HOMOGRAPHY) {
            r[0][0] = -x1; r[0][1] = -y1; r[0][2] = -1.f; r[0][3] = 0.f; r[0][4] = 0.f; r[0][5] = 0.f;
            r[0][6] = __fmul_rn(x2, x1); r[0][7] = __fmul_rn(x2, y1); r[0][8] = x2;
            r[1][0] = 0.f; r[1][1] = 0.f; r[1][2] = 0.f; r[1][3] = -x1; r[1][4] = -y1; r[1][5] = -1.f;
            r[1][6] = __fmul_rn(y2, x1); r[1][7] = __fmul_rn(y2, y1); r[1][8] = y2;
        } else {
            r[0][0] = __fmul_rn(x2, x1); r[0][1] = __fmul_rn(x2, y1); r[0][2] = x2; r[0][3] = __fmul_rn(y2, x1); r[0][4] = __fmul_rn(y2, y1);
            r[0][5] = y2; r[0][6] = x1; r[0][7] = y1; r[0][8] = 1.f;
#pragma unroll
            for (int q = 0; q < 9; q++) r[1][q] = 0.f;
        }
        LoAatAcc<NROWS, G, 0, CNT>::run(acc, r);
    });
#pragma unroll
    for (int c = 0; c < CNT; c++) tree[(G + 4 * c) * REFIT_THREADS + l] = acc[c];
}

// Estimator::EstimateModelNonMinimalSample on `n` point ids -> sh.model, sh.ok: the normalised DLT / eight-point path of the two-view
// estimators; lines are the specialisation below.
template <int EST>
__device__ void cta_nonminimal(const float* __restrict__ pts, const int* ids, int n, LoShared& sh) {
    const int t = threadIdx.x;
    const int l = t & (REFIT_THREADS - 1), grp = t >> 8;                // virtual lane, thread group (LO_THREADS = 4 x REFIT_THREADS)
    static_assert(LO_THREADS == 4 * REFIT_THREADS, "four thread groups share the 256 virtual lanes");
    const float fn = (float)n;
    float* treef = reinterpret_cast<float*>(sh.tree);
    __syncthreads();                                                   // everyone has read the previous call's sh.ok / sh.model
    if (t == 0) sh.ok = 0;
    if (n < 4) { __syncthreads(); return; }                            // uniform
    // ---- normalising transformations: group g sums coordinate g ----
    {
        float a = 0.f;
        lo_lane_points<EST>(pts, ids, n, l, [&](const float4& p) { a = __fadd_rn(a, grp == 0 ? p.x : grp == 1 ? p.y : grp == 2 ? p.z : p.w); });
        treef[grp * REFIT_THREADS + l] = a;
    }
    lo_tree256<float>(treef, 4);
    float m[4];
    for (int k = 0; k < 4; k++) m[k] = __fdiv_rn(treef[k * REFIT_THREADS], fn);
    __syncthreads();
    if (grp < 2) {                                                     // group 0: mean distance in image 1, group 1: in image 2
        float d = 0.f;
        const float mx = grp == 0 ? m[0] : m[2], my = grp == 0 ? m[1] : m[3];
        lo_lane_points<EST>(pts, ids, n, l, [&](const float4& p) {
            const sf a = sf(grp == 0 ? p.x : p.z) - sf(mx), b = sf(grp == 0 ? p.y : p.w) - sf(my);
            d = __fadd_rn(d, ssqrt(a * a + b * b).v);
        });
        treef[grp * REFIT_THREADS + l] = d;
    }
    lo_tree256<float>(treef, 2);
    const float d1 = treef[0], d2 = treef[REFIT_THREADS];
    __syncthreads();
    const double SQRT2 = 1.41421356237309504880;
    const float s1 = (float)(sd(SQRT2) / sd((double)__fdiv_rn(d1, fn))).v, s2 = (float)(sd(SQRT2) / sd((double)__fdiv_rn(d2, fn))).v;
    const float t1x = (-sf(m[0]) * sf(s1)).v, t1y = (-sf(m[1]) * sf(s1)).v, t2x = (-sf(m[2]) * sf(s2)).v, t2y = (-sf(m[3]) * sf(s2)).v;
    if (!isfinite(s1) || !isfinite(s2)) return;                        // uniform (every thread holds the same values)
    // ---- A'A: one pass over the points; group g accumulates the entries g, g + 4, ... of the upper triangle ----
    switch (grp) {                                                     // warp-uniform
        case 0: lo_aat_group<EST, 0>(pts, ids, n, l, s1, t1x, t1y, s2, t2x, t2y, sh.tree); break;
        case 1: lo_aat_group<EST, 1>(pts, ids, n, l, s1, t1x, t1y, s2, t2x, t2y, sh.tree); break;
        case 2: lo_aat_group<EST, 2>(pts, ids, n, l, s1, t1x, t1y, s2, t2x, t2y, sh.tree); break;
        default: lo_aat_group<EST, 3>(pts, ids, n, l, s1, t1x, t1y, s2, t2x, t2y, sh.tree); break;
    }
    lo_tree256<double>(sh.tree, 45);
    if (t < 45) {
        int i = 0, e = t;
        while (e >= 9 - i) { e -= 9 - i; i++; }
        const int j = i + e;
        const double v = sh.tree[t * REFIT_THREADS];
        sh.S[i * 9 + j] = v; sh.S[j * 9 + i] = v;
    }
    __syncthreads();
    if (t < 32) refit_smallest_eigenvector_warp(sh.S, 9, sh.h, sh.V);
    if (t == 0) {
        const double* h = sh.h;
        sd M[9], R[9];
        const sd S1((double)s1), T1x((double)t1x), T1y((double)t1y), S2((double)s2), T2x((double)t2x), T2y((double)t2y);
        for (int i = 0; i < 3; i++) {
            M[3 * i] = sd(h[3 * i]) * S1; M[3 * i + 1] = sd(h[3 * i + 1]) * S1;
            M[3 * i + 2] = (sd(h[3 * i]) * T1x + sd(h[3 * i + 1]) * T1y) + sd(h[3 * i + 2]);
        }
        bool ok = true;
        if (EST == USAC_EST_HOMOGRAPHY) {
            const sd is2 = sd(1.0) / S2, ux = -(T2x * is2), uy = -(T2y * is2);
            for (int j = 0; j < 3; j++) { R[j] = is2 * M[j] + ux * M[6 + j]; R[3 + j] = is2 * M[3 + j] + uy * M[6 + j]; R[6 + j] = M[6 + j]; }
            const sd inv = sd(1.0) / R[8];
            for (int i = 0; i < 9; i++) { const double v = (R[i] * inv).v; if (!dfinite(v)) ok = false; sh.model[i] = (float)v; }
            sh.model[8] = 1.f;
        } else {
            for (int j = 0; j < 3; j++) { R[j] = S2 * M[j]; R[3 + j] = S2 * M[3 + j]; R[6 + j] = (T2x * M[j] + T2y * M[3 + j]) + M[6 + j]; }
            const bool scale = fabsf((float)R[8].v) > 1.1920929e-07f;     // FLT_EPSILON
            const sd inv = scale ? sd(1.0) / R[8] : sd(1.0);
            for (int i = 0; i < 9; i++) { const double v = (R[i] * inv).v; if (!dfinite(v)) ok = false; sh.model[i] = (float)v; }
        }
        sh.ok = ok ? 1 : 0;
    }
    __syncthreads();
}

// Line2d (line2d_estimator.hpp:59-106): the five sums x, y, xy, xx, yy over the points. Group g accumulates sum g and, group 0, also
// sum 4 - each sum's addends in its lane's order - then one fixed tree over the five, then the closed form (line_from_sums) on thread 0.
template <>
__device__ void cta_nonminimal<USAC_EST_LINE2D>(const float* __restrict__ pts, const int* ids, int n, LoShared& sh) {
    const int t = threadIdx.x;
    const int l = t & (REFIT_THREADS - 1), grp = t >> 8;
    float* treef = reinterpret_cast<float*>(sh.tree);
    __syncthreads();                                                   // everyone has read the previous call's sh.ok / sh.model
    if (t == 0) sh.ok = 0;
    if (n < 2) { __syncthreads(); return; }                            // uniform
    float a = 0.f, yy = 0.f;
    lo_lane_points<USAC_EST_LINE2D>(pts, ids, n, l, [&](const float2& p) {
        a = __fadd_rn(a, grp == 0 ? p.x : grp == 1 ? p.y : grp == 2 ? __fmul_rn(p.x, p.y) : __fmul_rn(p.x, p.x));
        if (grp == 0) yy = __fadd_rn(yy, __fmul_rn(p.y, p.y));
    });
    treef[grp * REFIT_THREADS + l] = a;
    if (grp == 0) treef[4 * REFIT_THREADS + l] = yy;
    lo_tree256<float>(treef, 5);
    if (t == 0) {
        float r[5];
        for (int k = 0; k < 5; k++) r[k] = treef[k * REFIT_THREADS];
        sh.ok = line_from_sums(r, n, sh.model) ? 1 : 0;
    }
    __syncthreads();
}

// Estimator::EstimateModelNonMinimalSample as a kernel of its own (usac_gpu_estimate_nonminimal, the final refit): the CTA-wide
// form above, for every estimator.
template <int EST>
__global__ void __launch_bounds__(LO_THREADS, 1) nonminimal_cta_kernel(const float* __restrict__ pts, const int* __restrict__ ids, int n,
                                                                       float* __restrict__ model_out, int* __restrict__ ok_out) {
    extern __shared__ __align__(16) unsigned char lo_smem[];
    LoShared& sh = *reinterpret_cast<LoShared*>(lo_smem);
    cta_nonminimal<EST>(pts, ids, n, sh);
    __syncthreads();
    if (threadIdx.x == 0) {
        *ok_out = sh.ok;
        if (sh.ok) for (int i = 0; i < (EST == USAC_EST_LINE2D ? 3 : 9); i++) model_out[i] = sh.model[i];
    }
}

// Quality::getNumberInliers(score, model, thr, get_inliers = true, ids) (quality.hpp:60-101): sh.cnt, sh.sum, ids in ascending order.
// Same arithmetic as inliers_sum_kernel (score.cuh).
template <int EST>
__device__ void cta_score(const float* __restrict__ aos, int n, const float* model, float thr, const ProblemDesc& pd, int* ids, LoShared& sh) {
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) {
        float rec[USAC_REC_STRIDE];
        make_record(EST, model, thr, pd, rec);
        for (int i = 0; i < USAC_REC_STRIDE; i++) sh.rec[i] = rec[i];
    }
    __syncthreads();
    float acc = 0.f;
    int base = 0;                                                      // inliers so far (the same value in every thread)
    for (int start = 0, buf = 0; start < n; start += LO_THREADS, buf ^= 1) {
        const int i = start + t;
        bool in = false;
        if (i < n) {
            float e;
            if constexpr (usac_point_dim(EST) == 2) { const float2 p = reinterpret_cast<const float2*>(aos)[i]; e = strict_error<EST>(sh.rec, p.x, p.y, 0.f, 0.f); }
            else { const float4 p = reinterpret_cast<const float4*>(aos)[i]; e = strict_error<EST>(sh.rec, p.x, p.y, p.z, p.w); }
            in = e < thr;
            if (in) acc = __fadd_rn(acc, e);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) sh.warp_tot[buf][warp] = __popc(bal);
        __syncthreads();                                               // the one barrier per block: the other buffer is free again by the next one
        int incl = sh.warp_tot[buf][lane];                             // lane l holds warp l's count: scan over the 32 warps by shuffles
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        const int upto = __shfl_sync(0xffffffffu, incl, warp);        // inclusive count of warps 0 .. warp
        const int before = upto - __popc(bal);
        if (in) ids[base + before + __popc(bal & ((1u << lane) - 1))] = i;
        base += total;
    }
    sh.part[t] = acc;
    __syncthreads();
    for (int s = LO_THREADS / 2; s >= 32; s >>= 1) {
        if (t < s) sh.part[t] = __fadd_rn(sh.part[t], sh.part[t + s]);
        __syncthreads();
    }
    if (warp == 0) {
        for (int s = 16; s > 0; s >>= 1) {
            if (lane < s) sh.part[lane] = __fadd_rn(sh.part[lane], sh.part[lane + s]);
            __syncwarp();
        }
    }
    __syncthreads();
    if (t == 0) { sh.cnt = base; sh.sum = sh.part[0]; }
    __threadfence_block();
    __syncthreads();
}

// 14 distinct positions in [0, count): two Philox draws (8 + 6), the second mapped past the first (LoRunner::fit_random_subset)
__device__ void lo_subset(unsigned long long seed, unsigned long long calls, int k, int count, const int* from, int* sample) {
    int pos[16], a[8], b[8];
    philox_unique(seed, calls, 7, count, k < 8 ? k : 8, a);
    for (int i = 0; i < (k < 8 ? k : 8); i++) pos[i] = a[i];
    if (k > 8) {
        philox_unique(seed, calls, 8, count - 8, k - 8, b);
        int sorted[8];
        for (int i = 0; i < 8; i++) sorted[i] = a[i];
        for (int i = 1; i < 8; i++) { const int v = sorted[i]; int j = i - 1; while (j >= 0 && sorted[j] > v) { sorted[j + 1] = sorted[j]; j--; } sorted[j + 1] = v; }
        for (int i = 0; i < k - 8; i++) {
            int v = b[i];
            for (int q = 0; q < 8; q++) if (v >= sorted[q]) v++;
            pos[8 + i] = v;
        }
    }
    for (int i = 0; i < k; i++) sample[i] = from[pos[i]];
}

__device__ __forceinline__ bool lo_bigger(int ia, float sa, int ib, float sb) { return ia > ib || (ia == ib && sa > sb); }

// One inner iteration of InnerLocalOptimization::GetModelScore (inner_local_optimization.hpp:85-131 with the iterative stage,
// iterative_local_optimization.hpp:61-135) from the state (best score, pool A of `avail` inliers, running threshold, call counter).
// Returns 1 when the inner loop ends here (`break`), else 0; `improved` = the candidate (sh.model, B[0 .. lo_inl)) beats the best.
template <int EST>
__device__ int lo_inner_iteration(const LoArgs& a, const ProblemDesc& pd, LoShared& sh, const int* A, int* B, int best_inl, float best_sum, int avail,
                                  float& lo_thr, unsigned long long& calls, unsigned& inner_done, unsigned& iterative_done,
                                  bool& improved, int& lo_inl, float& lo_sum) {
    const int t = threadIdx.x;
    improved = false; lo_inl = 0; lo_sum = 0.f;
    if (avail > a.sample_limit) {
        if (t == 0) lo_subset(a.seed, calls, a.sample_limit, avail, A, sh.sample);
        calls++;
        __syncthreads();
        cta_nonminimal<EST>(a.aos, sh.sample, a.sample_limit, sh);
        if (!sh.ok) return 0;                                          // continue
    } else {
        cta_nonminimal<EST>(a.aos, A, avail, sh);
        if (!sh.ok) return 1;                                          // break
    }
    lo_thr = (unsigned)a.mult * lo_thr;                                 // inner_local_optimization.hpp:101
    cta_score<EST>(a.aos, a.n, sh.model, lo_thr, pd, B, sh);
    lo_inl = sh.cnt;
    lo_sum = sh.sum;
    if (lo_inl <= a.m) return 0;                                       // continue
    // ---- IterativeLocalOptimization::GetModelScore ----
    for (int k = 0; k < a.iter_iters; k++) {
        lo_thr -= a.step;
        if (lo_inl <= a.m) break;
        if (a.kind == 2) {                                             // GetScoreLimited
            if (lo_inl > a.sample_limit) {
                if (t == 0) lo_subset(a.seed, calls, a.sample_limit, lo_inl, B, sh.sample);
                calls++;
                __syncthreads();
                cta_nonminimal<EST>(a.aos, sh.sample, a.sample_limit, sh);
                if (!sh.ok) continue;
            } else {
                cta_nonminimal<EST>(a.aos, B, lo_inl, sh);
                if (!sh.ok) break;
            }
            cta_score<EST>(a.aos, a.n, sh.model, lo_thr, pd, B, sh);
            lo_inl = sh.cnt; lo_sum = sh.sum;
        } else {                                                       // GetScoreUnlimited
            cta_nonminimal<EST>(a.aos, B, lo_inl, sh);
            if (!sh.ok) break;
            cta_score<EST>(a.aos, a.n, sh.model, lo_thr, pd, B, sh);
            lo_inl = sh.cnt; lo_sum = sh.sum;
            if (lo_bigger(best_inl, best_sum, lo_inl, lo_sum)) break;
        }
        iterative_done++;
    }
    bool fail = false;
    if (fabsf(lo_thr - a.theta) > 0.00001) { fail = true; lo_thr = a.theta; }
    improved = !fail && lo_bigger(lo_inl, lo_sum, best_inl, best_sum);
    inner_done++;
    return 0;
}

template <int EST>
__global__ void __launch_bounds__(LO_THREADS, 1) lo_kernel(const LoArgs a) {
    extern __shared__ __align__(16) unsigned char lo_smem[];
    LoShared& sh = *reinterpret_cast<LoShared*>(lo_smem);
    const int t = threadIdx.x;
    const ProblemDesc pd = a.prob[a.problem];
    // every thread follows the same control flow: the decisions depend on values that all threads read from shared / global memory
    // behind a CTA barrier
    int best_inl = a.io->inliers;
    float best_sum = a.io->score, lo_thr = a.io->lo_thr;
    unsigned long long calls = a.io->calls;
    unsigned inner_done = 0, iterative_done = 0;
    if (t < 9) sh.best_model[t] = a.io->model[t];
    __syncthreads();
    if (best_inl >= 12) {                                              // inner_local_optimization.hpp:76
        cta_score<EST>(a.aos, a.n, sh.best_model, a.theta, pd, a.A, sh);   // quality->getInliers(best_model)
        int avail = min(best_inl, sh.cnt);                             // ids present in A (never index past the list)
        for (int it = 0; it < a.inner_iters; it++) {
            bool improved;
            int lo_inl;
            float lo_sum;
            if (lo_inner_iteration<EST>(a, pd, sh, a.A, a.B, best_inl, best_sum, avail, lo_thr, calls, inner_done, iterative_done, improved, lo_inl, lo_sum)) break;
            if (improved) {
                __syncthreads();
                if (t < 9) sh.best_model[t] = sh.model[t];
                for (int i = t; i < lo_inl; i += LO_THREADS) a.A[i] = a.B[i];
                best_inl = lo_inl; best_sum = lo_sum; avail = lo_inl;
                __threadfence_block();
                __syncthreads();
            }
        }
    }
    __syncthreads();
    if (t == 0) {
        for (int i = 0; i < 9; i++) a.io->model[i] = sh.best_model[i];
        a.io->inliers = best_inl; a.io->score = best_sum; a.io->lo_thr = lo_thr; a.io->calls = calls;
        a.io->inner_done = inner_done; a.io->iterative_done = iterative_done;
    }
}

// ------------------------------------------------------------------------------------------------------------------------------
// The same LO call with its inner iterations executed SPECULATIVELY side by side. An inner iteration changes the state the next one
// starts from only when it improves the best model (rare: a few of the 20) - otherwise the next iteration's inputs are known in
// advance: the same pool A, the running threshold back at theta, the call counter advanced by the iteration's subset draws. So a
// WAVE runs all remaining iterations at once, one CTA each, on those predicted inputs; a commit kernel then walks them in order,
// accepts every iteration whose assumed inputs equal the actual state, stops at the first improvement (which it applies: model,
// pool, counters) or misprediction, and the next wave starts behind it. Every accepted iteration ran the sequential code on the
// sequential inputs, so the result is that of lo_kernel bit for bit; an LO call costs (improvements + 1) waves of ~5 dependent
// fit-and-score steps instead of 20 x 5.
// ------------------------------------------------------------------------------------------------------------------------------
struct LoWaveState {
    float best_model[9];
    int best_inl;
    float best_sum;
    int avail;
    float lo_thr;
    unsigned long long calls;
    unsigned inner_done, iterative_done;
    int next_it, finished;
};
struct LoSpec {                   // one speculatively executed inner iteration
    unsigned long long calls_in, calls_out;
    float lo_thr_in, lo_thr_out;
    int status, improved, lo_inl;
    float lo_sum;
    float model[9];
    unsigned d_inner, d_iter;
};
#define LO_WAVE_VARIANTS 6       // predicted running thresholds tried per iteration (grid.y of the wave)
struct LoWaveArgs {
    LoArgs a;
    LoWaveState* ws;
    LoSpec* spec;                 // [inner_iters][LO_WAVE_VARIANTS]
    int* Bwave;                   // [inner_iters][LO_WAVE_VARIANTS][n] candidate inlier lists
};

// best model -> pool A, avail (quality->getInliers(best_model)); state from the io record
template <int EST>
__global__ void __launch_bounds__(LO_THREADS, 1) lo_pool_kernel(const LoWaveArgs w) {
    extern __shared__ __align__(16) unsigned char lo_smem[];
    LoShared& sh = *reinterpret_cast<LoShared*>(lo_smem);
    const LoArgs& a = w.a;
    const int t = threadIdx.x;
    const ProblemDesc pd = a.prob[a.problem];
    if (t < 9) sh.best_model[t] = a.io->model[t];
    __syncthreads();
    cta_score<EST>(a.aos, a.n, sh.best_model, a.theta, pd, a.A, sh);
    if (t == 0) {
        LoWaveState& s = *w.ws;
        for (int i = 0; i < 9; i++) s.best_model[i] = a.io->model[i];
        s.best_inl = a.io->inliers; s.best_sum = a.io->score; s.avail = min(a.io->inliers, sh.cnt);
        s.lo_thr = a.io->lo_thr; s.calls = a.io->calls; s.inner_done = 0; s.iterative_done = 0; s.next_it = 0; s.finished = 0;
    }
}

// subset draws an iteration is expected to make (the prediction of the next iteration's call counter)
__device__ __forceinline__ int lo_expected_draws(const LoArgs& a, int avail) {
    return (avail > a.sample_limit ? 1 : 0) + (a.kind == 2 ? a.iter_iters : 0);
}
// the running threshold after an iteration that goes through all its steps (the statements of lo_inner_iteration, one rounding each)
__device__ __forceinline__ float lo_thr_after_full_iteration(const LoArgs& a, float x) {
    x = __fmul_rn((float)(unsigned)a.mult, x);
    for (int k = 0; k < a.iter_iters; k++) x = __fsub_rn(x, a.step);
    if (fabsf(__fsub_rn(x, a.theta)) > 0.00001) x = a.theta;
    return x;
}
// Predicted running threshold of iteration next_it + b, variant v. An iteration leaves either the value of the full path or theta
// (reset after an early exit of the iterative stage), so the candidates are: v = 0 the full-path chain from the actual value,
// v = j + 1 the full-path chain restarted from theta j iterations ago. Returns false for a variant that repeats an earlier one.
__device__ __forceinline__ bool lo_predicted_threshold(const LoArgs& a, float actual, int b, int v, float& out) {
    float cand[LO_WAVE_VARIANTS];
    int nc = 0;
    {
        float x = actual;
        for (int i = 0; i < b; i++) x = lo_thr_after_full_iteration(a, x);
        cand[nc++] = x;
    }
    if (b > 0) {
        float x = a.theta;
        for (int j = 0; j < LO_WAVE_VARIANTS - 1 && j < b; j++) {       // restarted from theta j iterations ago
            if (j > 0) x = lo_thr_after_full_iteration(a, x);
            cand[nc++] = x;
        }
    }
    if (v >= nc) return false;
    for (int i = 0; i < v; i++) if (__float_as_uint(cand[i]) == __float_as_uint(cand[v])) return false;
    out = cand[v];
    return true;
}

template <int EST>
__global__ void __launch_bounds__(LO_THREADS, 1) lo_wave_kernel(const LoWaveArgs w) {
    extern __shared__ __align__(16) unsigned char lo_smem[];
    LoShared& sh = *reinterpret_cast<LoShared*>(lo_smem);
    const LoArgs& a = w.a;
    const ProblemDesc pd = a.prob[a.problem];
    const LoWaveState s = *w.ws;                                     // written by the previous kernel in the stream
    const int b = blockIdx.x, v = blockIdx.y;                        // iteration s.next_it + b, threshold variant v
    LoSpec& o = w.spec[b * LO_WAVE_VARIANTS + v];
    float lo_thr;
    const bool run = !s.finished && s.next_it + b < a.inner_iters && lo_predicted_threshold(a, s.lo_thr, b, v, lo_thr);
    if (!run) {                                                      // uniform over the CTA
        if (threadIdx.x == 0) o.status = -1;                         // nothing ran here
        return;
    }
    unsigned long long calls = s.calls + (unsigned long long)b * (unsigned long long)lo_expected_draws(a, s.avail);
    const unsigned long long calls_in = calls;
    const float lo_thr_in = lo_thr;
    unsigned d_inner = 0, d_iter = 0;
    bool improved;
    int lo_inl;
    float lo_sum;
    int* B = w.Bwave + ((size_t)b * LO_WAVE_VARIANTS + v) * a.n;
    const int status = lo_inner_iteration<EST>(a, pd, sh, a.A, B, s.best_inl, s.best_sum, s.avail, lo_thr, calls, d_inner, d_iter, improved, lo_inl, lo_sum);
    __syncthreads();
    if (threadIdx.x == 0) {
        o.calls_in = calls_in; o.calls_out = calls; o.lo_thr_in = lo_thr_in; o.lo_thr_out = lo_thr;
        o.status = status; o.improved = improved ? 1 : 0; o.lo_inl = lo_inl; o.lo_sum = lo_sum;
        for (int i = 0; i < 9; i++) o.model[i] = sh.model[i];
        o.d_inner = d_inner; o.d_iter = d_iter;
    }
}

// walk the wave in iteration order (one CTA): accept, apply the first improvement, stop at a misprediction
__global__ void __launch_bounds__(LO_THREADS) lo_commit_kernel(const LoWaveArgs w) {
    __shared__ int s_copy_from, s_copy_n;
    const LoArgs& a = w.a;
    LoWaveState& s = *w.ws;
    if (threadIdx.x == 0) {
        s_copy_from = -1; s_copy_n = 0;
        if (!s.finished) {
            int it = s.next_it;
            const int it0 = it;
            for (; it < a.inner_iters; it++) {
                int hit = -1;                                          // the variant that ran on the actual inputs
                for (int v = 0; v < LO_WAVE_VARIANTS && hit < 0; v++) {
                    const LoSpec& c = w.spec[(it - it0) * LO_WAVE_VARIANTS + v];
                    if (c.status >= 0 && c.calls_in == s.calls && __float_as_uint(c.lo_thr_in) == __float_as_uint(s.lo_thr)) hit = v;
                }
                if (hit < 0) break;                                    // ran on other inputs: the next wave starts here
                const LoSpec& o = w.spec[(it - it0) * LO_WAVE_VARIANTS + hit];
                s.calls = o.calls_out; s.lo_thr = o.lo_thr_out; s.inner_done += o.d_inner; s.iterative_done += o.d_iter;
                if (o.status) { s.finished = 1; it++; break; }         // the inner loop's `break`
                if (o.improved) {
                    for (int i = 0; i < 9; i++) s.best_model[i] = o.model[i];
                    s.best_inl = o.lo_inl; s.best_sum = o.lo_sum; s.avail = o.lo_inl;
                    s_copy_from = (it - it0) * LO_WAVE_VARIANTS + hit; s_copy_n = o.lo_inl;
                    it++;
                    break;                                             // the later iterations of the wave saw the old state
                }
            }
            s.next_it = it;
            if (it >= a.inner_iters) s.finished = 1;
        }
    }
    __syncthreads();
    if (s_copy_from >= 0) {
        const int* B = w.Bwave + (size_t)s_copy_from * a.n;
        for (int i = threadIdx.x; i < s_copy_n; i += blockDim.x) a.A[i] = B[i];
    }
    __syncthreads();
    if (threadIdx.x == 0 && s.finished) {
        for (int i = 0; i < 9; i++) a.io->model[i] = s.best_model[i];
        a.io->inliers = s.best_inl; a.io->score = s.best_sum; a.io->lo_thr = s.lo_thr; a.io->calls = s.calls;
        a.io->inner_done = s.inner_done; a.io->iterative_done = s.iterative_done;
    }
}
