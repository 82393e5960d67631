// pipeline.cuh - the kernels around the scoring kernel for one round of K samples per problem:
//   sample_kernel  -> solve_kernel -> prepare_kernel -> score_kernel -> reduce_kernel -> [all-gather] -> select_kernel
// One host sync per round (the FitState records are copied back after select_kernel).
#pragma once
#include "strict_math.cuh"

struct RoundArgs {
    const ProblemDesc* prob;
    const int* active;           // slot -> problem id
    FitState* state;             // per problem
    const float* aos;
    int est, K, S, m, mstride;   // samples per round, models per sample, sample size, K*S
    int e5_all_roots;            // essential: every cheirality-valid root is a model (S = USAC_E5_MAX_ROOTS), else the first one
    int midx_shift;              // per-sample score packing: model index above bit midx_shift (30: up to 3 models, 28: up to 10)
    // sampler
    int sampler, rng, neighbors;
    uint64_t seed;
    const int* table; unsigned table_rows;     // USAC_RNG_TABLE (problem 0)
    const unsigned* growth;                    // PROSAC growth functions (ProblemDesc::growth_off)
    const int* knn; const int* cell_of_point; const int* members; const int* rank_in_cell; const int* cell_start;
    unsigned* cursors;                         // NAPSAC use counters
    int* seeds;                                // [slot][K] NAPSAC seed points of the round
    // buffers, all [slot][...]
    int* samples;                // [K][m]
    float* models_raw;           // [K][S][9]
    int* nmodels;                // [K]
    int* offsets;                // [K]  exclusive prefix sum of nmodels
    float* recs;                 // [K*S][USAC_REC_STRIDE]
    int* mvalid;                 // [1]
    uint2* items;                // compact work-item list of the scoring kernel: (slot, chunk << 16 | model group), only groups that hold models
    unsigned* item_count;        // [0] = number of items (zeroed by the host before the round), [1] = the scoring kernel's draw counter
    int* part_cnt; float* part_sum; int nchunks;   // [nchunks][K*S]
    uint2* sample_scores;        // [K] per-sample best (cnt | midx << midx_shift, sum bits); with nranks>1: [nranks][ceil(K/nranks)]
    // fit parameters
    float thr, confidence;
    unsigned max_iterations;
    const unsigned* term_tables; // standard termination bound by inlier count (ProblemDesc::term_off)
    int rank, nranks;
    // SPRT (sprt.cuh)
    int sprt;
    const int* pool;             // shuffled point pools (ProblemDesc::pool_off)
    struct SprtModelResult* sprt_res;   // [slot][K*S]
    int* done_out;               // [slot] FitState::done after the round (the only thing the host reads per round)
    unsigned before_sprt;        // model.hpp:39 max_hypothesis_test_before_sprt
    int limit_remaining;         // 1: samples the sequential loop can no longer reach (index >= max_iters - iters at the start of
                                 // the round; the bound never grows) are not solved or scored
    // hypothesis sharding over peer memory (NVLink): the reduce kernels store this rank's per-sample scores straight into every
    // rank's exchange window and raise a flag there; select_kernel waits for the flags of all ranks. No collective call.
    void* const* peer_win;       // [nranks] exchange windows (PeerWindow layout below), own included; nullptr = exchange by the host's hook
    void* peer_self;             // this rank's window
    unsigned peer_seq;           // sequence number of this round (same on every rank, grows by one per round for the life of the windows)
    unsigned peer_cap;           // uint2 entries per parity buffer
    unsigned* peer_counter;      // CTAs of the reduce kernel that have stored their part
    int* peer_error;             // set when a wait timed out
    unsigned long long hyp_base_p1;   // 0: the hypothesis id of sample j is FitState::samples_drawn + j; else (hyp_base_p1 - 1) + j (solve-ahead
                                      // blocks launched before the state has advanced that far)
};

// Exchange window of one rank: flags[2][64] (sequence number last published by rank r, per parity), then two buffers of
// peer_cap packed scores laid out [rank][slot][ceil(K / nranks)]. Two parities: a rank can be at most one round ahead of the
// slowest one, because it needs everybody's part of round s before it can publish round s + 1.
#define USAC_PEER_HEADER_BYTES 1024
#define USAC_PEER_MAX_RANKS 64
__device__ __forceinline__ uint2* peer_data(void* win, unsigned seq, unsigned cap) {
    return reinterpret_cast<uint2*>(reinterpret_cast<char*>(win) + USAC_PEER_HEADER_BYTES) + (size_t)(seq & 1u) * cap;
}
__device__ __forceinline__ unsigned* peer_flags(void* win, unsigned seq) {
    return reinterpret_cast<unsigned*>(win) + (seq & 1u) * USAC_PEER_MAX_RANKS;
}
// one packed score -> the same place in every rank's window
__device__ __forceinline__ void peer_store(const RoundArgs& a, size_t idx, uint2 v) {
    for (int r = 0; r < a.nranks; r++) peer_data(a.peer_win[r], a.peer_seq, a.peer_cap)[idx] = v;
}
// end of a reduce kernel (every thread of every CTA calls it): the last CTA to arrive raises this rank's flag everywhere
__device__ __forceinline__ void peer_publish(const RoundArgs& a) {
    __threadfence_system();                                          // this thread's remote stores are visible system-wide ...
    __syncthreads();                                                 // ... before thread 0 counts the CTA in
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y * gridDim.z;
        if (atomicAdd(a.peer_counter, 1u) == total - 1u) {
            *a.peer_counter = 0u;
            __threadfence_system();
            for (int r = 0; r < a.nranks; r++) {
                unsigned* f = peer_flags(a.peer_win[r], a.peer_seq) + a.rank;
                asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(f), "r"(a.peer_seq) : "memory");
            }
        }
    }
}
// start of select_kernel: until every rank has published this round (2 s limit: a rank that never arrives must not hang the GPU)
__device__ __forceinline__ void peer_wait(const RoundArgs& a) {
    if ((int)threadIdx.x < a.nranks) {
        const unsigned* f = peer_flags(a.peer_self, a.peer_seq) + threadIdx.x;
        unsigned long long t0 = 0, t1 = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            unsigned v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if ((int)(v - a.peer_seq) >= 0) break;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 2000000000ull) { *a.peer_error = 1; break; }
            __nanosleep(200);
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------------
// Guard-band constants of the fast scoring path (see score.cuh). u = 2^-24. All bounds are deliberately loose
// (worst-case linear error accumulation); a looser band only sends a few more points through the strict path.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void make_record(int est, const float* model, float thr, const ProblemDesc& pd, float* rec) {
    const float u = 5.9604645e-8f;
#pragma unroll
    for (int i = 0; i < USAC_REC_STRIDE; i++) rec[i] = 0.f;
    const int w = est == USAC_EST_LINE2D ? 3 : 9;
    for (int i = 0; i < w; i++) rec[i] = model[i];
    rec[REC_THR] = thr;
    const float* f = model;
    if (est == USAC_EST_HOMOGRAPHY) {
        cv_inv3x3(model, rec + REC_HINV);
        const float* g = rec + REC_HINV;
        // |fl32 reference value of 2*err  -  fast value| <= c0 + K1 |1/nz| + K2 |1/mz| for every point that either
        // arithmetic puts at or below the threshold (first order in u, derivation in DESIGN.md section 4.2):
        //   projections: reference 3u*A, fast (FMA) 2u*A, A = |h_i1 x| + |h_i2 y| + |h_i3| <= b*;
        //   quotient: reference u, fast 4u (product, rcp.approx 2^-23, product);  norm: reference 2u, fast 3u.
        // c0 is folded into the first term with |1/nz| >= 1/bz1.
        const float T2 = 2.f * thr;
        const float bx1 = fabsf(f[0]) * pd.mx1 + fabsf(f[1]) * pd.my1 + fabsf(f[2]);
        const float by1 = fabsf(f[3]) * pd.mx1 + fabsf(f[4]) * pd.my1 + fabsf(f[5]);
        const float bz1 = fabsf(f[6]) * pd.mx1 + fabsf(f[7]) * pd.my1 + fabsf(f[8]);
        const float bx2 = fabsf(g[0]) * pd.mx2 + fabsf(g[1]) * pd.my2 + fabsf(g[2]);
        const float by2 = fabsf(g[3]) * pd.mx2 + fabsf(g[4]) * pd.my2 + fabsf(g[5]);
        const float bz2 = fabsf(g[6]) * pd.mx2 + fabsf(g[7]) * pd.my2 + fabsf(g[8]);
        const float g8 = 8.f * u;
        const float K1 = g8 * ((bx1 + by1) + (pd.mx2 + pd.my2 + 2.1f * T2) * bz1);
        const float K2 = g8 * ((bx2 + by2) + (pd.mx1 + pd.my1 + 2.1f * T2) * bz2);
        const float c0 = g8 * (pd.mx1 + pd.my1 + pd.mx2 + pd.my2 + 4.2f * T2) + 32.f * u * T2;
        rec[REC_BAND] = 1.001f * (K1 + c0 * bz1);
        rec[REC_BAND + 1] = 1.001f * K2;
    } else if (est == USAC_EST_FUNDAMENTAL) {
        const float ba = fabsf(f[0]) * pd.mx1 + fabsf(f[1]) * pd.my1 + fabsf(f[2]);
        const float bb = fabsf(f[3]) * pd.mx1 + fabsf(f[4]) * pd.my1 + fabsf(f[5]);
        const float bc = fabsf(f[0]) * pd.mx2 + fabsf(f[3]) * pd.my2 + fabsf(f[6]);
        const float bd = fabsf(f[1]) * pd.mx2 + fabsf(f[4]) * pd.my2 + fabsf(f[7]);
        const float bn = pd.mx2 * ba + pd.my2 * bb + fabsf(f[6]) * pd.mx1 + fabsf(f[7]) * pd.my1 + fabsf(f[8]);
        const float dn = 18.f * u * bn, dabcd = 5.f * u * (ba + bb + bc + bd);
        const float eta = 1e-3f * thr;
        const float gq = 1.5f * sqrtf(thr) * dn + thr * dabcd;
        rec[REC_BAND] = eta + 16.f * u * thr;                 // * den
        rec[REC_BAND + 1] = gq * gq / eta + dn * dn;          // + const
    } else if (est == USAC_EST_ESSENTIAL) {
        const float T = 2.f * thr;
        const float bl1 = fabsf(f[0]) * pd.mx2 + fabsf(f[3]) * pd.my2 + fabsf(f[6]);
        const float bl2 = fabsf(f[1]) * pd.mx2 + fabsf(f[4]) * pd.my2 + fabsf(f[7]);
        const float bl3 = fabsf(f[2]) * pd.mx2 + fabsf(f[5]) * pd.my2 + fabsf(f[8]);
        const float bt1 = fabsf(f[0]) * pd.mx1 + fabsf(f[1]) * pd.my1 + fabsf(f[2]);
        const float bt2 = fabsf(f[3]) * pd.mx1 + fabsf(f[4]) * pd.my1 + fabsf(f[5]);
        const float bt3 = fabsf(f[6]) * pd.mx1 + fabsf(f[7]) * pd.my1 + fabsf(f[8]);
        const float ba1 = pd.mx1 * bl1 + pd.my1 * bl2 + bl3, bb1 = pd.mx2 * bt1 + pd.my2 * bt2 + bt3;
        rec[REC_BAND] = 10.f * u * ba1 + 10.f * u * T * (bl1 + bl2);       // * 1/|l12|
        rec[REC_BAND + 1] = 10.f * u * bb1 + 10.f * u * T * (bt1 + bt2);   // * 1/|t12|
        rec[REC_BAND + 2] = 32.f * u * T;
    } else {
        rec[REC_BAND] = 5.f * u * (fabsf(f[0]) * pd.mx1 + fabsf(f[1]) * pd.my1 + fabsf(f[2])) + 2.f * u * thr;
    }
}

// records for host-supplied models (usac_gpu_score): one thread per model, no compaction
__global__ void prepare_models_kernel(int est, const float* __restrict__ models, int M, int model_stride, float thr,
                                      const ProblemDesc* prob, int problem, float* __restrict__ recs) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= M) return;
    float rec[USAC_REC_STRIDE];
    make_record(est, models + (size_t)q * model_stride, thr, prob[problem], rec);
    float4* dst = reinterpret_cast<float4*>(recs + (size_t)q * USAC_REC_STRIDE);
#pragma unroll
    for (int i = 0; i < USAC_REC_STRIDE / 4; i++) dst[i] = make_float4(rec[4 * i], rec[4 * i + 1], rec[4 * i + 2], rec[4 * i + 3]);
}

// ---------------------------------------------------------------------------------------------------------------
// Samplers (uniform_sampler.hpp, prosac_sampler.hpp, napsac_sampler.hpp). One thread per sample of the round.
// ---------------------------------------------------------------------------------------------------------------

// PROSAC: subset size after the call with hypothesis counter t (prosac_sampler.hpp:147-156): min{n >= m : g[n-1] >= t}
__device__ __forceinline__ unsigned prosac_subset(const unsigned* __restrict__ g, unsigned n_points, unsigned m, unsigned t) {
    unsigned lo = m, hi = n_points;          // answer in [m, n_points]
    while (lo < hi) {
        const unsigned mid = (lo + hi) >> 1;
        if (g[mid - 1] >= t) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// NAPSAC seed points of the round (napsac_sampler.hpp:77, 103-108)
__global__ void napsac_seed_kernel(const RoundArgs a) {
    const int slot = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.K) return;
    const int pid = a.active[slot];
    const ProblemDesc pd = a.prob[pid];
    const uint64_t hyp = (a.hyp_base_p1 ? (uint64_t)(a.hyp_base_p1 - 1) : (uint64_t)a.state[pid].samples_drawn) + j;
    int p = 0;
    if (a.sampler == USAC_SAMPLER_PROGRESSIVE_NAPSAC) {
        if (hyp >= pnapsac_length(pd)) p = -1;                             // global phase: no centre, nothing counted
        else philox_unique(a.seed, hyp, 5, pd.n, 1, &p);
    } else if (a.neighbors == USAC_NEIGH_KNN) {
        philox_unique(a.seed, hyp, 4, pd.n, 1, &p);
    } else {
        // napsac_sampler.hpp:100-128: redraw the seed until its cell holds enough neighbours; a call that finds none in n draws switches
        // the sampler to uniform sampling FOR THE REST OF THE RUN (do_uniform). The hypothesis id of the first such call lives in the
        // last entry of the cursor segment (0xffffffff = none): every sample from that id on is uniform, whatever its own search says.
        unsigned* first_uniform = a.cursors + pd.cursor_off + 3 * (size_t)pd.n;
        if ((unsigned long long)hyp >= (unsigned long long)*reinterpret_cast<volatile unsigned*>(first_uniform)) p = -1;
        else {
            int tries = 0;
            for (; tries < pd.n; tries++) {
                philox_unique(a.seed, hyp, 16 + (uint32_t)tries, pd.n, 1, &p);
                const int c = a.cell_of_point[pd.grid_off + p];
                const int cnt = a.cell_start[pd.cell_start_off + c + 1] - a.cell_start[pd.cell_start_off + c] - 1;
                if (cnt >= a.m) break;
            }
            if (tries == pd.n) { p = -1; atomicMin(first_uniform, (unsigned)hyp); }
        }
    }
    a.seeds[(size_t)slot * a.K + j] = p;
    // how often the round uses each seed point (second half of the cursor segment, all zero between rounds): a seed used once -
    // the common case - needs no search for earlier uses in sample_kernel
    if (p >= 0) {
        atomicAdd(&a.cursors[pd.cursor_off + pd.n + p], 1u);
        atomicMax(&a.cursors[pd.cursor_off + 2 * (size_t)pd.n + p], (unsigned)(a.K - j));   // third part of the segment: K - (first sample of the round
    }                                                                                         // that uses this seed); 0 = none
}

__global__ void napsac_commit_kernel(const RoundArgs a) {
    const int slot = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.K) return;
    const int pid = a.active[slot];
    const int p = a.seeds[(size_t)slot * a.K + j];
    if (p >= 0) {
        const ProblemDesc pd = a.prob[pid];
        const uint64_t hyp = (a.hyp_base_p1 ? (uint64_t)(a.hyp_base_p1 - 1) : (uint64_t)a.state[pid].samples_drawn) + j;
        const bool uniform_by_now = a.neighbors != USAC_NEIGH_KNN && hyp >= (uint64_t)a.cursors[pd.cursor_off + 3 * (size_t)pd.n];
        // NAPSAC counts consumed neighbours, Progressive NAPSAC counts uses of the centre; a sample drawn uniformly consumed none
        const unsigned step = a.sampler == USAC_SAMPLER_PROGRESSIVE_NAPSAC ? 1u : (unsigned)(a.m - 1);
        if (!uniform_by_now) atomicAdd(&a.cursors[pd.cursor_off + p], step);
        a.cursors[pd.cursor_off + pd.n + p] = 0u;                     // use count and first user back to zero for the next round
        a.cursors[pd.cursor_off + 2 * (size_t)pd.n + p] = 0u;
    }
}

// How many samples of this round before sample j share its seed point p (napsac_seed_kernel's use count and first user answer the
// common cases without a search)
__device__ __forceinline__ unsigned earlier_uses_in_round(const RoundArgs& a, const ProblemDesc& pd, const int* seeds, int j, int p) {
    const unsigned uses = a.cursors[pd.cursor_off + pd.n + p];
    if (uses == 2u)                                                                  // the round draws this seed twice: am I the second one?
        return ((unsigned)j > (unsigned)a.K - a.cursors[pd.cursor_off + 2 * (size_t)pd.n + p]) ? 1u : 0u;
    if (uses <= 1u) return 0u;
    unsigned earlier = 0;                                                            // rarer still: count the earlier uses within this round
    int i = 0;
    for (; i + 8 <= j; i += 8) {
        int v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = seeds[i + u];
#pragma unroll
        for (int u = 0; u < 8; u++) earlier += (v[u] == p);
    }
    for (; i < j; i++) earlier += (seeds[i] == p);
    return earlier;
}

// Progressive NAPSAC neighbourhood size for the t-th use of a centre (t >= 1): min(k, min{s >= r : C(s, r) >= t}), r = m - 1.
// PROSAC's growth rule over the centre's own distance-ordered list. C stays below t <= 2^32 until the last step, so the product
// never leaves 64 bits.
__device__ __forceinline__ int pnapsac_size(unsigned t, int r, int k) {
    int s = r;
    unsigned long long C = 1;                                                        // C(r, r)
    while (s < k && C < (unsigned long long)t) { C = C * (unsigned long long)(s + 1) / (unsigned long long)(s + 1 - r); s++; }
    return s;
}

__global__ void sample_kernel(const RoundArgs a) {
    const int slot = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.K) return;
    const int pid = a.active[slot];
    const ProblemDesc pd = a.prob[pid];
    FitState& st = a.state[pid];
    const uint64_t hyp = (a.hyp_base_p1 ? (uint64_t)(a.hyp_base_p1 - 1) : (uint64_t)st.samples_drawn) + j;
    int s[8];
    const int m = a.m, n = pd.n;
    if (a.rng == USAC_RNG_TABLE && pid == 0 && hyp < a.table_rows) {
        for (int i = 0; i < m; i++) s[i] = a.table[hyp * m + i];
    } else if (a.sampler == USAC_SAMPLER_PROSAC) {
        // prosac_sampler.hpp:117-172 replayed in closed form. Sequential rule for the call with counter t and subset
        // size n_prev: n_prev > L -> draw m from [0, L] and leave (t, n) alone; else n = n_prev + (t > g[n_prev-1]),
        // draw m-1 from [0, n-2] plus point n-1, t++. While the sampler stays in PROSAC mode t_j = t0 + j and
        // n_j = max(n0, F(t_j)), F(t) = min{n : g[n-1] >= t}; once n_prev exceeds L everything freezes.
        const unsigned* g = a.growth + pd.growth_off;
        const unsigned t0 = st.prosac_t, n0 = st.prosac_n, L = st.prosac_term_len;
        auto n_before = [&](int jj) -> unsigned { return jj == 0 ? n0 : max(n0, prosac_subset(g, n, m, t0 + jj - 1)); };
        unsigned n_prev = n_before(j);
        const bool term_mode = n_prev > L;
        unsigned t_next, n_next;
        if (term_mode) {
            int lo = 0, hi = j;                                   // first call of the round in termination mode
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (n_before(mid) > L) hi = mid; else lo = mid + 1; }
            n_prev = n_before(lo);
            philox_unique(a.seed, hyp, 2, (int)min(L + 1, (unsigned)n), m, s);          // closed range [0, L], clipped to the data
            t_next = t0 + lo; n_next = n_prev;
        } else {
            const unsigned nn = max(n0, prosac_subset(g, n, m, t0 + j));
            philox_unique(a.seed, hyp, 3, (int)nn - 1, m - 1, s);                       // closed range [0, nn-2]
            s[m - 1] = (int)nn - 1;
            t_next = t0 + j + 1; n_next = nn;
        }
        if (j == a.K - 1) { st.prosac_t_next = t_next; st.prosac_n_next = n_next; st.prosac_largest_next = max(st.prosac_largest, n_next); }
    } else if (a.sampler == USAC_SAMPLER_PROGRESSIVE_NAPSAC) {
        // DESIGN.md section 4.8: the t-th use of centre p draws from its s(t) nearest neighbours and always takes the s-th one;
        // t = uses before this round + earlier uses in this round + 1 (the sequential count, whatever the round size)
        const int* seeds = a.seeds + (size_t)slot * a.K;
        const int p = seeds[j];
        if (p < 0) {
            philox_unique(a.seed, hyp, 0, n, m, s);                                        // global phase: the uniform sampler's sample
        } else {
            const unsigned t = a.cursors[pd.cursor_off + p] + earlier_uses_in_round(a, pd, seeds, j, p) + 1u;
            const int sz = pnapsac_size(t, m - 1, pd.knn);
            const int* row = a.knn + pd.knn_off + (size_t)pd.knn * p;
            s[0] = p;
            s[m - 1] = row[sz - 1];
            if (m > 2) {
                int jj[8];
                philox_unique(a.seed, hyp, 6, sz - 1, m - 2, jj);                          // distinct ranks in [0, s-2]
                for (int i = 0; i < m - 2; i++) s[1 + i] = row[jj[i]];
            }
        }
    } else if (a.sampler == USAC_SAMPLER_NAPSAC) {
        const int* seeds = a.seeds + (size_t)slot * a.K;
        const int p = seeds[j];
        const bool uniform_by_now = a.neighbors != USAC_NEIGH_KNN && hyp >= (uint64_t)a.cursors[pd.cursor_off + 3 * (size_t)n];   // do_uniform
        if (p < 0 || uniform_by_now) {
            philox_unique(a.seed, hyp, 0, n, m, s);
        } else {
            const unsigned c = a.cursors[pd.cursor_off + p] + earlier_uses_in_round(a, pd, seeds, j, p) * (unsigned)(m - 1);
            s[0] = p;
            if (a.neighbors == USAC_NEIGH_KNN) {
                const int* row = a.knn + pd.knn_off + (size_t)pd.knn * p;
                for (int i = 1; i < m; i++) s[i] = row[pd.knn - 1 - (int)((c + i - 1) % (unsigned)pd.knn)];   // farthest first, cyclic
            } else {
                const int cell = a.cell_of_point[pd.grid_off + p];
                const int cs = a.cell_start[pd.cell_start_off + cell];
                const int cnt = a.cell_start[pd.cell_start_off + cell + 1] - cs - 1;
                const int rk = a.rank_in_cell[pd.grid_off + p];
                for (int i = 1; i < m; i++) {
                    const int pos = (int)((c + i - 1) % (unsigned)cnt);
                    s[i] = a.members[pd.grid_off + cs + pos + (pos >= rk ? 1 : 0)];       // other cell members, ascending
                }
            }
        }
    } else {
        philox_unique(a.seed, hyp, 0, n, m, s);
    }
    int* dst = a.samples + ((size_t)slot * a.K + j) * m;
    for (int i = 0; i < m; i++) dst[i] = s[i];
}

// ---------------------------------------------------------------------------------------------------------------
// Minimal solvers: one thread per sample (Estimator::EstimateModel, estimator.hpp:19)
// ---------------------------------------------------------------------------------------------------------------
// How far the sequential loop `while (iters < max_iters)` (ransac.cpp:58) can still get: max_iters - and, while max_iters is the value
// the standard criterion CAPS at (max_iterations: the initial bound, or a best model whose w^m is below 0.0005), the peak of the
// termination table, because the next better model may answer an uncapped, larger bound (found by the parity sweep: max_iterations
// 50, round size 32: the sequential loop went on to sample 61, the round had dropped samples 50..63 as out of reach).
__device__ __forceinline__ unsigned samples_in_reach(const RoundArgs& a, const ProblemDesc& pd, const FitState& st) {
    unsigned reach = st.max_iters;
    if (a.term_tables && pd.term_off >= 0 && st.max_iters == a.max_iterations) reach = max(reach, a.term_tables[pd.term_off + (size_t)pd.n + 1]);
    return reach;
}
template <int EST>
__global__ void __launch_bounds__(64) solve_kernel(const RoundArgs a) {
    const int slot = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.K) return;
    int* nm = a.nmodels + (size_t)slot * a.K + j;
    if (a.nranks > 1 && (j % a.nranks) != a.rank) { *nm = 0; return; }     // another rank's hypothesis
    const int pid = a.active[slot];
    const ProblemDesc pd = a.prob[pid];
    if (a.limit_remaining) {
        const FitState& st = a.state[pid];
        const unsigned reach = samples_in_reach(a, pd, st);
        if (reach <= st.iters || (unsigned)j >= reach - st.iters) { *nm = 0; return; }
    }
    const float* pts = a.aos + (size_t)pd.aos_off * (EST == USAC_EST_LINE2D ? 2 : 4);
    int s[8];
    const int* src = a.samples + ((size_t)slot * a.K + j) * a.m;
    for (int i = 0; i < a.m; i++) s[i] = src[i];
    float out[27];
    const int k = solve_minimal<EST>(pts, s, out);
    float* dst = a.models_raw + ((size_t)slot * a.K + j) * a.S * 9;
    for (int i = 0; i < k * 9; i++) dst[i] = out[i];
    *nm = k;
}

// Essential matrices: one WARP per sample (essential.cuh, solve_essential5_warp) - the one-thread form of the five-point solver
// is latency bound at ~3 ms per sample, the warp form spreads its independent pieces over the lanes (bit-identical results).
#define E5_WARPS_PER_CTA 4
#ifndef E5_MIN_CTAS
#define E5_MIN_CTAS 1            // resident CTAs per SM the register allocation aims at (255 registers -> 2 CTAs = 8 warps per SM)
#endif
__global__ void __launch_bounds__(32 * E5_WARPS_PER_CTA, E5_MIN_CTAS) solve_kernel_e5_warp(const RoundArgs a) {
    __shared__ double sm[E5_WARPS_PER_CTA][E5_WARP_DOUBLES];
    const int slot = blockIdx.y, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * E5_WARPS_PER_CTA + w;
    if (j >= a.K) return;                                               // whole warps leave together
    int* nm = a.nmodels + (size_t)slot * a.K + j;
    if (a.nranks > 1 && (j % a.nranks) != a.rank) { if (lane == 0) *nm = 0; return; }
    const int pid = a.active[slot];
    const ProblemDesc pd = a.prob[pid];
    if (a.limit_remaining) {
        const FitState& st = a.state[pid];
        const unsigned reach = samples_in_reach(a, pd, st);
        if (reach <= st.iters || (unsigned)j >= reach - st.iters) { if (lane == 0) *nm = 0; return; }
    }
    const float* pts = a.aos + (size_t)pd.aos_off * 4;
    int s[8];
    const int* src = a.samples + ((size_t)slot * a.K + j) * a.m;
    for (int i = 0; i < a.m; i++) s[i] = src[i];
    float* dst = a.models_raw + ((size_t)slot * a.K + j) * a.S * 9;
    const int k = solve_essential5_warp(pts, s, dst, sm[w], a.e5_all_roots);
    if (lane == 0) *nm = k;
}
// S = 1: the first valid root per sample (usac_gpu_estimate); S = USAC_E5_MAX_ROOTS with all_roots (usac_gpu_estimate_essential_roots)
__global__ void __launch_bounds__(32 * E5_WARPS_PER_CTA, E5_MIN_CTAS) estimate_kernel_e5_warp(const float* __restrict__ pts, const int* __restrict__ samples, int K,
                                                                                int S, int all_roots, float* __restrict__ models,
                                                                                int* __restrict__ nmodels) {
    __shared__ double sm[E5_WARPS_PER_CTA][E5_WARP_DOUBLES];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * E5_WARPS_PER_CTA + w;
    if (j >= K) return;
    int s[8];
    for (int i = 0; i < 5; i++) s[i] = samples[(size_t)j * 5 + i];
    float* dst = models + (size_t)j * S * 9;
    for (int i = lane; i < S * 9; i += 32) dst[i] = 0.f;
    __syncwarp();
    const int k = solve_essential5_warp(pts, s, dst, sm[w], all_roots);
    if (lane == 0) nmodels[j] = k;
}

// standalone Estimator API (usac_gpu_estimate)
template <int EST>
__global__ void __launch_bounds__(64) estimate_kernel(const float* __restrict__ pts, const int* __restrict__ samples, int K, int m, int S,
                                                     float* __restrict__ models, int* __restrict__ nmodels) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= K) return;
    int s[8];
    for (int i = 0; i < m; i++) s[i] = samples[(size_t)j * m + i];
    float out[27];
    for (int i = 0; i < 27; i++) out[i] = 0.f;
    const int k = solve_minimal<EST>(pts, s, out);
    for (int i = 0; i < S * 9; i++) models[(size_t)j * S * 9 + i] = out[i];
    nmodels[j] = k;
}

// ---------------------------------------------------------------------------------------------------------------
// prepare: compact the valid models of the round in (sample, root) order and build their scoring records
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int block_exclusive_scan(int v, int* total, int* sm /* >= 33 ints */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int w = lane < nw ? sm[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
        sm[lane] = w;
    }
    __syncthreads();
    const int before = (warp > 0 ? sm[warp - 1] : 0) + x - v;
    *total = sm[nw - 1];
    __syncthreads();
    return before;
}

__global__ void __launch_bounds__(1024) prepare_kernel(const RoundArgs a) {
    __shared__ int sm[33];
    const int slot = blockIdx.x;
    const int pid = a.active[slot];
    const ProblemDesc pd = a.prob[pid];
    const int per = (a.K + blockDim.x - 1) / blockDim.x;
    const int j0 = threadIdx.x * per, j1 = min(j0 + per, a.K);
    const int* nm = a.nmodels + (size_t)slot * a.K;
    int local = 0;
    for (int j = j0; j < j1; j++) local += nm[j];
    int total;
    int off = block_exclusive_scan(local, &total, sm);
    float rec[USAC_REC_STRIDE];
    for (int j = j0; j < j1; j++) {
        a.offsets[(size_t)slot * a.K + j] = off;
        const int k = nm[j];
        for (int i = 0; i < k; i++) {
            make_record(a.est, a.models_raw + (((size_t)slot * a.K + j) * a.S + i) * 9, a.thr, pd, rec);
            float4* dst = reinterpret_cast<float4*>(a.recs + ((size_t)slot * a.mstride + off + i) * USAC_REC_STRIDE);
#pragma unroll
            for (int w = 0; w < USAC_REC_STRIDE / 4; w++) dst[w] = make_float4(rec[4 * w], rec[4 * w + 1], rec[4 * w + 2], rec[4 * w + 3]);
        }
        off += k;
    }
    if (threadIdx.x == 0) a.mvalid[slot] = total;
    // Work items of the scoring kernel for this slot: (point chunk, group of 32 models) for the groups that exist. Fundamental
    // matrices pass the oriented-epipolar filter for a fraction of the samples only, the five-point solver returns 0 or 1 model
    // (0..10 with e5_all_roots, 0.44 per sample on C4):
    // a grid over K x S model slots would be mostly empty groups.
    if (a.items) {
        __shared__ unsigned s_base;
        const unsigned ngroups = (unsigned)(total + 31) / 32u, count = ngroups * (unsigned)a.nchunks;
        if (threadIdx.x == 0) s_base = atomicAdd(a.item_count, count);
        __syncthreads();
        for (unsigned i = threadIdx.x; i < count; i += blockDim.x)          // model group fastest: neighbouring warps share the point tiles in L2
            a.items[s_base + i] = make_uint2((unsigned)slot, ((i / ngroups) << 16) | (i % ngroups));
    }
}

// ---------------------------------------------------------------------------------------------------------------
// reduce: per-sample best score (sum the chunk partials in fixed order -> deterministic), packed for the exchange
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool score_bigger(int ca, float sa, int cb, float sb) {   // Score::bigger, quality.hpp:22-26
    return ca > cb || (ca == cb && sa > sb);
}
// Per-sample score word: the inlier count below bit midx_shift, the index of the sample's best model above it; the field's
// all-ones value marks a sample without a model. Counts of an all-roots fit are < 2^28 (usac_gpu_fit checks n).
__device__ __forceinline__ unsigned pack_cnt_midx(const RoundArgs& a, int cnt, int midx) { return (unsigned)cnt | ((unsigned)midx << a.midx_shift); }
__device__ __forceinline__ int packed_cnt(const RoundArgs& a, unsigned x) { return (int)(x & ((1u << a.midx_shift) - 1u)); }
__device__ __forceinline__ int packed_midx(const RoundArgs& a, unsigned x) { return (int)(x >> a.midx_shift); }
__device__ __forceinline__ int midx_none(const RoundArgs& a) { return (int)(0xffffffffu >> a.midx_shift); }

__global__ void reduce_kernel(const RoundArgs a) {
    const int slot = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < a.K && !(a.nranks > 1 && (j % a.nranks) != a.rank)) {
        const int k = a.nmodels[(size_t)slot * a.K + j];
        const int off = a.offsets[(size_t)slot * a.K + j];
        int bc = -1, bi = 0;
        float bs = 0.f;
        for (int i = 0; i < k; i++) {
            int c = 0;
            float s = 0.f;
            for (int ch = 0; ch < a.nchunks; ch++) {
                const size_t o = ((size_t)slot * a.nchunks + ch) * a.mstride + off + i;
                c += a.part_cnt[o];
                s += a.part_sum[o];
            }
            if (bc < 0 || score_bigger(c, s, bc, bs)) { bc = c; bs = s; bi = i; }
        }
        if (bc < 0) { bc = 0; bs = 0.f; bi = midx_none(a); }             // no model: "nothing to compare"
        const int per_rank = (a.K + a.nranks - 1) / a.nranks;
        const size_t dst = (a.nranks > 1) ? ((size_t)slot * per_rank + j / a.nranks) : ((size_t)slot * a.K + j);
        const uint2 v = make_uint2(pack_cnt_midx(a, bc, bi), __float_as_uint(bs));
        if (a.peer_win) peer_store(a, (size_t)a.rank * gridDim.y * per_rank + dst, v);
        else a.sample_scores[dst] = v;
    }
    if (a.peer_win) peer_publish(a);
}

// The same for many point chunks (one large problem: hundreds of partials per model): a CTA of 8 warps owns 32 samples
// (lane <-> sample, coalesced), warp w sums the chunks w, w+8, ... and the eight partial sums are added in warp order
// (fixed order -> deterministic). SMAX >= a.S.
template <int SMAX>
__global__ void __launch_bounds__(256) reduce_chunks_kernel(const RoundArgs a) {
    __shared__ int s_c[8][SMAX][32];
    __shared__ float s_s[8][SMAX][32];
    const int slot = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int own = blockIdx.x * 32 + lane;                            // this rank's samples, densely: j = own * nranks + rank
    const int j = a.nranks > 1 ? own * a.nranks + a.rank : own;
    const bool mine = j < a.K;
    const int k = mine ? a.nmodels[(size_t)slot * a.K + j] : 0;
    const int off = mine ? a.offsets[(size_t)slot * a.K + j] : 0;
    for (int i = 0; i < SMAX; i++) {
        int c = 0;
        float s = 0.f;
        if (i < k)
            for (int ch = warp; ch < a.nchunks; ch += 8) {
                const size_t o = ((size_t)slot * a.nchunks + ch) * a.mstride + off + i;
                c += a.part_cnt[o];
                s += a.part_sum[o];
            }
        s_c[warp][i][lane] = c;
        s_s[warp][i][lane] = s;
    }
    __syncthreads();
    if (warp == 0 && mine) {
        int bc = -1, bi = 0;
        float bs = 0.f;
        for (int i = 0; i < k; i++) {
            int c = 0;
            float s = 0.f;
            for (int w = 0; w < 8; w++) { c += s_c[w][i][lane]; s += s_s[w][i][lane]; }
            if (bc < 0 || score_bigger(c, s, bc, bs)) { bc = c; bs = s; bi = i; }
        }
        if (bc < 0) { bc = 0; bs = 0.f; bi = midx_none(a); }
        const int per_rank = (a.K + a.nranks - 1) / a.nranks;
        const size_t dst = (a.nranks > 1) ? ((size_t)slot * per_rank + own) : ((size_t)slot * a.K + j);
        const uint2 v = make_uint2(pack_cnt_midx(a, bc, bi), __float_as_uint(bs));
        if (a.peer_win) peer_store(a, (size_t)a.rank * gridDim.y * per_rank + dst, v);
        else a.sample_scores[dst] = v;
    }
    if (a.peer_win) peer_publish(a);
}

// ---------------------------------------------------------------------------------------------------------------
// select: best-update and adaptive termination with the reference's sequential semantics (ransac.cpp:58-139):
// the prefix best over the samples of the round, the first sample t at which iters reaches max_iters, the result
// as of that sample. One CTA per problem.
// ---------------------------------------------------------------------------------------------------------------
struct SelKey { unsigned long long key; int j; };
__device__ __forceinline__ SelKey sel_max(SelKey a, SelKey b) { return (b.key > a.key) ? b : a; }   // ties keep the earlier

__global__ void __launch_bounds__(256) select_kernel(const RoundArgs a, const uint2* __restrict__ scores_all) {
    __shared__ unsigned long long s_key[8];
    __shared__ int s_j[8];
    __shared__ int s_stop[8];
    __shared__ int s_T;
    __shared__ unsigned s_useful;
    const int slot = blockIdx.x;
    const int pid = a.active[slot];
    FitState& st = a.state[pid];
    if (a.peer_win) peer_wait(a);                                   // every rank's scores of this round have landed in this rank's window
    if (st.done) return;                                            // a round enqueued ahead of the host's knowledge: the fit has already ended
    const ProblemDesc pd = a.prob[pid];
    const unsigned* table = a.term_tables + pd.term_off;
    const int K = a.K, R = a.nranks;
    const int per_rank = (K + R - 1) / R;
    const uint2* sc = scores_all;
    const bool peer = a.peer_win != nullptr;
    if (peer) sc = peer_data(a.peer_self, a.peer_seq, a.peer_cap);
    auto load = [&](int j) -> uint2 {
        if (peer) return __ldcv(sc + ((size_t)(j % R) * gridDim.x + slot) * per_rank + j / R);   // written by other GPUs: never from L1
        return (R > 1) ? sc[((size_t)(j % R) * gridDim.x + slot) * per_rank + j / R] : sc[(size_t)slot * K + j];
    };
    const unsigned long long carry_key = score_key(st.best_cnt, st.best_sum);
    const unsigned iters0 = st.iters, carry_max = st.max_iters;
    const int none = midx_none(a);

    const int per = (K + blockDim.x - 1) / blockDim.x;
    const int j0 = threadIdx.x * per, j1 = min(j0 + per, K);
    SelKey mine = {0ull, -1};
    for (int j = j0; j < j1; j++) {
        const uint2 v = load(j);
        if (packed_midx(a, v.x) == none) continue;
        SelKey c = {score_key(packed_cnt(a, v.x), __uint_as_float(v.y)), j};
        mine = sel_max(mine, c);
    }
    // exclusive prefix over threads of the "leftmost maximum" (associative): shuffle scan inside each warp, then the
    // totals of the earlier warps
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    SelKey inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const SelKey left = {__shfl_up_sync(0xffffffffu, inc.key, o), __shfl_up_sync(0xffffffffu, inc.j, o)};
        if (lane >= o) inc = sel_max(left, inc);
    }
    if (lane == 31) { s_key[warp] = inc.key; s_j[warp] = inc.j; }
    __syncthreads();
    SelKey run = {carry_key, -1};
    for (int w = 0; w < warp; w++) { const SelKey c = {s_key[w], s_j[w]}; run = sel_max(run, c); }
    {
        const SelKey excl = {__shfl_up_sync(0xffffffffu, inc.key, 1), __shfl_up_sync(0xffffffffu, inc.j, 1)};
        if (lane > 0) run = sel_max(run, excl);
    }
    // walk own samples with the running prefix best; find the first sample at which the loop condition fails
    int stop = K;           // K = no stop in my range
    SelKey at_stop = run;
    for (int j = j0; j < j1; j++) {
        const uint2 v = load(j);
        if (packed_midx(a, v.x) != none) { SelKey c = {score_key(packed_cnt(a, v.x), __uint_as_float(v.y)), j}; run = sel_max(run, c); }
        const unsigned mi = (run.j < 0) ? carry_max : table[(unsigned)(run.key >> 32)];
        if (iters0 + (unsigned)j + 1u >= mi) { stop = j; at_stop = run; break; }
    }
    {
        int wmin = stop;
#pragma unroll
        for (int o = 16; o; o >>= 1) wmin = min(wmin, __shfl_xor_sync(0xffffffffu, wmin, o));
        if (lane == 0) s_stop[warp] = wmin;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int T = K;
        for (int t = 0; t < (int)(blockDim.x >> 5); t++) T = min(T, s_stop[t]);
        s_T = T;
        s_useful = 0;
    }
    __syncthreads();
    const int T = s_T;
    {   // models this rank scored for samples 0..T: what the sequential loop would have evaluated too
        unsigned u = 0;
        const int* nmod = a.nmodels + (size_t)slot * K;
        for (int j = j0; j < j1 && j <= T; j++) u += (unsigned)nmod[j];
        if (u) atomicAdd(&s_useful, u);
    }
    __syncthreads();
    // the owner of T (or the last thread when the round did not terminate) publishes the result
    const bool owner = (T < K) ? (stop == T) : (threadIdx.x == blockDim.x - 1);
    if (owner) {
        const SelKey best = (T < K) ? at_stop : run;
        if (best.j >= 0) {
            const uint2 v = load(best.j);
            st.best_cnt = packed_cnt(a, v.x);
            st.best_sum = __uint_as_float(v.y);
            st.best_hyp = (long long)st.samples_drawn + best.j;
            st.best_midx = packed_midx(a, v.x);
            st.max_iters = table[(unsigned)st.best_cnt];
        }
        st.iters = iters0 + (unsigned)min(T + 1, K);
        st.done = (T < K) || !(st.iters < st.max_iters);
        st.samples_drawn += (unsigned)K;
        st.rounds += 1;
        st.round_pending = 1;                                       // winner_kernel finishes this round
        st.useful_evals += (unsigned long long)s_useful * (unsigned long long)pd.n;
    }
}

// Round epilogue, one thread per problem: the winning model is re-derived from its sample (the solvers are
// deterministic), so no model has to travel between ranks; sampler state of the round is committed.
template <int EST>
__global__ void winner_kernel(const RoundArgs a, int slots) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= slots) return;
    const int pid = a.active[slot];
    FitState& st = a.state[pid];
    if (!st.round_pending) { if (a.done_out) a.done_out[slot] = st.done; return; }   // round enqueued after the fit had ended: select_kernel skipped it
    st.round_pending = 0;
    const ProblemDesc pd = a.prob[pid];
    const long long first = (long long)st.samples_drawn - a.K;       // select_kernel already advanced samples_drawn
    if (st.best_hyp >= first) {
        const int j = (int)(st.best_hyp - first);
        const int w = EST == USAC_EST_LINE2D ? 3 : 9;
        if (a.nranks == 1 || (j % a.nranks) == a.rank) {            // this rank solved the sample: the model is in HBM
            const float* src = a.models_raw + (((size_t)slot * a.K + j) * a.S + st.best_midx) * 9;
            for (int i = 0; i < w; i++) st.best_model[i] = src[i];
        } else {                                                    // another rank's sample: re-derive (deterministic solver)
            int s[8];
            const int* src = a.samples + ((size_t)slot * a.K + j) * a.m;
            for (int i = 0; i < a.m; i++) s[i] = src[i];
            float out[EST == USAC_EST_ESSENTIAL ? 9 * USAC_E5_MAX_ROOTS : 27];
            const float* pts = a.aos + (size_t)pd.aos_off * (EST == USAC_EST_LINE2D ? 2 : 4);
            const int k = solve_minimal<EST>(pts, s, out, a.e5_all_roots);
            if (st.best_midx < k) for (int i = 0; i < w; i++) st.best_model[i] = out[9 * st.best_midx + i];
        }
    }
    if (a.done_out) a.done_out[slot] = st.done;
    st.evals += (unsigned long long)a.mvalid[slot] * (unsigned long long)pd.n;
    st.prosac_t = st.prosac_t_next; st.prosac_n = st.prosac_n_next; st.prosac_largest = st.prosac_largest_next;
}
