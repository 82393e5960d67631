// score_sq.cuh - the scoring kernel for homography / fundamental / essential models: a division-free rejection test in the
// hot loop, and a per-warp SURVIVOR QUEUE for everything it cannot reject.
//
// Replaces Quality::getNumberInliers (quality.hpp:60-101) looping the virtual Estimator::GetError.
//
// Observation (ncu, profiles/r2_*): for the models a RANSAC round produces, more than 99 % of the (model, point)
// evaluations are outliers that a cheap one-sided test proves to be outliers (FastModel<EST>::reject: 9 - 18 packed FP32x2
// instructions per pair of points, no MUFU, no division), yet in the round-1 kernel one surviving evaluation out of the 64 of
// a (warp, point pair) sent the whole warp through the second phase (8 MUFU + ~30 more instructions; 45 % of the kernel's
// time for the homography, and a warp-wide exit from the loop whenever a value fell inside the guard band). Here the hot
// loop does nothing but the rejection test. A lane whose point is NOT a proven outlier appends the point index to ITS OWN
// queue in shared memory (USAC_SQ_LANE_CAP entries per lane, stored lane-interleaved so the stores never conflict): one
// predicated store and one predicated pointer increment per value, no cross-lane dependency (one vote per trip skips even
// that when no lane has a survivor, the common case for homographies) - and the loop goes on. When some lane's queue could
// overflow during the next trip (and at the end of the work item) the warp drains all 32
// queues together: a warp scan of the per-lane counts turns them into one dense list, processed 32 entries at a time, every
// lane evaluating one (model, point) pair of the queue with the REFERENCE'S EXACT ARITHMETIC (strict_error<EST>: one
// rounding per operator, IEEE division and square root), reading the model record of the owning lane from L1. The inlier
// count is therefore exact by construction (the only approximation is one-sided: `reject` may only claim an outlier when the
// guard-band analysis of pipeline.cuh proves it), there is no second fast evaluator and no band test on the accept side.
// The error sum is accumulated in fixed point (err / thr in units of 2^-36): the drain adds the 14 high and 22 low bits with
// native 32-bit shared-memory atomics, and after every drain each lane folds its own model's partials into a 64-bit register.
// Integer sums are order independent, hence deterministic, and closer to the real sum than the reference's sequential float sum.
#pragma once
#include "score.cuh"

// Tuning knobs (A/B on one box, profiles/README.md): the trip-level vote pays for homographies (63 % of the trips have no survivor
// in the whole warp) and costs for the epipolar metrics (a third of the trips); drawing the next work item one item ahead
// was slower than drawing it when needed.
#ifndef USAC_SQ_TRIPVOTE
#define USAC_SQ_TRIPVOTE 2                 // 0: never, 1: always, 2: homography only - one vote per trip skips the pushes when no lane has a survivor
#endif
#ifndef USAC_SQ_PREFETCH
#define USAC_SQ_PREFETCH 0                 // 1: the next work item is drawn one item ahead
#endif
#define USAC_SQ_LANE_CAP 16                // queue entries per lane (a trip of USAC_PPI pairs pushes at most 2 * USAC_PPI per lane)
#define USAC_SQ_FIXED_BITS 36
#define USAC_SQ_LO_BITS 22                 // a drain handles <= 32 * USAC_SQ_LANE_CAP entries: 512 * 2^22 and 512 * 2^14 both fit 32 bits

// append `entry` to this lane's queue when `pred` holds (predicated store + predicated pointer increment; the slots of a lane
// are 128 bytes apart). No memory clobber on purpose: the tile loads of the other instruction streams may move across it; the
// queue is only read by sq_drain, behind a compiler barrier.
__device__ __forceinline__ void sq_push(bool pred, uint32_t& qaddr, uint32_t entry) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %1, 0;\n\t"
        "@p st.shared.u32 [%0], %2;\n\t"
        "@p add.u32 %0, %0, 128;\n\t}"
        : "+r"(qaddr)
        : "r"((uint32_t)pred), "r"(entry));
}

// Drain: lane l holds cnt entries q[k * 32 + l], k < cnt. The 32 lists are processed as one dense list, 32 entries at a time.
template <int EST>
__device__ __noinline__ void sq_drain(const uint32_t* __restrict__ q, uint32_t cnt, uint32_t* pre, const float* __restrict__ recs_group,
                                      const float* __restrict__ aos, int n, double scale, uint32_t* mcnt, uint32_t* mlo, uint32_t* mhi) {
    const int lane = threadIdx.x & 31;
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    pre[lane] = incl - cnt;                                            // exclusive prefix: first dense position of lane's entries
    __syncwarp();
    // two batches of 32 entries per trip: their point / record loads (L2 / L1 latency) are in flight together
    for (uint32_t base = 0; base < total; base += 64) {
        int l[2], idx[2];
        bool on[2];
        float4 p[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t t = base + 32u * h + lane;
            on[h] = t < total;
            l[h] = 0; idx[h] = 0;
            if (on[h]) {
                int ll = 0;                                            // owner: the largest l with pre[l] <= t
#pragma unroll
                for (int step = 16; step; step >>= 1) if (pre[ll + step] <= t) ll += step;
                l[h] = ll;
                idx[h] = (int)q[(t - pre[ll]) * 32 + ll];
                on[h] = idx[h] < n;                                    // NaN padding of an odd point count
            }
            p[h] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (on[h]) {
                if (EST == USAC_EST_LINE2D) { const float2 v = reinterpret_cast<const float2*>(aos)[idx[h]]; p[h] = make_float4(v.x, v.y, 0.f, 0.f); }
                else p[h] = reinterpret_cast<const float4*>(aos)[idx[h]];
            }
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if (!on[h]) continue;
            const float* rec = recs_group + (size_t)l[h] * USAC_REC_STRIDE;
            const float err = strict_error<EST>(rec, p[h].x, p[h].y, p[h].z, p[h].w);
            if (err < rec[REC_THR]) {                                  // quality.hpp:90-94, strict `<`, NaN is an outlier
                const unsigned long long fix = __double2ull_rn((double)err * scale);
                atomicAdd(&mcnt[l[h]], 1u);
                atomicAdd(&mlo[l[h]], (uint32_t)(fix & ((1u << USAC_SQ_LO_BITS) - 1u)));
                atomicAdd(&mhi[l[h]], (uint32_t)(fix >> USAC_SQ_LO_BITS));
            }
        }
    }
}

template <int EST>
__global__ void __launch_bounds__(USAC_SCORE_THREADS, USAC_SQ_MIN_CTAS) score_sq_kernel(const ScoreArgs a) {
    constexpr int PAIR_FLOATS = (EST == USAC_EST_LINE2D) ? 4 : 8;
    constexpr int NWARPS = USAC_SCORE_THREADS / 32;
    static_assert(USAC_SQ_LANE_CAP >= 4 * USAC_PPI, "a lane's queue must hold two trips of pushes");
    __shared__ __align__(128) float tile_all[NWARPS][USAC_WARP_STAGES][USAC_TILE_PAIRS * PAIR_FLOATS];
    __shared__ __align__(8) uint64_t full_all[NWARPS][USAC_WARP_STAGES];
    __shared__ __align__(128) uint32_t queue_all[NWARPS][USAC_SQ_LANE_CAP * 32];
    __shared__ uint32_t macc_all[NWARPS][4][32];                    // per model of the warp: inlier count, low / high part of the error sum; [3] = scan scratch

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float (*tile)[USAC_TILE_PAIRS * PAIR_FLOATS] = tile_all[warp];
    uint64_t* full = full_all[warp];
    uint32_t* queue = queue_all[warp];
    uint32_t* mcnt = macc_all[warp][0];
    uint32_t* mlo = macc_all[warp][1];
    uint32_t* mhi = macc_all[warp][2];
    uint32_t* pre = macc_all[warp][3];
    const uint32_t q_first = smem_u32(queue) + 4u * (uint32_t)lane;                          // this lane's slot 0
    const uint32_t q_limit = q_first + 128u * (USAC_SQ_LANE_CAP - 2 * USAC_PPI);             // beyond this a trip of pushes might not fit
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < USAC_WARP_STAGES; s++) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();

    const int mgroups = a.mblocks * NWARPS;
    const unsigned total = a.items ? *a.item_count : (unsigned)a.slots * (unsigned)a.nchunks * (unsigned)mgroups;
    uint32_t g = 0;                                                  // tiles consumed so far by this warp (uniform)

    unsigned pending = 0;                                            // lane 0: the next work item, drawn one item ahead so that the
    if (USAC_SQ_PREFETCH && lane == 0) pending = atomicAdd(a.work, 1u) - a.work_base;    // round trip of the atomic hides behind the current item
    for (;;) {
        if (!USAC_SQ_PREFETCH && lane == 0) pending = atomicAdd(a.work, 1u) - a.work_base;
        const unsigned item = __shfl_sync(0xffffffffu, pending, 0);
        int slot, chunk, mgroup;
        if (!score_item(a, item, total, mgroups, slot, chunk, mgroup)) break;
        if (USAC_SQ_PREFETCH && lane == 0) pending = atomicAdd(a.work, 1u) - a.work_base;   // every warp overdraws exactly once (accounted by the host)
        const int M = a.mvalid ? a.mvalid[slot] : a.M;
        if (mgroup * 32 >= M) continue;                              // uniform per warp
        const ProblemDesc pd = a.prob[a.active ? a.active[slot] : slot];
        const int m = mgroup * 32 + lane;
        const bool live = m < M;
        const float* recs_group = a.recs + ((size_t)slot * a.mstride + (size_t)mgroup * 32) * USAC_REC_STRIDE;
        const float* rec = recs_group + (size_t)(live ? lane : 0) * USAC_REC_STRIDE;
        const size_t out = ((size_t)slot * a.nchunks + chunk) * a.mstride + m;

        const int pair_begin = chunk * a.chunk_pairs;
        const int npairs = min(pair_begin + a.chunk_pairs, pd.n_pairs) - pair_begin;
        if (npairs <= 0) {                                           // ragged batch: this problem is shorter than the chunk grid
            if (live) { a.part_cnt[out] = 0; a.part_sum[out] = 0.f; }
            continue;
        }
        const int ntiles = (npairs + USAC_TILE_PAIRS - 1) / USAC_TILE_PAIRS;
        const float* src = a.pairs + ((size_t)pd.pair_off + pair_begin) * PAIR_FLOATS;

        if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the stages were last read through the generic proxy
            for (int k = 0; k < USAC_WARP_STAGES && k < ntiles; k++) {
                const int s = (g + k) % USAC_WARP_STAGES;
                const uint32_t bytes = min(USAC_TILE_PAIRS, npairs - k * USAC_TILE_PAIRS) * PAIR_FLOATS * 4;
                mbar_expect_tx(&full[s], bytes);
                bulk_copy_g2s(tile[s], src + (size_t)k * USAC_TILE_PAIRS * PAIR_FLOATS, bytes, &full[s]);
            }
        }
        mcnt[lane] = 0u; mlo[lane] = 0u; mhi[lane] = 0u;
        uint32_t acc_cnt = 0;                                        // this lane's model: totals of the drains so far
        unsigned long long acc_sum = 0;
        __syncwarp();

        FastModel<EST> fm;
        fm.load(rec);
        const float thr = rec[REC_THR];
        const double scale = (double)(1ull << USAC_SQ_FIXED_BITS) / (double)thr;
        const float* aos = a.aos + (size_t)pd.aos_off * (EST == USAC_EST_LINE2D ? 2 : 4);
        uint32_t qaddr = q_first;                                    // shared-space address of this lane's next free slot

        // drain the queues and fold this lane's partials (its own slots of the shared arrays) into its registers
        auto drain = [&]() {
            asm volatile("" ::: "memory");
            __syncwarp();
            sq_drain<EST>(queue, (qaddr - q_first) >> 7, pre, recs_group, aos, pd.n, scale, mcnt, mlo, mhi);
            __syncwarp();
            acc_cnt += mcnt[lane];
            acc_sum += ((unsigned long long)mhi[lane] << USAC_SQ_LO_BITS) + mlo[lane];
            mcnt[lane] = 0u; mlo[lane] = 0u; mhi[lane] = 0u;
            qaddr = q_first;
            __syncwarp();
        };

        for (int k = 0; k < ntiles; k++) {
            const int s = (g + k) % USAC_WARP_STAGES;
            mbar_wait(&full[s], ((g + k) / USAC_WARP_STAGES) & 1);
            const int np = min(USAC_TILE_PAIRS, npairs - k * USAC_TILE_PAIRS);
            const float4* tp = reinterpret_cast<const float4*>(tile[s]);
            uint32_t ebase = (uint32_t)(2 * (pair_begin + k * USAC_TILE_PAIRS));   // index of the first point of the trip within the problem
            auto load_pair = [&](int j, float4& A, float4& B) {
                if (EST == USAC_EST_LINE2D) { A = tp[j]; B = A; }
                else { A = tp[2 * j]; B = tp[2 * j + 1]; }
            };
            int j = 0;
#pragma unroll 1
            for (; j + USAC_PPI <= np; j += USAC_PPI) {
                float2 z[USAC_PPI], zb[USAC_PPI];                                   // proven outlier <=> z > zb
#pragma unroll
                for (int q = 0; q < USAC_PPI; q++) {                               // independent instruction streams
                    float4 A, B;
                    load_pair(j + q, A, B);
                    z[q] = fm.reject(A, B, zb[q]);
                }
                bool lane_any = false;
#pragma unroll
                for (int q = 0; q < USAC_PPI; q++) lane_any = lane_any || !(z[q].x > zb[q].x) || !(z[q].y > zb[q].y);
                // one vote for the whole trip: in most trips every point is a proven outlier for every model of the warp
                if (!USAC_SQ_TRIPVOTE || (EST != USAC_EST_HOMOGRAPHY && USAC_SQ_TRIPVOTE == 2) || __any_sync(0xffffffffu, lane_any && live)) {
#pragma unroll
                    for (int q = 0; q < USAC_PPI; q++) {                           // everything that is not a proven outlier goes to the queue
                        sq_push(!(z[q].x > zb[q].x) && live, qaddr, ebase + 2 * q);
                        sq_push(!(z[q].y > zb[q].y) && live, qaddr, ebase + 2 * q + 1);
                    }
                    if (__any_sync(0xffffffffu, qaddr > q_limit)) drain();           // rare: some lane's queue is nearly full
                }
                ebase += 2 * USAC_PPI;
            }
            if (j < np) {                                                           // tail of the tile: fewer than USAC_PPI pairs
                const int rest = np - j;
#pragma unroll
                for (int q = 0; q < USAC_PPI; q++) {
                    if (q < rest) {
                        float4 A, B;
                        load_pair(j + q, A, B);
                        float2 zb;
                        const float2 z = fm.reject(A, B, zb);
                        sq_push(!(z.x > zb.x) && live, qaddr, ebase + 2 * q);
                        sq_push(!(z.y > zb.y) && live, qaddr, ebase + 2 * q + 1);
                    }
                }
                if (__any_sync(0xffffffffu, qaddr > q_limit)) drain();
            }
            // every lane is done with the stage: re-arm it and fetch the tile USAC_WARP_STAGES ahead
            __syncwarp();
            if (lane == 0 && k + USAC_WARP_STAGES < ntiles) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                const int nk = k + USAC_WARP_STAGES;
                const uint32_t bytes = min(USAC_TILE_PAIRS, npairs - nk * USAC_TILE_PAIRS) * PAIR_FLOATS * 4;
                mbar_expect_tx(&full[s], bytes);
                bulk_copy_g2s(tile[s], src + (size_t)nk * USAC_TILE_PAIRS * PAIR_FLOATS, bytes, &full[s]);
            }
        }
        g += (uint32_t)ntiles;
        if (__any_sync(0xffffffffu, qaddr != q_first)) drain();
        if (live) {
            a.part_cnt[out] = (int)acc_cnt;
            a.part_sum[out] = (float)((double)acc_sum / scale);
        }
        __syncwarp();                                                // all lanes left the item before its stages are refilled
    }
}
