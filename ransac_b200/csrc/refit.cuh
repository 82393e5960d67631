// refit.cuh - non-minimal estimation on a list of point ids (Estimator::EstimateModelNonMinimalSample) for the final refit
// of Ransac::run (ransac.cpp:157-207):
//   homography   homography_estimator.hpp:67-75 -> DLt::NormalizedDLT (dlt/normalized_dlt.cpp:7-23, dlt/dlt.cpp:55-101)
//   fundamental  fundamental_estimator.hpp:65-75 -> EightPointsAlgorithm (fundamental/eight_points.cpp:4-100)
//   essential    essential_estimator.hpp:64-74 (the same eight-point solver)
//   line2d       line2d_estimator.hpp:59-106 (PCA)
// with GetNormalizingTransformation (dlt/normalizing_transformation.cpp:7-112).
//
// The kernel is the CTA-wide form in lo.cuh (cta_nonminimal, nonminimal_cta_kernel); this file holds its building blocks. Every
// sum over the points is a "lane sum": virtual lane l (of 256) adds elements l, l+256, ... in order, then the 256 partials are
// combined by a fixed binary tree (stride 128 ... 1) - the host restatement used by the parity
// tests adds in exactly this order, so the models are bit-identical. A is formed in float like the reference, A'A (45 unique
// entries) is accumulated in double, and the null vector is the eigenvector of its smallest eigenvalue (cyclic Jacobi sweeps, at most 12, ended by the first sweep without a rotation) instead of cv::SVD on A. All arithmetic strict (no FMA contraction).
#pragma once
#include "strict_math.cuh"

#define REFIT_THREADS 256

// Eigenvector of the smallest eigenvalue of the symmetric n x n matrix S (n odd, <= 9; S, V in shared memory): at most 12 Jacobi
// sweeps in the round-robin order, executed by the first warp. Round r rotates the (n-1)/2 disjoint pairs {(r+k) mod n, (r-k) mod n}:
// their angles are computed side by side (one lane each) from the matrix at the start of the round, then lane (pair, k) updates
// element k of the pair's two columns, then of its two rows and of V - 9 dependent steps per sweep instead of 36 (the angle is
// a chain of three divisions and two square roots in double). Every element sees exactly the operations of the sequential loops
// of the host restatement, which uses the same round order.
__device__ void refit_smallest_eigenvector_warp(double* S, int n, double* vec, double* V) {
    const int lane = threadIdx.x & 31;
    const int half = (n - 1) / 2;                                        // n odd (9): disjoint pairs per round
    for (int i = lane; i < n * n; i += 32) V[i] = (i / n == i % n) ? 1.0 : 0.0;
    __syncwarp();
    for (int sweep = 0; sweep < 12; sweep++) {
        int rotations = 0;                                               // a sweep without a rotation: converged (uniform over the warp)
        for (int r = 0; r < n; r++) {
            // lane e < half computes the angle of pair e of this round from the matrix as it stands
            int p = 0, q = 0;
            double c = 1.0, s = 0.0;
            bool on = false;
            if (lane < half) {
                p = (r + lane + 1) % n; q = (r - lane - 1 + n) % n;
                if (p > q) { const int t = p; p = q; q = t; }
                const sd apq(S[p * n + q]);
                const sd big(fmax(fabs(S[p * n + p]), fabs(S[q * n + q])));       // |apq| <= 1e-12 max(|app|, |aqq|): enough for the eigenvector
                if (apq.v != 0.0 && !((apq * apq).v <= (sd(1e-24) * (big * big)).v)) {
                    // t = sgn(d) b / (|d| + sqrt(d^2 + b^2)), c = sqrt(w) (1 / w), w = t^2 + 1: three dependent div / sqrt, not five
                    const sd d = sd(S[q * n + q]) - sd(S[p * n + p]), b = sd(2.0) * apq;
                    const sd rr = dsqrt(d * d + b * b);
                    const sd t0 = b / (sd(fabs(d.v)) + rr);
                    const sd t = d.v < 0.0 ? -t0 : t0;
                    const sd w = t * t + sd(1.0);
                    const sd cc = dsqrt(w) * (sd(1.0) / w), ss = t * cc;
                    if (dfinite(cc.v) && dfinite(ss.v)) { c = cc.v; s = ss.v; on = true; }
                }
            }
            const unsigned live = __ballot_sync(0xffffffffu, on);
            __syncwarp();                                                // every angle has been computed from the old matrix
            rotations += __popc(live);
            if (!live) continue;                                         // uniform
            // element updates: lane = (pair e, index k), half * n of them in passes of the whole warp
            for (int base = 0; base < half * n; base += 32) {            // columns p, q of S
                const int w = base + lane;
                const bool act = w < half * n;
                const int e = act ? w / n : 0, k = act ? w % n : 0;
                const int pe = __shfl_sync(0xffffffffu, p, e), qe = __shfl_sync(0xffffffffu, q, e);
                const double ce = __shfl_sync(0xffffffffu, c, e), se = __shfl_sync(0xffffffffu, s, e);
                if (act && ((live >> e) & 1u)) {
                    const sd a(S[k * n + pe]), b(S[k * n + qe]);
                    S[k * n + pe] = (sd(ce) * a - sd(se) * b).v;
                    S[k * n + qe] = (sd(se) * a + sd(ce) * b).v;
                }
            }
            __syncwarp();
            for (int base = 0; base < half * n; base += 32) {            // rows p, q of S; columns p, q of V
                const int w = base + lane;
                const bool act = w < half * n;
                const int e = act ? w / n : 0, k = act ? w % n : 0;
                const int pe = __shfl_sync(0xffffffffu, p, e), qe = __shfl_sync(0xffffffffu, q, e);
                const double ce = __shfl_sync(0xffffffffu, c, e), se = __shfl_sync(0xffffffffu, s, e);
                if (act && ((live >> e) & 1u)) {
                    const sd a(S[pe * n + k]), b(S[qe * n + k]);
                    S[pe * n + k] = (sd(ce) * a - sd(se) * b).v;
                    S[qe * n + k] = (sd(se) * a + sd(ce) * b).v;
                    const sd va(V[k * n + pe]), vb(V[k * n + qe]);
                    V[k * n + pe] = (sd(ce) * va - sd(se) * vb).v;
                    V[k * n + qe] = (sd(se) * va + sd(ce) * vb).v;
                }
            }
            __syncwarp();
        }
        if (!rotations) break;
    }
    int best = 0;
    for (int i = 1; i < n; i++) if (S[i * n + i] < S[best * n + best]) best = i;
    if (lane < n) vec[lane] = V[lane * n + best];
    __syncwarp();
}

// Line2d non-minimal fit (line2d_estimator.hpp:59-106) from the five lane sums r = (x, y, xy, xx, yy) of n points: mean, scatter,
// the eigenvector of the scatter's smaller eigenvalue (closed form in double) as the normal (A, B), c = -A mx - B my -> model[0..2].
// Returns whether all three are finite. Every operation is one rounding, in the order of the host restatement the tests use.
__device__ __forceinline__ bool line_from_sums(const float* r, int n, float* model) {
    const sf sx(r[0]), sy(r[1]), sxy(r[2]), sx2(r[3]), sy2(r[4]), N((float)n);
    const sf mx = sx / N, my = sy / N;
    const sf c00 = sx2 - sf(2.f) * sx * mx + N * mx * mx;
    const sf c01 = sxy - sx * my - sy * mx + N * mx * my;
    const sf c11 = sy2 - sf(2.f) * sy * my + N * my * my;
    const sd p((double)c00.v), q((double)c01.v), rr((double)c11.v);
    const sd half = sd(0.5) * (p - rr), rad = dsqrt(half * half + q * q), lam = sd(0.5) * (p + rr) - rad;
    sd vx = q, vy = lam - p;
    const sd wx = lam - rr, wy = q;
    if ((wx * wx + wy * wy).v > (vx * vx + vy * vy).v) { vx = wx; vy = wy; }
    const sd nn = dsqrt(vx * vx + vy * vy);
    if (!(nn.v > 0.0)) { vx = sd(1.0); vy = sd(0.0); } else { vx = vx / nn; vy = vy / nn; }
    const sf A((float)vx.v), B((float)vy.v);
    const float c = (-A * mx - B * my).v;
    model[0] = A.v; model[1] = B.v; model[2] = c;
    return isfinite(A.v) && isfinite(B.v) && isfinite(c);
}
