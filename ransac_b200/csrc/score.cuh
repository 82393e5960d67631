// score.cuh - the fused scoring kernel: M models x N points -> (inlier count, error sum) per model.
//
// Replaces Quality::getNumberInliers (quality.hpp:60-101) looping the virtual Estimator::GetError.
//
// Mapping: one thread owns one model (register resident); a warp of 32 models walks a chunk of the point set that is
// staged through the warp's own shared-memory ring in tiles of USAC_TILE_PAIRS point pairs by 1-D bulk async copies
// (cp.async.bulk -> UBLKCP, completion on an mbarrier), USAC_WARP_STAGES deep. Points are stored pair-interleaved ([x1a x1b y1a y1b x2a x2b y2a y2b] per pair) so that one broadcast
// LDS.128 feeds two points straight into the packed FP32x2 pipe (FFMA2/FMUL2/FADD2, sm_100): the residual costs ~28
// packed instructions per pair for a homography, which makes the kernel FMA-pipe bound rather than issue bound.
//
// Exactness: the packed path uses FMA contraction and approximate MUFU rcp/sqrt, so its error value differs from the
// reference's one-rounding-per-operator float32 value in the low bits. Each model record carries a rigorous bound on
// that difference (prepare_kernel, "guard band"); a point whose fast value is closer to the threshold than the bound
// is re-evaluated with strict_error<EST>() - the reference's exact arithmetic - so the inlier COUNT is bit-exact. The
// error SUM is accumulated from the fast values (tolerance 1e-4 relative, BASELINE.json).
#pragma once
#include "strict_math.cuh"

__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_sqrt(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_rsqrt(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float2 dup(float x) { return make_float2(x, x); }   // folds into the scalar-broadcast operand form of FFMA2
// max(|a|, |b|), NaN if either is NaN (fmaxf would return the other operand): one FMNMX.NAN with |.| operands on the ALU pipe
__device__ __forceinline__ float abs_max_nan(float a, float b) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(fabsf(a)), "f"(fabsf(b))); return r; }

// ---- mbarrier / bulk-copy helpers (PTX ISA 8.x, sm_90+) ---------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- per-estimator fast evaluators --------------------------------------------------------------------------------
// eval(): given one pair of points returns, per lane,
//   t   : decision value, t < 0 <=> inlier by the fast path (homography/essential: 2*err - 2*thr, fundamental:
//         n^2 - thr*den, line: err - thr);
//   s   : guard band (>= 0): the fast decision is trusted only when |t| > s, otherwise the point is re-evaluated with
//         the reference's exact arithmetic (strict_em);
//   w   : (fundamental only) 1/den, so that min(t,0)*w = err - thr.
// The kernel accumulates em = min(t, 0) [* w] (NaN-safe: fminf drops a NaN) and counts its sign bits; finish() turns
// (sum of em, count) into the reference's error sum of the inliers.

template <int EST> struct FastModel;

template <> struct FastModel<USAC_EST_HOMOGRAPHY> {
    static constexpr bool WEIGHTED = false;
    // rows 0,1 negated so that dx = x2 - nx/nz is a single FFMA2; scalars are broadcast by the FFMA2 operand form
    float a11, a12, a13, a21, a22, a23, h31, h32, h33;
    float b11, b12, b13, b21, b22, b23, g31, g32, g33;
    float negT, k1, k2;
    __device__ __forceinline__ void load(const float* r) {
        a11 = -r[0]; a12 = -r[1]; a13 = -r[2]; a21 = -r[3]; a22 = -r[4]; a23 = -r[5]; h31 = r[6]; h32 = r[7]; h33 = r[8];
        b11 = -r[9]; b12 = -r[10]; b13 = -r[11]; b21 = -r[12]; b22 = -r[13]; b23 = -r[14]; g31 = r[15]; g32 = r[16]; g33 = r[17];
        negT = -2.f * r[REC_THR]; k1 = r[REC_BAND]; k2 = r[REC_BAND + 1];
        T2p = 2.f * r[REC_THR] * 1.0000019f;
    }
    // Two phases. The symmetric transfer error is (d1 + d2)/2 with d1, d2 >= 0, so a point whose FORWARD distance alone
    // exceeds 2*thr by more than the forward guard band is an outlier whatever the backward distance is (also when the
    // backward term is NaN: the reference's sum is then NaN and fails `err < thr` as well). phase1 decides that without a
    // division or a square root, on the distance scaled by nz:
    //     d1 > 2 thr + k1/|nz|   <=>   (x2 nz - nx)^2 + (y2 nz - ny)^2 > (2 thr |nz| + k1)^2
    // (12 packed FMA-pipe instructions, no MUFU). The rounding error of the left-hand side is smaller than that of the
    // quotient form the band k1 was derived for (one rounding of x2*nz - nx instead of product, rcp.approx, product), and
    // T2p = 2 thr (1 + 2^-19) absorbs the roundings of the comparison itself. The kernel runs phase2 (d1 itself and the
    // backward half, all 8 MUFU) only for the pairs of points on which some lane of the warp still needs it - for the
    // random-sample hypotheses of a RANSAC round that is a small minority.
    static constexpr bool TWO_PHASE = true;
    float T2p;
    struct P1 { float2 sa, nz; };                                          // sa = (d1 nz)^2
    __device__ __forceinline__ void phase1(const float4 A, const float4 B, P1& s) const {
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 nz = __ffma2_rn(dup(h31), X1, __ffma2_rn(dup(h32), Y1, dup(h33)));
        const float2 nx = __ffma2_rn(dup(a11), X1, __ffma2_rn(dup(a12), Y1, dup(a13)));   // -(h11 x1 + h12 y1 + h13)
        const float2 ny = __ffma2_rn(dup(a21), X1, __ffma2_rn(dup(a22), Y1, dup(a23)));
        const float2 ax = __ffma2_rn(X2, nz, nx), ay = __ffma2_rn(Y2, nz, ny);           // nz * (x2 - nx/nz)
        s.sa = __ffma2_rn(ay, ay, __fmul2_rn(ax, ax));
        s.nz = nz;
    }
    __device__ __forceinline__ void sure(const P1& s, bool& ox, bool& oy) const {       // false for NaN
        const float2 az = make_float2(fabsf(s.nz.x), fabsf(s.nz.y));
        const float2 c = __ffma2_rn(dup(T2p), az, dup(k1));
        const float2 c2 = __fmul2_rn(c, c);
        ox = s.sa.x > c2.x; oy = s.sa.y > c2.y;
    }
    __device__ __forceinline__ void phase2(const float4 A, const float4 B, const P1& s, float2& t, float2& band) const {
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 r1 = make_float2(fabsf(fast_rcp(s.nz.x)), fabsf(fast_rcp(s.nz.y)));
        const float2 d1 = __fmul2_rn(make_float2(fast_sqrt(s.sa.x), fast_sqrt(s.sa.y)), r1);
        const float2 mz = __ffma2_rn(dup(g31), X2, __ffma2_rn(dup(g32), Y2, dup(g33)));
        const float2 mx = __ffma2_rn(dup(b11), X2, __ffma2_rn(dup(b12), Y2, dup(b13)));
        const float2 my = __ffma2_rn(dup(b21), X2, __ffma2_rn(dup(b22), Y2, dup(b23)));
        const float2 r2 = make_float2(fast_rcp(mz.x), fast_rcp(mz.y));
        const float2 ex = __ffma2_rn(mx, r2, X1), ey = __ffma2_rn(my, r2, Y1);
        const float2 sb = __ffma2_rn(ey, ey, __fmul2_rn(ex, ex));
        const float2 d2 = make_float2(fast_sqrt(sb.x), fast_sqrt(sb.y));
        t = __fadd2_rn(__fadd2_rn(d1, dup(negT)), d2);                     // 2*err - 2*thr
        const float2 p2 = __fmul2_rn(dup(k2), r2);
        band = __ffma2_rn(dup(k1), r1, make_float2(fabsf(p2.x), fabsf(p2.y)));
    }
    __device__ __forceinline__ void eval(const float4 A, const float4 B, float2& t, float2& s, float2& w) const {
        P1 st;
        bool ox, oy;
        phase1(A, B, st);
        sure(st, ox, oy);
        phase2(A, B, st, t, s);
        // a lane that phase1 already proves an outlier is decided, whatever the backward half says (it may be NaN)
        if (ox) { t.x = 1.f; s.x = 0.f; }
        if (oy) { t.y = 1.f; s.y = 0.f; }
        w = t;
    }
    // score_sq.cuh: the point is a PROVEN outlier iff the returned value is > bound (a NaN proves nothing). Max-norm form of the
    // forward distance: max(|x2 nz - nx|, |y2 nz - ny|) > 2 thr |nz| + k1, 9 packed FMA-pipe instructions per pair (the
    // maximum and the comparison go to the ALU pipe). It rejects a subset of what the disc of phase1/sure rejects: |ax| > c
    // implies that the rounded ax^2 + ay^2 exceeds c^2 (DESIGN.md section 4.2), so it is sound with the same band; the square
    // lets through at most 4/pi of the disc's survivors. max.NaN keeps a NaN in either coordinate a survivor, as the disc did.
    __device__ __forceinline__ float2 reject(const float4 A, const float4 B, float2& bound) const {
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 nz = __ffma2_rn(dup(h31), X1, __ffma2_rn(dup(h32), Y1, dup(h33)));
        const float2 nx = __ffma2_rn(dup(a11), X1, __ffma2_rn(dup(a12), Y1, dup(a13)));   // -(h11 x1 + h12 y1 + h13)
        const float2 ny = __ffma2_rn(dup(a21), X1, __ffma2_rn(dup(a22), Y1, dup(a23)));
        const float2 ax = __ffma2_rn(X2, nz, nx), ay = __ffma2_rn(Y2, nz, ny);           // nz * (x2 - nx/nz)
        bound = __ffma2_rn(dup(T2p), make_float2(fabsf(nz.x), fabsf(nz.y)), dup(k1));
        return make_float2(abs_max_nan(ax.x, ay.x), abs_max_nan(ax.y, ay.y));
    }
    static __device__ __forceinline__ float finish(float sum_em, int cnt, float thr) { return 0.5f * (sum_em + (float)cnt * (2.f * thr)); }
    static __device__ __forceinline__ float strict_to_em(float err, float thr) { return 2.f * err - 2.f * thr; }
};

template <> struct FastModel<USAC_EST_FUNDAMENTAL> {
    // Two phases, like the homography evaluator, but the split is different: the squared Sampson error n^2/den needs no division
    // for the DECISION (n^2 - thr*den < 0), only for the error sum of the inliers. phase1 computes n^2 and den (18 packed
    // FMA-pipe instructions per pair of points, no MUFU); `sure` proves the outlier with the guard band folded into the
    // constants: n^2 - (thr + b1)*den > b0 (one more FFMA2, chained compare). Only the pairs on which some model of the warp
    // has a point that is NOT a proven outlier - an inlier or a point inside the band - run phase2: the exact decision value,
    // the band, 1/den for the sum, counting and accumulation.
#ifdef USAC_F_SINGLE_PHASE   /* tuning experiment (tools/): the round-1 single-phase form */
    static constexpr bool TWO_PHASE = false;
#else
    static constexpr bool TWO_PHASE = true;
#endif
    static constexpr bool WEIGHTED = true;                                 // em = min(t, 0) * w
    float f11, f12, f13, f21, f22, f23, f31, f32, f33, negthr, b1, b0, negthrP, b0P;
    __device__ __forceinline__ void load(const float* r) {
        f11 = r[0]; f12 = r[1]; f13 = r[2]; f21 = r[3]; f22 = r[4]; f23 = r[5]; f31 = r[6]; f32 = r[7]; f33 = r[8];
        negthr = -r[REC_THR]; b1 = r[REC_BAND]; b0 = r[REC_BAND + 1];
        // sure-outlier test n^2 - thrP*den > b0P: both constants rounded UP by 2^-18 relative, far more than the roundings of
        // the folded form (2^-23 each), so every point it rejects also satisfies t > s of the two-sided band test
        negthrP = -(r[REC_THR] + b1) * 1.0000039f;
        b0P = b0 * 1.0000039f + 1e-37f;
    }
    struct P1 { float2 n2, den; };
    __device__ __forceinline__ void phase1(const float4 A, const float4 B, P1& s) const {
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 a = __ffma2_rn(dup(f11), X1, __ffma2_rn(dup(f12), Y1, dup(f13)));
        const float2 b = __ffma2_rn(dup(f21), X1, __ffma2_rn(dup(f22), Y1, dup(f23)));
        const float2 c = __ffma2_rn(dup(f11), X2, __ffma2_rn(dup(f21), Y2, dup(f31)));
        const float2 d = __ffma2_rn(dup(f12), X2, __ffma2_rn(dup(f22), Y2, dup(f32)));
        const float2 n = __ffma2_rn(X2, a, __ffma2_rn(Y2, b, __ffma2_rn(dup(f31), X1, __ffma2_rn(dup(f32), Y1, dup(f33)))));
        s.n2 = __fmul2_rn(n, n);
        s.den = __ffma2_rn(d, d, __ffma2_rn(c, c, __ffma2_rn(b, b, __fmul2_rn(a, a))));
    }
    __device__ __forceinline__ void sure(const P1& s, bool& ox, bool& oy) const {       // false for NaN
        const float2 u = __ffma2_rn(dup(negthrP), s.den, s.n2);
        ox = u.x > b0P; oy = u.y > b0P;
    }
    __device__ __forceinline__ void phase2(const float4, const float4, const P1& s, float2& t, float2& band) const {
        t = __ffma2_rn(dup(negthr), s.den, s.n2);     // n^2 - thr*den  (< 0 <=> n^2/den < thr, no division)
        band = __ffma2_rn(dup(b1), s.den, dup(b0));
    }
    __device__ __forceinline__ float2 weight(const P1& s) const { return make_float2(fast_rcp(s.den.x), fast_rcp(s.den.y)); }
    // score_sq.cuh: proven outlier iff the returned value is > bound = 0: (n^2 - b0P) - thrP den, 18 packed instructions
    __device__ __forceinline__ float2 reject(const float4 A, const float4 B, float2& bound) const {
        bound = make_float2(0.f, 0.f);
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 a = __ffma2_rn(dup(f11), X1, __ffma2_rn(dup(f12), Y1, dup(f13)));
        const float2 b = __ffma2_rn(dup(f21), X1, __ffma2_rn(dup(f22), Y1, dup(f23)));
        const float2 c = __ffma2_rn(dup(f11), X2, __ffma2_rn(dup(f21), Y2, dup(f31)));
        const float2 d = __ffma2_rn(dup(f12), X2, __ffma2_rn(dup(f22), Y2, dup(f32)));
        const float2 cp = __ffma2_rn(dup(f31), X1, __ffma2_rn(dup(f32), Y1, dup(f33)));
        const float2 n = __ffma2_rn(X2, a, __ffma2_rn(Y2, b, cp));    // (two scalar FFMA per product instead of the three-pair FFMA2: no gain, A/B r2m)
        const float2 den = __ffma2_rn(d, d, __ffma2_rn(c, c, __ffma2_rn(b, b, __fmul2_rn(a, a))));
        return __ffma2_rn(dup(negthrP), den, __ffma2_rn(n, n, dup(-b0P)));
    }
    __device__ __forceinline__ void eval(const float4 A, const float4 B, float2& t, float2& s, float2& w) const {
        P1 st;
        phase1(A, B, st);
        phase2(A, B, st, t, s);
        w = weight(st);                                                    // only the error sum needs the quotient
    }
    static __device__ __forceinline__ float finish(float sum_em, int cnt, float thr) { return sum_em + (float)cnt * thr; }
    static __device__ __forceinline__ float strict_to_em(float err, float thr) { return err - thr; }
};

template <> struct FastModel<USAC_EST_ESSENTIAL> {
    static constexpr bool WEIGHTED = false;
    float e11, e12, e13, e21, e22, e23, e31, e32, e33, negT, ka, kb, k0, negka, C2;
    __device__ __forceinline__ void load(const float* r) {
        e11 = r[0]; e12 = r[1]; e13 = r[2]; e21 = r[3]; e22 = r[4]; e23 = r[5]; e31 = r[6]; e32 = r[7]; e33 = r[8];
        negT = -2.f * r[REC_THR]; ka = r[REC_BAND]; kb = r[REC_BAND + 1]; k0 = r[REC_BAND + 2];
        negka = -ka;
        const float c = (2.f * r[REC_THR] + k0) * 1.0000039f;             // rounded up by 2^-18: covers the roundings of the squared form
        C2 = c * c * 1.0000039f;
    }
    // score_sq.cuh: the one-sided test of phase1/sure without the rsqrt. da = |a1| / L with L = |l12|; da alone beyond
    // 2 thr + (ka / L + k0) proves the outlier:  |a1| / L - 2 thr > ka / L + k0  <=>  v := |a1| - ka > (2 thr + k0) L
    // <=>  v |v| > (2 thr + k0)^2 L^2  (the left side keeps the sign of v, the right side is >= 0). 13 packed instructions, no MUFU.
    // Proven outlier iff the returned value is > bound = 0.
    __device__ __forceinline__ float2 reject(const float4 A, const float4 B, float2& bound) const {
        bound = make_float2(0.f, 0.f);
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 l1 = __ffma2_rn(dup(e11), X2, __ffma2_rn(dup(e21), Y2, dup(e31)));
        const float2 l2 = __ffma2_rn(dup(e12), X2, __ffma2_rn(dup(e22), Y2, dup(e32)));
        const float2 l3 = __ffma2_rn(dup(e13), X2, __ffma2_rn(dup(e23), Y2, dup(e33)));
        const float2 a1 = __ffma2_rn(l1, X1, __ffma2_rn(l2, Y1, l3));
        const float2 a2 = __ffma2_rn(l2, l2, __fmul2_rn(l1, l1));
        const float2 v = __fadd2_rn(make_float2(fabsf(a1.x), fabsf(a1.y)), dup(negka));
        const float2 m = __fmul2_rn(dup(C2), a2);
        return __ffma2_rn(v, make_float2(fabsf(v.x), fabsf(v.y)), make_float2(-m.x, -m.y));   // > 0: proven outlier
    }
    // Two phases, as for the homography: err = (da + db)/2 with da = |p1.l|/|l12| (l = E^T p2) and db >= 0, so da alone
    // beyond 2*thr + (its band + the band of the final sum) proves the outlier; phase2 adds the other epipolar distance.
    #ifdef USAC_E_SINGLE_PHASE   /* tuning experiment (tools/): evaluate both halves for every pair */
    static constexpr bool TWO_PHASE = false;
#else
    static constexpr bool TWO_PHASE = true;
#endif
    struct P1 { float2 u, p1; };                                           // u = da - 2*thr, p1 = ka/|l12| + k0 (>= 0)
    __device__ __forceinline__ void phase1(const float4 A, const float4 B, P1& s) const {
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 l1 = __ffma2_rn(dup(e11), X2, __ffma2_rn(dup(e21), Y2, dup(e31)));
        const float2 l2 = __ffma2_rn(dup(e12), X2, __ffma2_rn(dup(e22), Y2, dup(e32)));
        const float2 l3 = __ffma2_rn(dup(e13), X2, __ffma2_rn(dup(e23), Y2, dup(e33)));
        const float2 a1 = __ffma2_rn(l1, X1, __ffma2_rn(l2, Y1, l3));
        const float2 a2 = __ffma2_rn(l2, l2, __fmul2_rn(l1, l1));
        const float2 ra = make_float2(fast_rsqrt(a2.x), fast_rsqrt(a2.y));
        const float2 pa = __fmul2_rn(a1, ra);
        s.u = make_float2(fabsf(pa.x) + negT, fabsf(pa.y) + negT);
        s.p1 = __ffma2_rn(dup(ka), ra, dup(k0));
    }
    __device__ __forceinline__ void sure(const P1& s, bool& ox, bool& oy) const {       // false for NaN
        ox = s.u.x > fabsf(s.p1.x); oy = s.u.y > fabsf(s.p1.y);
    }
    __device__ __forceinline__ void phase2(const float4 A, const float4 B, const P1& s, float2& t, float2& band) const {
        const float2 X1 = make_float2(A.x, A.y), Y1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y), Y2 = make_float2(B.z, B.w);
        const float2 t1 = __ffma2_rn(dup(e11), X1, __ffma2_rn(dup(e12), Y1, dup(e13)));
        const float2 t2 = __ffma2_rn(dup(e21), X1, __ffma2_rn(dup(e22), Y1, dup(e23)));
        const float2 t3 = __ffma2_rn(dup(e31), X1, __ffma2_rn(dup(e32), Y1, dup(e33)));
        const float2 b1 = __ffma2_rn(t1, X2, __ffma2_rn(t2, Y2, t3));
        const float2 b2 = __ffma2_rn(t2, t2, __fmul2_rn(t1, t1));
        const float2 rb = make_float2(fast_rsqrt(b2.x), fast_rsqrt(b2.y));
        const float2 pb = __fmul2_rn(b1, rb);
        t = make_float2(s.u.x + fabsf(pb.x), s.u.y + fabsf(pb.y));        // 2*err - 2*thr
        band = __ffma2_rn(dup(kb), rb, s.p1);
    }
    __device__ __forceinline__ void eval(const float4 A, const float4 B, float2& t, float2& s, float2& w) const {
        P1 st;
        bool ox, oy;
        phase1(A, B, st);
        sure(st, ox, oy);
        phase2(A, B, st, t, s);
        if (ox) { t.x = 1.f; s.x = 0.f; }
        if (oy) { t.y = 1.f; s.y = 0.f; }
        w = t;
    }
    static __device__ __forceinline__ float finish(float sum_em, int cnt, float thr) { return 0.5f * (sum_em + (float)cnt * (2.f * thr)); }
    static __device__ __forceinline__ float strict_to_em(float err, float thr) { return 2.f * err - 2.f * thr; }
};

template <> struct FastModel<USAC_EST_LINE2D> {
    static constexpr bool TWO_PHASE = false;
    static constexpr bool WEIGHTED = false;
    float a, b, c, negthr, band;
    __device__ __forceinline__ void load(const float* r) { a = r[0]; b = r[1]; c = r[2]; negthr = -r[REC_THR]; band = r[REC_BAND]; }
    // line pairs are [xa xb ya yb]: one float4 per pair (B unused)
    __device__ __forceinline__ void eval(const float4 A, const float4, float2& t, float2& s, float2& w) const {
        const float2 X = make_float2(A.x, A.y), Y = make_float2(A.z, A.w);
        const float2 v = __ffma2_rn(dup(a), X, __ffma2_rn(dup(b), Y, dup(c)));
        t = make_float2(fabsf(v.x) + negthr, fabsf(v.y) + negthr);
        s = dup(band);
        w = t;
    }
    __device__ __forceinline__ float2 reject(const float4 A, const float4, float2& bound) const {   // score_sq.cuh: > bound = 0: proven outlier
        bound = make_float2(0.f, 0.f);
        const float2 X = make_float2(A.x, A.y), Y = make_float2(A.z, A.w);
        const float2 v = __ffma2_rn(dup(a), X, __ffma2_rn(dup(b), Y, dup(c)));
        return make_float2(fabsf(v.x) + (negthr - band), fabsf(v.y) + (negthr - band));
    }
    static __device__ __forceinline__ float finish(float sum_em, int cnt, float thr) { return sum_em + (float)cnt * thr; }
    static __device__ __forceinline__ float strict_to_em(float err, float thr) { return err - thr; }
};

struct ScoreArgs {
    const float* pairs;          // pair-interleaved points of all problems
    const float* aos;            // original AoS points (strict re-evaluation reads these)
    const ProblemDesc* prob;
    const int* active;           // slot -> problem id (NULL: identity)
    const float* recs;           // [slot][mstride][USAC_REC_STRIDE]
    const int* mvalid;           // [slot] models to score (NULL: M for all)
    int M, mstride;              // models per problem (upper bound) and record/partial stride
    int chunk_pairs, nchunks;    // point pairs per work item along the point axis
    int mblocks, slots;          // work items = slots x nchunks x mblocks (model block fastest: neighbours share points)
    int* part_cnt;               // [slot][nchunks][mstride]
    float* part_sum;
    unsigned* work;              // global work-item counter, never reset: this launch's items are work - work_base
    unsigned work_base;
    const uint2* items;          // optional compact item list written by prepare_kernel (slot, chunk << 16 | model group); NULL: dense grid
    const unsigned* item_count;  // number of entries of `items` (device side: the host does not know how many models a round produced)
};

// work item -> (slot, chunk, model group); false when the item is past the end
__device__ __forceinline__ bool score_item(const ScoreArgs& a, unsigned item, unsigned total, int mgroups, int& slot, int& chunk, int& mgroup) {
    if (item >= total) return false;
    if (a.items) {
        const uint2 it = a.items[item];
        slot = (int)it.x; chunk = (int)(it.y >> 16); mgroup = (int)(it.y & 0xffffu);
    } else {
        mgroup = (int)(item % (unsigned)mgroups);
        const unsigned rest = item / (unsigned)mgroups;
        chunk = (int)(rest % (unsigned)a.nchunks); slot = (int)(rest / (unsigned)a.nchunks);
    }
    return true;
}

// Slow path of one lane: the reference's exact arithmetic for point `idx` of the problem. Returns the lane's `em`
// contribution: negative (its sign bit is the inlier flag) for an inlier, +0 otherwise. Pure, so the hot loop keeps
// everything in registers.
template <int EST>
__device__ __noinline__ float strict_em(const float* __restrict__ rec, const float* __restrict__ aos, int idx, int n) {
    if (idx >= n) return 0.f;
    const float thr = rec[REC_THR];
    float err;
    if (EST == USAC_EST_LINE2D) {
        const float2 p = reinterpret_cast<const float2*>(aos)[idx];
        err = strict_error<EST>(rec, p.x, p.y, 0.f, 0.f);
    } else {
        const float4 p = reinterpret_cast<const float4*>(aos)[idx];
        err = strict_error<EST>(rec, p.x, p.y, p.z, p.w);
    }
    // err < thr  =>  strict_to_em < 0 exactly (2*err and 2*thr are exact, the difference of distinct floats is non-zero)
    return (err < thr) ? FastModel<EST>::strict_to_em(err, thr) : 0.f;
}

// Persistent kernel of independent warps: every warp draws work items (slot, point chunk, group of 32 models) from a global
// counter and streams the item's points through its OWN USAC_WARP_STAGES-deep ring of shared-memory tiles filled by 1-D bulk
// async copies (completion on the warp's `full` mbarriers). Warps never wait for each other - no CTA barrier, no shared
// counters: a warp whose models need the slow phases (good models, degenerate models) does not hold back its neighbours,
// and the dynamic hand-out levels the tail. The four warps of a CTA mostly draw neighbouring items (the model group is the
// fastest index), so their tile fetches hit the same L2 lines.
template <int EST>
__global__ void __launch_bounds__(USAC_SCORE_THREADS, USAC_SCORE_MIN_CTAS) score_kernel(const ScoreArgs a) {
    constexpr int PAIR_FLOATS = (EST == USAC_EST_LINE2D) ? 4 : 8;
    constexpr int NWARPS = USAC_SCORE_THREADS / 32;
    __shared__ __align__(128) float tile_all[NWARPS][USAC_WARP_STAGES][USAC_TILE_PAIRS * PAIR_FLOATS];
    __shared__ __align__(8) uint64_t full_all[NWARPS][USAC_WARP_STAGES];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float (*tile)[USAC_TILE_PAIRS * PAIR_FLOATS] = tile_all[warp];
    uint64_t* full = full_all[warp];
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

    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(a.work, 1u) - a.work_base;   // every warp overdraws exactly once (accounted by the host)
        item = __shfl_sync(0xffffffffu, item, 0);
        int slot, chunk, mgroup;
        if (!score_item(a, item, total, mgroups, slot, chunk, mgroup)) break;
        const int M = a.mvalid ? a.mvalid[slot] : a.M;
        if (mgroup * 32 >= M) continue;                              // uniform per warp
        const ProblemDesc pd = a.prob[a.active ? a.active[slot] : slot];
        const int m = mgroup * 32 + lane;
        const bool live = m < M;
        const float* rec = a.recs + ((size_t)slot * a.mstride + (live ? m : 0)) * USAC_REC_STRIDE;
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

        FastModel<EST> fm;
        fm.load(rec);
        const float* aos = a.aos + (size_t)pd.aos_off * (EST == USAC_EST_LINE2D ? 2 : 4);
        unsigned cnt = 0;
        float2 sum[USAC_PPI];
#pragma unroll
        for (int q = 0; q < USAC_PPI; q++) sum[q] = make_float2(0.f, 0.f);

        for (int k = 0; k < ntiles; k++) {
            const int s = (g + k) % USAC_WARP_STAGES;
            mbar_wait(&full[s], ((g + k) / USAC_WARP_STAGES) & 1);
            const int np = min(USAC_TILE_PAIRS, npairs - k * USAC_TILE_PAIRS);
            const float4* tp = reinterpret_cast<const float4*>(tile[s]);
            const int idx0 = 2 * (pair_begin + k * USAC_TILE_PAIRS);
            // Hot loop with a warp-uniform exit: USAC_PPI pairs (2*USAC_PPI points) per trip, evaluated as independent
            // instruction streams. When any lane of the warp cannot decide one of them from the fast value the whole
            // warp leaves the loop, these pairs are redone one by one - undecided lanes re-evaluate with the reference's
            // arithmetic (a real function call, kept out of the loop body so that it does not clobber the loop's uniform
            // registers) - and the loop resumes behind them.
            auto load_pair = [&](int j, float4& A, float4& B) {
                if (EST == USAC_EST_LINE2D) { A = tp[j]; B = A; }
                else { A = tp[2 * j]; B = tp[2 * j + 1]; }
            };
            int j = 0;
            while (j < np) {
#pragma unroll 1
                for (; j + USAC_PPI <= np; j += USAC_PPI) {
                    float2 em[USAC_PPI];
                    bool unsure = false;
                    if constexpr (FastModel<EST>::TWO_PHASE) {
                        typename FastModel<EST>::P1 st[USAC_PPI];
                        bool lane_any = false;
#pragma unroll
                        for (int q = 0; q < USAC_PPI; q++) {                                    // forward halves, independent streams
                            float4 A, B;
                            load_pair(j + q, A, B);
                            fm.phase1(A, B, st[q]);
                            bool ox, oy;
                            fm.sure(st[q], ox, oy);
                            lane_any = lane_any || !ox || !oy;
                        }
                        // one vote for the whole trip: in most trips every point is a proven outlier for every model of the
                        // warp - nothing to count, nothing to add
                        if (!__any_sync(0xffffffffu, lane_any)) continue;
#pragma unroll
                        for (int q = 0; q < USAC_PPI; q++) {
                            em[q] = make_float2(0.f, 0.f);
                            bool ox, oy;
                            fm.sure(st[q], ox, oy);
                            if (__any_sync(0xffffffffu, !ox || !oy)) {                          // warp-uniform
                                float4 A, B;
                                load_pair(j + q, A, B);
                                float2 t, sb;
                                fm.phase2(A, B, st[q], t, sb);
                                unsure = unsure || (!ox && !(fabsf(t.x) > sb.x)) || (!oy && !(fabsf(t.y) > sb.y));
                                if constexpr (FastModel<EST>::WEIGHTED) t = __fmul2_rn(t, fm.weight(st[q]));   // weights are >= 0; inf/NaN * (t >= 0) is dropped by fminf
                                em[q] = make_float2(ox ? 0.f : fminf(t.x, 0.f), oy ? 0.f : fminf(t.y, 0.f));
                            }
                        }
                    } else {
#pragma unroll
                        for (int q = 0; q < USAC_PPI; q++) {
                            float4 A, B;
                            load_pair(j + q, A, B);
                            float2 t, sb, w;
                            fm.eval(A, B, t, sb, w);
                            unsure = unsure || !(fabsf(t.x) > sb.x) || !(fabsf(t.y) > sb.y);   // also catches NaN
                            if constexpr (FastModel<EST>::WEIGHTED) t = __fmul2_rn(t, w);
                            em[q] = make_float2(fminf(t.x, 0.f), fminf(t.y, 0.f));
                        }
                    }
                    if (__any_sync(0xffffffffu, unsure)) break;
#pragma unroll
                    for (int q = 0; q < USAC_PPI; q++) {
                        cnt += (__float_as_uint(em[q].x) >> 31) + (__float_as_uint(em[q].y) >> 31);
                        sum[q] = __fadd2_rn(sum[q], em[q]);
                    }
                }
                const int jend = min(j + USAC_PPI, np);
#pragma unroll 1
                for (; j < jend; j++) {
                    float4 A, B;
                    load_pair(j, A, B);
                    float2 t, sb, w;
                    fm.eval(A, B, t, sb, w);
                    const bool ux = !(fabsf(t.x) > sb.x), uy = !(fabsf(t.y) > sb.y);
                    if constexpr (FastModel<EST>::WEIGHTED) t = __fmul2_rn(t, w);
                    float2 e1 = make_float2(fminf(t.x, 0.f), fminf(t.y, 0.f));
                    if (ux) e1.x = strict_em<EST>(rec, aos, idx0 + 2 * j, pd.n);
                    if (uy) e1.y = strict_em<EST>(rec, aos, idx0 + 2 * j + 1, pd.n);
                    cnt += (__float_as_uint(e1.x) >> 31) + (__float_as_uint(e1.y) >> 31);
                    sum[0] = __fadd2_rn(sum[0], e1);
                }
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
        if (live) {
            a.part_cnt[out] = (int)cnt;
            float tot = 0.f;
#pragma unroll
            for (int q = 0; q < USAC_PPI; q++) tot += sum[q].x + sum[q].y;
            a.part_sum[out] = FastModel<EST>::finish(tot, (int)cnt, rec[REC_THR]);
        }
        __syncwarp();                                                // all lanes left the item before its stages are refilled
    }
}

// Reference-arithmetic scoring of every point (no fast path): used by usac_gpu_errors and as the in-library
// cross-check of the fast kernel in tests. One thread per point.
template <int EST>
__global__ void errors_kernel(const float* __restrict__ aos, int n, const float* __restrict__ rec, float* __restrict__ err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (EST == USAC_EST_LINE2D) {
        const float2 p = reinterpret_cast<const float2*>(aos)[i];
        err[i] = strict_error<EST>(rec, p.x, p.y, 0.f, 0.f);
    } else {
        const float4 p = reinterpret_cast<const float4*>(aos)[i];
        err[i] = strict_error<EST>(rec, p.x, p.y, p.z, p.w);
    }
}

// Quality::getInliers (quality.hpp:108-121): ids of the inliers in ascending order. One CTA, ordered block scan.
template <int EST>
__global__ void __launch_bounds__(1024) inliers_kernel(const float* __restrict__ aos, int n, const float* __restrict__ rec, float thr,
                                                       int* __restrict__ ids, int* __restrict__ count) {
    __shared__ int warp_tot[32];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int start = 0; start < n; start += 1024) {
        const int i = start + threadIdx.x;
        bool in = false;
        if (i < n) {
            float e;
            if (EST == USAC_EST_LINE2D) { const float2 p = reinterpret_cast<const float2*>(aos)[i]; e = strict_error<EST>(rec, p.x, p.y, 0.f, 0.f); }
            else { const float4 p = reinterpret_cast<const float4*>(aos)[i]; e = strict_error<EST>(rec, p.x, p.y, p.z, p.w); }
            in = e < thr;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < 32; w++) { const int v = warp_tot[w]; if (w < warp) before += v; total += v; }
        if (in) ids[base + before + __popc(bal & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (threadIdx.x == 0) base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

// The same list for large problems (1M points = 977 blocks of the loop above, one after the other: 1.5 ms) in three small launches:
// flags + per-block counts over a grid, one CTA scanning the block counts, and the scatter from the stored flags. Every decision is
// the same strict_error comparison, so the list is identical to the one-CTA kernel's.
template <int EST>
__global__ void __launch_bounds__(1024) inliers_flags_kernel(const float* __restrict__ aos, int n, const float* __restrict__ rec, float thr,
                                                             unsigned* __restrict__ ballots, int* __restrict__ block_counts) {
    __shared__ int warp_tot[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * 1024 + threadIdx.x;
    bool in = false;
    if (i < n) {
        float e;
        if (EST == USAC_EST_LINE2D) { const float2 p = reinterpret_cast<const float2*>(aos)[i]; e = strict_error<EST>(rec, p.x, p.y, 0.f, 0.f); }
        else { const float4 p = reinterpret_cast<const float4*>(aos)[i]; e = strict_error<EST>(rec, p.x, p.y, p.z, p.w); }
        in = e < thr;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, in);
    if (lane == 0) { ballots[blockIdx.x * 32 + warp] = bal; warp_tot[warp] = __popc(bal); }
    __syncthreads();
    if (warp == 0) {
        int v = warp_tot[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) block_counts[blockIdx.x] = v;
    }
}
// exclusive scan of the block counts in place (one CTA), total -> *count
__global__ void __launch_bounds__(1024) inliers_scan_kernel(int* __restrict__ block_counts, int nblocks, int* __restrict__ count) {
    __shared__ int sm[33];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nblocks; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const int v = b < nblocks ? block_counts[b] : 0;
        int total;
        const int off = block_exclusive_scan(v, &total, sm);
        if (b < nblocks) block_counts[b] = base + off;
        __syncthreads();
        if (threadIdx.x == 0) base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}
__global__ void __launch_bounds__(1024) inliers_scatter_kernel(const unsigned* __restrict__ ballots, const int* __restrict__ block_offsets, int n,
                                                               int* __restrict__ ids) {
    __shared__ int warp_off[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp == 0) {                                                  // exclusive scan of the 32 warp counts of this block
        const int v = __popc(ballots[blockIdx.x * 32 + lane]);
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
        warp_off[lane] = incl - v;
    }
    __syncthreads();
    const unsigned bal = ballots[blockIdx.x * 32 + warp];
    const int i = blockIdx.x * 1024 + threadIdx.x;
    if (i < n && ((bal >> lane) & 1u)) ids[block_offsets[blockIdx.x] + warp_off[warp] + __popc(bal & ((1u << lane) - 1))] = i;
}

// Quality::getNumberInliers(score, model, thr, get_inliers = true, ids) (quality.hpp:60-101) for local optimisation: ids in
// ascending order, count, and the error sum as a lane sum (thread t adds the errors of its inliers t, t+1024, ... in order,
// then a fixed binary tree over the 1024 lanes) - the order the parity tests' host restatement uses. stat = {count, sum bits}.
template <int EST>
__global__ void __launch_bounds__(1024) inliers_sum_kernel(const float* __restrict__ aos, int n, const float* __restrict__ rec, float thr,
                                                           int* __restrict__ ids, int* __restrict__ stat) {
    __shared__ int warp_tot[32];
    __shared__ int base;
    __shared__ float part[1024];
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float acc = 0.f;
    for (int start = 0; start < n; start += 1024) {
        const int i = start + threadIdx.x;
        bool in = false;
        if (i < n) {
            float e;
            if (EST == USAC_EST_LINE2D) { const float2 p = reinterpret_cast<const float2*>(aos)[i]; e = strict_error<EST>(rec, p.x, p.y, 0.f, 0.f); }
            else { const float4 p = reinterpret_cast<const float4*>(aos)[i]; e = strict_error<EST>(rec, p.x, p.y, p.z, p.w); }
            in = e < thr;
            if (in) acc = __fadd_rn(acc, e);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < 32; w++) { const int v = warp_tot[w]; if (w < warp) before += v; total += v; }
        if (in) ids[base + before + __popc(bal & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (threadIdx.x == 0) base += total;
        __syncthreads();
    }
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) part[threadIdx.x] = __fadd_rn(part[threadIdx.x], part[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) { stat[0] = base; stat[1] = __float_as_int(part[0]); }
}

__global__ void gather_ids_kernel(const int* __restrict__ from, const int* __restrict__ pos, int k, int* __restrict__ out) {
    const int i = threadIdx.x;
    if (i < k) out[i] = from[pos[i]];
}
