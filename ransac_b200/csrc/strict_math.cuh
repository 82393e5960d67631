// strict_math.cuh - IEEE, one-rounding-per-operator arithmetic (no FMA contraction) for everything that has to be
// bit-identical to the reference's x86-64 SSE float/double code: the error functions (homography_estimator.hpp:85-110,
// fundamental_estimator.hpp:101-117, essential_estimator.hpp:76-107, line2d_estimator.hpp:154-156), the 3x3 inverse of
// setModelParameters and the minimal solvers. nvcc contracts a*b+c into FMA by default; the wrapper types below route
// every operator through the *_rn intrinsics, which are never contracted.
#pragma once
#include "common.cuh"

struct sf {   // strict float
    float v;
    __device__ __forceinline__ sf() {}
    __device__ __forceinline__ sf(float x) : v(x) {}
};
__device__ __forceinline__ sf operator+(sf a, sf b) { return sf(__fadd_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator-(sf a, sf b) { return sf(__fsub_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator*(sf a, sf b) { return sf(__fmul_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator/(sf a, sf b) { return sf(__fdiv_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator-(sf a) { return sf(-a.v); }
__device__ __forceinline__ sf ssqrt(sf a) { return sf(__fsqrt_rn(a.v)); }
__device__ __forceinline__ sf sabs(sf a) { return sf(fabsf(a.v)); }

struct sd {   // strict double
    double v;
    __device__ __forceinline__ sd() {}
    __device__ __forceinline__ sd(double x) : v(x) {}
};
__device__ __forceinline__ sd operator+(sd a, sd b) { return sd(__dadd_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator-(sd a, sd b) { return sd(__dsub_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator*(sd a, sd b) { return sd(__dmul_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator/(sd a, sd b) { return sd(__ddiv_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator-(sd a) { return sd(-a.v); }
__device__ __forceinline__ sd dsqrt(sd a) { return sd(__dsqrt_rn(a.v)); }
__device__ __forceinline__ bool dfinite(double x) { return isfinite(x); }

// ---------------------------------------------------------------------------------------------------------------
// Error functions, reference operation order (SURVEY.md appendix A). p = model record (REC_MODEL.., REC_HINV..).
// ---------------------------------------------------------------------------------------------------------------
template <int EST>
__device__ __forceinline__ float strict_error(const float* __restrict__ p, float x1f, float y1f, float x2f, float y2f) {
    const sf x1(x1f), y1(y1f), x2(x2f), y2(y2f);
    if (EST == USAC_EST_LINE2D) {   // line2d_estimator.hpp:154-156 (x1f,y1f = x,y)
        return sabs(sf(p[0]) * x1 + sf(p[1]) * y1 + sf(p[2])).v;
    } else if (EST == USAC_EST_HOMOGRAPHY) {   // homography_estimator.hpp:85-110
        sf ex = sf(p[0]) * x1 + sf(p[1]) * y1 + sf(p[2]);
        sf ey = sf(p[3]) * x1 + sf(p[4]) * y1 + sf(p[5]);
        sf ez = sf(p[6]) * x1 + sf(p[7]) * y1 + sf(p[8]);
        ex = ex / ez; ey = ey / ez;
        sf fx = sf(p[9]) * x2 + sf(p[10]) * y2 + sf(p[11]);
        sf fy = sf(p[12]) * x2 + sf(p[13]) * y2 + sf(p[14]);
        sf fz = sf(p[15]) * x2 + sf(p[16]) * y2 + sf(p[17]);
        fx = fx / fz; fy = fy / fz;
        sf e = ssqrt((x2 - ex) * (x2 - ex) + (y2 - ey) * (y2 - ey)) + ssqrt((x1 - fx) * (x1 - fx) + (y1 - fy) * (y1 - fy));
        return (e / sf(2.f)).v;
    } else if (EST == USAC_EST_FUNDAMENTAL) {   // fundamental_estimator.hpp:101-117
        sf a = sf(p[0]) * x1 + sf(p[1]) * y1 + sf(p[2]);
        sf b = sf(p[3]) * x1 + sf(p[4]) * y1 + sf(p[5]);
        sf c = sf(p[0]) * x2 + sf(p[3]) * y2 + sf(p[6]);
        sf d = sf(p[1]) * x2 + sf(p[4]) * y2 + sf(p[7]);
        sf n = x2 * a + y2 * b + sf(p[6]) * x1 + sf(p[7]) * y1 + sf(p[8]);
        return ((n * n) / (a * a + b * b + c * c + d * d)).v;
    } else {   // essential_estimator.hpp:76-107
        sf l1 = sf(p[0]) * x2 + sf(p[3]) * y2 + sf(p[6]);
        sf l2 = sf(p[1]) * x2 + sf(p[4]) * y2 + sf(p[7]);
        sf l3 = sf(p[2]) * x2 + sf(p[5]) * y2 + sf(p[8]);
        sf t1 = sf(p[0]) * x1 + sf(p[1]) * y1 + sf(p[2]);
        sf t2 = sf(p[3]) * x1 + sf(p[4]) * y1 + sf(p[5]);
        sf t3 = sf(p[6]) * x1 + sf(p[7]) * y1 + sf(p[8]);
        sf a1 = l1 * x1 + l2 * y1 + l3;
        sf a2 = ssqrt(l1 * l1 + l2 * l2);
        sf b1 = t1 * x2 + t2 * y2 + t3;
        sf b2 = ssqrt(t1 * t1 + t2 * t2);
        return ((sabs(a1 / a2) + sabs(b1 / b2)) / sf(2.f)).v;
    }
}

// cv::Mat::inv() of a 3x3 CV_32F (OpenCV core lapack.cpp, n==3 branch): cofactors and determinant in double, 1/det,
// rounded to float; det == 0 -> all zeros. Call site: homography_estimator.hpp:35.
__device__ __forceinline__ void cv_inv3x3(const float* m, float* out) {
    const sd a00(m[0]), a01(m[1]), a02(m[2]), a10(m[3]), a11(m[4]), a12(m[5]), a20(m[6]), a21(m[7]), a22(m[8]);
    sd d = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20);
    if (d.v == 0.0) {
#pragma unroll
        for (int i = 0; i < 9; i++) out[i] = 0.f;
        return;
    }
    d = sd(1.0) / d;
    out[0] = (float)((a11 * a22 - a12 * a21) * d).v;
    out[1] = (float)((a02 * a21 - a01 * a22) * d).v;
    out[2] = (float)((a01 * a12 - a02 * a11) * d).v;
    out[3] = (float)((a12 * a20 - a10 * a22) * d).v;
    out[4] = (float)((a00 * a22 - a02 * a20) * d).v;
    out[5] = (float)((a02 * a10 - a00 * a12) * d).v;
    out[6] = (float)((a10 * a21 - a11 * a20) * d).v;
    out[7] = (float)((a01 * a20 - a00 * a21) * d).v;
    out[8] = (float)((a00 * a11 - a01 * a10) * d).v;
}

// ---------------------------------------------------------------------------------------------------------------
// Minimal solvers (one thread per sample). Operation order is the contract of DESIGN.md S1-S4.
// ---------------------------------------------------------------------------------------------------------------

// Gauss-Jordan with partial (row) pivoting on a ROWS x 9 double system held in REGISTERS: every loop is fully unrolled so
// that all indices are compile-time constants, and the pivot row is brought into place by predicated swaps (only columns
// >= k are live). The matrix is passed as two arrays (rows 0..3 and 4..ROWS-1): nvcc keeps a local array in registers only
// up to ~300 bytes, a single 8x9 double array stays in local memory (measured: 720-byte stack frame, 3x slower kernel).
// Same operations in the same order as the host restatement used by the parity tests: pivot = first row r >= k
// maximising |A[r][k]|; scale row k by 1/pivot; A[r][j] -= A[r][k]*A[k][j] (product rounded, then difference rounded).
// On success row k is the k-th reduced row: the entries of the free columns ROWS..8 are valid.
#define GJ_AT(r, j) (*((r) < 4 ? &T[(r)][(j)] : &B[(r) - 4][(j)]))
template <int ROWS>
__device__ __forceinline__ bool gauss_jordan9(double (&T)[4][9], double (&B)[ROWS - 4][9]) {
#pragma unroll
    for (int k = 0; k < ROWS; k++) {
        int piv = k;
        double best = fabs(GJ_AT(k, k));
#pragma unroll
        for (int r = k + 1; r < ROWS; r++) {
            const double v = fabs(GJ_AT(r, k));
            if (v > best) { best = v; piv = r; }
        }
        if (!(best > 0.0) || !dfinite(best)) return false;
#pragma unroll
        for (int r = k + 1; r < ROWS; r++) {
            const bool sw = piv == r;
#pragma unroll
            for (int j = k; j < 9; j++) {
                const double a = GJ_AT(k, j), b = GJ_AT(r, j);
                GJ_AT(k, j) = sw ? b : a;
                GJ_AT(r, j) = sw ? a : b;
            }
        }
        const sd inv = sd(1.0) / sd(GJ_AT(k, k));
#pragma unroll
        for (int j = k + 1; j < 9; j++) GJ_AT(k, j) = (sd(GJ_AT(k, j)) * inv).v;
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
            if (r == k) continue;
            const sd f(GJ_AT(r, k));
#pragma unroll
            for (int j = k + 1; j < 9; j++) GJ_AT(r, j) = (sd(GJ_AT(r, j)) - f * sd(GJ_AT(k, j))).v;
        }
    }
    return true;
}

// line2d_estimator.hpp:36-54
__device__ __forceinline__ int solve_line2d(const float* __restrict__ pts, const int* s, float* out) {
    const float2 p1 = reinterpret_cast<const float2*>(pts)[s[0]], p2 = reinterpret_cast<const float2*>(pts)[s[1]];
    sf a = sf(p1.y) - sf(p2.y);
    sf b = sf(p2.x) - sf(p1.x);
    const sf mag = ssqrt(a * a + b * b);
    a = a / mag;
    b = b / mag;
    const sf c = (sf(p1.x) * sf(p2.y) - sf(p2.x) * sf(p1.y)) / mag;
    out[0] = a.v; out[1] = b.v; out[2] = c.v;
    return 1;
}

// Four-point homography: Hartley normalisation as GetNormalizingTransformation (normalizing_transformation.cpp:7-112),
// DLT rows (dlt.cpp:55-101), true null vector, H = T2^-1 Hn T1, /h33 (normalized_dlt.cpp:18-20). DESIGN.md S2.
__device__ int solve_homography4(const float* __restrict__ pts, const int* s, float* out) {
    float4 p[4];
#pragma unroll
    for (int i = 0; i < 4; i++) p[i] = reinterpret_cast<const float4*>(pts)[s[i]];
    sf m1x(0.f), m1y(0.f), m2x(0.f), m2y(0.f);
#pragma unroll
    for (int i = 0; i < 4; i++) { m1x = m1x + sf(p[i].x); m1y = m1y + sf(p[i].y); m2x = m2x + sf(p[i].z); m2y = m2y + sf(p[i].w); }
    m1x = m1x / sf(4.f); m1y = m1y / sf(4.f); m2x = m2x / sf(4.f); m2y = m2y / sf(4.f);
    sf d1(0.f), d2(0.f);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const sf ax = sf(p[i].x) - m1x, ay = sf(p[i].y) - m1y, bx = sf(p[i].z) - m2x, by = sf(p[i].w) - m2y;
        d1 = d1 + ssqrt(ax * ax + ay * ay);
        d2 = d2 + ssqrt(bx * bx + by * by);
    }
    const double SQRT2 = 1.41421356237309504880;   // M_SQRT2
    const float s1 = (float)(sd(SQRT2) / sd((double)(d1 / sf(4.f)).v)).v;
    const float s2 = (float)(sd(SQRT2) / sd((double)(d2 / sf(4.f)).v)).v;
    const float t1x = (-m1x * sf(s1)).v, t1y = (-m1y * sf(s1)).v, t2x = (-m2x * sf(s2)).v, t2y = (-m2y * sf(s2)).v;

    double T[4][9], B[4][9];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const sd x1 = sd((double)s1) * sd((double)p[i].x) + sd((double)t1x), y1 = sd((double)s1) * sd((double)p[i].y) + sd((double)t1y);
        const sd x2 = sd((double)s2) * sd((double)p[i].z) + sd((double)t2x), y2 = sd((double)s2) * sd((double)p[i].w) + sd((double)t2y);
        const int a = 2 * i, b = 2 * i + 1;
        GJ_AT(a, 0) = -x1.v; GJ_AT(a, 1) = -y1.v; GJ_AT(a, 2) = -1; GJ_AT(a, 3) = 0; GJ_AT(a, 4) = 0; GJ_AT(a, 5) = 0;
        GJ_AT(a, 6) = (x2 * x1).v; GJ_AT(a, 7) = (x2 * y1).v; GJ_AT(a, 8) = x2.v;
        GJ_AT(b, 0) = 0; GJ_AT(b, 1) = 0; GJ_AT(b, 2) = 0; GJ_AT(b, 3) = -x1.v; GJ_AT(b, 4) = -y1.v; GJ_AT(b, 5) = -1;
        GJ_AT(b, 6) = (y2 * x1).v; GJ_AT(b, 7) = (y2 * y1).v; GJ_AT(b, 8) = y2.v;
    }
    if (!gauss_jordan9<8>(T, B)) return 0;
    sd h[9];
#pragma unroll
    for (int i = 0; i < 8; i++) h[i] = -sd(GJ_AT(i, 8));
    h[8] = sd(1.0);
    sd M[9];
#pragma unroll
    for (int i = 0; i < 3; i++) {
        M[3 * i] = h[3 * i] * sd((double)s1);
        M[3 * i + 1] = h[3 * i + 1] * sd((double)s1);
        M[3 * i + 2] = h[3 * i] * sd((double)t1x) + h[3 * i + 1] * sd((double)t1y) + h[3 * i + 2];
    }
    const sd is2 = sd(1.0) / sd((double)s2);
    const sd ux = -(sd((double)t2x) * is2), uy = -(sd((double)t2y) * is2);
    sd H[9];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        H[j] = is2 * M[j] + ux * M[6 + j];
        H[3 + j] = is2 * M[3 + j] + uy * M[6 + j];
        H[6 + j] = M[6 + j];
    }
    const sd inv = sd(1.0) / H[8];
#pragma unroll
    for (int i = 0; i < 9; i++) {
        const double v = (H[i] * inv).v;
        if (!dfinite(v)) return 0;
        out[i] = (float)v;
    }
    out[8] = 1.f;
    return 1;
}

__device__ __forceinline__ sd det3(const sd* m) {
    return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}
__device__ __forceinline__ double cubic_eval(sd a, sd b, sd c, sd x) { return (((x + a) * x + b) * x + c).v; }

__device__ double cubic_bisect(sd a, sd b, sd c, double l, double r) {
    const double pl = cubic_eval(a, b, c, sd(l));
    if (pl == 0.0) return l;
    const double pr = cubic_eval(a, b, c, sd(r));
    if (pr == 0.0) return r;
    const bool neg_left = pl < 0.0;
#pragma unroll 1
    for (int it = 0; it < 2200; it++) {
        const double m = (sd(0.5) * (sd(l) + sd(r))).v;
        if (m == l || m == r) break;
        const double pm = cubic_eval(a, b, c, sd(m));
        if (pm == 0.0) return m;
        if ((pm < 0.0) == neg_left) l = m; else r = m;
    }
    return (sd(0.5) * (sd(l) + sd(r))).v;
}

// Real roots of c0 x^3 + c1 x^2 + c2 x + c3 with cv::solveCubic's count/order semantics (seven_points.cpp:131);
// bracketing + bisection so that only + - * / sqrt are used. DESIGN.md S4.
__device__ int solve_cubic(const sd* co, double* roots) {
    roots[0] = roots[1] = roots[2] = 0.0;
    const sd a0 = co[0];
    if (a0.v == 0.0) {
        const sd a1 = co[1], a2 = co[2], a3 = co[3];
        if (a1.v == 0.0) {
            if (a2.v == 0.0) return a3.v == 0.0 ? -1 : 0;
            roots[0] = (-a3 / a2).v;
            return 1;
        }
        sd d = a2 * a2 - sd(4.0) * a1 * a3;
        if (d.v < 0.0) return 0;
        d = dsqrt(d);
        const sd q1 = (-a2 + d) * sd(0.5), q2 = (a2 + d) * sd(-0.5);
        if (fabs(q1.v) > fabs(q2.v)) { roots[0] = (q1 / a1).v; roots[1] = (a3 / q1).v; }
        else { roots[0] = (q2 / a1).v; roots[1] = (a3 / q2).v; }
        return d.v > 0.0 ? 2 : 1;
    }
    const sd inv = sd(1.0) / a0;
    const sd a = co[1] * inv, b = co[2] * inv, c = co[3] * inv;
    if (!dfinite(a.v) || !dfinite(b.v) || !dfinite(c.v)) return 0;
    double B = fabs(a.v);
    if (fabs(b.v) > B) B = fabs(b.v);
    if (fabs(c.v) > B) B = fabs(c.v);
    B = (sd(B) + sd(1.0)).v;
    const sd disc = a * a - sd(3.0) * b;
    if (!(disc.v > 0.0)) { roots[0] = cubic_bisect(a, b, c, -B, B); return 1; }
    const sd sq = dsqrt(disc);
    const double xlo = ((-a - sq) / sd(3.0)).v, xhi = ((-a + sq) / sd(3.0)).v;
    const double plo = cubic_eval(a, b, c, sd(xlo)), phi = cubic_eval(a, b, c, sd(xhi));
    if (plo < 0.0) { roots[0] = cubic_bisect(a, b, c, xhi, B); return 1; }
    if (phi > 0.0) { roots[0] = cubic_bisect(a, b, c, -B, xlo); return 1; }
    if (plo == 0.0 && phi == 0.0) { roots[0] = xlo; return 1; }
    if (plo == 0.0) { roots[0] = cubic_bisect(a, b, c, xhi, B); roots[1] = xlo; return 2; }
    if (phi == 0.0) { roots[0] = cubic_bisect(a, b, c, -B, xlo); roots[1] = xhi; return 2; }
    const double r_small = cubic_bisect(a, b, c, -B, xlo);
    const double r_mid = cubic_bisect(a, b, c, xlo, xhi);
    const double r_large = cubic_bisect(a, b, c, xhi, B);
    roots[0] = r_small; roots[1] = r_large; roots[2] = r_mid;
    return 3;
}

// Oriented epipolar constraint, fundamental_estimator.hpp:189-231 (float).
__device__ bool fundamental_is_valid(const float4* p, const float* F) {
    sf ec[3];
    ec[0] = sf(F[1]) * sf(F[8]) - sf(F[2]) * sf(F[7]);
    ec[1] = sf(F[2]) * sf(F[6]) - sf(F[0]) * sf(F[8]);
    ec[2] = sf(F[0]) * sf(F[7]) - sf(F[1]) * sf(F[6]);
    bool big = false;
#pragma unroll
    for (int i = 0; i < 3; i++)
        if ((double)ec[i].v > 1.9984e-15 || (double)ec[i].v < -1.9984e-15) { big = true; break; }
    if (!big) {
        ec[0] = sf(F[4]) * sf(F[8]) - sf(F[5]) * sf(F[7]);
        ec[1] = sf(F[5]) * sf(F[6]) - sf(F[3]) * sf(F[8]);
        ec[2] = sf(F[3]) * sf(F[7]) - sf(F[4]) * sf(F[6]);
    }
    sf sig1(0.f);
#pragma unroll
    for (int i = 0; i < 7; i++) {
        const sf y1(p[i].y), x2(p[i].z), y2(p[i].w);
        const sf s1 = sf(F[0]) * x2 + sf(F[3]) * y2 + sf(F[6]);
        const sf s2 = ec[1] - ec[2] * y1;
        const sf sig = s1 * s2;
        if (i == 0) sig1 = sig;
        else if ((sig1 * sig).v < 0.f) return false;
    }
    return true;
}

// Seven-point algorithm (seven_points.cpp:49-156) + validity filter (fundamental_estimator.hpp:48-63). DESIGN.md S3.
__device__ int solve_fundamental7(const float* __restrict__ pts, const int* s, float* out) {
    float4 p[7];
    double T[4][9], B[3][9];
#pragma unroll
    for (int i = 0; i < 7; i++) {
        p[i] = reinterpret_cast<const float4*>(pts)[s[i]];
        const sd x1((double)p[i].x), y1((double)p[i].y), x2((double)p[i].z), y2((double)p[i].w);
        GJ_AT(i, 0) = (x2 * x1).v; GJ_AT(i, 1) = (x2 * y1).v; GJ_AT(i, 2) = x2.v; GJ_AT(i, 3) = (y2 * x1).v; GJ_AT(i, 4) = (y2 * y1).v;
        GJ_AT(i, 5) = y2.v; GJ_AT(i, 6) = x1.v; GJ_AT(i, 7) = y1.v; GJ_AT(i, 8) = 1;
    }
    if (!gauss_jordan9<7>(T, B)) return 0;
    sd f1[9], f2[9];
#pragma unroll
    for (int i = 0; i < 7; i++) { f2[i] = -sd(GJ_AT(i, 8)); f1[i] = -sd(GJ_AT(i, 7)) - f2[i]; }
    f2[7] = sd(0.0); f2[8] = sd(1.0);
    f1[7] = sd(1.0) - f2[7]; f1[8] = sd(0.0) - f2[8];

    sd c[4];
    c[0] = det3(f1);
    c[3] = det3(f2);
    c[1] = sd(0.0); c[2] = sd(0.0);
    sd m[9];
#pragma unroll
    for (int row = 0; row < 3; row++) {
#pragma unroll
        for (int i = 0; i < 9; i++) m[i] = (i / 3 == row) ? f2[i] : f1[i];
        c[1] = c[1] + det3(m);
#pragma unroll
        for (int i = 0; i < 9; i++) m[i] = (i / 3 == row) ? f1[i] : f2[i];
        c[2] = c[2] + det3(m);
    }
    double r[3];
    const int nroots = solve_cubic(c, r);
    if (nroots < 1) return 0;
    int valid = 0;
    for (int k = 0; k < nroots; k++) {
        sd lambda(r[k]), mu(1.0);
        const sd sc = f1[8] * sd(r[k]) + f2[8];
        float F[9];
        if (fabs(sc.v) > 2.2204460492503131e-16) {   // DBL_EPSILON, seven_points.cpp:144
            mu = sd(1.0) / sc;
            lambda = lambda * mu;
            F[8] = 1.f;
        } else {
            F[8] = 0.f;
        }
        bool finite = true;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const double v = (f1[i] * lambda + f2[i] * mu).v;
            if (!dfinite(v)) finite = false;
            F[i] = (float)v;
        }
        if (!finite) continue;
        if (fundamental_is_valid(p, F)) {
#pragma unroll
            for (int i = 0; i < 9; i++) out[9 * valid + i] = F[i];
            valid++;
        }
    }
    return valid;
}

__device__ int solve_essential5(const float* __restrict__ pts, const int* s, float* out, int all_roots);   // essential.cuh

// out: up to 3 models (fundamental), up to USAC_E5_MAX_ROOTS with e5_all_roots, else one
template <int EST>
__device__ __forceinline__ int solve_minimal(const float* __restrict__ pts, const int* s, float* out, int e5_all_roots = 0) {
    if (EST == USAC_EST_LINE2D) return solve_line2d(pts, s, out);
    if (EST == USAC_EST_HOMOGRAPHY) return solve_homography4(pts, s, out);
    if (EST == USAC_EST_FUNDAMENTAL) return solve_fundamental7(pts, s, out);
    return solve_essential5(pts, s, out, e5_all_roots);
}
