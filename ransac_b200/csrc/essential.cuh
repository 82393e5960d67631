// essential.cuh - five-point essential-matrix solver, one thread per sample, double precision, strict IEEE arithmetic.
//
// Replaces EssentialEstimator::EstimateModel -> EssentialSolver::FivePoints -> Solve5PointEssential
// (essential_estimator.hpp:52-62, essential/five_points.cpp:13-274): 5x9 design matrix (:48-63), 4-D null space
// E = x*B0 + y*B1 + z*B2 + B3 (:65-105), the ten cubic constraints 2EE'E - tr(EE')E = 0, det E = 0 as a 10x10 matrix M(z) over
// [x^3 y^3 x^2y xy^2 x^2 y^2 xy x y 1] (essential/mblock.hpp), det M(z) by interpolation (:117-138), its real roots
// (:140-157), per root the null vector of M(z) -> x, y -> E (:181-204) and the cheirality vote of the five points over the
// four (R, t) decompositions (:206-252); 0 or 1 model, cast to float (:28).
//
// Deterministic choices where the reference depends on cv::SVD / Jenkins-Traub internals (DESIGN.md section 4.5): null
// spaces by Gauss-Jordan with partial pivoting, made orthonormal by modified Gram-Schmidt; two interpolations on 11 nodes
// in [-1, 1] (p(z) for |z| <= 1.05, the reversed polynomial for the rest) by Newton divided differences; real roots by
// derivative bracketing + bisection, visited by ascending |z|; eight Gauss-Newton steps on the ten constraints per root;
// closed-form (R, t) = (cof(E) -/+ [t]x E, +/-t) and least-squares depths for the vote. Operation order is a contract with
// the host restatement used by the parity tests: the models are bit-identical.
#pragma once
#include "strict_math.cuh"

namespace e5 {

__device__ __constant__ signed char MONO[20][3] = {{3, 0, 0}, {0, 3, 0}, {2, 1, 0}, {1, 2, 0}, {2, 0, 0}, {2, 0, 1}, {0, 2, 0}, {0, 2, 1}, {1, 1, 0}, {1, 1, 1},
                                                   {1, 0, 0}, {1, 0, 1}, {1, 0, 2}, {0, 1, 0}, {0, 1, 1}, {0, 1, 2}, {0, 0, 0}, {0, 0, 1}, {0, 0, 2}, {0, 0, 3}};
__device__ __constant__ signed char COL_FIRST[10] = {0, 1, 2, 3, 4, 6, 8, 10, 13, 16};
__device__ __constant__ signed char COL_DEG[10] = {0, 0, 0, 0, 1, 1, 1, 2, 2, 3};
__device__ __constant__ signed char LL[4][4] = {{0, 3, 4, 6}, {3, 1, 5, 7}, {4, 5, 2, 8}, {6, 7, 8, 9}};                 // linear x linear -> quadratic
__device__ __constant__ signed char QL[10][4] = {{0, 2, 5, 4}, {3, 1, 7, 6}, {12, 15, 19, 18}, {2, 3, 9, 8}, {5, 9, 12, 11},
                                                 {9, 7, 15, 14}, {4, 8, 11, 10}, {8, 6, 14, 13}, {11, 14, 18, 17}, {10, 13, 17, 16}};   // quadratic x linear -> cubic

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
// one copy of the IEEE division sequence: the solver is ~11 000 instructions when everything is inlined, more than the instruction
// cache holds - the warps of an SM are at different places of it and 'no instruction' was the top stall reason (ncu)
__device__ __noinline__ double dvd(double a, double b) { return __ddiv_rn(a, b); }

__device__ __noinline__ void acc_ll(double* q, const double* a, const double* b, double s) {
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) { const int k = LL[i][j]; q[k] = add(q[k], mul(mul(a[i], b[j]), s)); }
}
__device__ __noinline__ void acc_ql(double* c, const double* q, const double* l, double s) {
    for (int i = 0; i < 10; i++)
        for (int j = 0; j < 4; j++) { const int k = QL[i][j]; c[k] = add(c[k], mul(mul(q[i], l[j]), s)); }
}

__device__ __noinline__ double det_lu(double* a, int n) {
    double det = 1.0;
#pragma unroll 1
    for (int k = 0; k < n; k++) {
        int piv = k;
        double best = fabs(a[k * n + k]);
        for (int r = k + 1; r < n; r++) { const double v = fabs(a[r * n + k]); if (v > best) { best = v; piv = r; } }
        if (!(best > 0.0)) return 0.0;
        if (piv != k) { for (int j = 0; j < n; j++) { const double t = a[k * n + j]; a[k * n + j] = a[piv * n + j]; a[piv * n + j] = t; } det = -det; }
        det = mul(det, a[k * n + k]);
        const double inv = dvd(1.0, a[k * n + k]);
        for (int r = k + 1; r < n; r++) {
            const double f = mul(a[r * n + k], inv);
            for (int j = k + 1; j < n; j++) a[r * n + j] = sub(a[r * n + j], mul(f, a[k * n + j]));
        }
    }
    return det;
}

__device__ __noinline__ double horner(const double* c, int deg, double x) {
    double v = c[deg];
    for (int i = deg - 1; i >= 0; i--) v = add(mul(v, x), c[i]);
    return v;
}
__device__ __noinline__ double horner_rev(const double* c, int deg, double w) {
    double v = c[0];
    for (int i = 1; i <= deg; i++) v = add(mul(v, w), c[i]);
    return v;
}

// safeguarded Newton (see the host restatement): Newton steps inside the bracket, bisection when Newton leaves it or stops halving it
__device__ __noinline__ double bisect(const double* c, const double* dc, int deg, double l, double r, double pl) {
    if (pl == 0.0) return l;
    double xl = pl < 0.0 ? l : r, xh = pl < 0.0 ? r : l;
    double x = mul(0.5, add(l, r)), dxold = fabs(sub(r, l)), dx = dxold;
    double f = horner(c, deg, x), df = horner(dc, deg - 1, x);
    for (int it = 0; it < 200; it++) {
        if (f == 0.0) return x;
        const double a = sub(mul(sub(x, xh), df), f), b = sub(mul(sub(x, xl), df), f);
        const bool newton = (mul(a, b) <= 0.0) && (fabs(mul(2.0, f)) <= fabs(mul(dxold, df)));
        dxold = dx;
        if (!newton) {
            dx = mul(0.5, sub(xh, xl));
            x = add(xl, dx);
            if (xl == x) return x;
        } else {
            dx = dvd(f, df);
            const double t = x;
            x = sub(x, dx);
            if (t == x) return x;
        }
        if (fabs(dx) <= mul(4.4e-16, fabs(x))) return x;
        f = horner(c, deg, x);
        df = horner(dc, deg - 1, x);
        if (f < 0.0) xl = x; else xh = x;
    }
    return x;
}

__device__ int real_roots(const double* c, int deg, double* roots) {
    if (deg < 1) return 0;
    double bound = 0.0;
    for (int i = 0; i < deg; i++) { const double v = fabs(dvd(c[i], c[deg])); if (v > bound) bound = v; }
    bound = add(bound, 1.0);
    if (!(bound < 1e300)) return 0;
    double der[11][11];
    for (int i = 0; i <= deg; i++) der[deg][i] = c[i];
    for (int d = deg; d > 1; d--)
        for (int i = 0; i < d; i++) der[d - 1][i] = mul(der[d][i + 1], (double)(i + 1));
    double prev[11], cur[11];
    int nprev = 1;
    prev[0] = -dvd(der[1][0], der[1][1]);
    if (!(fabs(prev[0]) <= bound)) nprev = 0;
    for (int d = 2; d <= deg; d++) {
        const double* p = der[d];
        int ncur = 0;
        double left = -bound, pl = horner(p, d, left);
        for (int s = 0; s <= nprev; s++) {
            const double right = s < nprev ? prev[s] : bound;
            const double pr = horner(p, d, right);
            if (pl == 0.0) { cur[ncur++] = left; }
            else if (pr != 0.0 && ((pl < 0.0) != (pr < 0.0))) { cur[ncur++] = bisect(p, der[d - 1], d, left, right, pl); }
            left = right; pl = pr;
        }
        if (pl == 0.0) cur[ncur++] = left;
        for (int i = 0; i < ncur; i++) prev[i] = cur[i];
        nprev = ncur;
    }
    for (int i = 0; i < nprev; i++) roots[i] = prev[i];
    return nprev;
}

// Gauss-Jordan null space of the 5 x 9 design matrix (rows x 9, row-major, destroyed): same operations as gauss_jordan9
// and as the host restatement; basis vector q has v[5+q] = 1, v[i<5] = -A[i][5+q].
__device__ __noinline__ bool null_space5(double* A, double* basis) {
#pragma unroll 1
    for (int k = 0; k < 5; k++) {
        int piv = k;
        double best = fabs(A[k * 9 + k]);
        for (int r = k + 1; r < 5; r++) { const double v = fabs(A[r * 9 + k]); if (v > best) { best = v; piv = r; } }
        if (!(best > 0.0) || !dfinite(best)) return false;
        if (piv != k) for (int j = 0; j < 9; j++) { const double t = A[k * 9 + j]; A[k * 9 + j] = A[piv * 9 + j]; A[piv * 9 + j] = t; }
        const double inv = dvd(1.0, A[k * 9 + k]);
        for (int j = k + 1; j < 9; j++) A[k * 9 + j] = mul(A[k * 9 + j], inv);
        for (int r = 0; r < 5; r++) {
            if (r == k) continue;
            const double f = A[r * 9 + k];
            for (int j = k + 1; j < 9; j++) A[r * 9 + j] = sub(A[r * 9 + j], mul(f, A[k * 9 + j]));
        }
    }
    for (int q = 0; q < 4; q++) {
        double* v = basis + q * 9;
        for (int i = 0; i < 5; i++) v[i] = -A[i * 9 + 5 + q];
        for (int i = 5; i < 9; i++) v[i] = (i == 5 + q) ? 1.0 : 0.0;
    }
    return true;
}

}  // namespace e5

// ---------------------------------------------------------------------------------------------------------------
// The solver in stages. The one-thread form (solve_essential5) runs them in sequence; the one-warp form
// (solve_essential5_warp) spreads the independent pieces over the lanes - 22 determinants, the root brackets of every
// derivative level, the candidate roots - each piece still evaluated by ONE lane with the same operations in the same
// order, so both forms (and the host restatement of the parity tests) return bit-identical models.
// ---------------------------------------------------------------------------------------------------------------
namespace e5 {

// stage 1: points -> X = [x1[5] y1[5] x2[5] y2[5]], L[9][4] (E_ij as linear forms), C[10][20] (the ten cubic constraints)
// stage 1 in pieces (the warp form runs the nine Q blocks and the ten constraint rows on separate lanes; the one-thread form calls
// them in a loop - the same operations in the same order per block / row)
__device__ __noinline__ bool stage_basis(const float* __restrict__ pts, const int* s, double* X, double (*L)[4]) {
    double A[45];
    double *x1 = X, *y1 = X + 5, *x2 = X + 10, *y2 = X + 15;
#pragma unroll 1
    for (int i = 0; i < 5; i++) {
        const float4 p = reinterpret_cast<const float4*>(pts)[s[i]];
        x1[i] = p.x; y1[i] = p.y; x2[i] = p.z; y2[i] = p.w;
        double* r = A + 9 * i;
        r[0] = mul(x1[i], x2[i]); r[1] = mul(x2[i], y1[i]); r[2] = x2[i]; r[3] = mul(x1[i], y2[i]); r[4] = mul(y1[i], y2[i]); r[5] = y2[i];
        r[6] = x1[i]; r[7] = y1[i]; r[8] = 1.0;
    }
    double Bs[36];
    if (!null_space5(A, Bs)) return false;
#pragma unroll 1
    for (int a = 3; a >= 0; a--) {                                        // modified Gram-Schmidt, last vector first
        double* v = Bs + 9 * a;
#pragma unroll 1
        for (int b = 3; b > a; b--) {
            const double* u = Bs + 9 * b;
            double dot = 0.0;
            for (int e = 0; e < 9; e++) dot = add(dot, mul(v[e], u[e]));
            for (int e = 0; e < 9; e++) v[e] = sub(v[e], mul(dot, u[e]));
        }
        double nn = 0.0;
        for (int e = 0; e < 9; e++) nn = add(nn, mul(v[e], v[e]));
        if (!(nn > 0.0)) return false;
        const double inv = dvd(1.0, __dsqrt_rn(nn));
        for (int e = 0; e < 9; e++) v[e] = mul(v[e], inv);
    }
    for (int e = 0; e < 9; e++) for (int q = 0; q < 4; q++) L[e][q] = Bs[q * 9 + e];
    return true;
}
// Q[i][j] = sum_k L[3i+k] x L[3j+k] (quadratic forms of E E'): block b = 3 i + j -> Qb[10]
__device__ __noinline__ void stage_q_block(const double (*L)[4], int b, double* Qb) {
    const int i = b / 3, j = b % 3;
    for (int m = 0; m < 10; m++) Qb[m] = 0.0;
#pragma unroll 1
    for (int k = 0; k < 3; k++) acc_ll(Qb, L[3 * i + k], L[3 * j + k], 1.0);
}
// constraint row r < 9 (2 E E' E - tr(E E') E, entry (i, j) = (r / 3, r % 3)) or r = 9 (det E): Cr[20]
__device__ __noinline__ void stage_c_row(const double (*L)[4], const double* Q /* [9][10] */, const double* tr, int r, double* Cr) {
    for (int m = 0; m < 20; m++) Cr[m] = 0.0;
    if (r < 9) {
        const int i = r / 3, j = r % 3;
#pragma unroll 1
        for (int k = 0; k < 3; k++) acc_ql(Cr, Q + 10 * (3 * i + k), L[3 * k + j], 2.0);
        acc_ql(Cr, tr, L[3 * i + j], -1.0);
    } else {
        double m0[10], m1[10], m2[10];
        for (int m = 0; m < 10; m++) { m0[m] = 0.0; m1[m] = 0.0; m2[m] = 0.0; }
        acc_ll(m0, L[4], L[8], 1.0); acc_ll(m0, L[5], L[7], -1.0);
        acc_ll(m1, L[3], L[8], 1.0); acc_ll(m1, L[5], L[6], -1.0);
        acc_ll(m2, L[3], L[7], 1.0); acc_ll(m2, L[4], L[6], -1.0);
        acc_ql(Cr, m0, L[0], 1.0); acc_ql(Cr, m1, L[1], -1.0); acc_ql(Cr, m2, L[2], 1.0);
    }
}
__device__ bool stage_constraints(const float* __restrict__ pts, const int* s, double* X, double (*L)[4], double (*C)[20]) {
    if (!stage_basis(pts, s, X, L)) return false;
    double Q[90], tr[10];
#pragma unroll 1
    for (int b = 0; b < 9; b++) stage_q_block(L, b, Q + 10 * b);
    for (int m = 0; m < 10; m++) tr[m] = add(add(Q[m], Q[40 + m]), Q[80 + m]);
#pragma unroll 1
    for (int r = 0; r < 10; r++) stage_c_row(L, Q, tr, r, C[r]);
    return true;
}

// stage 2: det M(z) (pass 0) or det(M(1/w) diag(w^deg)) (pass 1) at node t of the 11 equispaced nodes in [-1, 1]
__device__ __noinline__ double stage_det(const double (*C)[20], int pass, int t) {
    double Mz[100];
    const double z = dvd((double)(t - 5), 5.0);
#pragma unroll 1
    for (int r = 0; r < 10; r++)
#pragma unroll 1
        for (int c = 0; c < 10; c++)
            Mz[r * 10 + c] = pass == 0 ? horner(&C[r][COL_FIRST[c]], COL_DEG[c], z) : horner_rev(&C[r][COL_FIRST[c]], COL_DEG[c], z);
    return det_lu(Mz, 10);
}

// stage 3: 11 determinant values -> monomial coefficients (Newton divided differences); returns the degree after trimming,
// 0 when there is nothing to solve, -1 when a coefficient is not finite (the solver then returns no model)
__device__ __noinline__ int stage_coefficients(double* dd, double* coef) {
    double zs[11];
    for (int t = 0; t < 11; t++) zs[t] = dvd((double)(t - 5), 5.0);
#pragma unroll 1
    for (int lev = 1; lev < 11; lev++)
#pragma unroll 1
        for (int t = 10; t >= lev; t--) dd[t] = dvd(sub(dd[t], dd[t - 1]), sub(zs[t], zs[t - lev]));
    for (int i = 0; i < 11; i++) coef[i] = 0.0;
    coef[0] = dd[10];
#pragma unroll 1
    for (int t = 9; t >= 0; t--) {
        for (int i = 10; i >= 1; i--) coef[i] = sub(coef[i - 1], mul(coef[i], zs[t]));
        coef[0] = sub(dd[t], mul(coef[0], zs[t]));
    }
    int deg = 10;
    double cmax = 0.0;
    bool finite = true;
    for (int i = 0; i <= 10; i++) { if (!dfinite(coef[i])) finite = false; if (fabs(coef[i]) > cmax) cmax = fabs(coef[i]); }
    if (!finite) return -1;
    while (deg > 0 && !(fabs(coef[deg]) > mul(1e-13, cmax))) deg--;
    return deg;
}

// stage 4 helper: keep the roots of pass 0 with |z| <= 1.05 and the reciprocals of the roots of pass 1 with |w| < 1/1.05
__device__ int stage_collect(int pass, const double* rr, int nr, double* roots, int nroots) {
    for (int i = 0; i < nr; i++) {
        if (pass == 0) { if (fabs(rr[i]) <= 1.05) roots[nroots++] = rr[i]; }
        else if (fabs(rr[i]) < dvd(1.0, 1.05) && rr[i] != 0.0) roots[nroots++] = dvd(1.0, rr[i]);
    }
    return nroots;
}
__device__ void stage_sort(double* roots, int& nroots) {                 // ascending |z|, stable
    if (nroots > 10) nroots = 10;
    for (int i = 1; i < nroots; i++) {
        const double v = roots[i];
        int j = i - 1;
        while (j >= 0 && fabs(roots[j]) > fabs(v)) { roots[j + 1] = roots[j]; j--; }
        roots[j + 1] = v;
    }
}

// stage 5: one root z -> x, y (Gauss-Jordan on [M(z) | last column]), eight Gauss-Newton steps, E, cheirality vote.
// In pieces, so that the warp form can spread the Gauss-Newton rows of all roots over its lanes: the pieces do the same
// operations in the same order whoever calls them.
__device__ __noinline__ bool stage_root_init(const double (*C)[20], double z, double* u) {
    double Mz[100];
#pragma unroll 1
    for (int r = 0; r < 10; r++)
#pragma unroll 1
        for (int c = 0; c < 10; c++) Mz[r * 10 + c] = horner(&C[r][COL_FIRST[c]], COL_DEG[c], z);
#pragma unroll 1
    for (int k = 0; k < 9; k++) {
        int piv = k;
        double best = fabs(Mz[k * 10 + k]);
        for (int r = k + 1; r < 10; r++) { const double v = fabs(Mz[r * 10 + k]); if (v > best) { best = v; piv = r; } }
        if (!(best > 0.0) || !dfinite(best)) return false;
        if (piv != k) for (int j = 0; j < 10; j++) { const double t = Mz[k * 10 + j]; Mz[k * 10 + j] = Mz[piv * 10 + j]; Mz[piv * 10 + j] = t; }
        const double inv = dvd(1.0, Mz[k * 10 + k]);
        for (int j = k + 1; j < 10; j++) Mz[k * 10 + j] = mul(Mz[k * 10 + j], inv);
        for (int r = 0; r < 10; r++) {
            if (r == k) continue;
            const double f = Mz[r * 10 + k];
            for (int j = k + 1; j < 10; j++) Mz[r * 10 + j] = sub(Mz[r * 10 + j], mul(f, Mz[k * 10 + j]));
        }
    }
    u[0] = -Mz[7 * 10 + 9]; u[1] = -Mz[8 * 10 + 9]; u[2] = z;
    return true;
}
// value and gradient of constraint row `Cr` (20 monomial coefficients) at u: out = {val, g0, g1, g2}
__device__ __noinline__ void stage_gn_row(const double* Cr, const double* u, double* out) {
    double pw[3][4];
    for (int a = 0; a < 3; a++) { pw[a][0] = 1.0; pw[a][1] = u[a]; pw[a][2] = mul(u[a], u[a]); pw[a][3] = mul(pw[a][2], u[a]); }
    double val = 0.0, g[3] = {0, 0, 0};
#pragma unroll 1
    for (int m = 0; m < 20; m++) {
        const int e[3] = {MONO[m][0], MONO[m][1], MONO[m][2]};
        const double c = Cr[m];
        val = add(val, mul(c, mul(mul(pw[0][e[0]], pw[1][e[1]]), pw[2][e[2]])));
        for (int a = 0; a < 3; a++) {
            if (e[a] == 0) continue;
            double t = (double)e[a];
            for (int b = 0; b < 3; b++) t = mul(t, pw[b][b == a ? e[b] - 1 : e[b]]);
            g[a] = add(g[a], mul(c, t));
        }
    }
    out[0] = val; out[1] = g[0]; out[2] = g[1]; out[3] = g[2];
}
// one Gauss-Newton update from the ten rows (rows[r] = {val, g0, g1, g2}, added in row order); false = the iteration stops here
__device__ __noinline__ bool stage_gn_step(const double* rows, double* u) {
    double JtJ[6] = {0, 0, 0, 0, 0, 0}, Jtr[3] = {0, 0, 0};
    for (int r = 0; r < 10; r++) {
        const double val = rows[4 * r], g[3] = {rows[4 * r + 1], rows[4 * r + 2], rows[4 * r + 3]};
        JtJ[0] = add(JtJ[0], mul(g[0], g[0])); JtJ[1] = add(JtJ[1], mul(g[0], g[1])); JtJ[2] = add(JtJ[2], mul(g[0], g[2]));
        JtJ[3] = add(JtJ[3], mul(g[1], g[1])); JtJ[4] = add(JtJ[4], mul(g[1], g[2])); JtJ[5] = add(JtJ[5], mul(g[2], g[2]));
        Jtr[0] = add(Jtr[0], mul(g[0], val)); Jtr[1] = add(Jtr[1], mul(g[1], val)); Jtr[2] = add(Jtr[2], mul(g[2], val));
    }
    const double a = JtJ[0], b = JtJ[1], c = JtJ[2], d = JtJ[3], e = JtJ[4], f = JtJ[5];
    const double c00 = sub(mul(d, f), mul(e, e)), c01 = sub(mul(c, e), mul(b, f)), c02 = sub(mul(b, e), mul(c, d));
    const double c11 = sub(mul(a, f), mul(c, c)), c12 = sub(mul(b, c), mul(a, e)), c22 = sub(mul(a, d), mul(b, b));
    const double det = add(add(mul(a, c00), mul(b, c01)), mul(c, c02));
    if (!(fabs(det) > 0.0) || !dfinite(det)) return false;
    const double dx = dvd(add(add(mul(c00, Jtr[0]), mul(c01, Jtr[1])), mul(c02, Jtr[2])), det);
    const double dy = dvd(add(add(mul(c01, Jtr[0]), mul(c11, Jtr[1])), mul(c12, Jtr[2])), det);
    const double dz = dvd(add(add(mul(c02, Jtr[0]), mul(c12, Jtr[1])), mul(c22, Jtr[2])), det);
    if (!dfinite(dx) || !dfinite(dy) || !dfinite(dz)) return false;
    u[0] = sub(u[0], dx); u[1] = sub(u[1], dy); u[2] = sub(u[2], dz);
    return true;
}
__device__ __noinline__ bool stage_root_finish(const double (*L)[4], const double* X, const double* u, double* E) {
    const double *x1 = X, *y1 = X + 5, *x2 = X + 10, *y2 = X + 15;
    bool finite = true;
    for (int e = 0; e < 9; e++) {
        double v = mul(L[e][0], u[0]);
        v = add(v, mul(L[e][1], u[1]));
        v = add(v, mul(L[e][2], u[2]));
        v = add(v, L[e][3]);
        E[e] = v;
        if (!dfinite(v)) finite = false;
    }
    if (!finite) return false;
    double n2 = 0.0;
    for (int e = 0; e < 9; e++) n2 = add(n2, mul(E[e], E[e]));
    const double sc = __dsqrt_rn(mul(0.5, n2));
    if (!(sc > 0.0)) return false;
    double En[9];
    for (int e = 0; e < 9; e++) En[e] = dvd(E[e], sc);
    double tv[3] = {0, 0, 0}, tbest = -1.0;
    for (int a = 0; a < 3; a++) {
        const int b = (a + 1) % 3;
        const double cx = sub(mul(En[3 + a], En[6 + b]), mul(En[6 + a], En[3 + b]));
        const double cy = sub(mul(En[6 + a], En[0 + b]), mul(En[0 + a], En[6 + b]));
        const double cz = sub(mul(En[0 + a], En[3 + b]), mul(En[3 + a], En[0 + b]));
        const double nn = add(add(mul(cx, cx), mul(cy, cy)), mul(cz, cz));
        if (nn > tbest) { tbest = nn; tv[0] = cx; tv[1] = cy; tv[2] = cz; }
    }
    if (!(tbest > 0.0)) return false;
    { const double inv = dvd(1.0, __dsqrt_rn(tbest)); tv[0] = mul(tv[0], inv); tv[1] = mul(tv[1], inv); tv[2] = mul(tv[2], inv); }
    double cof[9], tE[9];
    cof[0] = sub(mul(En[4], En[8]), mul(En[5], En[7])); cof[1] = sub(mul(En[5], En[6]), mul(En[3], En[8])); cof[2] = sub(mul(En[3], En[7]), mul(En[4], En[6]));
    cof[3] = sub(mul(En[2], En[7]), mul(En[1], En[8])); cof[4] = sub(mul(En[0], En[8]), mul(En[2], En[6])); cof[5] = sub(mul(En[1], En[6]), mul(En[0], En[7]));
    cof[6] = sub(mul(En[1], En[5]), mul(En[2], En[4])); cof[7] = sub(mul(En[2], En[3]), mul(En[0], En[5])); cof[8] = sub(mul(En[0], En[4]), mul(En[1], En[3]));
    for (int c = 0; c < 3; c++) {
        tE[0 + c] = sub(mul(tv[1], En[6 + c]), mul(tv[2], En[3 + c]));
        tE[3 + c] = sub(mul(tv[2], En[0 + c]), mul(tv[0], En[6 + c]));
        tE[6 + c] = sub(mul(tv[0], En[3 + c]), mul(tv[1], En[0 + c]));
    }
#pragma unroll 1
    for (int cam = 0; cam < 4; cam++) {
        double R[9], t[3];
        const double rs = (cam < 2) ? -1.0 : 1.0, ts = (cam & 1) ? -1.0 : 1.0;
        for (int e = 0; e < 9; e++) R[e] = add(cof[e], mul(rs, tE[e]));
        for (int e = 0; e < 3; e++) t[e] = mul(ts, tv[e]);
        int infront = 0;
        for (int k = 0; k < 5; k++) {
            const double a0 = add(add(mul(R[0], x1[k]), mul(R[1], y1[k])), R[2]);
            const double a1 = add(add(mul(R[3], x1[k]), mul(R[4], y1[k])), R[5]);
            const double a2 = add(add(mul(R[6], x1[k]), mul(R[7], y1[k])), R[8]);
            const double b0 = x2[k], b1 = y2[k], b2 = 1.0;
            const double aa = add(add(mul(a0, a0), mul(a1, a1)), mul(a2, a2)), bb = add(add(mul(b0, b0), mul(b1, b1)), mul(b2, b2));
            const double ab = add(add(mul(a0, b0), mul(a1, b1)), mul(a2, b2));
            const double at = add(add(mul(a0, t[0]), mul(a1, t[1])), mul(a2, t[2])), bt = add(add(mul(b0, t[0]), mul(b1, t[1])), mul(b2, t[2]));
            const double det = sub(mul(aa, bb), mul(ab, ab));
            const double l1 = dvd(sub(mul(ab, bt), mul(bb, at)), det), l2 = dvd(sub(mul(aa, bt), mul(ab, at)), det);
            if (l1 > 0.0 && l2 > 0.0) infront++; else break;
        }
        if (infront == 5) return true;
    }
    return false;
}
__device__ bool stage_root(const double (*C)[20], const double (*L)[4], const double* X, double z, double* E) {
    double u[3];
    if (!stage_root_init(C, z, u)) return false;
    for (int it = 0; it < 8; it++) {                                  // Gauss-Newton on the ten constraints
        double rows[40];
        for (int r = 0; r < 10; r++) stage_gn_row(C[r], u, rows + 4 * r);
        if (!stage_gn_step(rows, u)) break;
    }
    return stage_root_finish(L, X, u, E);
}

}  // namespace e5

// one thread per sample. all_roots = 0: the first root that passes the cheirality vote (the reference's rule), out[9];
// all_roots = 1: every such root in visiting order, out[k * 9], k <= 10
__device__ __noinline__ int solve_essential5(const float* __restrict__ pts, const int* s, float* out, int all_roots) {
    using namespace e5;
    double X[20], L[9][4], C[10][20];
    if (!stage_constraints(pts, s, X, L, C)) return 0;
    double roots[20];
    int nroots = 0;
    for (int pass = 0; pass < 2; pass++) {
        double dd[11], coef[11], rr[10];
        for (int t = 0; t < 11; t++) dd[t] = stage_det(C, pass, t);
        const int deg = stage_coefficients(dd, coef);
        if (deg < 0) return 0;
        if (deg < 1) continue;
        const int nr = real_roots(coef, deg, rr);
        nroots = stage_collect(pass, rr, nr, roots, nroots);
    }
    stage_sort(roots, nroots);
    int k = 0;
    for (int ri = 0; ri < nroots; ri++) {
        double E[9];
        if (stage_root(C, L, X, roots[ri], E)) {
            for (int e = 0; e < 9; e++) out[9 * k + e] = (float)E[e];
            k++;
            if (!all_roots) break;
        }
    }
    return k;
}

// one warp per sample: `sm` points to E5_WARP_DOUBLES doubles of shared memory owned by this warp. Every lane returns the
// model count; the lane that owns the winning root writes `out` (all_roots: every lane with a valid root writes its E at
// out + 9 * (valid roots of the lanes below it), so the models are compacted in visiting order).
#define E5_WARP_DOUBLES (20 + 36 + 200 + 22 + 22 + 242 + 24 + 24 + 20 + 60 + 800)
__device__ int solve_essential5_warp(const float* __restrict__ pts, const int* s, float* out, double* sm, int all_roots) {
    using namespace e5;
    const int lane = threadIdx.x & 31;
    double* X = sm;                                                    // 20
    double (*L)[4] = reinterpret_cast<double (*)[4]>(sm + 20);         // 36
    double (*C)[20] = reinterpret_cast<double (*)[20]>(sm + 56);       // 200
    double* dd = sm + 256;                                             // 2 x 11
    double* coef = sm + 278;                                           // 2 x 11
    double* der = sm + 300;                                            // 2 x 11 x 11 derivative tables
    double* prev = sm + 542;                                           // 2 x 12 roots of the previous level
    double* cur = sm + 566;                                            // 2 x 12
    double* roots = sm + 590;                                          // 20
    double* U = sm + 610;                                              // 20 x 3 Gauss-Newton iterates of the roots
    double* rows = sm + 670;                                           // 20 roots x 10 constraint rows x {val, g0, g1, g2}
    __shared__ int sh_i[8][8];                                         // per warp: ok, deg0, deg1, nprev0, nprev1, nroots
    int* si = sh_i[(threadIdx.x >> 5) & 7];
    if (lane == 0) si[0] = stage_basis(pts, s, X, L) ? 1 : 0;
    __syncwarp();
    if (!si[0]) return 0;
    {                                                                  // the nine Q blocks, then the ten constraint rows, one lane each
        double* Q = rows;                                              // 90 + 10 doubles of the region stage 5 uses later
        double* tr = rows + 90;
        if (lane < 9) stage_q_block(L, lane, Q + 10 * lane);
        __syncwarp();
        if (lane < 10) tr[lane] = add(add(Q[lane], Q[40 + lane]), Q[80 + lane]);
        __syncwarp();
        if (lane < 10) stage_c_row(L, Q, tr, lane, C[lane]);
        __syncwarp();
    }
    if (lane < 22) dd[lane] = stage_det(C, lane / 11, lane % 11);
    __syncwarp();
    if (lane < 2) {
        const int deg = stage_coefficients(dd + 11 * lane, coef + 11 * lane);
        si[1 + lane] = deg;
        if (deg >= 1) {                                                // derivative tables + the root of the linear one (real_roots)
            double* D = der + 121 * lane;
            const double* c = coef + 11 * lane;
            double bound = 0.0;
            for (int i = 0; i < deg; i++) { const double v = fabs(dvd(c[i], c[deg])); if (v > bound) bound = v; }
            bound = add(bound, 1.0);
            for (int i = 0; i <= deg; i++) D[deg * 11 + i] = c[i];
            for (int d = deg; d > 1; d--)
                for (int i = 0; i < d; i++) D[(d - 1) * 11 + i] = mul(D[d * 11 + i + 1], (double)(i + 1));
            double* P = prev + 12 * lane;
            P[11] = bound;
            int np = 1;
            P[0] = -dvd(D[1 * 11 + 0], D[1 * 11 + 1]);
            if (!(fabs(P[0]) <= bound)) np = 0;
            if (!(bound < 1e300)) { np = 0; si[1 + lane] = 0; }         // real_roots returns no roots
            si[3 + lane] = np;
        }
    }
    __syncwarp();
    if (si[1] < 0 || si[2] < 0) return 0;
    // derivative levels 2..deg of both polynomials: lane (16*pass + k) owns bracket k of the level
    const int pass = lane >> 4, k = lane & 15;
    const int deg = si[1 + pass];
    const int maxdeg = max(si[1], si[2]);
    for (int d = 2; d <= maxdeg; d++) {
        bool has = false;
        double val = 0.0;
        const int np = (d <= deg) ? si[3 + pass] : 0;
        if (d <= deg && k <= np + 1) {
            const double* p = der + 121 * pass + 11 * d;
            const double* P = prev + 12 * pass;
            const double bound = P[11];
            if (k <= np) {
                const double left = k == 0 ? -bound : P[k - 1], right = k < np ? P[k] : bound;
                const double pl = horner(p, d, left), pr = horner(p, d, right);
                if (pl == 0.0) { has = true; val = left; }
                else if (pr != 0.0 && ((pl < 0.0) != (pr < 0.0))) { has = true; val = bisect(p, p - 11, d, left, right, pl); }
            } else if (horner(p, d, bound) == 0.0) { has = true; val = bound; }   // the closing `if (pl == 0.0)` of real_roots
        }
        const unsigned bal = __ballot_sync(0xffffffffu, has);
        const unsigned mine = (bal >> (16 * pass)) & 0xffffu;
        if (has) cur[12 * pass + __popc(mine & ((1u << k) - 1))] = val;
        __syncwarp();
        if (d <= deg) {
            const int nc = __popc(mine);
            if (k < nc) prev[12 * pass + k] = cur[12 * pass + k];
            if (k == 0) si[3 + pass] = nc;
        }
        __syncwarp();
    }
    if (lane == 0) {
        int nroots = 0;
        for (int ps = 0; ps < 2; ps++)
            if (si[1 + ps] >= 1) nroots = stage_collect(ps, prev + 12 * ps, si[3 + ps], roots, nroots);
        stage_sort(roots, nroots);
        si[5] = nroots;
    }
    __syncwarp();
    const int nroots = si[5];
    // stage 5 with the Gauss-Newton rows of ALL roots spread over the lanes (lane <-> (root, row), 10 rows per root), each root's
    // own lane adds its ten rows in order and updates its iterate - the arithmetic of stage_root, ~4 dependent rows instead of 10
    double u[3] = {0, 0, 0};
    bool alive = lane < nroots;
    if (alive) alive = stage_root_init(C, roots[lane], u);
    bool iterating = alive;
    for (int it = 0; it < 8; it++) {
        const unsigned going = __ballot_sync(0xffffffffu, iterating);
        if (!going) break;                                             // uniform
        if (iterating) { U[3 * lane] = u[0]; U[3 * lane + 1] = u[1]; U[3 * lane + 2] = u[2]; }
        __syncwarp();
        for (int base = 0; base < 10 * nroots; base += 32) {
            const int w = base + lane;
            if (w < 10 * nroots && ((going >> (w / 10)) & 1u)) stage_gn_row(C[w % 10], U + 3 * (w / 10), rows + 4 * w);
        }
        __syncwarp();
        if (iterating) iterating = stage_gn_step(rows + 40 * lane, u);
        __syncwarp();
    }
    double E[9];
    const bool ok = alive && stage_root_finish(L, X, u, E);
    const unsigned win = __ballot_sync(0xffffffffu, ok);
    if (!win) return 0;
    if (all_roots) {
        if (ok) {
            float* dst = out + 9 * __popc(win & ((1u << lane) - 1u));
            for (int e = 0; e < 9; e++) dst[e] = (float)E[e];
        }
        return __popc(win);
    }
    if (lane == __ffs(win) - 1) for (int e = 0; e < 9; e++) out[e] = (float)E[e];
    return 1;
}
