// ref_shim_entry.cpp - C entry points over the stand-in OpenCV numerics of oracle/ref_shim/ (cvshim.hpp) alone, so that they can be
// held against the real OpenCV (tests/golden/svd_cv.npz, eig_cv.npz, cv_primitives.npz) without the reference's sources. Built by
// oracle/Makefile into libref_shim.so with the flags of the reference build (Makefile.ref). TEST INFRASTRUCTURE ONLY.
#include <cstring>

#include "ref_shim/cvshim.hpp"

extern "C" {

// ---- the stand-in cv::SVD itself (oracle/ref_shim/cvshim.hpp), so that it can be held against the real OpenCV on the matrices the
// reference feeds it (tests/golden/svd_cv.npz): A is rows x cols in double, converted to float32 when !depth64; flags as cv::SVD
// (4 = FULL_UV). dims = {len(w), u.rows, u.cols, vt.rows, vt.cols}.
int ref_shim_svd(const double* A, int rows, int cols, int depth64, int flags, double* w, double* u, double* vt, int* dims) {
    cv::Mat M(rows, cols, depth64 ? CV_64F : CV_32F);
    for (int r = 0; r < rows; r++)
        for (int c = 0; c < cols; c++) {
            if (depth64) M.at<double>(r, c) = A[(size_t)r * cols + c];
            else M.at<float>(r, c) = (float)A[(size_t)r * cols + c];
        }
    cv::Mat W, U, Vt;
    cv::SVD::compute(M, W, U, Vt, flags);
    auto get = [&](const cv::Mat& m, int r, int c) { return depth64 ? m.at<double>(r, c) : (double)m.at<float>(r, c); };
    dims[0] = W.rows * W.cols; dims[1] = U.rows; dims[2] = U.cols; dims[3] = Vt.rows; dims[4] = Vt.cols;
    for (int i = 0; i < dims[0]; i++) w[i] = W.rows > 1 ? get(W, i, 0) : get(W, 0, i);
    for (int r = 0; r < U.rows; r++) for (int c = 0; c < U.cols; c++) u[(size_t)r * U.cols + c] = get(U, r, c);
    for (int r = 0; r < Vt.rows; r++) for (int c = 0; c < Vt.cols; c++) vt[(size_t)r * Vt.cols + c] = get(Vt, r, c);
    return 0;
}

// ---- the other stand-in numerical routines the path calls: cv::eigen (line2d_estimator.hpp:93), cv::solveCubic (seven_points.cpp:131),
// cv::invert / Mat::inv of a float 3 x 3 (homography_estimator.hpp:35) - held against cv2 fixtures in tests/test_ref_build.py
int ref_shim_eigen(const double* A, int n, int depth64, double* evals, double* evecs) {
    cv::Mat M(n, n, depth64 ? CV_64F : CV_32F);
    for (int r = 0; r < n; r++)
        for (int c = 0; c < n; c++) { if (depth64) M.at<double>(r, c) = A[r * n + c]; else M.at<float>(r, c) = (float)A[r * n + c]; }
    cv::Mat D, V;
    if (!cv::eigen(M, D, V)) return 0;
    for (int i = 0; i < n; i++) {
        evals[i] = depth64 ? D.at<double>(i) : (double)D.at<float>(i);
        for (int c = 0; c < n; c++) evecs[i * n + c] = depth64 ? V.at<double>(i, c) : (double)V.at<float>(i, c);
    }
    return 1;
}
int ref_shim_cubic(const double* coeffs4, double* roots3) {
    cv::Mat_<double> c(1, 4), r(1, 3);
    for (int i = 0; i < 4; i++) c(0, i) = coeffs4[i];
    for (int i = 0; i < 3; i++) r(0, i) = 0;
    const int n = cv::solveCubic(c, r);
    for (int i = 0; i < 3; i++) roots3[i] = r(0, i);
    return n;
}
int ref_shim_inv3(const float* in9, float* out9) {
    cv::Mat_<float> m(3, 3);
    std::memcpy(m.data, in9, 36);
    cv::Mat inv = m.inv();
    for (int i = 0; i < 9; i++) out9[i] = inv.at<float>(i);
    return 0;
}

}   // extern "C"
