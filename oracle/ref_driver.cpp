// ref_driver.cpp - C entry points over the REFERENCE'S OWN classes, compiled from the sources where they lie under
// /root/reference (oracle/Makefile.ref; OpenCV / Eigen / nanoflann answered by the stand-ins in oracle/ref_shim/).
// The result, oracle/_ref/libusac_ref.so, is what the oracle restatement is validated against (tests/test_ref_build.py) and may
// serve as the CPU baseline of bench.py. TEST INFRASTRUCTURE ONLY: nothing in ransac_b200/ links or loads it.
//
// `private`/`protected` are opened for this translation unit so that the tests can read the state the reference keeps
// private (the SPRT pool and test history, the samplers' counters); no reference code is modified.
#include <algorithm>
#include <cassert>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <map>
#include <memory>
#include <random>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>
#include <omp.h>
#include "ref_shim/cvshim.hpp"
#include "ref_shim/Eigen/Dense"
#include "ref_shim/nanoflann.hpp"
#define private public
#define protected public
#include "usac/ransac/ransac.hpp"
#include "usac/estimator/essential/rpoly.hpp"
#include "usac/utils/utils.hpp"
#undef private
#undef protected

#include <cstdint>
#include <cstring>

namespace {
cv::Mat borrow(const float* pts, int n, int dim) { return cv::Mat(n, dim, CV_32F, const_cast<float*>(pts)); }
ESTIMATOR est_of(int e) { return e == 1 ? Line2d : e == 2 ? Homography : e == 3 ? Fundamental : Essential; }
int sample_size_of(int e) { return e == 1 ? 2 : e == 2 ? 4 : e == 3 ? 7 : 5; }
cv::Mat model_mat(int est, const float* m) {
    cv::Mat_<float> d = est == 1 ? cv::Mat_<float>(1, 3) : cv::Mat_<float>(3, 3);
    std::memcpy(d.data, m, sizeof(float) * (est == 1 ? 3 : 9));
    return d;
}
Estimator* make_estimator(int est, const cv::Mat& pts) {
    Estimator* e = nullptr;
    initEstimator(e, est_of(est), pts);                              // init.cpp:3-21
    return e;
}
}   // namespace

extern "C" {

// ---- Estimator::GetError for every point (homography/fundamental/essential/line2d_estimator.hpp) -------------------------------
int ref_errors(int est, const float* pts, int n, const float* model, float* out) {
    cv::Mat P = borrow(pts, n, est == 1 ? 2 : 4);
    Estimator* e = make_estimator(est, P);
    e->setModelParameters(model_mat(est, model));
    for (int i = 0; i < n; i++) out[i] = e->GetError((unsigned)i);
    delete e;
    return 0;
}

// ---- Quality::getNumberInliers (quality.hpp:60-101) ---------------------------------------------------------------------------
int ref_score(int est, const float* pts, int n, const float* model, float thr, int* count, float* sum, int* ids) {
    cv::Mat P = borrow(pts, n, est == 1 ? 2 : 4);
    Estimator* e = make_estimator(est, P);
    Quality q;
    q.init((unsigned)n, thr, e);
    Score s;
    q.getNumberInliers(&s, model_mat(est, model), thr, ids != nullptr, ids);
    *count = s.inlier_number; *sum = s.score;
    delete e;
    return 0;
}

// ---- Estimator::EstimateModel (estimator.hpp:19): up to 10 model slots like ransac.cpp:19-33 ------------------------------------
int ref_solve_minimal(int est, const float* pts, int n, const int* sample, float* models_out) {
    cv::Mat P = borrow(pts, n, est == 1 ? 2 : 4);
    Estimator* e = make_estimator(est, P);
    Model cfg(2.f, (unsigned)sample_size_of(est), 0.95f, 5, est_of(est), Uniform);
    std::vector<Model*> models;
    for (int i = 0; i < 10; i++) models.push_back(new Model(&cfg));
    const unsigned k = e->EstimateModel(sample, models);
    const int w = est == 1 ? 3 : 9;
    for (unsigned i = 0; i < k; i++) {
        cv::Mat d = models[i]->returnDescriptor();
        for (int j = 0; j < w; j++) models_out[9 * i + j] = d.at<float>(j);
    }
    for (Model* m : models) delete m;
    delete e;
    return (int)k;
}

// ---- Estimator::EstimateModelNonMinimalSample (estimator.hpp:22) ----------------------------------------------------------------
int ref_nonminimal(int est, const float* pts, int n, const int* ids, int count, float* model_out) {
    cv::Mat P = borrow(pts, n, est == 1 ? 2 : 4);
    Estimator* e = make_estimator(est, P);
    Model cfg(2.f, (unsigned)sample_size_of(est), 0.95f, 5, est_of(est), Uniform);
    Model out(&cfg);
    const bool ok = e->EstimateModelNonMinimalSample(ids, (unsigned)count, out);
    if (ok) { cv::Mat d = out.returnDescriptor(); for (int j = 0; j < (est == 1 ? 3 : 9); j++) model_out[j] = d.at<float>(j); }
    delete e;
    return ok ? 1 : 0;
}

// ---- StandardTerminationCriteria::getUpBoundIterations (standard_termination_criteria.hpp:52-62) -------------------------------
unsigned ref_standard_termination(unsigned inliers, unsigned n, int m, float conf, unsigned max_it) {
    Model cfg(2.f, (unsigned)m, conf, 5, Homography, Uniform);
    cfg.max_iterations = max_it;
    StandardTerminationCriteria t(&cfg, n);
    return t.getUpBoundIterations(inliers);
}

// ---- UniformSampler (uniform_sampler.hpp:42-54) over glibc random() seeded with srand(seed) ----------------------------------
void ref_uniform_samples(unsigned seed, int n, int m, int K, int* out) {
    srand(seed);
    UniformSampler s(false);
    s.setSampleSize((unsigned)m);
    s.setPointsSize((unsigned)n);
    for (int j = 0; j < K; j++) s.generateSample(out + (size_t)j * m);
}

// ---- ProsacSampler (prosac_sampler.hpp:62-172): growth function, and K samples with the termination length held at
// `termination_length` (0 = n); subset_out[j] / hyp_out[j] = the sampler's subset size and counter t after sample j ------------
void ref_prosac_samples(unsigned rd_seed, int n, int m, int K, unsigned termination_length, int* out, unsigned* growth_out,
                        unsigned* subset_out, unsigned* hyp_out, unsigned* largest_out) {
    usac_ref_random_device_seed() = rd_seed;
    ProsacSampler s;
    s.initProsacSampler((unsigned)m, (unsigned)n);
    unsigned tl = termination_length ? termination_length : (unsigned)n;
    s.setTerminationLength(&tl);
    for (int i = 0; i < n; i++) growth_out[i] = s.getGrowthFunction()[i];
    for (int j = 0; j < K; j++) {
        s.generateSample(out + (size_t)j * m);
        subset_out[j] = s.subset_size; hyp_out[j] = s.hypCount; largest_out[j] = s.largest_sample_size;
    }
}

// ---- SPRT (sprt.hpp): the pool shuffle of the constructor under srand(seed), then verifyModelAndGetModelScore over a given
// sequence of models. Model q is hypothesis hyp[q]; `maximum_score` is the running best like ransac.cpp:73,103-118. ------------
int ref_sprt_sequence(int est, const float* pts, int n, float thr, unsigned seed, unsigned max_it, const float* models, int M, const int* hyp,
                      int* good_out, int* inl_out, unsigned* pool_idx_after, unsigned* bound_after, double* hist_out, int* nhist, int* pool_out) {
    cv::Mat P = borrow(pts, n, est == 1 ? 2 : 4);
    Estimator* e = make_estimator(est, P);
    Model cfg(thr, (unsigned)sample_size_of(est), 0.95f, 5, est_of(est), Uniform);
    cfg.max_iterations = max_it;
    cfg.reset_random_generator = false;
    srand(seed);
    SPRT sprt(&cfg, e, (unsigned)n);
    for (int i = 0; i < n; i++) pool_out[i] = (int)sprt.points_random_pool[i];
    Model mod(&cfg);
    int best = 0;
    for (int q = 0; q < M; q++) {
        mod.setDescriptor(model_mat(est, models + 9 * q));
        Score sc;
        sc.inlier_number = -1; sc.score = -1;
        const bool good = sprt.verifyModelAndGetModelScore(&mod, hyp[q], (unsigned)best, &sc);
        good_out[q] = good;
        inl_out[q] = (good || hyp[q] < (int)cfg.max_hypothesis_test_before_sprt) ? sc.inlier_number : -1;
        bound_after[q] = 0xffffffffu;
        if (inl_out[q] > best) { best = inl_out[q]; bound_after[q] = sprt.getUpperBoundIterations(best); }
        pool_idx_after[q] = sprt.random_pool_idx;
    }
    *nhist = (int)sprt.sprt_histories.size();
    for (int i = 0; i < *nhist && i < 4096; i++) {
        hist_out[4 * i] = sprt.sprt_histories[i]->epsilon; hist_out[4 * i + 1] = sprt.sprt_histories[i]->delta;
        hist_out[4 * i + 2] = sprt.sprt_histories[i]->A; hist_out[4 * i + 3] = sprt.sprt_histories[i]->k;
    }
    delete e;
    return 0;
}

// ---- ProsacTerminationCriteria (prosac_termination_criteria.hpp:44-201) over a sequence of best-model updates ------------------
int ref_prosac_termination_sequence(int est, const float* pts, int n, float thr, float conf, unsigned max_it, const float* models, int M,
                                    const unsigned* hyp_count, const unsigned* largest, unsigned* max_samples_out, unsigned* term_len_out) {
    cv::Mat P = borrow(pts, n, 4);
    Estimator* e = make_estimator(est, P);
    Model cfg(thr, (unsigned)sample_size_of(est), conf, 5, est_of(est), Prosac);
    cfg.max_iterations = max_it;
    ProsacSampler s;
    s.initProsacSampler((unsigned)sample_size_of(est), (unsigned)n);
    ProsacTerminationCriteria t(s.getGrowthFunction(), &cfg, (unsigned)n, e);
    unsigned lss = 0;
    t.setLargestSampleSize(&lss);
    for (int q = 0; q < M; q++) {
        lss = largest[q];
        max_samples_out[q] = t.getUpBoundIterations(hyp_count[q], model_mat(est, models + 9 * q));
        term_len_out[q] = *t.getStoppingLength();
    }
    delete e;
    return 0;
}

// ---- neighbourhoods (nearest_neighbors.cpp:69-128, 160-201) ----------------------------------------------------------------------
// grid: lists flattened in point order, offsets[n+1]
int ref_grid_neighbors(const float* pts, int n, int cell, int* flat_out, long long capacity, long long* offsets) {
    cv::Mat P = borrow(pts, n, 4);
    std::vector<std::vector<int>> nb;
    NearestNeighbors::getGridNearestNeighbors(P, cell, nb);
    long long pos = 0;
    for (int i = 0; i < n; i++) {
        offsets[i] = pos;
        for (int v : nb[i]) { if (pos < capacity) flat_out[pos] = v; pos++; }
    }
    offsets[n] = pos;
    return pos <= capacity ? 0 : 1;
}
int ref_knn(const float* pts, int n, int dim, int k, int* out) {
    cv::Mat P = borrow(pts, n, dim);
    cv::Mat nn, dists;
    NearestNeighbors::getNearestNeighbors_nanoflann(P, k, nn, false, dists);
    std::memcpy(out, nn.data, sizeof(int) * (size_t)n * k);
    return 0;
}

// ---- Jenkins-Traub (essential/rpoly.cpp): roots of a real polynomial, highest power first --------------------------------------
int ref_rpoly(const double* coeffs, int degree, double* zeror, double* zeroi) {
    double op[101];
    for (int i = 0; i <= degree; i++) op[i] = coeffs[i];
    int deg = degree;
    rpoly_ak1(op, &deg, zeror, zeroi);
    return deg;
}

// ---- the whole driver: Ransac::Ransac + Ransac::run (ransac.hpp:41-93, ransac.cpp:14-238) ----------------------------------------
struct ref_run_result {
    float model[9];
    int inliers;                // RansacOutput::getNumberOfInliers (after the refit loop)
    unsigned iterations, lo_inner, lo_iterative;
    long long time_us;
};
int ref_ransac_run(int est, int sampler, int neighbors, int sprt, int lo, const float* pts, int n, float thr, float conf, unsigned max_it,
                   unsigned knn, int cell, unsigned seed, unsigned rd_seed, ref_run_result* out, int* inliers_out) {
    cv::Mat P = borrow(pts, n, est == 1 ? 2 : 4);
    Model cfg(thr, (unsigned)sample_size_of(est), conf, knn, est_of(est),
              sampler == 1 ? Uniform : sampler == 3 ? Napsac : sampler == 4 ? Prosac : NullS);
    cfg.max_iterations = max_it;
    cfg.reset_random_generator = false;          // the reproducible configuration (test_homography_fitting.cpp:57): nothing calls srand(time)
    cfg.sprt = sprt != 0;
    cfg.lo = lo == 1 ? InItLORsc : lo == 2 ? InItFLORsc : NullLO;
    cfg.neighborsType = neighbors == 1 ? Nanoflann : neighbors == 2 ? Grid : NullN;
    cfg.cell_size = cell;
    srand(seed);
    usac_ref_random_device_seed() = rd_seed;
    Ransac r(&cfg, P);
    r.run();
    RansacOutput* o = r.getRansacOutput();
    std::memset(out, 0, sizeof(*out));
    cv::Mat d = o->getModel()->returnDescriptor();
    for (int j = 0; j < (est == 1 ? 3 : 9); j++) out->model[j] = d.at<float>(j);
    out->inliers = (int)o->getNumberOfInliers();
    out->iterations = o->getNumberOfMainIterations();
    out->lo_inner = o->getLOInnerIters();
    out->lo_iterative = o->getLOIterativeIters();
    out->time_us = o->getTimeMicroSeconds();
    if (inliers_out) { std::vector<int> in = o->getInliers(); for (int i = 0; i < out->inliers && i < (int)in.size(); i++) inliers_out[i] = in[i]; }
    return 0;
}

}   // extern "C"
