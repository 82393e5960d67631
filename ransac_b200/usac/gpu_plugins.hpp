// gpu_plugins.hpp - GPU-backed implementations of the plugin surface. Every method forwards to the C ABI of
// libusac_gpu.so (include/usac_gpu.h); there is NO CPU implementation behind any of them - when the library cannot
// create a context (no sm_100 device) construction fails and the caller gets the library's error text.
#pragma once
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>

#include "../../include/usac_gpu.h"
#include "plugin.hpp"

inline int usac_estimator_code(ESTIMATOR e) {
    switch (e) {
        case Line2d: return USAC_EST_LINE2D;
        case Homography: return USAC_EST_HOMOGRAPHY;
        case Fundamental: return USAC_EST_FUNDAMENTAL;
        case Essential: return USAC_EST_ESSENTIAL;
        default: return 0;
    }
}
inline int usac_sampler_code(SAMPLER s) {
    switch (s) {
        case Uniform: return USAC_SAMPLER_UNIFORM;
        case Napsac: return USAC_SAMPLER_NAPSAC;
        case Prosac: return USAC_SAMPLER_PROSAC;
        case ProgressiveNAPSAC: return USAC_SAMPLER_PROGRESSIVE_NAPSAC;
        default: return 0;
    }
}

// Owns the device context and the uploaded copy of the points (the reference BORROWS the cv::Mat memory for the lifetime of
// the estimator, ransac.hpp:41; the device copy is taken once here).
class GpuDevice {
public:
    usac_gpu_ctx* ctx = nullptr;
    int estimator = 0, points_size = 0, dim = 4;
    GpuDevice(int device, ESTIMATOR est, const cv::Mat& points) {
        estimator = usac_estimator_code(est);
        if (!estimator) throw std::runtime_error("GpuDevice: unknown estimator");
        dim = est == Line2d ? 2 : 4;
        if (points.empty() || points.cols != dim) throw std::runtime_error("GpuDevice: points must be N x " + std::to_string(dim) + " float32");
        if (usac_gpu_create(&ctx, device) != USAC_OK) throw std::runtime_error(std::string("usac_gpu_create: ") + usac_gpu_last_error(nullptr));
        points_size = points.rows;
        check(usac_gpu_set_points(ctx, estimator, points.ptr(), &points_size, 1), "usac_gpu_set_points");
        host_points = points.ptr();
        registry()[host_points] = this;
    }
    ~GpuDevice() {
        auto it = registry().find(host_points);
        if (it != registry().end() && it->second == this) registry().erase(it);
        usac_gpu_destroy(ctx);
    }
    // The reference's factories receive the points matrix, not a device (init.cpp:3-51): the device that uploaded a matrix is
    // found again through the address of its data (the reference borrows that same pointer for the estimator's lifetime).
    static GpuDevice* find(const cv::Mat& points) {
        auto it = registry().find(points.ptr());
        return it == registry().end() ? nullptr : it->second;
    }
    const float* host_points = nullptr;
    GpuDevice(const GpuDevice&) = delete;
    GpuDevice& operator=(const GpuDevice&) = delete;
    void check(int rc, const char* what) const {
        if (rc != USAC_OK) throw std::runtime_error(std::string(what) + ": " + usac_gpu_last_error(ctx));
    }
private:
    static std::map<const float*, GpuDevice*>& registry() { static std::map<const float*, GpuDevice*> r; return r; }
};

// Estimator (estimator.hpp:19-40): EstimateModel = the device minimal solver on one sample (usac_gpu_estimate, K = 1;
// usac_gpu_estimate_essential_roots when the models carry Model::gpu_essential_all_roots);
// setModelParameters + GetError(pidx) = usac_gpu_errors (all N errors in the reference's exact arithmetic, cached).
class GpuEstimator : public Estimator {
    GpuDevice* dev;
    bool owns_device;
    std::vector<float> errors;
    bool errors_valid = false;
    float model_params[9];
public:
    explicit GpuEstimator(GpuDevice* d, bool owns_device_ = false) : dev(d), owns_device(owns_device_), errors((size_t)d->points_size) {}
    ~GpuEstimator() override { if (owns_device) delete dev; }
    int SampleNumber() override { return dev->estimator == USAC_EST_LINE2D ? 2 : dev->estimator == USAC_EST_HOMOGRAPHY ? 4 : dev->estimator == USAC_EST_FUNDAMENTAL ? 7 : 5; }
    unsigned int EstimateModel(const int* const sample, std::vector<Model*>& models) override {
        float out[USAC_E5_MAX_ROOTS * 9];
        int n = 0;
        if (dev->estimator == USAC_EST_ESSENTIAL && !models.empty() && models[0]->gpu_essential_all_roots)
            dev->check(usac_gpu_estimate_essential_roots(dev->ctx, 0, sample, 1, out, &n), "usac_gpu_estimate_essential_roots");
        else
            dev->check(usac_gpu_estimate(dev->ctx, 0, sample, 1, out, &n), "usac_gpu_estimate");
        const bool line = dev->estimator == USAC_EST_LINE2D;
        for (int i = 0; i < n && i < (int)models.size(); i++) {
            cv::Mat d = line ? cv::Mat(1, 3) : cv::Mat(3, 3);
            for (int k = 0; k < (line ? 3 : 9); k++) d.ptr()[k] = out[9 * i + k];
            models[i]->setDescriptor(d);
        }
        return (unsigned int)n;
    }
    // batched form used by the fused path and by callers that want K samples per call
    unsigned int EstimateModels(const int* samples, int K, float* models_out, int* nmodels_out) {
        dev->check(usac_gpu_estimate(dev->ctx, 0, samples, K, models_out, nmodels_out), "usac_gpu_estimate");
        return (unsigned int)K;
    }
    bool EstimateModelNonMinimalSample(const int* const sample, unsigned int sample_size, Model& model) override {
        float out[9];
        int ok = 0;
        dev->check(usac_gpu_estimate_nonminimal(dev->ctx, 0, sample, (int)sample_size, out, &ok), "usac_gpu_estimate_nonminimal");
        if (!ok) return false;
        const bool line = dev->estimator == USAC_EST_LINE2D;
        cv::Mat d = line ? cv::Mat(1, 3) : cv::Mat(3, 3);
        for (int k = 0; k < (line ? 3 : 9); k++) d.ptr()[k] = out[k];
        model.setDescriptor(d);
        return true;
    }
    void setModelParameters(const cv::Mat& model) override {
        const int w = dev->estimator == USAC_EST_LINE2D ? 3 : 9;
        for (int k = 0; k < w; k++) model_params[k] = model.ptr()[k];
        errors_valid = false;
    }
    float GetError(unsigned int pidx) override {
        if (!errors_valid) {
            dev->check(usac_gpu_errors(dev->ctx, 0, model_params, errors.data()), "usac_gpu_errors");
            errors_valid = true;
        }
        return errors[pidx];
    }
    GpuDevice* device() { return dev; }
};

// Quality (quality.hpp:49-121): one usac_gpu_score call per model (M = 1), or M models per call through the batched form.
class GpuQuality : public Quality {
    GpuDevice* dev;
public:
    explicit GpuQuality(GpuDevice* d) : dev(d) {}
    void getNumberInliers(Score* score, const cv::Mat& model, float threshold_ = 0, bool get_inliers = false, int* inliers = nullptr,
                          bool /*parallel*/ = false) override {
        if (threshold_ == 0) threshold_ = threshold;
        dev->check(usac_gpu_score(dev->ctx, 0, model.ptr(), 1, threshold_, &score->inlier_number, &score->score), "usac_gpu_score");
        if (get_inliers) {
            int n = 0;
            dev->check(usac_gpu_get_inliers(dev->ctx, 0, model.ptr(), threshold_, inliers, &n), "usac_gpu_get_inliers");
        }
    }
    void getNumberInliersBatch(const float* models, int M, float threshold_, int* inlier_numbers, float* scores) {
        dev->check(usac_gpu_score(dev->ctx, 0, models, M, threshold_ == 0 ? threshold : threshold_, inlier_numbers, scores), "usac_gpu_score");
    }
    void getInliers(const cv::Mat& model, int* inliers) override {
        assert(isinit);
        int n = 0;
        dev->check(usac_gpu_get_inliers(dev->ctx, 0, model.ptr(), threshold, inliers, &n), "usac_gpu_get_inliers");
    }
};

// Sampler (sampler.hpp:21): samples are drawn on the device in blocks (usac_gpu_sample) and handed out one per call.
// Hypothesis h always gets the same index set for a given seed (counter-based Philox), whatever the block size.
class GpuSampler : public Sampler {
    GpuDevice* dev;
    usac_sampler_cfg cfg;
    std::vector<int> block;
    int block_size, cursor;
    unsigned long long next_hyp = 0;
    // PROSAC (prosac_sampler.hpp:19-60): growth function, the stopping length shared with ProsacTerminationCriteria, and the
    // largest subset size reached so far. While the stopping length can change between samples the sampler draws one sample per
    // device call (block size 1), so that every sample sees the current value like the reference's.
    std::vector<unsigned int> growth_function;
    unsigned int* termination_length = nullptr;
    unsigned int largest_sample_size = 0, subset_size = 0, hyp_count = 1;
public:
    GpuSampler(GpuDevice* d, const Model* model, int block_size_ = 256) : dev(d), block_size(block_size_), cursor(block_size_) {
        sample_size = model->sample_size; points_size = (unsigned int)d->points_size;
        cfg.sampler = usac_sampler_code(model->sampler); cfg.rng = USAC_RNG_PHILOX; cfg.seed = model->seed;
        cfg.neighbors = model->neighborsType == Grid ? USAC_NEIGH_GRID : model->neighborsType == Nanoflann ? USAC_NEIGH_KNN : USAC_NEIGH_NONE;
        cfg.prosac_termination_length = 0; cfg.prosac_hyp_count = 0;
        if (cfg.sampler == USAC_SAMPLER_PROSAC) {
            growth_function.resize(points_size);
            usac_prosac_growth_function(points_size, sample_size, growth_function.data());
            largest_sample_size = subset_size = sample_size;
            block_size = 1; cursor = 1;
        }
        block.resize((size_t)block_size * sample_size);
    }
    void setTerminationLength(unsigned int* p) { termination_length = p; }
    unsigned int* getGrowthFunction() { return growth_function.data(); }
    unsigned int* getLargestSampleSize() { return &largest_sample_size; }
    void generateSample(int* sample) override {
        if (cursor == block_size) {
            if (cfg.sampler == USAC_SAMPLER_PROSAC) {
                const unsigned int L = termination_length ? *termination_length : points_size;
                if (!(subset_size > L)) {                                   // prosac_sampler.hpp:141-156: counters move only outside termination mode
                    if (hyp_count > growth_function[subset_size - 1]) {
                        if (++subset_size > points_size) subset_size = points_size;
                        if (largest_sample_size < subset_size) largest_sample_size = subset_size;
                    }
                    cfg.prosac_hyp_count = hyp_count;
                    hyp_count++;
                } else {
                    cfg.prosac_hyp_count = hyp_count;
                }
                cfg.prosac_termination_length = L;
            }
            dev->check(usac_gpu_sample(dev->ctx, 0, &cfg, next_hyp, block_size, block.data()), "usac_gpu_sample");
            cursor = 0;
        }
        for (unsigned int i = 0; i < sample_size; i++) sample[i] = block[(size_t)cursor * sample_size + i];
        cursor++; next_hyp++; k_iterations++;
    }
    bool isInit() override { return true; }
    const usac_sampler_cfg& config() const { return cfg; }
};

// standard_termination_criteria.hpp:52-62 - plain host arithmetic (float, truncation), exactly the table usac_gpu_fit uploads.
class StandardTerminationCriteria : public TerminationCriteria {
    float log_1_p;
    unsigned int sample_size, points_size, max_iterations;
public:
    StandardTerminationCriteria(const Model* const model, unsigned int points_size_)
        : log_1_p((float)logf(1 - model->desired_prob)), sample_size(model->sample_size), points_size(points_size_),
          max_iterations(model->max_iterations) { isinit = true; }
    unsigned int getUpBoundIterations(unsigned int inlier_size) override { return getUpBoundIterations(inlier_size, points_size); }
    unsigned int getUpBoundIterations(unsigned int inlier_size, unsigned int n) override {
        const float w = (float)inlier_size / n;
        float p = w * w;
        for (int k = (int)sample_size; k > 2; k--) p *= w;
        if (p < 0.0005f) return max_iterations;
        return (unsigned int)(log_1_p / logf(1 - p));
    }
};
