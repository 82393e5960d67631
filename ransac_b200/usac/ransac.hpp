// ransac.hpp - the driver, same construction and accessors as usac/ransac/ransac.hpp:17-118; run() has two forms:
//   run()            the GPU hypothesis batch: the whole loop of ransac.cpp:58-139 in usac_gpu_fit (rounds of K samples, one
//                    host sync per round; SPRT, PROSAC termination and LO included), the refit loop of ransac.cpp:157-207 in
//                    usac_gpu_refit, then the final inlier list;
//   run_sequential() the reference's one-hypothesis-at-a-time loop (ransac.cpp:58-139) over the virtual plugin interfaces -
//                    Sampler, Estimator, Quality, SPRT, TerminationCriteria / ProsacTerminationCriteria, LocalOptimization -
//                    each call forwarding to the C ABI: the drop-in at plugin granularity. Without SPRT, run() with
//                    Model::gpu_round_size = 1 is the same loop (and without PROSAC every round size is). With SPRT a round freezes
//                    the test and starts model q of the round at pool offset cursor + 32 q (rounds-of-K semantics, DESIGN 4.4), while
//                    the sequential walk starts where the last one stopped: about one SPRT fit in ten ends differently even at
//                    K = 1 (tools/stress_harness.py checks each form against its own CPU restatement).
#pragma once
#include <chrono>

#include "init.hpp"
#include "ransac_output.hpp"

class Ransac {
protected:
    Model* model;
    GpuDevice* device = nullptr;
    Quality* quality = nullptr;
    Sampler* sampler = nullptr;
    TerminationCriteria* termination_criteria = nullptr;
    RansacOutput* ransac_output = nullptr;
    Estimator* estimator = nullptr;
    LocalOptimization* local_optimization = nullptr;
    SPRT* sprt = nullptr;
    unsigned int points_size;
    usac_fit_result last_fit{};
public:
    Ransac(Model* model_, cv::InputArray points_, int gpu = 0) : model(model_) {                 // ransac.hpp:41-93
        assert(model != nullptr);
        const cv::Mat& pts = points_.getMat();
        points_size = (unsigned int)pts.rows;
        initEstimator(estimator, model->estimator, pts, gpu);
        device = static_cast<GpuEstimator*>(estimator)->device();
        initSampler(sampler, model, pts);
        quality = new GpuQuality(device);
        quality->init(points_size, model->threshold, estimator);
        initLocalOptimization(local_optimization, model, estimator, quality, points_size);
        if (model->sampler == Prosac) initProsacTerminationCriteria(termination_criteria, sampler, model, estimator, points_size);
        else initTerminationCriteria(termination_criteria, model, points_size);
        if (model->sprt) sprt = new SPRT(model, estimator, points_size);                          // uploads the shuffled pool
    }
    ~Ransac() { delete sprt; delete local_optimization; delete sampler; delete quality; delete termination_criteria; delete ransac_output; delete estimator; }
    Ransac(const Ransac&) = delete;

    void setSampler(Sampler* s) { sampler = s; }
    void setModel(Model* m) { model = m; }
    void setTerminationCriteria(TerminationCriteria* t) { termination_criteria = t; }
    void setQuality(Quality* q) { quality = q; }
    Quality* getQuality() { return quality; }
    RansacOutput* getRansacOutput() { return ransac_output; }
    const usac_fit_result& lastFit() const { return last_fit; }

    void run() {
        auto t0 = std::chrono::steady_clock::now();
        GpuSampler* gs = dynamic_cast<GpuSampler*>(sampler);
        if (!gs) throw std::runtime_error("Ransac::run: the fused path needs the GPU sampler (a custom Sampler installed with setSampler works with run_sequential())");
        usac_fit_cfg cfg{};
        cfg.sampler = gs->config();
        cfg.sampler.prosac_termination_length = 0; cfg.sampler.prosac_hyp_count = 0;
        cfg.threshold = model->threshold; cfg.confidence = model->desired_prob; cfg.max_iterations = model->max_iterations;
        cfg.sprt = model->sprt; cfg.round_size = model->gpu_round_size; cfg.rank = 0; cfg.nranks = 1;
        cfg.lo = (int)model->lo;                                                         // NullLO 0, InItLORsc 1, InItFLORsc 2 (model.hpp:13)
        cfg.lo_sample_size = model->lo_sample_size; cfg.lo_inner_iterations = model->lo_inner_iterations;       // Model::setLOParametres
        cfg.lo_iterative_iterations = model->lo_iterative_iterations; cfg.lo_threshold_multiplier = model->lo_threshold_multiplier;
        cfg.max_hypothesis_test_before_sprt = model->max_hypothesis_test_before_sprt;
        cfg.essential_roots = model->gpu_essential_all_roots ? USAC_E5_ROOTS_ALL_VALID : USAC_E5_ROOTS_FIRST_VALID;
        device->check(usac_gpu_fit(device->ctx, &cfg, &last_fit), "usac_gpu_fit");
        if (last_fit.inliers <= 0) throw std::runtime_error("Ransac: best score is 0");           // ransac.cpp:143-147
        usac_refit_result rf{};                                                                   // ransac.cpp:157-207 on the device
        device->check(usac_gpu_refit(device->ctx, 0, last_fit.model, last_fit.inliers, model->threshold, &rf), "usac_gpu_refit");
        finish(rf.model, rf.inliers, last_fit.iterations, t0, last_fit.lo_inner_iters, last_fit.lo_iterative_iters);
    }

    // ransac.cpp:14-139 statement for statement over the plugin interfaces
    void run_sequential() {
        auto t0 = std::chrono::steady_clock::now();
        Score best, cur;
        std::vector<Model*> models;
        // ransac.cpp:19-33 (the five-point solver returns one model, or every valid root with gpu_essential_all_roots)
        const int nmod = model->estimator == Fundamental ? 3 : (model->estimator == Essential && model->gpu_essential_all_roots) ? USAC_E5_MAX_ROOTS : 1;
        for (int i = 0; i < nmod; i++) models.push_back(new Model(model));
        Model best_model(model);
        std::vector<int> sample((size_t)estimator->SampleNumber());
        const bool is_prosac = model->sampler == Prosac, is_sprt = model->sprt, LO = local_optimization != nullptr;
        unsigned int iters = 0, max_iters = model->max_iterations;
        while (iters < max_iters) {
            sampler->generateSample(sample.data());
            const unsigned int n = estimator->EstimateModel(sample.data(), models);
            for (unsigned int i = 0; i < n; i++) {
                if (is_sprt) {
                    const bool good = sprt->verifyModelAndGetModelScore(models[i], (int)iters, (unsigned int)best.inlier_number, &cur);
                    if (!good && iters >= model->max_hypothesis_test_before_sprt) { iters++; continue; }     // ransac.cpp:77-85
                } else {
                    quality->getNumberInliers(&cur, models[i]->returnDescriptor());
                }
                if (cur.bigger(&best)) {
                    if (LO) local_optimization->GetModelScore(models[i], &cur);            // ransac.cpp:108-112
                    best.copyFrom(&cur);
                    best_model.setDescriptor(models[i]->returnDescriptor());
                    if (is_prosac) max_iters = static_cast<ProsacTerminationCriteria*>(termination_criteria)->getUpBoundIterations(iters, best_model.returnDescriptor());
                    else max_iters = termination_criteria->getUpBoundIterations((unsigned int)best.inlier_number);
                    if (is_sprt) max_iters = std::min(max_iters, sprt->getUpperBoundIterations(best.inlier_number));   // ransac.cpp:129-133
                }
            }
            iters++;
        }
        for (Model* m : models) delete m;
        if (best.inlier_number == 0) throw std::runtime_error("Ransac: best score is 0");   // the reference exit(111)s, ransac.cpp:143-147
        last_fit = usac_fit_result{};
        last_fit.inliers = best.inlier_number; last_fit.score = best.score; last_fit.iterations = iters;
        const cv::Mat d = best_model.returnDescriptor();
        for (int k = 0; k < d.rows * d.cols; k++) last_fit.model[k] = d.ptr()[k];
        unsigned int lo_inner = 0, lo_iterative = 0;
        if (InnerLocalOptimization* ilo = dynamic_cast<InnerLocalOptimization*>(local_optimization)) { lo_inner = ilo->lo_inner_iters; lo_iterative = ilo->lo_iterative_iters; }
        last_fit.lo_inner_iters = lo_inner; last_fit.lo_iterative_iters = lo_iterative;
        // the refit loop of ransac.cpp:157-207 over the virtual plugin calls
        std::vector<int> max_inliers(points_size);
        quality->getInliers(best_model.returnDescriptor(), max_inliers.data());
        Model non_minimal(model);
        unsigned int previous = 0;
        // under SPRT best.inlier_number is a count over the whole pool for accepted models, i.e. the number of entries of the list
        for (unsigned int norm = 0; norm < 4; norm++) {
            if (!estimator->EstimateModelNonMinimalSample(max_inliers.data(), (unsigned int)best.inlier_number, non_minimal)) break;
            quality->getNumberInliers(&cur, non_minimal.returnDescriptor(), model->threshold, true, max_inliers.data());
            if ((float)cur.inlier_number / best.inlier_number < 0.8) break;
            if ((unsigned int)cur.inlier_number <= previous) break;
            previous = (unsigned int)cur.inlier_number;
            best.copyFrom(&cur);
            best_model.setDescriptor(non_minimal.returnDescriptor());
        }
        const cv::Mat fd = best_model.returnDescriptor();
        float params[9] = {0};
        for (int k = 0; k < fd.rows * fd.cols; k++) params[k] = fd.ptr()[k];
        finish(params, best.inlier_number, iters, t0, lo_inner, lo_iterative);
    }

private:
    void finish(const float* params, int inlier_number, unsigned int iters, std::chrono::steady_clock::time_point t0,
                unsigned int lo_inner = 0, unsigned int lo_iterative = 0) {
        if (inlier_number <= 0) throw std::runtime_error("Ransac: best score is 0");
        const bool line = model->estimator == Line2d;
        cv::Mat d = line ? cv::Mat(1, 3) : cv::Mat(3, 3);
        for (int k = 0; k < (line ? 3 : 9); k++) d.ptr()[k] = params[k];
        Model best(model);
        best.setDescriptor(d);
        std::vector<int> inliers(points_size);
        quality->getInliers(d, inliers.data());                                       // ransac.cpp:210
        const long us = (long)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        delete ransac_output;
        ransac_output = new RansacOutput(&best, inliers.data(), us, (unsigned int)inlier_number, iters, lo_inner, lo_iterative, 0);
    }
};
