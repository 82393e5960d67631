// init.hpp - the factory functions of the reference (usac/ransac/init.cpp:3-83, init.hpp), same names and signatures, selecting
// the GPU-backed plugins. Like the reference they report an unknown enum and exit(111) (init.cpp:17-19, 48-50) - here by throwing,
// which the harness turns into exit code 111. Samplers the reference does not finish (Evsac / ProsacNapsac: commented out / empty
// branch in init.cpp:40-47) are refused, never silently replaced by uniform sampling. ProgressiveNAPSAC, a stub in the reference
// (progressive_sampler.hpp:149-172 never fills its sample), is built as DESIGN.md section 4.8 defines it, over kNN neighbourhoods.
#pragma once
#include "gpu_plugins.hpp"
#include "local_optimization.hpp"
#include "prosac_termination_criteria.hpp"
#include "sprt.hpp"

inline void initEstimator(Estimator*& estimator, ESTIMATOR est, const cv::Mat& points, int gpu = 0) {
    if (est != Line2d && est != Homography && est != Fundamental && est != Essential) throw std::runtime_error("UNKOWN Estimator IN Init Estimator");
    estimator = new GpuEstimator(new GpuDevice(gpu, est, points), /*owns_device=*/true);      // uploads the points (the reference borrows them)
}

inline void initSampler(Sampler*& sampler, const Model* const model, const cv::Mat& points) {
    if (model->sampler != Uniform && model->sampler != Prosac && model->sampler != Napsac && model->sampler != ProgressiveNAPSAC)
        throw std::runtime_error("UNKOWN Sampler IN Init Sampler (Uniform, Prosac, Napsac and ProgressiveNAPSAC are built; Evsac / ProsacNapsac are unfinished in the reference)");
    GpuDevice* dev = GpuDevice::find(points);
    if (!dev) throw std::runtime_error("initSampler: call initEstimator on these points first (it uploads them)");
    if (model->sampler == Napsac) {                                                           // ransac.hpp:61-78 (neighbourhood search)
        if (model->neighborsType == Grid) dev->check(usac_gpu_set_neighbors_grid(dev->ctx, 0, model->cell_size), "usac_gpu_set_neighbors_grid");
        else if (model->neighborsType == Nanoflann) dev->check(usac_gpu_build_neighbors_knn(dev->ctx, 0, (int)model->k_nearest_neighbors), "usac_gpu_build_neighbors_knn");
        else throw std::runtime_error("initSampler: Napsac needs Model::setNeighborsType(Grid | Nanoflann)");
    }
    if (model->sampler == ProgressiveNAPSAC) {                                                // grows each centre's distance-ordered list
        if (model->neighborsType != Nanoflann) throw std::runtime_error("initSampler: ProgressiveNAPSAC needs Model::setNeighborsType(Nanoflann)");
        dev->check(usac_gpu_build_neighbors_knn(dev->ctx, 0, (int)model->k_nearest_neighbors), "usac_gpu_build_neighbors_knn");
        dev->check(usac_gpu_set_pnapsac_length(dev->ctx, 0, model->gpu_pnapsac_local_samples), "usac_gpu_set_pnapsac_length");
    }
    sampler = new GpuSampler(dev, model);
}

inline void initTerminationCriteria(TerminationCriteria*& termination_criteria, const Model* const model, unsigned int points_size) {
    termination_criteria = new StandardTerminationCriteria(model, points_size);
}

inline void initProsacTerminationCriteria(TerminationCriteria*& termination_criteria, Sampler*& prosac_sampler, const Model* const model,
                                          Estimator* estimator, unsigned int points_size) {
    GpuSampler* ps = dynamic_cast<GpuSampler*>(prosac_sampler);
    if (!ps || ps->config().sampler != USAC_SAMPLER_PROSAC) throw std::runtime_error("initProsacTerminationCriteria: needs the PROSAC sampler");
    ProsacTerminationCriteria* t = new ProsacTerminationCriteria(ps->getGrowthFunction(), model, points_size, estimator);
    termination_criteria = t;
    ps->setTerminationLength(t->getStoppingLength());                                         // init.cpp:62-65: the two share their state by pointer
    t->setLargestSampleSize(ps->getLargestSampleSize());
}

inline void initLocalOptimization(LocalOptimization*& local_optimization, Model* model, Estimator* estimator, Quality* quality, unsigned int points_size) {
    if (model->lo == InItLORsc || model->lo == InItFLORsc) local_optimization = new InnerLocalOptimization(model, estimator, quality, points_size);
    else if (model->lo == GC || model->lo == IRLS) throw std::runtime_error("initLocalOptimization: graph-cut / IRLS local optimisation is outside the GPU layer (SURVEY.md section 2, rows 21-22)");
    else local_optimization = nullptr;
}
