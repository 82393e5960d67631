// model.hpp - run configuration + model descriptor. Mirrors usac/model.hpp:10-143 of the reference (same enum values,
// field names, defaults and setters), minus the debug-only dataset fields.
#pragma once
#include <string>

#include "mat.hpp"

enum ESTIMATOR { NullE, Line2d, Homography, Fundamental, Essential };
enum SAMPLER { NullS, Uniform, ProgressiveNAPSAC, Napsac, Prosac, Evsac, ProsacNapsac };
enum NeighborsSearch { NullN, Nanoflann, Grid };
enum LocOpt { NullLO, InItLORsc, InItFLORsc, GC, IRLS };

class Model {
public:
    float threshold = 2;
    float desired_prob = 0.95f;
    unsigned int sample_size = 0;
    unsigned int min_iterations = 20;
    unsigned int max_iterations = 10000;
    unsigned int k_nearest_neighbors = 5;
    LocOpt lo = NullLO;
    unsigned int lo_sample_size = 14, lo_iterative_iterations = 4, lo_inner_iterations = 20, lo_threshold_multiplier = 10;
    float spatial_coherence_gc = 0.1f;
    ESTIMATOR estimator = NullE;
    SAMPLER sampler = NullS;
    bool sprt = false;
    unsigned int max_hypothesis_test_before_sprt = 20;
    NeighborsSearch neighborsType = NullN;
    int cell_size = 50;
    bool reset_random_generator = true;
    std::string img_name;
    // additions of the GPU host layer (not in the reference): explicit sampler seed and round size of the fused loop, and
    // (essential only) every cheirality-valid five-point root as a model instead of the reference's first one
    unsigned long long seed = 1;
    int gpu_round_size = 0;
    bool gpu_essential_all_roots = false;

    Model(const Model* const other) { copyFrom(other); }
    Model(float threshold_, unsigned int sample_number_, float desired_prob_, unsigned int knn, ESTIMATOR estimator_, SAMPLER sampler_)
        : threshold(threshold_), desired_prob(desired_prob_), sample_size(sample_number_), k_nearest_neighbors(knn),
          estimator(estimator_), sampler(sampler_) {}

    void ResetRandomGenerator(bool reset) { reset_random_generator = reset; }
    void setNeighborsType(NeighborsSearch t) { neighborsType = t; }
    void setCellSize(int c) { cell_size = c; }
    void setSprt(bool s) { sprt = s; }
    void setGpuEssentialAllRoots(bool a) { gpu_essential_all_roots = a; }
    void setLOParametres(unsigned int it, unsigned int inner, unsigned int mult) {
        lo_iterative_iterations = it; lo_inner_iterations = inner; lo_threshold_multiplier = mult;
    }
    void setDescriptor(const cv::Mat& desc) { descriptor = desc.clone(); }        // deep copy, model.hpp:93-96
    cv::Mat returnDescriptor() const { return descriptor; }
    void setThreshold(float t) { threshold = t; }
    void setSampleNumber(float n) { sample_size = (unsigned int)n; }
    void setDesiredProbability(float p) { desired_prob = p; }
    void setKNearestNeighbors(int k) { k_nearest_neighbors = (unsigned int)k; }
    void copyFrom(const Model* const m) {                                          // everything but the descriptor, model.hpp:119-141
        threshold = m->threshold; sample_size = m->sample_size; desired_prob = m->desired_prob;
        max_iterations = m->max_iterations; min_iterations = m->min_iterations; estimator = m->estimator; sampler = m->sampler;
        k_nearest_neighbors = m->k_nearest_neighbors; lo_sample_size = m->lo_sample_size;
        lo_iterative_iterations = m->lo_iterative_iterations; lo_inner_iterations = m->lo_inner_iterations;
        lo_threshold_multiplier = m->lo_threshold_multiplier; reset_random_generator = m->reset_random_generator;
        lo = m->lo; sprt = m->sprt; spatial_coherence_gc = m->spatial_coherence_gc; cell_size = m->cell_size;
        neighborsType = m->neighborsType; max_hypothesis_test_before_sprt = m->max_hypothesis_test_before_sprt;
        seed = m->seed; gpu_round_size = m->gpu_round_size; gpu_essential_all_roots = m->gpu_essential_all_roots;
    }

private:
    cv::Mat descriptor;
};
