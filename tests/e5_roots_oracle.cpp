/*
 * e5_roots_oracle.cpp - the CPU oracle's fit loop with every cheirality-valid five-point root as a model: the reference the tests
 * of usac_fit_cfg::essential_roots = USAC_E5_ROOTS_ALL_VALID compare against. TEST INFRASTRUCTURE ONLY, built by e5_roots_oracle.py
 * into a temporary directory together with the unmodified oracle sources (oracle/), whose SPRT, PROSAC termination and LO it reuses.
 *
 * orc_ransac_e5_all_roots is oracle/usac_oracle_ransac.cpp:orc_ransac with three differences: an essential sample yields every root
 * that passes the cheirality vote, in visiting order (orc_essential5_candidates filtered by its valid flags, cast to float), up to
 * 10; a round therefore holds S = 10 model slots per essential sample (SPRT pool walk of model q = j*S + i from cursor + 32 q);
 * the model buffer holds 10 models. Everything else - best update per model in order, iterations counting samples, SPRT, LO,
 * termination - is the oracle's code as it stands.
 */
/* the oracle's loop and its SPRT / PROSAC-termination classes; its own orc_ransac is compiled under another name here */
#define orc_ransac orc_ransac_first_valid_root
#include "../oracle/usac_oracle_ransac.cpp"
#undef orc_ransac

#define E5_MAX_ROOTS 10

/* every cheirality-valid candidate, in visiting order, as float32 (models_out: up to 10 x 9 floats); returns the count */
extern "C" int essential5_all_roots(const float* points, const int* sample, float* models_out) {
    double Es[E5_MAX_ROOTS * 9];
    int valid[E5_MAX_ROOTS];
    const int n = orc_essential5_candidates(points, sample, Es, valid);
    int k = 0;
    for (int i = 0; i < n; i++)
        if (valid[i]) {
            for (int e = 0; e < 9; e++) models_out[9 * k + e] = (float)Es[9 * i + e];
            k++;
        }
    return k;
}

extern "C" int orc_ransac_e5_all_roots(const orc_config* cfg, const float* points, int n, orc_result* out) {
    const int est = cfg->estimator;
    const int m = est == ORC_EST_LINE2D ? 2 : est == ORC_EST_HOMOGRAPHY ? 4 : est == ORC_EST_FUNDAMENTAL ? 7 : 5;
    const int S = est == ORC_EST_FUNDAMENTAL ? 3 : est == ORC_EST_ESSENTIAL ? E5_MAX_ROOTS : 1;
    const int msize = est == ORC_EST_LINE2D ? 3 : 9;
    memset(out, 0, sizeof(*out));
    out->best_hyp = -1;

    orc_sampler* sampler = orc_sampler_new(cfg->sampler, cfg->rng == ORC_RNG_TABLE ? ORC_RNG_PHILOX : cfg->rng, n, m, cfg->seed);
    if (cfg->sampler == ORC_SAMPLER_NAPSAC) {
        if (cfg->neighbors == ORC_NEIGH_GRID) orc_sampler_set_grid(sampler, points, cfg->cell_size);
        else orc_sampler_set_knn(sampler, cfg->knn_table, cfg->knn);
    }
    const bool is_prosac = cfg->sampler == ORC_SAMPLER_PROSAC;
    ProsacTermination pterm;
    if (is_prosac) pterm.init(orc_sampler_growth_function(sampler), n, m, cfg->threshold, cfg->confidence, cfg->max_iterations);

    Sprt sprt;
    if (cfg->sprt) {
        /* Ransac ctor order (ransac.hpp:50-92): sampler first, SPRT last; both draw from the one glibc stream */
        sprt.init(est, cfg->threshold, n, m, cfg->max_iterations, [&]() { return orc_sampler_glibc_next(sampler); });
    }

    int best_inl = 0;
    float best_score = 0;
    float best_model[9] = {0};
    unsigned iters = 0, max_iters = cfg->max_iterations;
    unsigned long long evals = 0;
    unsigned models_scored = 0;
    uint64_t hyp = 0;   /* samples drawn so far */
    ErrFn f;
    std::vector<unsigned char> inl_mask;

    auto draw = [&](int* sample) {
        if (cfg->rng == ORC_RNG_TABLE) {
            if (hyp < cfg->sample_table_rows) memcpy(sample, cfg->sample_table + (size_t)hyp * m, sizeof(int) * m);
            else orc_sampler_generate(sampler, hyp, sample);
        } else {
            if (is_prosac) orc_sampler_set_termination_length(sampler, pterm.termination_length);
            orc_sampler_generate(sampler, hyp, sample);
        }
        hyp++;
    };
    orc_lo* lo = cfg->lo ? orc_lo_new(est, points, n, cfg->threshold, cfg->lo, cfg->seed) : nullptr;
    auto on_new_best = [&](const float* model_in, int inl, float score, long long h, int mi) {
        float lo_model[9] = {0};
        memcpy(lo_model, model_in, sizeof(float) * msize);
        if (lo) orc_lo_get_model_score(lo, lo_model, &inl, &score);                 /* ransac.cpp:108-110 */
        const float* model = lo_model;
        best_inl = inl; best_score = score;
        memcpy(best_model, model, sizeof(float) * msize);
        out->best_hyp = h; out->best_model_idx = mi;
        if (is_prosac) {                                              /* ransac.cpp:123-125 */
            inl_mask.resize(n);
            f.set(est, model);
            for (int i = 0; i < n; i++) inl_mask[i] = f(points, (unsigned)i) < cfg->threshold;
            max_iters = pterm.update(iters, inl_mask, orc_sampler_largest_sample_size(sampler));
        } else {
            max_iters = orc_standard_termination((unsigned)best_inl, (unsigned)n, m, cfg->confidence, cfg->max_iterations);
        }
        if (cfg->sprt) max_iters = std::min(max_iters, sprt.getUpperBoundIterations(best_inl));   /* :129-133 */
    };

    int sample[8];
    float models[E5_MAX_ROOTS * 9];
    auto solve = [&](const int* smp, float* mdl) {                    /* Appendix B quirk 1 as a switch */
        if (cfg->ref_thin_svd && est == ORC_EST_HOMOGRAPHY) return orc_solve_homography_dlt4p_thin(points, smp, mdl);
        if (est == ORC_EST_ESSENTIAL) return essential5_all_roots(points, smp, mdl);
        return orc_solve_minimal(est, points, smp, mdl);
    };

    if (cfg->batch <= 0) {
        /* ---------------- reference-sequential ---------------- */
        while (iters < max_iters) {
            draw(sample);
            int nm = solve(sample, models);
            for (int i = 0; i < nm; i++) {
                int cur_inl = 0; float cur_score = 0;
                const float* mdl = models + 9 * i;
                if (cfg->sprt) {
                    f.set(est, mdl);
                    /* NOTE: on a rejection after the first 20 hypotheses the reference leaves current_score
                     * untouched and `continue`s (ransac.cpp:77-85), so stale values are never compared. */
                    bool good = sprt.verify(f, points, (int)iters, (unsigned)best_inl, cur_inl, cur_score, evals);
                    models_scored++;
                    if (!good && iters >= 20) { iters++; continue; }
                } else {
                    orc_score(est, points, n, mdl, cfg->threshold, &cur_inl, &cur_score, nullptr, 0, nullptr);
                    evals += n; models_scored++;
                }
                if (bigger(cur_inl, cur_score, best_inl, best_score)) on_new_best(mdl, cur_inl, cur_score, (long long)hyp - 1, i);
            }
            iters++;
        }
    } else {
        /* ---------------- batched(K) ---------------- */
        const int K = cfg->batch;
        std::vector<int> samples((size_t)K * m);
        std::vector<float> rmodels((size_t)K * S * 9);
        std::vector<int> nmodels(K), r_inl((size_t)K * S), r_good((size_t)K * S), r_tested_inl((size_t)K * S), r_tested_pts((size_t)K * S);
        std::vector<float> r_score((size_t)K * S);
        unsigned cursor = 0;
        bool done = false;
        while (!done && iters < max_iters) {
            const uint64_t hyp0 = hyp;
            if (is_prosac) orc_sampler_set_termination_length(sampler, pterm.termination_length);
            for (int j = 0; j < K; j++) {
                if (cfg->rng == ORC_RNG_TABLE && hyp < cfg->sample_table_rows)
                    memcpy(&samples[(size_t)j * m], cfg->sample_table + (size_t)hyp * m, sizeof(int) * m);
                else
                    orc_sampler_generate(sampler, hyp, &samples[(size_t)j * m]);
                hyp++;
                nmodels[j] = solve(&samples[(size_t)j * m], &rmodels[(size_t)j * S * 9]);
            }
            const SprtTest frozen = cfg->sprt ? sprt.hist[sprt.cur] : SprtTest();
            for (int j = 0; j < K; j++) {
                for (int i = 0; i < nmodels[j]; i++) {
                    const size_t q = (size_t)j * S + i;
                    const float* mdl = &rmodels[q * 9];
                    if (cfg->sprt) {
                        f.set(est, mdl);
                        unsigned tp, ti, end;
                        unsigned start = (unsigned)(((unsigned long long)cursor + 32ull * q) % (unsigned)n);
                        bool good = sprt.walk(f, points, frozen, start, tp, ti, end, evals);
                        r_good[q] = good; r_tested_inl[q] = (int)ti; r_tested_pts[q] = (int)tp;
                        r_inl[q] = (int)ti;
                        if (!good && hyp0 + j < 20) r_inl[q] = (int)(ti + sprt.count_rest(f, points, tp, end, evals));
                        r_score[q] = (float)r_inl[q];
                    } else {
                        orc_score(est, points, n, mdl, cfg->threshold, &r_inl[q], &r_score[q], nullptr, 0, nullptr);
                        evals += n;
                        r_good[q] = 1;
                    }
                    models_scored++;
                }
            }
            /* replay */
            const unsigned iters_round_start = iters;
            long long last_improving_inl = -1;
            unsigned long long rej_inl = 0, rej_pts = 0;
            for (int j = 0; j < K; j++) {
                if (!(iters < max_iters)) { done = true; break; }
                for (int i = 0; i < nmodels[j]; i++) {
                    const size_t q = (size_t)j * S + i;
                    if (cfg->sprt) {
                        if (r_good[q]) { if (r_tested_inl[q] > best_inl) last_improving_inl = r_tested_inl[q]; }
                        else { rej_inl += r_tested_inl[q]; rej_pts += r_tested_pts[q]; }
                        if (!r_good[q] && iters >= 20) { iters++; continue; }
                    }
                    if (bigger(r_inl[q], r_score[q], best_inl, best_score))
                        on_new_best(&rmodels[q * 9], r_inl[q], r_score[q], (long long)(hyp0 + j), i);
                }
                iters++;
            }
            if (cfg->sprt) {
                const SprtTest t = sprt.hist[sprt.cur];
                double eps = t.epsilon, delta = t.delta;
                bool redesign = false;
                if (last_improving_inl >= 0) { eps = (float)last_improving_inl / n; redesign = true; }
                if (rej_pts > 0) {
                    float delta_estimated = (float)rej_inl / (unsigned)rej_pts;
                    if (delta_estimated > 0 && std::fabs(t.delta - delta_estimated) / t.delta > 0.05) { delta = delta_estimated; redesign = true; }
                }
                if (redesign) sprt.push_test(eps, delta, (int)iters_round_start);
                cursor = (unsigned)(((unsigned long long)cursor + 32ull * K * S) % (unsigned)n);
            }
        }
    }

    memcpy(out->model, best_model, sizeof(float) * msize);
    out->inliers = best_inl;
    out->score = best_score;
    out->iterations = iters;
    out->samples_drawn = (unsigned)hyp;
    out->evals = evals;
    out->models_scored = models_scored;
    if (lo) { unsigned a, b; unsigned long long c; orc_lo_counters(lo, &a, &b, &c); out->lo_inner = a; out->lo_iterative = b; orc_lo_free(lo); }
    orc_sampler_free(sampler);
    return best_inl > 0 ? 0 : 1;   /* ransac.cpp:143-147: the reference exits(111) when nothing was found */
}
