// usac_harness.cpp - the reference's test harness shape (test/test.cpp:5-60: build a Model, construct Ransac(model, points),
// run(), print RansacOutput) over the GPU plugin layer. Points come from the reference's dataset files (reader.hpp = detector/Reader.h):
//   --format pts    first line N, then N rows `x1 y1 x2 y2` (`x y` for lines): dataset/homography/sift_update/*_pts.txt (default)
//   --format nby6   rows `x1 y1 1 x2 y2 1` (Reader::getPointsNby6)
//   --format nby7   rows `x1 y1 z1 x2 y2 z2 isinlier` (Reader::read_points + getInliers; the flags give the GT inlier count)
//   --format evd    header + `x1,y1,x2,y2,FGINN,SNN,detector,descriptor,is_correct` (Reader::readEVDPointsInliers)
//   --format line2d `width height noise a b c N` + N rows `x y` (dataset/GetImage.h:88-116; the GT line gives the GT inlier count)
//   --gt-model F    3 x 3 ground-truth model (Reader::getMatrix3x3, the *_model.txt files): GT inliers = points under the threshold
//   usac_harness <points file> <line2d|homography|fundamental|essential> <uniform|prosac|napsac> <threshold> <confidence> [seed]
//                [--format F] [--gt-model file] [--read-only] [--sequential|--both] [--sprt] [--lo 1|2] [--round K] [--max-iter N] [--knn K]
//                [--all-roots]
//                [--report] [--runs N --csv out.csv [--gt-inliers G]]
// --read-only parses the input, prints `read n=.. dim=.. checksum=.. flagged_inliers=..` and exits (no GPU needed).
// Prints one `key=value` line per result (model as IEEE bit patterns, inlier ids as a hash) for the parity tests; --report adds the
// human-readable block of Tests::test (test/test.cpp:38-53); --runs/--csv writes one statistics row in the column layout of
// Logging::saveHeadOfCSV / saveResultsCSV (helper/Logging.h:47-97) over N runs with seeds seed .. seed+N-1.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <fstream>
#include <numeric>

#include "ransac.hpp"
#include "reader.hpp"

static void report(const char* tag, Ransac& r, const Model& m);
static void report_block(Ransac& r, const Model& m);
static void report(const char* tag, Ransac& r, const Model& m) {
    RansacOutput* o = r.getRansacOutput();
    const cv::Mat d = o->getModel()->returnDescriptor();
    std::printf("%s iterations=%u inliers=%u time_us=%ld model_bits=", tag, o->getNumberOfMainIterations(), o->getNumberOfInliers(), o->getTimeMicroSeconds());
    for (int k = 0; k < d.rows * d.cols; k++) { unsigned u; float f = d.ptr()[k]; std::memcpy(&u, &f, 4); std::printf("%08x%s", u, k + 1 < d.rows * d.cols ? "," : ""); }
    unsigned long long h = 1469598103934665603ull;                                   // FNV-1a over the inlier ids
    for (int id : o->getInliers()) { h ^= (unsigned)id; h *= 1099511628211ull; }
    std::printf(" inlier_hash=%016llx score=%.9g\n", h, (double)r.lastFit().score);
    (void)m;
}

static const char* sampler_name(SAMPLER s) { return s == Uniform ? "uniform" : s == Prosac ? "prosac" : s == Napsac ? "napsac" : "unknown"; }
static const char* estimator_name(ESTIMATOR e) { return e == Line2d ? "line2d" : e == Homography ? "homography" : e == Fundamental ? "fundamental" : "essential"; }

static void report_block(Ransac& r, const Model& m) {                               // test/test.cpp:38-53
    RansacOutput* o = r.getRansacOutput();
    const long us = o->getTimeMicroSeconds();
    std::cout << sampler_name(m.sampler) << "_" << estimator_name(m.estimator) << "\n";
    std::cout << "\ttime: " << us / 1000000 << " secs, " << (us / 1000) % 1000 << " ms, " << us % 1000 << " mcs\n";
    std::cout << "\tMain iterations: " << o->getNumberOfMainIterations() << "\n";
    std::cout << "\tLO iterations: " << o->getLOIters() << " (where " << o->getLOInnerIters() << " (inner iters) and " << o->getLOIterativeIters()
              << " (iterative iters) and " << o->getGCIters() << " (GC iters))\n";
    std::cout << "\tpoints under threshold: " << o->getNumberOfInliers() << "\n";
    std::cout << "Best model = ...\n" << o->getModel()->returnDescriptor() << "\n";
}

struct Stat { double avg, std_dev, med; };
static Stat stat_of(std::vector<double> v) {
    Stat s{0, 0, 0};
    if (v.empty()) return s;
    s.avg = std::accumulate(v.begin(), v.end(), 0.0) / v.size();
    for (double x : v) s.std_dev += (x - s.avg) * (x - s.avg);
    s.std_dev = v.size() > 1 ? std::sqrt(s.std_dev / (v.size() - 1)) : 0.0;
    std::sort(v.begin(), v.end());
    s.med = v.size() % 2 ? v[v.size() / 2] : 0.5 * (v[v.size() / 2 - 1] + v[v.size() / 2]);
    return s;
}

int main(int argc, char** argv) {
    if (argc < 6 || !std::strcmp(argv[1], "--help")) {
        std::fprintf(stderr, "usage: %s <points.txt> <line2d|homography|fundamental|essential> <uniform|prosac|napsac> <threshold> <confidence> [seed] [--sequential|--both] [--sprt] [--lo 1|2] [--round K] [--max-iter N] [--knn K] [--all-roots] [--report] [--runs N --csv out.csv [--gt-inliers G]]\n", argv[0]);
        return argc < 2 ? 2 : (!std::strcmp(argv[1], "--help") ? 0 : 2);
    }
    const std::string est = argv[2], smp = argv[3];
    const ESTIMATOR e = est == "line2d" ? Line2d : est == "homography" ? Homography : est == "fundamental" ? Fundamental : est == "essential" ? Essential : NullE;
    const SAMPLER s = smp == "uniform" ? Uniform : smp == "prosac" ? Prosac : smp == "napsac" ? Napsac : NullS;
    if (e == NullE || s == NullS) { std::fprintf(stderr, "unknown estimator/sampler\n"); return 2; }
    const int dim = e == Line2d ? 2 : 4;
    std::string format = "pts";
    const char* gt_model_file = nullptr;
    bool read_only = false;
    for (int i = 6; i < argc; i++) {
        if (!std::strcmp(argv[i], "--format") && i + 1 < argc) format = argv[i + 1];
        if (!std::strcmp(argv[i], "--gt-model") && i + 1 < argc) gt_model_file = argv[i + 1];
        if (!std::strcmp(argv[i], "--read-only")) read_only = true;
    }
    cv::Mat points, gt_model;
    std::vector<int> flagged;
    int flagged_known = 0;
    try {
        if (format == "pts" && dim == 4) { if (!Reader::LoadPointsFromFile(points, argv[1])) { std::fprintf(stderr, "cannot read %s\n", argv[1]); return 2; } }
        else if (format == "pts") {                                   // N, then N rows `x y`
            std::ifstream in(argv[1]);
            int n = 0;
            if (!(in >> n) || n <= 0) { std::fprintf(stderr, "cannot read %s\n", argv[1]); return 2; }
            points = cv::Mat(n, 2);
            for (int i = 0; i < 2 * n; i++) if (!(in >> points.ptr()[i])) { std::fprintf(stderr, "short points file\n"); return 2; }
        }
        else if (format == "nby6") Reader::getPointsNby6(argv[1], points);
        else if (format == "nby7") {
            cv::Mat p1, p2;
            Reader::read_points(p1, p2, argv[1]);
            Reader::getInliers(argv[1], flagged);
            flagged_known = 1;
            points = cv::Mat(p1.rows, 4);
            for (int i = 0; i < p1.rows; i++) { points.at(i, 0) = p1.at(i, 0); points.at(i, 1) = p1.at(i, 1); points.at(i, 2) = p2.at(i, 0); points.at(i, 3) = p2.at(i, 1); }
        }
        else if (format == "evd") { Reader::readEVDPointsInliers(points, flagged, argv[1]); flagged_known = 1; }
        else if (format == "line2d") { if (!Reader::readLine2d(points, gt_model, argv[1])) { std::fprintf(stderr, "cannot read %s\n", argv[1]); return 2; } }
        else { std::fprintf(stderr, "unknown --format %s\n", format.c_str()); return 2; }
        if (gt_model_file) Reader::getMatrix3x3(gt_model_file, gt_model);
    } catch (const std::exception& ex) { std::fprintf(stderr, "usac_harness: %s\n", ex.what()); return 2; }
    if (points.rows <= 0 || points.cols != dim) { std::fprintf(stderr, "%s: no %d-column points read (format %s)\n", argv[1], dim, format.c_str()); return 2; }
    if (read_only) {
        unsigned long long h = 1469598103934665603ull;
        for (int i = 0; i < points.rows * points.cols; i++) { unsigned u; std::memcpy(&u, points.ptr() + i, 4); h ^= u; h *= 1099511628211ull; }
        std::printf("read n=%d dim=%d checksum=%016llx flagged_inliers=%d gt_model=%d\n", points.rows, points.cols, h, flagged_known ? (int)flagged.size() : -1,
                    gt_model.empty() ? 0 : gt_model.rows * gt_model.cols);
        return 0;
    }
    const unsigned m = e == Line2d ? 2 : e == Homography ? 4 : e == Fundamental ? 7 : 5;
    Model model((float)std::atof(argv[4]), m, (float)std::atof(argv[5]), 5, e, s);
    bool sequential = false, both = false, want_report = false;
    int runs = 0, gt_inliers = 0, knn = 0;
    const char* csv = nullptr;
    for (int i = 6; i < argc; i++) {
        if (!std::strcmp(argv[i], "--sequential")) sequential = true;
        else if (!std::strcmp(argv[i], "--both")) both = true;
        else if (!std::strcmp(argv[i], "--report")) want_report = true;
        else if (!std::strcmp(argv[i], "--lo") && i + 1 < argc) model.lo = std::atoi(argv[++i]) == 2 ? InItFLORsc : InItLORsc;
        else if (!std::strcmp(argv[i], "--runs") && i + 1 < argc) runs = std::atoi(argv[++i]);
        else if (!std::strcmp(argv[i], "--csv") && i + 1 < argc) csv = argv[++i];
        else if (!std::strcmp(argv[i], "--gt-inliers") && i + 1 < argc) gt_inliers = std::atoi(argv[++i]);
        else if (!std::strcmp(argv[i], "--knn") && i + 1 < argc) knn = std::atoi(argv[++i]);
        else if (!std::strcmp(argv[i], "--sprt")) model.setSprt(true);
        else if (!std::strcmp(argv[i], "--all-roots")) model.setGpuEssentialAllRoots(true);   // essential: every cheirality-valid root
        else if (!std::strcmp(argv[i], "--round") && i + 1 < argc) model.gpu_round_size = std::atoi(argv[++i]);
        else if (!std::strcmp(argv[i], "--max-iter") && i + 1 < argc) model.max_iterations = (unsigned)std::atoi(argv[++i]);
        else if ((!std::strcmp(argv[i], "--format") || !std::strcmp(argv[i], "--gt-model")) && i + 1 < argc) i++;
        else if (!std::strcmp(argv[i], "--read-only")) {}
        else model.seed = std::strtoull(argv[i], nullptr, 10);
    }
    model.setCellSize(50);
    if (s == Napsac) model.setNeighborsType(knn > 0 ? Nanoflann : Grid);
    if (knn > 0) model.setKNearestNeighbors(knn);
    try {
        if (gt_inliers == 0 && flagged_known) gt_inliers = (int)flagged.size();
        if (gt_inliers == 0 && !gt_model.empty()) {                            // GT inliers = points of the GT model under the threshold (Quality)
            Ransac r(&model, points);
            Score sc;
            r.getQuality()->getNumberInliers(&sc, gt_model);
            gt_inliers = sc.inlier_number;
            std::printf("gt_model inliers=%d\n", gt_inliers);
        }
        if (runs > 0 && csv) {                                                  // Tests::getStatisticalResults, test/tests.h:148-150
            std::vector<double> inl, it, lo, us;
            int worst = 1 << 30, f10 = 0, f25 = 0, f50 = 0;
            Ransac r(&model, points);
            const unsigned long long seed0 = model.seed;
            for (int k = 0; k < runs; k++) {
                model.seed = seed0 + k;
                Ransac rk(&model, points);
                rk.run();
                RansacOutput* o = rk.getRansacOutput();
                inl.push_back(o->getNumberOfInliers()); it.push_back(o->getNumberOfMainIterations()); lo.push_back(o->getLOIters());
                us.push_back((double)o->getTimeMicroSeconds());
                worst = std::min(worst, (int)o->getNumberOfInliers());
                if (gt_inliers > 0) { const double q = (double)o->getNumberOfInliers() / gt_inliers; f10 += q < 0.1; f25 += q < 0.25; f50 += q < 0.5; }
            }
            const Stat si = stat_of(inl), st = stat_of(it), sl = stat_of(lo), su = stat_of(us);
            std::ofstream f(csv);
            f << sampler_name(model.sampler) << "_" << estimator_name(model.estimator) << "\n";
            f << "Runs for each image = " << runs << "\nThreshold for each image = " << model.threshold << "\nDesired probability for each image = "
              << model.desired_prob << "\nInner Iterative LO = " << (model.lo == InItLORsc) << "\nInner Iterative Fxing LO = " << (model.lo == InItFLORsc)
              << "\nGraph Cut LO = 0\nSPRT = " << model.sprt << "\n\n\n";
            f << "Filename,GT Inl,Avg num inl/gt,Std dev num inl,Med num inl,Avg num iters,Std dev num iters,Med num iters,Avg num LO iters,"
                 "Std dev num LO iters,Med num LO iters,Avg time (mcs),Std dev time,Med time,Avg err,Std dev err,Med err,Worst case num Inl,"
                 "Worst case Err,Num fails (<10%),Num fails (<25%),Num fails (<50%)\n";
            f << argv[1] << "," << gt_inliers << "," << si.avg << "," << si.std_dev << "," << si.med << "," << st.avg << "," << st.std_dev << "," << st.med
              << "," << sl.avg << "," << sl.std_dev << "," << sl.med << "," << su.avg << "," << su.std_dev << "," << su.med << ",,,," << worst << ",,"
              << f10 << "," << f25 << "," << f50 << "\n";
            std::printf("stats runs=%d avg_inliers=%.3f avg_iterations=%.3f avg_lo=%.3f avg_time_us=%.1f worst_inliers=%d\n", runs, si.avg, st.avg, sl.avg, su.avg, worst);
            return 0;
        }
        if (!sequential || both) { Ransac r(&model, points); r.run(); report("fused", r, model); if (want_report) report_block(r, model); }
        if (sequential || both) { Ransac r(&model, points); r.run_sequential(); report("sequential", r, model); if (want_report) report_block(r, model); }
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "usac_harness: %s\n", ex.what());
        return 111;                                                                  // the reference's fatal exit code (init.cpp:17-19)
    }
    return 0;
}
