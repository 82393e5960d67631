// usac_gpu.cu - context, host orchestration and the C ABI of libusac_gpu.so (see include/usac_gpu.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC (ransac_b200/build.py)
#include <dlfcn.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "essential.cuh"
#include "pipeline.cuh"
#include "score.cuh"
#include "score_sq.cuh"
#include "sprt.cuh"
#include "refit.cuh"
#include "lo.cuh"
#include "knn.cuh"
#include "host_replay.hpp"

// ------------------------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------------------------
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;   // elements
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// pinned host staging (device -> host copies into pageable memory block the calling thread until the copy has run)
template <typename T>
struct PinnedBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMallocHost(&p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct SideUsed { size_t knn = 0, grid = 0, cell_start = 0, cursors = 0, pool = 0; };   // elements used in the appended side arrays

struct usac_gpu_ctx {
    SideUsed side;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    cudaDeviceProp prop;
    std::string err;
    void set_error(const char* what, const char* why) { err = std::string(what) + ": " + why; }

    // data
    int est = 0, est_prev = 0, P = 0;
    std::vector<ProblemDesc> h_prob;
    std::vector<ProblemDesc> h_prob_pushed;   // what d_prob holds (push_desc skips the upload when nothing changed)
    bool maxima_fetched = false;              // coordinate maxima (written by layout_kernel) copied into h_prob
    long long total_points = 0, total_pairs = 0;
    DevBuf<float> d_aos, d_pairs;
    DevBuf<ProblemDesc> d_prob;
    DevBuf<long long> d_pair_offs;
    DevBuf<FitState> d_state;
    FitState* h_state = nullptr; size_t h_state_cap = 0;     // pinned
    DevBuf<int> d_active, d_done;
    DevBuf<int> d_active2;                    // second active list: the lists of consecutive rounds are compacted on the device
    DevBuf<FitState> d_state_init;            // initial fit states of the current point sets (uploaded once, copied per fit)
    std::vector<long long> state_init_sig;
    int* h_active = nullptr; size_t h_active_cap = 0;        // pinned
    int* h_done = nullptr;                                   // pinned, same capacity as h_active
    // side structures
    DevBuf<int> d_knn, d_cell_of_point, d_members, d_rank, d_cell_start, d_pool;
    DevBuf<unsigned> d_cursors, d_growth, d_term;
    std::vector<int> h_pool_set;   // problems with an uploaded SPRT pool
    // round buffers
    DevBuf<int> d_samples, d_nmodels, d_offsets, d_mvalid, d_part_cnt, d_seeds, d_table;
    DevBuf<float> d_models_raw, d_recs, d_part_sum;
    DevBuf<uint2> d_scores, d_scores_all;
    DevBuf<SprtModelResult> d_sprt_res;
    DevBuf<SprtCarry> d_sprt_carry;          // walks handed from sprt_walk_kernel to sprt_tail_kernel
    DevBuf<unsigned> d_sprt_count;
    cudaStream_t stream2 = nullptr;           // solve-ahead blocks of the SPRT replay path run here, beside the rounds of the previous block
    cudaEvent_t ev_block[2] = {nullptr, nullptr};
    cudaEvent_t ev_round = nullptr;
    DevBuf<int> d_lo_bwave;                   // speculative LO waves (lo.cuh): candidate inlier lists, per-iteration records, state
    DevBuf<LoSpec> d_lo_spec;
    DevBuf<LoWaveState> d_lo_ws;
    PinnedBuf<LoWaveState> h_lo_ws;
    DevBuf<LoWaveArgs> d_lo_calls;            // batched LO steps: one record per pending call, its LoIO and the model it starts from
    PinnedBuf<LoWaveArgs> h_lo_calls;
    PinnedBuf<LoIO> h_lo_io;
    DevBuf<long long> d_lo_src;
    PinnedBuf<long long> h_lo_src;
    DevBuf<unsigned> d_inl_ballots;          // inlier flags of a large problem (launch_inliers)
    DevBuf<int> d_inl_counts;
    PinnedBuf<int> h_rp_nmodels;              // replay path: the round's results on the host
    PinnedBuf<SprtModelResult> h_rp_res;
    PinnedBuf<int2> h_rp_scores;
    PinnedBuf<float> h_rp_models;
    PinnedBuf<FitState> h_rp_state;
    DevBuf<int2> d_model_scores;
    DevBuf<float> d_pool_pts;          // the points in SPRT pool order (same offsets as d_aos)
    DevBuf<unsigned long long> d_grid_keys;   // grid build scratch: 2n keys
    DevBuf<int> d_grid_ints;                  // grid build scratch: 4n ints + 1
    DevBuf<unsigned char> d_grid_temp;        // CUB temporary storage
    DevBuf<unsigned> d_work;                  // work-item counter of the scoring kernel (monotone; see launch_score)
    DevBuf<uint2> d_items;                    // compact work-item list of a round (prepare_kernel -> scoring kernel)
    DevBuf<unsigned> d_item_count;            // [0] items in d_items, [1] draw counter of that launch; zeroed before every round
    unsigned work_next = 0;
    DevBuf<int> d_knn_cells;                  // kNN build scratch: cell_start of the search grid
    DevBuf<float4> d_knn_pts;                 // kNN build scratch: points in cell order
    // scoring API buffers
    DevBuf<float> d_q_models, d_q_recs, d_q_sum, d_q_err;
    DevBuf<int> d_q_cnt, d_q_ids, d_q_ids2, d_q_ok, d_lo_ids_a, d_lo_ids_b, d_lo_small;
    DevBuf<float> d_q_model2;
    DevBuf<LoIO> d_lo_io;
    // exchange
    usac_allgather_fn allgather = nullptr;
    void* allgather_user = nullptr;
    void* nccl_lib = nullptr;
    void* nccl_comm = nullptr;
    // exchange over peer memory (usac_gpu_peer_*): this rank's window, the windows of all ranks, round sequence number
    void* peer_self = nullptr;
    unsigned peer_cap = 0;                    // uint2 entries per parity buffer
    std::vector<void*> peer_opened;           // windows mapped with cudaIpcOpenMemHandle (closed in destroy)
    DevBuf<void*> d_peer_win;
    DevBuf<unsigned> d_peer_counter;
    DevBuf<int> d_peer_error;
    int* h_peer_error = nullptr;              // pinned
    int peer_rank = -1, peer_nranks = 0;
    unsigned peer_seq = 0;
    unsigned long long peer_rounds = 0;       // rounds exchanged through the windows (diagnostics)
    // termination tables of the last fit (rebuilt only when (n, m, confidence, max_iterations) change)
    std::map<std::tuple<int, int, float, unsigned>, std::vector<unsigned>> term_cache;
    std::vector<long long> term_signature;   // what d_term currently holds: (m, confidence bits, max_iterations, n of every problem)
    // timing
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> score_events;
    size_t score_events_used = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    float last_total_ms = 0, last_score_ms = 0;
    int last_launches = 0, last_score_launches = 0;

    // USAC_GPU_TRACE=2: per-kernel device times of a fit (events between the launches of the main loop), printed by rank-local stderr
    std::vector<std::pair<const char*, cudaEvent_t>> marks;
    size_t marks_used = 0;
    void mark(const char* name) {
        if (marks_used == marks.size()) { cudaEvent_t e; cudaEventCreate(&e); marks.push_back({name, e}); }
        marks[marks_used].first = name;
        cudaEventRecord(marks[marks_used].second, stream);
        marks_used++;
    }

    std::pair<cudaEvent_t, cudaEvent_t>& next_score_event() {
        if (score_events_used == score_events.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a); cudaEventCreate(&b);
            score_events.push_back({a, b});
        }
        return score_events[score_events_used++];
    }
};

static std::string g_create_error;
static cudaError_t set_lo_smem_attributes();

static int fail(usac_gpu_ctx* ctx, int code, const char* msg) {
    if (ctx) ctx->err = msg;
    return code;
}

extern "C" int usac_gpu_create(usac_gpu_ctx** out, int device) {
    if (!out) return USAC_ERR_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libusac_gpu has no CPU fallback)";
        return USAC_ERR_CUDA;
    }
    if (device < 0 || device >= count) { g_create_error = "device index out of range"; return USAC_ERR_ARG; }
    usac_gpu_ctx* c = new usac_gpu_ctx;
    c->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&c->prop, device)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete c;
        return USAC_ERR_CUDA;
    }
    if (c->prop.major < 10) {
        g_create_error = "libusac_gpu is built for sm_100a only; device is sm_" + std::to_string(c->prop.major * 10 + c->prop.minor);
        delete c;
        return USAC_ERR_CUDA;
    }
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete c;
        return USAC_ERR_CUDA;
    }
    cudaEventCreate(&c->ev0);
    cudaEventCreate(&c->ev1);
    // the LO / non-minimal kernels use more than 48 KB of dynamic shared memory: an opt-in of the device's context, set here after
    // cudaSetDevice so that every context on every device has it
    if ((e = set_lo_smem_attributes()) != cudaSuccess) {
        g_create_error = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e);
        usac_gpu_destroy(c);
        return USAC_ERR_CUDA;
    }
    if ((e = c->d_work.ensure(1)) != cudaSuccess || (e = cudaMemset(c->d_work.p, 0, sizeof(unsigned))) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete c;
        return USAC_ERR_CUDA;
    }
    *out = c;
    return USAC_OK;
}

extern "C" void usac_gpu_destroy(usac_gpu_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    for (int i = 0; i < 2; i++) if (c->ev_block[i]) cudaEventDestroy(c->ev_block[i]);
    if (c->ev_round) cudaEventDestroy(c->ev_round);
    for (void* w : c->peer_opened) cudaIpcCloseMemHandle(w);
    if (c->peer_self) cudaFree(c->peer_self);
    if (c->h_peer_error) cudaFreeHost(c->h_peer_error);
    c->d_peer_win.release(); c->d_peer_counter.release(); c->d_peer_error.release();
    if (c->nccl_comm && c->nccl_lib) {
        typedef int (*destroy_fn)(void*);
        destroy_fn f = (destroy_fn)dlsym(c->nccl_lib, "ncclCommDestroy");
        if (f) f(c->nccl_comm);
    }
    c->d_aos.release(); c->d_pairs.release(); c->d_prob.release(); c->d_pair_offs.release(); c->d_state.release(); c->d_active.release(); c->d_active2.release(); c->d_state_init.release();
    c->d_knn.release(); c->d_cell_of_point.release(); c->d_members.release(); c->d_rank.release(); c->d_cell_start.release();
    c->d_pool.release(); c->d_cursors.release(); c->d_growth.release(); c->d_term.release();
    c->d_samples.release(); c->d_nmodels.release(); c->d_offsets.release(); c->d_mvalid.release(); c->d_part_cnt.release();
    c->d_seeds.release(); c->d_table.release(); c->d_models_raw.release(); c->d_recs.release(); c->d_part_sum.release();
    c->d_scores.release(); c->d_scores_all.release(); c->d_sprt_res.release(); c->d_sprt_carry.release(); c->d_sprt_count.release(); c->d_inl_ballots.release(); c->d_inl_counts.release(); c->d_lo_bwave.release(); c->d_lo_spec.release(); c->d_lo_ws.release(); c->h_lo_ws.release(); c->d_lo_calls.release(); c->h_lo_calls.release(); c->h_lo_io.release(); c->d_lo_src.release(); c->h_lo_src.release(); c->h_rp_nmodels.release(); c->h_rp_res.release(); c->h_rp_scores.release(); c->h_rp_models.release(); c->h_rp_state.release(); c->d_model_scores.release(); c->d_pool_pts.release(); c->d_grid_keys.release(); c->d_grid_ints.release(); c->d_grid_temp.release(); c->d_knn_cells.release(); c->d_knn_pts.release(); c->d_work.release(); c->d_items.release(); c->d_item_count.release();
    c->d_q_models.release(); c->d_q_recs.release(); c->d_q_sum.release(); c->d_q_err.release(); c->d_q_cnt.release(); c->d_q_ids.release(); c->d_q_ids2.release(); c->d_q_ok.release(); c->d_q_model2.release(); c->d_lo_ids_a.release(); c->d_lo_ids_b.release(); c->d_lo_small.release(); c->d_lo_io.release();
    if (c->h_state) cudaFreeHost(c->h_state);
    if (c->h_active) cudaFreeHost(c->h_active);
    if (c->h_done) cudaFreeHost(c->h_done);
    c->d_done.release();
    for (auto& pr : c->score_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int usac_gpu_set_stream(usac_gpu_ctx* c, void* cuda_stream) {
    if (!c) return USAC_ERR_ARG;
    cudaSetDevice(c->device);
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    if (c->own_stream) cudaStreamDestroy(c->stream);
    c->stream = (cudaStream_t)cuda_stream;
    c->own_stream = false;
    return USAC_OK;
}

extern "C" const char* usac_gpu_last_error(const usac_gpu_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

extern "C" int usac_gpu_device_info(const usac_gpu_ctx* c, int info[4]) {
    if (!c || !info) return USAC_ERR_ARG;
    info[0] = c->prop.multiProcessorCount;
    info[1] = c->prop.clockRate;
    info[2] = c->prop.major * 10 + c->prop.minor;
    info[3] = c->prop.l2CacheSize;
    return USAC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// data upload: AoS copy + device-side re-layout into point pairs + per-column max |coordinate|
// ------------------------------------------------------------------------------------------------------------------
// per-column max |coordinate| of a problem: one atomic per warp when the whole warp belongs to one problem (the usual case;
// 4 atomics per thread on 4 addresses per problem made this kernel 5x slower than its memory traffic)
__device__ __forceinline__ void column_max(unsigned* dst, float v, bool uniform_warp) {
    unsigned bits = __float_as_uint(v);                      // |v| >= 0: the bit pattern is monotone
    if (uniform_warp) {
        bits = __reduce_max_sync(0xffffffffu, bits);
        if ((threadIdx.x & 31) == 0) atomicMax(dst, bits);
    } else {
        atomicMax(dst, bits);
    }
}

__global__ void layout_kernel(const float* __restrict__ aos, float* __restrict__ pairs, ProblemDesc* prob, int P, int dim,
                              const long long* __restrict__ pair_offs, long long total_pairs) {
    const long long gp = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = gp < total_pairs;
    int lo = 0, hi = P - 1;                       // problem owning global pair gp
    if (live) while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (pair_offs[mid] <= gp) lo = mid; else hi = mid - 1; }
    const int first = __shfl_sync(0xffffffffu, lo, 0);
    const bool uniform_warp = __all_sync(0xffffffffu, live && lo == first);
    if (!live) return;
    ProblemDesc& pd = prob[lo];
    const int j = (int)(gp - pd.pair_off);
    const int i0 = 2 * j, i1 = 2 * j + 1;
    const float nanv = __int_as_float(0x7fc00000);
    if (dim == 4) {
        const float4 a = reinterpret_cast<const float4*>(aos)[pd.aos_off + i0];
        const float4 b = (i1 < pd.n) ? reinterpret_cast<const float4*>(aos)[pd.aos_off + i1] : make_float4(nanv, nanv, nanv, nanv);
        float4* dst = reinterpret_cast<float4*>(pairs) + 2 * gp;
        dst[0] = make_float4(a.x, b.x, a.y, b.y);
        dst[1] = make_float4(a.z, b.z, a.w, b.w);
        float m1 = fabsf(a.x), m2 = fabsf(a.y), m3 = fabsf(a.z), m4 = fabsf(a.w);
        if (i1 < pd.n) { m1 = fmaxf(m1, fabsf(b.x)); m2 = fmaxf(m2, fabsf(b.y)); m3 = fmaxf(m3, fabsf(b.z)); m4 = fmaxf(m4, fabsf(b.w)); }
        column_max(reinterpret_cast<unsigned*>(&pd.mx1), m1, uniform_warp);
        column_max(reinterpret_cast<unsigned*>(&pd.my1), m2, uniform_warp);
        column_max(reinterpret_cast<unsigned*>(&pd.mx2), m3, uniform_warp);
        column_max(reinterpret_cast<unsigned*>(&pd.my2), m4, uniform_warp);
    } else {
        const float2 a = reinterpret_cast<const float2*>(aos)[pd.aos_off + i0];
        const float2 b = (i1 < pd.n) ? reinterpret_cast<const float2*>(aos)[pd.aos_off + i1] : make_float2(nanv, nanv);
        reinterpret_cast<float4*>(pairs)[gp] = make_float4(a.x, b.x, a.y, b.y);
        float m1 = fabsf(a.x), m2 = fabsf(a.y);
        if (i1 < pd.n) { m1 = fmaxf(m1, fabsf(b.x)); m2 = fmaxf(m2, fabsf(b.y)); }
        column_max(reinterpret_cast<unsigned*>(&pd.mx1), m1, uniform_warp);
        column_max(reinterpret_cast<unsigned*>(&pd.my1), m2, uniform_warp);
    }
}

extern "C" int usac_gpu_set_points(usac_gpu_ctx* c, int estimator, const float* points, const int* n_per_problem, int P) {
    if (!c || !points || !n_per_problem || P <= 0) return fail(c, USAC_ERR_ARG, "set_points: bad arguments");
    if (estimator < USAC_EST_LINE2D || estimator > USAC_EST_ESSENTIAL) return fail(c, USAC_ERR_ARG, "set_points: unknown estimator");
    cudaSetDevice(c->device);
    const int dim = usac_point_dim(estimator);
    // validate and lay out in locals first: the context changes only once nothing can fail any more, and a failure after that
    // point leaves it empty (P = 0) rather than half updated
    std::vector<ProblemDesc> desc(P);
    std::vector<long long> pair_offs(P);
    long long aos = 0, pairs = 0;
    const bool same_shape = c->h_prob.size() == (size_t)P && estimator == c->est;
    for (int p = 0; p < P; p++) {
        const int n = n_per_problem[p];
        if (n < usac_sample_size(estimator)) return fail(c, USAC_ERR_ARG, "set_points: a problem has fewer points than the minimal sample");
        ProblemDesc& d = desc[p];
        memset(&d, 0, sizeof(d));
        d.n = n; d.n_pairs = (n + 1) / 2; d.aos_off = aos; d.pair_off = pairs;
        d.growth_off = d.term_off = d.pool_off = d.knn_off = d.grid_off = d.cell_start_off = d.cursor_off = -1;
        if (same_shape && c->h_prob[p].n == n) d.term_off = c->h_prob[p].term_off;   // equally sized point sets keep their termination-table offsets
        pair_offs[p] = pairs;
        aos += n; pairs += d.n_pairs;
    }
    struct Rollback {                          // any early return below leaves an empty, consistent context
        usac_gpu_ctx* c; bool armed = true;
        ~Rollback() { if (armed) { c->P = 0; c->est = 0; c->h_prob.clear(); c->h_prob_pushed.clear(); c->total_points = c->total_pairs = 0; c->term_signature.clear(); c->state_init_sig.clear(); } }
    } rollback{c};
    const size_t pair_floats = (dim == 4) ? 8 : 4;
    CUDA_TRY(c, c->d_aos.ensure((size_t)aos * dim));
    CUDA_TRY(c, c->d_pairs.ensure((size_t)pairs * pair_floats));
    CUDA_TRY(c, c->d_prob.ensure(P));
    CUDA_TRY(c, c->d_pair_offs.ensure(P));
    CUDA_TRY(c, c->d_state.ensure(P));
    CUDA_TRY(c, c->d_active.ensure(P));
    CUDA_TRY(c, c->d_active2.ensure(P));
    if (c->d_state_init.cap < (size_t)P) {                  // the template survives a new upload of equally sized point sets
        CUDA_TRY(c, c->d_state_init.ensure(P));
        c->state_init_sig.clear();
    }
    CUDA_TRY(c, c->d_done.ensure(P));
    if (c->h_state_cap < (size_t)P) {
        if (c->h_state) cudaFreeHost(c->h_state);
        c->h_state = nullptr; c->h_state_cap = 0;
        CUDA_TRY(c, cudaMallocHost(&c->h_state, sizeof(FitState) * P));
        c->h_state_cap = P;
    }
    if (c->h_active_cap < (size_t)P) {
        if (c->h_active) cudaFreeHost(c->h_active);
        if (c->h_done) cudaFreeHost(c->h_done);
        c->h_active = c->h_done = nullptr; c->h_active_cap = 0;
        CUDA_TRY(c, cudaMallocHost(&c->h_active, sizeof(int) * P));
        CUDA_TRY(c, cudaMallocHost(&c->h_done, sizeof(int) * P));
        c->h_active_cap = P;
    }
    c->est_prev = c->est;
    c->est = estimator; c->P = P;
    c->h_prob = std::move(desc);
    c->h_prob_pushed.clear(); c->maxima_fetched = false;
    c->total_points = aos; c->total_pairs = pairs;
    c->h_pool_set.assign(P, 0);
    c->side = SideUsed();                 // neighbourhoods / pools belong to the previous point sets
    {   // the point upload goes in 4 MB pieces: the copy engine serves streams in submission order, and the few-KB uploads of
        // another context's running fit (its per-round active list) must not wait behind one 100+ MB transfer
        const size_t bytes = (size_t)aos * dim * sizeof(float), piece = (size_t)4 << 20;
        for (size_t off = 0; off < bytes; off += piece)
            CUDA_TRY(c, cudaMemcpyAsync(reinterpret_cast<char*>(c->d_aos.p) + off, reinterpret_cast<const char*>(points) + off,
                                        std::min(piece, bytes - off), cudaMemcpyHostToDevice, c->stream));
    }
    CUDA_TRY(c, cudaMemcpyAsync(c->d_prob.p, c->h_prob.data(), sizeof(ProblemDesc) * P, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_pair_offs.p, pair_offs.data(), sizeof(long long) * P, cudaMemcpyHostToDevice, c->stream));
    const int threads = 256;
    layout_kernel<<<(unsigned)((pairs + threads - 1) / threads), threads, 0, c->stream>>>(c->d_aos.p, c->d_pairs.p, c->d_prob.p, P, dim,
                                                                                          c->d_pair_offs.p, pairs);
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));   // pair_offs / h_prob staging are stack/heap temporaries
    c->h_prob_pushed = c->h_prob;                    // d_prob = this + the coordinate maxima layout_kernel has just written
    rollback.armed = false;
    return USAC_OK;
}

// push host-side descriptor fields that the host owns (offsets) without clobbering the device-computed maxima
static int push_desc(usac_gpu_ctx* c) {
    if (!c->maxima_fetched) {                                   // once per point set: the maxima layout_kernel computed
        std::vector<ProblemDesc> cur(c->P);
        CUDA_TRY(c, cudaMemcpyAsync(cur.data(), c->d_prob.p, sizeof(ProblemDesc) * c->P, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        for (int p = 0; p < c->P; p++) {
            ProblemDesc& h = c->h_prob[p];
            h.mx1 = cur[p].mx1; h.my1 = cur[p].my1; h.mx2 = cur[p].mx2; h.my2 = cur[p].my2;
            if (c->h_prob_pushed.size() == (size_t)c->P) {
                ProblemDesc& q = c->h_prob_pushed[p];
                q.mx1 = h.mx1; q.my1 = h.my1; q.mx2 = h.mx2; q.my2 = h.my2;
            }
        }
        c->maxima_fetched = true;
    }
    if (c->h_prob_pushed.size() == c->h_prob.size() &&
        memcmp(c->h_prob_pushed.data(), c->h_prob.data(), sizeof(ProblemDesc) * c->h_prob.size()) == 0)
        return USAC_OK;
    CUDA_TRY(c, cudaMemcpyAsync(c->d_prob.p, c->h_prob.data(), sizeof(ProblemDesc) * c->P, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->h_prob_pushed = c->h_prob;
    return USAC_OK;
}

// grow a device array of per-problem segments: returns the offset of a new segment of `count` elements
template <class T>
static cudaError_t append_segment(DevBuf<T>& buf, size_t& used, const T* host, size_t count, long long* off_out, cudaStream_t s) {
    if (used + count > buf.cap) {
        DevBuf<T> nb;
        cudaError_t e = nb.ensure(std::max((used + count) * 2, (size_t)1024));
        if (e != cudaSuccess) return e;
        if (used) cudaMemcpyAsync(nb.p, buf.p, used * sizeof(T), cudaMemcpyDeviceToDevice, s);
        cudaStreamSynchronize(s);
        buf.release();
        buf = nb;
    }
    cudaError_t e = host ? cudaMemcpyAsync(buf.p + used, host, count * sizeof(T), cudaMemcpyHostToDevice, s)
                         : cudaMemsetAsync(buf.p + used, 0, count * sizeof(T), s);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(s);
    *off_out = (long long)used;
    used += count;
    return e;
}


// reserve a segment of `count` elements at the end of a side array (contents undefined)
template <class T>
static cudaError_t reserve_segment(DevBuf<T>& buf, size_t used, size_t count, cudaStream_t s) {
    if (used + count <= buf.cap) return cudaSuccess;
    DevBuf<T> nb;
    cudaError_t e = nb.ensure(std::max((used + count) * 2, (size_t)1024));
    if (e != cudaSuccess) return e;
    if (used) cudaMemcpyAsync(nb.p, buf.p, used * sizeof(T), cudaMemcpyDeviceToDevice, s);
    cudaStreamSynchronize(s);
    buf.release();
    buf = nb;
    return cudaSuccess;
}

// segment of the kNN side array for a problem: an earlier table of the same size is overwritten in place (no leak on repeated calls)
static cudaError_t knn_segment(usac_gpu_ctx* c, ProblemDesc& d, int k, long long* off_out, bool* fresh) {
    SideUsed& u = c->side;
    if (d.knn_off >= 0 && d.knn == k) { *off_out = d.knn_off; *fresh = false; return cudaSuccess; }
    cudaError_t e = reserve_segment(c->d_knn, u.knn, (size_t)d.n * k, c->stream);
    if (e != cudaSuccess) return e;
    *off_out = (long long)u.knn; *fresh = true;
    return cudaSuccess;
}

extern "C" int usac_gpu_set_neighbors_knn(usac_gpu_ctx* c, int problem, const int* neighbors, int k) {
    if (!c || problem < 0 || problem >= c->P || !neighbors || k < 1) return fail(c, USAC_ERR_ARG, "set_neighbors_knn: bad arguments");
    if (k < usac_sample_size(c->est) - 1)
        return fail(c, USAC_ERR_ARG, "set_neighbors_knn: k must be at least sample size - 1 (napsac_sampler.hpp:49 asserts it: a smaller k repeats points within a sample)");
    cudaSetDevice(c->device);
    SideUsed& u = c->side;
    ProblemDesc& d = c->h_prob[problem];
    for (size_t i = 0; i < (size_t)d.n * k; i++)
        if (neighbors[i] < 0 || neighbors[i] >= d.n) return fail(c, USAC_ERR_ARG, "set_neighbors_knn: neighbour index out of range");
    long long off;
    bool fresh;
    CUDA_TRY(c, knn_segment(c, d, k, &off, &fresh));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_knn.p + off, neighbors, sizeof(int) * (size_t)d.n * k, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    if (fresh) u.knn += (size_t)d.n * k;
    d.knn_off = off;
    if (d.cursor_off < 0) CUDA_TRY(c, append_segment(c->d_cursors, u.cursors, (const unsigned*)nullptr, 3 * (size_t)d.n + 1, &d.cursor_off, c->stream));
    d.neigh_type = USAC_NEIGH_KNN; d.knn = k;
    return push_desc(c);
}

// ---- device-side grid build (nearest_neighbors.cpp:160-201): cell = (int(x1/c), int(y1/c), int(x2/c), int(y2/c)), truncation
// toward zero; a point's neighbours are the other members of its cell in ascending index order. Stored as CSR: points sorted
// by a 64-bit cell key (stable radix sort keeps the index order inside a cell) + the rank of each point in its cell.
__global__ void grid_keys_kernel(const float* __restrict__ aos, int n, float cell, unsigned long long* __restrict__ keys, int* __restrict__ idx,
                                 int* __restrict__ overflow) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = reinterpret_cast<const float4*>(aos)[i];
    const int c0 = (int)__fdiv_rn(p.x, cell), c1 = (int)__fdiv_rn(p.y, cell), c2 = (int)__fdiv_rn(p.z, cell), c3 = (int)__fdiv_rn(p.w, cell);
    if (max(max(abs(c0), abs(c1)), max(abs(c2), abs(c3))) >= 32768) *overflow = 1;
    keys[i] = ((unsigned long long)(unsigned)(c0 + 32768) << 48) | ((unsigned long long)(unsigned)(c1 + 32768) << 32) |
              ((unsigned long long)(unsigned)(c2 + 32768) << 16) | (unsigned long long)(unsigned)(c3 + 32768);
    idx[i] = i;
}
__global__ void grid_flags_kernel(const unsigned long long* __restrict__ skeys, int n, int* __restrict__ flags) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n) flags[q] = (q == 0 || skeys[q] != skeys[q - 1]) ? 1 : 0;
}
__global__ void grid_starts_kernel(const int* __restrict__ flags, const int* __restrict__ cellid1, int n, int* __restrict__ cell_start) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n && flags[q]) cell_start[cellid1[q] - 1] = q;
}
__global__ void grid_fill_tail_kernel(const int* __restrict__ cellid1, int n, int* __restrict__ cell_start) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= n && c >= cellid1[n - 1]) cell_start[c] = n;
}
__global__ void grid_scatter_kernel(const int* __restrict__ sidx, const int* __restrict__ cellid1, const int* __restrict__ cell_start, int n,
                                    int* __restrict__ cell_of_point, int* __restrict__ members, int* __restrict__ rank) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const int p = sidx[q], cid = cellid1[q] - 1;
    members[q] = p;
    cell_of_point[p] = cid;
    rank[p] = q - cell_start[cid];
}

// ---- device-side kNN build (nearest_neighbors.cpp:69-128), kernels in knn.cuh
template <int DIM>
static void launch_knn_query(int cap, int blocks, cudaStream_t st, const float4* spts, const int* sidx, const unsigned* skeys, const int* cell_start,
                             const knn::GridDesc* gd, int G, int n, int k, int* table) {
    if (cap <= 8) knn::query_kernel<DIM, 8><<<blocks, 128, 0, st>>>(spts, sidx, skeys, cell_start, gd, G, n, k, table);
    else if (cap <= 16) knn::query_kernel<DIM, 16><<<blocks, 128, 0, st>>>(spts, sidx, skeys, cell_start, gd, G, n, k, table);
    else knn::query_kernel<DIM, 32><<<blocks, 128, 0, st>>>(spts, sidx, skeys, cell_start, gd, G, n, k, table);
}

extern "C" int usac_gpu_build_neighbors_knn(usac_gpu_ctx* c, int problem, int k) {
    if (!c || problem < 0 || problem >= c->P || k < 1 || k > 31) return fail(c, USAC_ERR_ARG, "build_neighbors_knn: bad arguments (1 <= k <= 31)");
    cudaSetDevice(c->device);
    ProblemDesc& d = c->h_prob[problem];
    const int n = d.n, dim = usac_point_dim(c->est);
    if (n < k + 1) return fail(c, USAC_ERR_ARG, "build_neighbors_knn: needs at least k + 1 points");
    if (k < usac_sample_size(c->est) - 1) return fail(c, USAC_ERR_ARG, "build_neighbors_knn: k must be at least sample size - 1 (napsac_sampler.hpp:49)");
    SideUsed& u = c->side;
    long long knn_off;
    bool knn_fresh;
    CUDA_TRY(c, knn_segment(c, d, k, &knn_off, &knn_fresh));
    const int G = std::max(1, std::min(1024, (int)std::ceil(std::sqrt((double)n / 16.0))));
    const int ncells = G * G;
    CUDA_TRY(c, c->d_grid_keys.ensure((size_t)n + 8));                       // 2 x n unsigned keys + bbox + grid descriptor
    CUDA_TRY(c, c->d_grid_ints.ensure(2 * (size_t)n + 16));
    CUDA_TRY(c, c->d_knn_cells.ensure((size_t)ncells + 1));
    CUDA_TRY(c, c->d_knn_pts.ensure((size_t)n));
    unsigned* keys = reinterpret_cast<unsigned*>(c->d_grid_keys.p);
    unsigned* skeys = keys + n;
    int* idx = c->d_grid_ints.p;
    int* sidx = idx + n;
    int* bbox = sidx + n;
    knn::GridDesc* gd = reinterpret_cast<knn::GridDesc*>(bbox + 4);
    const float* pts = c->d_aos.p + (size_t)d.aos_off * dim;
    const int g = (n + 255) / 256;
    knn::bbox_init_kernel<<<1, 1, 0, c->stream>>>(bbox);
    knn::bbox_kernel<<<std::min(g, 4 * c->prop.multiProcessorCount), 256, 0, c->stream>>>(pts, n, dim, bbox);
    knn::grid_desc_kernel<<<1, 1, 0, c->stream>>>(bbox, G, gd);
    knn::cell_keys_kernel<<<g, 256, 0, c->stream>>>(pts, n, dim, gd, G, keys, idx);
    int bits = 1;
    while ((1 << bits) < ncells) bits++;
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, keys, skeys, idx, sidx, n, 0, bits, c->stream);
    CUDA_TRY(c, c->d_grid_temp.ensure(tb));
    CUDA_TRY(c, cub::DeviceRadixSort::SortPairs(c->d_grid_temp.p, tb, keys, skeys, idx, sidx, n, 0, bits, c->stream));
    knn::cell_start_kernel<<<(ncells + 1 + 255) / 256, 256, 0, c->stream>>>(skeys, n, ncells, c->d_knn_cells.p);
    knn::gather_kernel<<<g, 256, 0, c->stream>>>(pts, n, dim, sidx, c->d_knn_pts.p);
    int* table = c->d_knn.p + knn_off;
    if (dim == 4) launch_knn_query<4>(k + 1, (n + 127) / 128, c->stream, c->d_knn_pts.p, sidx, skeys, c->d_knn_cells.p, gd, G, n, k, table);
    else launch_knn_query<2>(k + 1, (n + 127) / 128, c->stream, c->d_knn_pts.p, sidx, skeys, c->d_knn_cells.p, gd, G, n, k, table);
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    d.knn_off = knn_off;
    if (knn_fresh) u.knn += (size_t)n * k;
    if (d.cursor_off < 0) CUDA_TRY(c, append_segment(c->d_cursors, u.cursors, (const unsigned*)nullptr, 3 * (size_t)n + 1, &d.cursor_off, c->stream));
    d.neigh_type = USAC_NEIGH_KNN; d.knn = k;
    return push_desc(c);
}

extern "C" int usac_gpu_get_neighbors_knn(usac_gpu_ctx* c, int problem, int* neighbors_out, int* k_out) {
    if (!c || problem < 0 || problem >= c->P || !neighbors_out || !k_out) return fail(c, USAC_ERR_ARG, "get_neighbors_knn: bad arguments");
    const ProblemDesc& d = c->h_prob[problem];
    if (d.neigh_type != USAC_NEIGH_KNN || d.knn_off < 0) return fail(c, USAC_ERR_ARG, "get_neighbors_knn: no kNN table installed for this problem");
    cudaSetDevice(c->device);
    CUDA_TRY(c, cudaMemcpyAsync(neighbors_out, c->d_knn.p + d.knn_off, (size_t)d.n * d.knn * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    *k_out = d.knn;
    return USAC_OK;
}

extern "C" int usac_gpu_set_pnapsac_length(usac_gpu_ctx* c, int problem, unsigned long long local_samples) {
    if (!c || problem < 0 || problem >= c->P) return fail(c, USAC_ERR_ARG, "set_pnapsac_length: bad arguments");
    cudaSetDevice(c->device);
    c->h_prob[problem].pn_len = local_samples;                     // 0: the default, 20 n
    return push_desc(c);
}

extern "C" int usac_gpu_set_neighbors_grid(usac_gpu_ctx* c, int problem, int cell_size) {
    if (!c || problem < 0 || problem >= c->P || cell_size <= 0) return fail(c, USAC_ERR_ARG, "set_neighbors_grid: bad arguments");
    if (usac_point_dim(c->est) != 4) return fail(c, USAC_ERR_ARG, "set_neighbors_grid: needs correspondences (nearest_neighbors.cpp:172 reads 4 columns)");
    cudaSetDevice(c->device);
    ProblemDesc& d = c->h_prob[problem];
    const int n = d.n;
    SideUsed& u = c->side;
    CUDA_TRY(c, reserve_segment(c->d_cell_of_point, u.grid, (size_t)n, c->stream));
    CUDA_TRY(c, reserve_segment(c->d_members, u.grid, (size_t)n, c->stream));
    CUDA_TRY(c, reserve_segment(c->d_rank, u.grid, (size_t)n, c->stream));
    CUDA_TRY(c, reserve_segment(c->d_cell_start, u.cell_start, (size_t)n + 1, c->stream));
    CUDA_TRY(c, c->d_grid_keys.ensure(2 * (size_t)n));
    CUDA_TRY(c, c->d_grid_ints.ensure(4 * (size_t)n + 1));
    struct { unsigned long long* p; } keys{c->d_grid_keys.p}, skeys{c->d_grid_keys.p + n};
    struct { int* p; } idx{c->d_grid_ints.p}, sidx{c->d_grid_ints.p + n}, flags{c->d_grid_ints.p + 2 * (size_t)n}, cellid1{c->d_grid_ints.p + 3 * (size_t)n},
        ovf{c->d_grid_ints.p + 4 * (size_t)n};
    CUDA_TRY(c, cudaMemsetAsync(ovf.p, 0, sizeof(int), c->stream));
    const int g = (n + 255) / 256;
    grid_keys_kernel<<<g, 256, 0, c->stream>>>(c->d_aos.p + (size_t)d.aos_off * 4, n, (float)cell_size, keys.p, idx.p, ovf.p);
    size_t tb1 = 0, tb2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb1, keys.p, skeys.p, idx.p, sidx.p, n, 0, 64, c->stream);
    cub::DeviceScan::InclusiveSum(nullptr, tb2, flags.p, cellid1.p, n, c->stream);
    CUDA_TRY(c, c->d_grid_temp.ensure(std::max(tb1, tb2)));
    struct { unsigned char* p; } temp{c->d_grid_temp.p};
    size_t tb = std::max(tb1, tb2);
    CUDA_TRY(c, cub::DeviceRadixSort::SortPairs(temp.p, tb, keys.p, skeys.p, idx.p, sidx.p, n, 0, 64, c->stream));
    grid_flags_kernel<<<g, 256, 0, c->stream>>>(skeys.p, n, flags.p);
    tb = std::max(tb1, tb2);
    CUDA_TRY(c, cub::DeviceScan::InclusiveSum(temp.p, tb, flags.p, cellid1.p, n, c->stream));
    int* cs = c->d_cell_start.p + u.cell_start;
    grid_fill_tail_kernel<<<(n + 1 + 255) / 256, 256, 0, c->stream>>>(cellid1.p, n, cs);
    grid_starts_kernel<<<g, 256, 0, c->stream>>>(flags.p, cellid1.p, n - 0, cs);
    grid_scatter_kernel<<<g, 256, 0, c->stream>>>(sidx.p, cellid1.p, cs, n, c->d_cell_of_point.p + u.grid, c->d_members.p + u.grid, c->d_rank.p + u.grid);
    int h_ovf = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&h_ovf, ovf.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    if (h_ovf) return fail(c, USAC_ERR_ARG, "set_neighbors_grid: cell coordinates exceed 16 bits (cell_size too small for this coordinate range)");
    d.grid_off = (long long)u.grid;
    d.cell_start_off = (long long)u.cell_start;
    u.grid += (size_t)n;
    u.cell_start += (size_t)n + 1;
    if (d.cursor_off < 0) CUDA_TRY(c, append_segment(c->d_cursors, u.cursors, (const unsigned*)nullptr, 3 * (size_t)n + 1, &d.cursor_off, c->stream));
    d.neigh_type = USAC_NEIGH_GRID;
    return push_desc(c);
}

extern "C" int usac_gpu_set_sprt_pool(usac_gpu_ctx* c, int problem, const int* pool) {
    if (!c || problem < 0 || problem >= c->P || !pool) return fail(c, USAC_ERR_ARG, "set_sprt_pool: bad arguments");
    cudaSetDevice(c->device);
    SideUsed& u = c->side;
    ProblemDesc& d = c->h_prob[problem];
    for (int i = 0; i < d.n; i++) if (pool[i] < 0 || pool[i] >= d.n) return fail(c, USAC_ERR_ARG, "set_sprt_pool: index out of range");
    CUDA_TRY(c, append_segment(c->d_pool, u.pool, pool, (size_t)d.n, &d.pool_off, c->stream));
    const int dim = usac_point_dim(c->est);
    CUDA_TRY(c, c->d_pool_pts.ensure((size_t)c->total_points * dim));
    pool_gather_kernel<<<(d.n + 255) / 256, 256, 0, c->stream>>>(c->d_aos.p + (size_t)d.aos_off * dim, c->d_pool.p + d.pool_off, d.n, dim,
                                                                  c->d_pool_pts.p + (size_t)d.aos_off * dim);
    CUDA_TRY(c, cudaGetLastError());
    c->h_pool_set[problem] = 1;
    return push_desc(c);
}

// ------------------------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------------------------
static void launch_score(usac_gpu_ctx* c, ScoreArgs a, int slots, int mblocks, bool dense_survivors = false) {
    a.mblocks = mblocks; a.slots = slots;
    constexpr int warps_per_cta = USAC_SCORE_THREADS / 32;
    const long long items = (long long)slots * a.nchunks * mblocks * warps_per_cta;            // one item = 32 models x one point chunk
    const unsigned grid = (unsigned)std::min<long long>((items + warps_per_cta - 1) / warps_per_cta,
                                                        (long long)c->prop.multiProcessorCount * USAC_SCORE_GRID_CTAS);
    // the kernel's warps draw items from a counter that is never reset: this launch owns [work_base, work_base + items),
    // and every warp draws exactly one value beyond that before it exits
    // homography / fundamental / essential models of a RANSAC round (nearly every evaluation a provable outlier): the
    // survivor-queue kernel (score_sq.cuh). The accumulate-in-the-loop kernel (score.cuh) keeps the cases where survivors are
    // dense or the arithmetic is trivial: caller-supplied models of the Quality API (typically good models: a third of the
    // points survive) and lines (3 flops per evaluation: the push would cost more than the arithmetic). Both are exact.
    // USAC_GPU_SCORE_LEGACY=1 / =2 force the loop / queue kernel for every launch (A/B runs, tools/).
    static const int legacy = [] { const char* e = getenv("USAC_GPU_SCORE_LEGACY"); return e ? atoi(e) : 0; }();
    const bool loop_kernel = legacy == 1 || c->est == USAC_EST_LINE2D || (dense_survivors && legacy != 2);
    unsigned grid_ctas = grid;
    if (a.items) {      // the round's compact item list: its length is known on the device only; the list's own draw counter starts at 0
        grid_ctas = (unsigned)c->prop.multiProcessorCount * (loop_kernel ? USAC_SCORE_GRID_CTAS : USAC_SQ_MIN_CTAS);
        a.work = c->d_item_count.p + 1; a.work_base = 0;
    } else {
        if (!loop_kernel) grid_ctas = (unsigned)std::min<long long>((items + warps_per_cta - 1) / warps_per_cta, (long long)c->prop.multiProcessorCount * USAC_SQ_MIN_CTAS);
        a.work = c->d_work.p; a.work_base = c->work_next;
        c->work_next += (unsigned)items + grid_ctas * warps_per_cta;
    }
    auto& ev = c->next_score_event();
    cudaEventRecord(ev.first, c->stream);
    if (loop_kernel) {
        switch (c->est) {
            case USAC_EST_LINE2D: score_kernel<USAC_EST_LINE2D><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
            case USAC_EST_HOMOGRAPHY: score_kernel<USAC_EST_HOMOGRAPHY><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
            case USAC_EST_FUNDAMENTAL: score_kernel<USAC_EST_FUNDAMENTAL><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
            default: score_kernel<USAC_EST_ESSENTIAL><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
        }
    } else {
        switch (c->est) {
            case USAC_EST_HOMOGRAPHY: score_sq_kernel<USAC_EST_HOMOGRAPHY><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
            case USAC_EST_FUNDAMENTAL: score_sq_kernel<USAC_EST_FUNDAMENTAL><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
            default: score_sq_kernel<USAC_EST_ESSENTIAL><<<grid_ctas, USAC_SCORE_THREADS, 0, c->stream>>>(a); break;
        }
    }
    if (!a.items && cudaPeekAtLastError() != cudaSuccess) c->work_next = a.work_base;   // not launched: the counter did not move (callers report the error)
    cudaEventRecord(ev.second, c->stream);
    c->last_launches++;
    c->last_score_launches++;
}

// Work items of the persistent scoring kernel = slots x nchunks x (mblocks x 4 groups of 32 models), drawn one at a time by
// SMs x USAC_SCORE_GRID_CTAS x 4 resident warps. With the dynamic hand-out the kernel ends at most one item time after the
// ideal, so the point axis is split until every warp gets ~16 items (a chunk stays >= 2 tiles: each item pays one exposed
// tile-fetch latency and 128 B of model record per lane).
static void plan_chunks(const usac_gpu_ctx* c, int slots, int mblocks, int max_pairs, int* chunk_pairs, int* nchunks) {
    static const int per_warp = [] { const char* e = getenv("USAC_GPU_ITEMS_PER_WARP"); const int v = e ? atoi(e) : 0; return v > 0 ? v : 16; }();
    const long long warps = (long long)c->prop.multiProcessorCount * std::max(USAC_SCORE_GRID_CTAS, USAC_SQ_MIN_CTAS) * (USAC_SCORE_THREADS / 32);
    const long long base = (long long)slots * mblocks * (USAC_SCORE_THREADS / 32);
    // a work item costs ~2 us before its first trip (draw, record load, first tile): items of a large problem stay >= 8 tiles
    static const int min_tiles_env = [] { const char* e = getenv("USAC_GPU_MIN_TILES"); return e ? atoi(e) : 0; }();   // tuning knob
    const int min_tiles = min_tiles_env > 0 ? min_tiles_env : (max_pairs >= 65536 ? 8 : 2);
    const int max_chunks = std::min(65535, std::max(1, max_pairs / (min_tiles * USAC_TILE_PAIRS)));
    int nc = (int)std::min<long long>((per_warp * warps + base - 1) / base, max_chunks);
    nc = std::max(nc, 1);
    int cp = (max_pairs + nc - 1) / nc;
    cp = ((cp + 1) / 2) * 2;
    nc = (max_pairs + cp - 1) / cp;
    *chunk_pairs = cp;
    *nchunks = std::max(nc, 1);
}

static void collect_timing(usac_gpu_ctx* c) {
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    c->last_total_ms = ms;
    float s = 0;
    for (size_t i = 0; i < c->score_events_used; i++) {
        float t = 0;
        cudaEventElapsedTime(&t, c->score_events[i].first, c->score_events[i].second);
        s += t;
    }
    c->last_score_ms = s;
}

// ------------------------------------------------------------------------------------------------------------------
// Quality API
// ------------------------------------------------------------------------------------------------------------------
// 256 threads = 8 warps x 32 models: warp w sums the chunks w, w+8, ...; the eight partials are added in warp order
__global__ void __launch_bounds__(256) final_reduce_kernel(const int* __restrict__ part_cnt, const float* __restrict__ part_sum, int M, int mstride,
                                                           int nchunks, int* __restrict__ cnt, float* __restrict__ sum) {
    __shared__ int s_c[8][32];
    __shared__ float s_s[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x * 32 + lane;
    int cc = 0;
    float s = 0.f;
    if (q < M)
        for (int ch = warp; ch < nchunks; ch += 8) { cc += part_cnt[(size_t)ch * mstride + q]; s += part_sum[(size_t)ch * mstride + q]; }
    s_c[warp][lane] = cc;
    s_s[warp][lane] = s;
    __syncthreads();
    if (warp != 0 || q >= M) return;
    cc = 0; s = 0.f;
    for (int w = 0; w < 8; w++) { cc += s_c[w][lane]; s += s_s[w][lane]; }
    cnt[q] = cc;
    sum[q] = s;
}

extern "C" int usac_gpu_score(usac_gpu_ctx* c, int problem, const float* models, int M, float threshold, int* inliers_out, float* sumerr_out) {
    if (!c || problem < 0 || problem >= c->P || !models || M < 0 || !(threshold > 0.f)) return fail(c, USAC_ERR_ARG, "score: bad arguments");
    if (M == 0) return USAC_OK;
    cudaSetDevice(c->device);
    const int w = c->est == USAC_EST_LINE2D ? 3 : 9;
    CUDA_TRY(c, c->d_q_models.ensure((size_t)M * w));
    CUDA_TRY(c, c->d_q_recs.ensure((size_t)M * USAC_REC_STRIDE));
    const ProblemDesc& d = c->h_prob[problem];
    const int mblocks = (M + USAC_SCORE_THREADS - 1) / USAC_SCORE_THREADS;
    int chunk_pairs, nchunks;
    plan_chunks(c, 1, mblocks, d.n_pairs, &chunk_pairs, &nchunks);
    CUDA_TRY(c, c->d_part_cnt.ensure((size_t)nchunks * M));
    CUDA_TRY(c, c->d_part_sum.ensure((size_t)nchunks * M));
    CUDA_TRY(c, c->d_q_cnt.ensure(M));
    CUDA_TRY(c, c->d_q_sum.ensure(M));
    c->score_events_used = 0; c->last_launches = 0; c->last_score_launches = 0;
    cudaEventRecord(c->ev0, c->stream);
    CUDA_TRY(c, cudaMemcpyAsync(c->d_q_models.p, models, sizeof(float) * w * M, cudaMemcpyHostToDevice, c->stream));
    c->h_active[0] = problem;
    CUDA_TRY(c, cudaMemcpyAsync(c->d_active.p, c->h_active, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    prepare_models_kernel<<<(M + 127) / 128, 128, 0, c->stream>>>(c->est, c->d_q_models.p, M, w, threshold, c->d_prob.p, problem, c->d_q_recs.p);
    c->last_launches++;
    ScoreArgs a{};
    a.pairs = c->d_pairs.p; a.aos = c->d_aos.p; a.prob = c->d_prob.p; a.active = c->d_active.p; a.recs = c->d_q_recs.p; a.mvalid = nullptr;
    a.M = M; a.mstride = M; a.chunk_pairs = chunk_pairs; a.nchunks = nchunks; a.part_cnt = c->d_part_cnt.p; a.part_sum = c->d_part_sum.p;
    launch_score(c, a, 1, mblocks, /*dense_survivors=*/true);
    final_reduce_kernel<<<(M + 31) / 32, 256, 0, c->stream>>>(c->d_part_cnt.p, c->d_part_sum.p, M, M, nchunks, c->d_q_cnt.p, c->d_q_sum.p);
    c->last_launches++;
    if (inliers_out) CUDA_TRY(c, cudaMemcpyAsync(inliers_out, c->d_q_cnt.p, sizeof(int) * M, cudaMemcpyDeviceToHost, c->stream));
    if (sumerr_out) CUDA_TRY(c, cudaMemcpyAsync(sumerr_out, c->d_q_sum.p, sizeof(float) * M, cudaMemcpyDeviceToHost, c->stream));
    cudaEventRecord(c->ev1, c->stream);
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    collect_timing(c);
    return USAC_OK;
}

static int upload_one_record(usac_gpu_ctx* c, int problem, const float* model, float thr) {
    const int w = c->est == USAC_EST_LINE2D ? 3 : 9;
    CUDA_TRY(c, c->d_q_models.ensure(9));
    CUDA_TRY(c, c->d_q_recs.ensure(USAC_REC_STRIDE));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_q_models.p, model, sizeof(float) * w, cudaMemcpyHostToDevice, c->stream));
    prepare_models_kernel<<<1, 32, 0, c->stream>>>(c->est, c->d_q_models.p, 1, w, thr, c->d_prob.p, problem, c->d_q_recs.p);
    return USAC_OK;
}

extern "C" int usac_gpu_errors(usac_gpu_ctx* c, int problem, const float* model, float* err_out) {
    if (!c || problem < 0 || problem >= c->P || !model || !err_out) return fail(c, USAC_ERR_ARG, "errors: bad arguments");
    cudaSetDevice(c->device);
    const ProblemDesc& d = c->h_prob[problem];
    const int dim = usac_point_dim(c->est);
    int rc = upload_one_record(c, problem, model, 1.f);
    if (rc) return rc;
    CUDA_TRY(c, c->d_q_err.ensure(d.n));
    const float* aos = c->d_aos.p + (size_t)d.aos_off * dim;
    const int g = (d.n + 255) / 256;
    switch (c->est) {
        case USAC_EST_LINE2D: errors_kernel<USAC_EST_LINE2D><<<g, 256, 0, c->stream>>>(aos, d.n, c->d_q_recs.p, c->d_q_err.p); break;
        case USAC_EST_HOMOGRAPHY: errors_kernel<USAC_EST_HOMOGRAPHY><<<g, 256, 0, c->stream>>>(aos, d.n, c->d_q_recs.p, c->d_q_err.p); break;
        case USAC_EST_FUNDAMENTAL: errors_kernel<USAC_EST_FUNDAMENTAL><<<g, 256, 0, c->stream>>>(aos, d.n, c->d_q_recs.p, c->d_q_err.p); break;
        default: errors_kernel<USAC_EST_ESSENTIAL><<<g, 256, 0, c->stream>>>(aos, d.n, c->d_q_recs.p, c->d_q_err.p); break;
    }
    CUDA_TRY(c, cudaMemcpyAsync(err_out, c->d_q_err.p, sizeof(float) * d.n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

// Quality::getInliers on the device: ordered ids + count. Small problems: one CTA (one launch); from 32768 points on: flags over a
// grid, a scan of the block counts, the scatter (three launches, ~20 us for 1M points instead of 1.5 ms).
template <int EST>
static int launch_inliers_est(usac_gpu_ctx* c, const float* aos, int n, const float* d_rec, float thr, int* d_ids, int* d_cnt) {
    if (n < 32768) {
        inliers_kernel<EST><<<1, 1024, 0, c->stream>>>(aos, n, d_rec, thr, d_ids, d_cnt);
        c->last_launches++;
        return USAC_OK;
    }
    const int nblocks = (n + 1023) / 1024;
    CUDA_TRY(c, c->d_inl_ballots.ensure((size_t)nblocks * 32));
    CUDA_TRY(c, c->d_inl_counts.ensure((size_t)nblocks));
    inliers_flags_kernel<EST><<<nblocks, 1024, 0, c->stream>>>(aos, n, d_rec, thr, c->d_inl_ballots.p, c->d_inl_counts.p);
    inliers_scan_kernel<<<1, 1024, 0, c->stream>>>(c->d_inl_counts.p, nblocks, d_cnt);
    inliers_scatter_kernel<<<nblocks, 1024, 0, c->stream>>>(c->d_inl_ballots.p, c->d_inl_counts.p, n, d_ids);
    c->last_launches += 3;
    return USAC_OK;
}
static int launch_inliers(usac_gpu_ctx* c, const float* aos, int n, const float* d_rec, float thr, int* d_ids, int* d_cnt) {
    switch (c->est) {
        case USAC_EST_LINE2D: return launch_inliers_est<USAC_EST_LINE2D>(c, aos, n, d_rec, thr, d_ids, d_cnt);
        case USAC_EST_HOMOGRAPHY: return launch_inliers_est<USAC_EST_HOMOGRAPHY>(c, aos, n, d_rec, thr, d_ids, d_cnt);
        case USAC_EST_FUNDAMENTAL: return launch_inliers_est<USAC_EST_FUNDAMENTAL>(c, aos, n, d_rec, thr, d_ids, d_cnt);
        default: return launch_inliers_est<USAC_EST_ESSENTIAL>(c, aos, n, d_rec, thr, d_ids, d_cnt);
    }
}

extern "C" int usac_gpu_get_inliers(usac_gpu_ctx* c, int problem, const float* model, float threshold, int* ids_out, int* n_out) {
    if (!c || problem < 0 || problem >= c->P || !model || !ids_out || !n_out || !(threshold > 0.f)) return fail(c, USAC_ERR_ARG, "get_inliers: bad arguments");
    cudaSetDevice(c->device);
    const ProblemDesc& d = c->h_prob[problem];
    const int dim = usac_point_dim(c->est);
    int rc = upload_one_record(c, problem, model, threshold);
    if (rc) return rc;
    CUDA_TRY(c, c->d_q_ids.ensure((size_t)d.n + 1));
    const float* aos = c->d_aos.p + (size_t)d.aos_off * dim;
    int* cnt = c->d_q_ids.p + d.n;
    rc = launch_inliers(c, aos, d.n, c->d_q_recs.p, threshold, c->d_q_ids.p, cnt);
    if (rc) return rc;
    CUDA_TRY(c, cudaMemcpyAsync(n_out, cnt, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    if (*n_out > 0) CUDA_TRY(c, cudaMemcpyAsync(ids_out, c->d_q_ids.p, sizeof(int) * (*n_out), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Non-minimal estimation and the final refit (ransac.cpp:157-207)
// ------------------------------------------------------------------------------------------------------------------
static int launch_nonminimal(usac_gpu_ctx* c, const float* aos, const int* d_ids, int n, float* d_model, int* d_ok) {
    switch (c->est) {
        case USAC_EST_LINE2D: nonminimal_cta_kernel<USAC_EST_LINE2D><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(aos, d_ids, n, d_model, d_ok); break;
        case USAC_EST_HOMOGRAPHY: nonminimal_cta_kernel<USAC_EST_HOMOGRAPHY><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(aos, d_ids, n, d_model, d_ok); break;
        case USAC_EST_FUNDAMENTAL: nonminimal_cta_kernel<USAC_EST_FUNDAMENTAL><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(aos, d_ids, n, d_model, d_ok); break;
        default: nonminimal_cta_kernel<USAC_EST_ESSENTIAL><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(aos, d_ids, n, d_model, d_ok); break;
    }
    c->last_launches++;
    CUDA_TRY(c, cudaPeekAtLastError());                           // a launch that did not start (no shared-memory opt-in, ...)
    return USAC_OK;
}

extern "C" int usac_gpu_estimate_nonminimal(usac_gpu_ctx* c, int problem, const int* ids, int count, float* model_out, int* ok_out) {
    if (!c || problem < 0 || problem >= c->P || !ids || count < 0 || !model_out || !ok_out) return fail(c, USAC_ERR_ARG, "estimate_nonminimal: bad arguments");
    cudaSetDevice(c->device);
    const ProblemDesc& d = c->h_prob[problem];
    for (int i = 0; i < count; i++) if (ids[i] < 0 || ids[i] >= d.n) return fail(c, USAC_ERR_ARG, "estimate_nonminimal: point id out of range");
    const int dim = usac_point_dim(c->est), w = c->est == USAC_EST_LINE2D ? 3 : 9;
    CUDA_TRY(c, c->d_q_ids.ensure((size_t)std::max(count, d.n) + 1));
    CUDA_TRY(c, c->d_q_model2.ensure(9));
    CUDA_TRY(c, c->d_q_ok.ensure(1));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_q_ids.p, ids, sizeof(int) * count, cudaMemcpyHostToDevice, c->stream));
    c->last_launches = 0;
    const int rc = launch_nonminimal(c, c->d_aos.p + (size_t)d.aos_off * dim, c->d_q_ids.p, count, c->d_q_model2.p, c->d_q_ok.p);
    if (rc) return rc;
    CUDA_TRY(c, cudaMemcpyAsync(model_out, c->d_q_model2.p, sizeof(float) * w, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(ok_out, c->d_q_ok.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

extern "C" int usac_gpu_refit(usac_gpu_ctx* c, int problem, const float* model_in, int best_inliers, float threshold, usac_refit_result* out) {
    if (!c || problem < 0 || problem >= c->P || !model_in || !out || !(threshold > 0.f) || best_inliers < 0) return fail(c, USAC_ERR_ARG, "refit: bad arguments");
    cudaSetDevice(c->device);
    const ProblemDesc& d = c->h_prob[problem];
    const int dim = usac_point_dim(c->est), w = c->est == USAC_EST_LINE2D ? 3 : 9;
    const float* aos = c->d_aos.p + (size_t)d.aos_off * dim;
    CUDA_TRY(c, c->d_q_ids.ensure((size_t)d.n + 1));
    CUDA_TRY(c, c->d_q_ids2.ensure((size_t)d.n + 1));
    CUDA_TRY(c, c->d_q_model2.ensure(9));
    CUDA_TRY(c, c->d_q_ok.ensure(1));
    c->last_launches = 0;
    int rc = upload_one_record(c, problem, model_in, threshold);
    if (rc) return rc;
    int* cur = c->d_q_ids.p;
    int* alt = c->d_q_ids2.p;
    rc = launch_inliers(c, aos, d.n, c->d_q_recs.p, threshold, cur, cur + d.n);            // quality->getInliers(best_model), ransac.cpp:163
    if (rc) return rc;
    memset(out, 0, sizeof(*out));
    for (int i = 0; i < w; i++) out->model[i] = model_in[i];
    int avail = 0;                                                                         // ids actually present in the list
    CUDA_TRY(c, cudaMemcpyAsync(&avail, cur + d.n, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    int best = std::min(best_inliers, avail), prev = 0;                                     // never read past the list (the reference would)
    for (int norm = 0; norm < 4; norm++) {
        float m2[9];
        int ok = 0, c2 = 0;
        rc = launch_nonminimal(c, aos, cur, best, c->d_q_model2.p, c->d_q_ok.p);           // :173
        if (rc) return rc;
        prepare_models_kernel<<<1, 32, 0, c->stream>>>(c->est, c->d_q_model2.p, 1, w, threshold, c->d_prob.p, problem, c->d_q_recs.p);
        rc = launch_inliers(c, aos, d.n, c->d_q_recs.p, threshold, alt, alt + d.n);        // :180 (count + ids of the refitted model)
        if (rc) return rc;
        c->last_launches++;
        CUDA_TRY(c, cudaMemcpyAsync(m2, c->d_q_model2.p, sizeof(float) * w, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(&ok, c->d_q_ok.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(&c2, alt + d.n, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        CUDA_TRY(c, cudaGetLastError());
        if (!ok) break;
        if ((float)c2 / best < 0.8f) break;                                                 // :187
        if ((unsigned)c2 <= (unsigned)prev) break;                                          // :195
        prev = c2; best = c2;
        std::swap(cur, alt);
        for (int i = 0; i < w; i++) out->model[i] = m2[i];
        out->accepted++;
    }
    out->inliers = best;
    return USAC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// host-side tables: StandardTerminationCriteria (standard_termination_criteria.hpp:52-62) and the PROSAC growth
// function (prosac_sampler.hpp:62-114). Host libm on purpose: the bound is a function of the inlier count only, so a
// table indexed by the count makes the device decision bit-identical to the host plugin's.
// ------------------------------------------------------------------------------------------------------------------
// Entry n + 1 is the table's PEAK. The bound is not monotone in the inlier count: below p = w^m < 0.0005 the criterion answers
// max_iterations (standard_termination_criteria.hpp:57), the first count past that answers up to log(1 - conf) / log(1 - 0.0005)
// (5990 at conf 0.95) - so with max_iterations below that figure a better model can RAISE the loop bound, and samples that look out
// of reach at the start of a round are reached after all (solve_kernel's limit_remaining test reads the peak for that case).
static void standard_termination_table(unsigned n, int m, float confidence, unsigned max_iterations, std::vector<unsigned>& out) {
    out.resize((size_t)n + 2);
    const float log_1_p = (float)logf(1 - confidence);
    auto fill = [&](unsigned lo, unsigned hi) {
        for (unsigned inl = lo; inl < hi; inl++) out[inl] = standard_termination_value(inl, n, m, log_1_p, max_iterations);
    };
    const unsigned total = n + 1;
    unsigned nthreads = total >= (1u << 16) ? std::min(16u, std::max(1u, std::thread::hardware_concurrency())) : 1u;
    if (nthreads <= 1) fill(0, total);
    else {
        std::vector<std::thread> pool;                   // 1M-point problems: a million logf calls, spread over the host cores
        const unsigned per = (total + nthreads - 1) / nthreads;
        for (unsigned t = 0; t < nthreads; t++) pool.emplace_back(fill, std::min(total, t * per), std::min(total, (t + 1) * per));
        for (auto& th : pool) th.join();
    }
    unsigned peak = 0;
    for (unsigned inl = 0; inl < total; inl++) peak = std::max(peak, out[inl]);
    out[total] = peak;
}

static void prosac_growth(unsigned n, unsigned m, std::vector<unsigned>& g) {
    g.resize(n);
    double T_n = 200000;
    for (unsigned i = 0; i < m; ++i) T_n *= (double)(m - i) / (n - i);
    unsigned T_n_prime = 1;
    for (unsigned i = 0; i < n; ++i) {
        if (i + 1 <= m) { g[i] = T_n_prime; continue; }
        double Tn_plus1 = (double)(i + 1) * T_n / (i + 1 - m);
        g[i] = T_n_prime + (unsigned)ceil(Tn_plus1 - T_n);
        T_n = Tn_plus1;
        T_n_prime = g[i];
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Sampler / Estimator APIs
// ------------------------------------------------------------------------------------------------------------------
// models per sample of a fit: the solver's maximum, or USAC_E5_MAX_ROOTS for an essential fit that keeps every valid root
static int fit_models_per_sample(int est, const usac_fit_cfg* cfg) {
    return cfg->essential_roots == USAC_E5_ROOTS_ALL_VALID ? USAC_E5_MAX_ROOTS : usac_models_per_sample(est);
}

static int ensure_round_buffers(usac_gpu_ctx* c, int slots, int K, int nchunks, int nranks, int S) {
    const int m = usac_sample_size(c->est);
    const size_t sk = (size_t)slots * K;
    CUDA_TRY(c, c->d_samples.ensure(sk * m));
    CUDA_TRY(c, c->d_nmodels.ensure(sk));
    CUDA_TRY(c, c->d_offsets.ensure(sk));
    CUDA_TRY(c, c->d_mvalid.ensure((size_t)slots + 1));          // + 1: the second buffer set of the solve-ahead path
    CUDA_TRY(c, c->d_models_raw.ensure(sk * S * 9));
    CUDA_TRY(c, c->d_recs.ensure(sk * S * USAC_REC_STRIDE));
    CUDA_TRY(c, c->d_part_cnt.ensure(sk * S * nchunks));
    CUDA_TRY(c, c->d_part_sum.ensure(sk * S * nchunks));
    CUDA_TRY(c, c->d_seeds.ensure(sk));
    const size_t per_rank = (K + nranks - 1) / nranks;
    CUDA_TRY(c, c->d_scores.ensure(std::max(sk, (size_t)slots * per_rank)));
    CUDA_TRY(c, c->d_scores_all.ensure((size_t)slots * per_rank * nranks));
    CUDA_TRY(c, c->d_sprt_res.ensure(sk * S));
    CUDA_TRY(c, c->d_items.ensure((size_t)slots * nchunks * ((size_t)(K * S + 31) / 32)));
    CUDA_TRY(c, c->d_item_count.ensure(2));
    return USAC_OK;
}

static int setup_sampler_side(usac_gpu_ctx* c, const usac_sampler_cfg& s, bool reset_cursors = true) {
    if (s.sampler == USAC_SAMPLER_PROSAC) {
        std::vector<unsigned> all, g;
        for (int p = 0; p < c->P; p++) {
            prosac_growth((unsigned)c->h_prob[p].n, (unsigned)usac_sample_size(c->est), g);
            c->h_prob[p].growth_off = (long long)all.size();
            all.insert(all.end(), g.begin(), g.end());
        }
        CUDA_TRY(c, c->d_growth.ensure(all.size()));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_growth.p, all.data(), sizeof(unsigned) * all.size(), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    if (s.sampler == USAC_SAMPLER_NAPSAC || s.sampler == USAC_SAMPLER_PROGRESSIVE_NAPSAC) {
        for (int p = 0; p < c->P; p++) {
            const ProblemDesc& d = c->h_prob[p];
            if (s.neighbors == USAC_NEIGH_KNN ? d.knn_off < 0 : d.grid_off < 0) return fail(c, USAC_ERR_STATE, "NAPSAC: neighbourhood of a problem was not set");
            if (reset_cursors) {
                CUDA_TRY(c, cudaMemsetAsync(c->d_cursors.p + d.cursor_off, 0, sizeof(unsigned) * d.n, c->stream));
                // last entry of the segment: the first hypothesis that found no usable neighbourhood (from there on the sampler is uniform)
                CUDA_TRY(c, cudaMemsetAsync(c->d_cursors.p + d.cursor_off + 3 * (size_t)d.n, 0xFF, sizeof(unsigned), c->stream));
            }
        }
    }
    return USAC_OK;
}

static void fill_round_args(usac_gpu_ctx* c, RoundArgs& a, const usac_sampler_cfg& s, int K, int S) {
    memset(&a, 0, sizeof(a));
    a.prob = c->d_prob.p; a.active = c->d_active.p; a.state = c->d_state.p; a.aos = c->d_aos.p;
    a.est = c->est; a.K = K; a.S = S; a.m = usac_sample_size(c->est); a.mstride = K * a.S;
    a.e5_all_roots = c->est == USAC_EST_ESSENTIAL && S == USAC_E5_MAX_ROOTS;
    a.midx_shift = S > 3 ? 28 : 30;
    a.sampler = s.sampler; a.rng = s.rng; a.neighbors = s.neighbors; a.seed = s.seed;
    a.growth = c->d_growth.p; a.knn = c->d_knn.p; a.cell_of_point = c->d_cell_of_point.p; a.members = c->d_members.p;
    a.rank_in_cell = c->d_rank.p; a.cell_start = c->d_cell_start.p; a.cursors = c->d_cursors.p; a.seeds = c->d_seeds.p;
    a.samples = c->d_samples.p; a.models_raw = c->d_models_raw.p; a.nmodels = c->d_nmodels.p; a.offsets = c->d_offsets.p;
    a.recs = c->d_recs.p; a.mvalid = c->d_mvalid.p; a.part_cnt = c->d_part_cnt.p; a.part_sum = c->d_part_sum.p;
    a.sample_scores = c->d_scores.p; a.term_tables = c->d_term.p; a.table = c->d_table.p;
    a.rank = 0; a.nranks = 1; a.nchunks = 1;
}

// Only the samplers that exist: Evsac / ProsacNapsac are not wired in the reference (init.cpp:23-50) - an unknown enum must not
// silently become uniform sampling. Progressive NAPSAC follows DESIGN.md section 4.8 (the reference's progressive_sampler.hpp:149-172
// never fills its sample).
static const char* check_sampler_cfg(const usac_sampler_cfg& s) {
    if (s.sampler != USAC_SAMPLER_UNIFORM && s.sampler != USAC_SAMPLER_NAPSAC && s.sampler != USAC_SAMPLER_PROSAC &&
        s.sampler != USAC_SAMPLER_PROGRESSIVE_NAPSAC)
        return "sampler must be USAC_SAMPLER_UNIFORM, USAC_SAMPLER_PROGRESSIVE_NAPSAC, USAC_SAMPLER_NAPSAC or USAC_SAMPLER_PROSAC";
    if (s.rng != USAC_RNG_PHILOX && s.rng != USAC_RNG_TABLE) return "rng must be USAC_RNG_PHILOX or USAC_RNG_TABLE";
    if (s.sampler == USAC_SAMPLER_NAPSAC && s.neighbors != USAC_NEIGH_KNN && s.neighbors != USAC_NEIGH_GRID)
        return "NAPSAC needs neighbors = USAC_NEIGH_KNN or USAC_NEIGH_GRID";
    if (s.sampler == USAC_SAMPLER_PROGRESSIVE_NAPSAC && s.neighbors != USAC_NEIGH_KNN)
        return "Progressive NAPSAC needs neighbors = USAC_NEIGH_KNN (it grows a distance-ordered neighbourhood; grid cells have no order)";
    return nullptr;
}

static void launch_sampler(usac_gpu_ctx* c, const RoundArgs& a, int slots) {
    dim3 g((a.K + 127) / 128, slots);
    const bool seeded = a.sampler == USAC_SAMPLER_NAPSAC || a.sampler == USAC_SAMPLER_PROGRESSIVE_NAPSAC;
    if (seeded) { napsac_seed_kernel<<<g, 128, 0, c->stream>>>(a); c->last_launches++; }
    sample_kernel<<<g, 128, 0, c->stream>>>(a);
    c->last_launches++;
    if (seeded) { napsac_commit_kernel<<<g, 128, 0, c->stream>>>(a); c->last_launches++; }
}

static void init_state(FitState& s, const ProblemDesc& d, int est, unsigned max_iterations, uint64_t first_hyp) {
    memset(&s, 0, sizeof(s));
    s.best_hyp = -1;
    s.max_iters = max_iterations;
    s.samples_drawn = (unsigned)first_hyp;
    s.prosac_t = s.prosac_t_next = 1;
    s.prosac_n = s.prosac_n_next = s.prosac_largest = s.prosac_largest_next = (unsigned)usac_sample_size(est);
    s.prosac_term_len = (unsigned)d.n;
    sprt_init_state(s, est);
}

extern "C" int usac_gpu_sample(usac_gpu_ctx* c, int problem, const usac_sampler_cfg* cfg, uint64_t first_hyp, int K, int* samples_out) {
    if (!c || !cfg || problem < 0 || problem >= c->P || K <= 0 || !samples_out) return fail(c, USAC_ERR_ARG, "sample: bad arguments");
    if (const char* why = check_sampler_cfg(*cfg)) return fail(c, USAC_ERR_ARG, why);
    if (cfg->rng == USAC_RNG_TABLE) return fail(c, USAC_ERR_ARG, "sample: table replay has nothing to generate");
    cudaSetDevice(c->device);
    int rc = ensure_round_buffers(c, 1, K, 1, 1, usac_models_per_sample(c->est));
    if (rc) return rc;
    rc = setup_sampler_side(c, *cfg, first_hyp == 0);   // NAPSAC cursors persist across calls that continue a stream
    if (rc) return rc;
    rc = push_desc(c);
    if (rc) return rc;
    FitState s;
    init_state(s, c->h_prob[problem], c->est, 0, first_hyp);
    if (cfg->sampler == USAC_SAMPLER_PROSAC) {
        if (cfg->prosac_termination_length) s.prosac_term_len = cfg->prosac_termination_length;
        if (cfg->prosac_hyp_count) {
            // subset size implied by the counter: the state a sequential sampler would be in before call t
            std::vector<unsigned> g;
            prosac_growth((unsigned)c->h_prob[problem].n, (unsigned)usac_sample_size(c->est), g);
            unsigned n = (unsigned)usac_sample_size(c->est);
            for (unsigned t = 1; t < cfg->prosac_hyp_count; t++) if (t > g[n - 1] && n < (unsigned)c->h_prob[problem].n) n++;
            s.prosac_t = cfg->prosac_hyp_count; s.prosac_n = n;
        }
    }
    c->h_state[problem] = s;
    CUDA_TRY(c, cudaMemcpyAsync(c->d_state.p + problem, c->h_state + problem, sizeof(FitState), cudaMemcpyHostToDevice, c->stream));
    c->h_active[0] = problem;
    CUDA_TRY(c, cudaMemcpyAsync(c->d_active.p, c->h_active, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    RoundArgs a;
    fill_round_args(c, a, *cfg, K, usac_models_per_sample(c->est));
    c->last_launches = 0;
    launch_sampler(c, a, 1);
    CUDA_TRY(c, cudaMemcpyAsync(samples_out, c->d_samples.p, sizeof(int) * K * a.m, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

// S models per sample in models_out: usac_models_per_sample, or USAC_E5_MAX_ROOTS with e5_all_roots
static int estimate_models(usac_gpu_ctx* c, int problem, const int* samples, int K, float* models_out, int* nmodels_out, bool e5_all_roots) {
    cudaSetDevice(c->device);
    const int S = e5_all_roots ? USAC_E5_MAX_ROOTS : usac_models_per_sample(c->est), m = usac_sample_size(c->est), dim = usac_point_dim(c->est);
    const ProblemDesc& d = c->h_prob[problem];
    for (size_t i = 0; i < (size_t)K * m; i++)
        if (samples[i] < 0 || samples[i] >= d.n) return fail(c, USAC_ERR_ARG, "estimate: sample index out of range");
    CUDA_TRY(c, c->d_samples.ensure((size_t)K * m));
    CUDA_TRY(c, c->d_models_raw.ensure((size_t)K * S * 9));
    CUDA_TRY(c, c->d_nmodels.ensure(K));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_samples.p, samples, sizeof(int) * K * m, cudaMemcpyHostToDevice, c->stream));
    const float* aos = c->d_aos.p + (size_t)d.aos_off * dim;
    const int g = (K + 63) / 64;
    switch (c->est) {
        case USAC_EST_LINE2D: estimate_kernel<USAC_EST_LINE2D><<<g, 64, 0, c->stream>>>(aos, c->d_samples.p, K, m, S, c->d_models_raw.p, c->d_nmodels.p); break;
        case USAC_EST_HOMOGRAPHY: estimate_kernel<USAC_EST_HOMOGRAPHY><<<g, 64, 0, c->stream>>>(aos, c->d_samples.p, K, m, S, c->d_models_raw.p, c->d_nmodels.p); break;
        case USAC_EST_FUNDAMENTAL: estimate_kernel<USAC_EST_FUNDAMENTAL><<<g, 64, 0, c->stream>>>(aos, c->d_samples.p, K, m, S, c->d_models_raw.p, c->d_nmodels.p); break;
        default:
            estimate_kernel_e5_warp<<<(K + E5_WARPS_PER_CTA - 1) / E5_WARPS_PER_CTA, 32 * E5_WARPS_PER_CTA, 0, c->stream>>>(aos, c->d_samples.p, K, S, e5_all_roots ? 1 : 0,
                                                                                                                c->d_models_raw.p, c->d_nmodels.p);
            break;
    }
    CUDA_TRY(c, cudaMemcpyAsync(models_out, c->d_models_raw.p, sizeof(float) * K * S * 9, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(nmodels_out, c->d_nmodels.p, sizeof(int) * K, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

extern "C" int usac_gpu_estimate(usac_gpu_ctx* c, int problem, const int* samples, int K, float* models_out, int* nmodels_out) {
    if (!c || problem < 0 || problem >= c->P || !samples || K <= 0 || !models_out || !nmodels_out) return fail(c, USAC_ERR_ARG, "estimate: bad arguments");
    return estimate_models(c, problem, samples, K, models_out, nmodels_out, false);
}

extern "C" int usac_gpu_estimate_essential_roots(usac_gpu_ctx* c, int problem, const int* samples, int K, float* models_out, int* nmodels_out) {
    if (!c || problem < 0 || problem >= c->P || !samples || K <= 0 || !models_out || !nmodels_out) return fail(c, USAC_ERR_ARG, "estimate_essential_roots: bad arguments");
    if (c->est != USAC_EST_ESSENTIAL) return fail(c, USAC_ERR_ARG, "estimate_essential_roots: the uploaded points are not an essential problem");
    return estimate_models(c, problem, samples, K, models_out, nmodels_out, true);
}

// ------------------------------------------------------------------------------------------------------------------
// fused fit
// ------------------------------------------------------------------------------------------------------------------
extern "C" int usac_gpu_set_allgather(usac_gpu_ctx* c, usac_allgather_fn fn, void* user) {
    if (!c) return USAC_ERR_ARG;
    c->allgather = fn; c->allgather_user = user;
    return USAC_OK;
}

template <int EST>
static void launch_round_est(usac_gpu_ctx* c, const RoundArgs& a, int slots, bool sprt) {
    if (EST == USAC_EST_ESSENTIAL) {
        dim3 gw((a.K + E5_WARPS_PER_CTA - 1) / E5_WARPS_PER_CTA, slots);
        solve_kernel_e5_warp<<<gw, 32 * E5_WARPS_PER_CTA, 0, c->stream>>>(a);
    } else {
        dim3 gs((a.K + 63) / 64, slots);
        solve_kernel<EST><<<gs, 64, 0, c->stream>>>(a);
    }
    c->last_launches++;
}
template <int EST>
static void launch_winner_est(usac_gpu_ctx* c, const RoundArgs& a, int slots) {
    winner_kernel<EST><<<(slots + 31) / 32, 32, 0, c->stream>>>(a, slots);
    c->last_launches++;
}

// ------------------------------------------------------------------------------------------------------------------
// LO-RANSAC: InnerLocalOptimization::GetModelScore + IterativeLocalOptimization (local_optimization/
// inner_local_optimization.hpp:74-133, iterative_local_optimization.hpp:61-135), kinds InItLORsc (1) and InItFLORsc (2).
// One LO call is one device loop (lo.cuh: lo_kernel, or the speculative waves lo_pool_kernel / lo_wave_kernel / lo_commit_kernel),
// called from the host round replay on every new best model. Random subsets: Philox keyed by (seed, call counter) in place of mt19937
// seeded from random_device (uniform_random_generator.hpp:11-47).
// ------------------------------------------------------------------------------------------------------------------
// dynamic shared memory above 48 KB for the kernels that hold a LoShared (usac_gpu_create: once per context, after cudaSetDevice).
// First use = instantiation order, which steers nvcc's inliner: the line kernels come after the two-view ones, whose code this
// keeps as it was before lines had LO, and the batch kernels after the single-call ones.
static cudaError_t set_lo_smem_attributes() {
    const int smem = (int)sizeof(LoShared);
    const void* kernels[] = {
        (const void*)lo_kernel<USAC_EST_HOMOGRAPHY>, (const void*)lo_kernel<USAC_EST_FUNDAMENTAL>,
        (const void*)lo_kernel<USAC_EST_ESSENTIAL>, (const void*)lo_kernel<USAC_EST_LINE2D>,
        (const void*)lo_pool_kernel<USAC_EST_HOMOGRAPHY>, (const void*)lo_pool_kernel<USAC_EST_FUNDAMENTAL>,
        (const void*)lo_pool_kernel<USAC_EST_ESSENTIAL>, (const void*)lo_pool_kernel<USAC_EST_LINE2D>,
        (const void*)lo_wave_kernel<USAC_EST_HOMOGRAPHY>, (const void*)lo_wave_kernel<USAC_EST_FUNDAMENTAL>,
        (const void*)lo_wave_kernel<USAC_EST_ESSENTIAL>, (const void*)lo_wave_kernel<USAC_EST_LINE2D>,
        (const void*)lo_batch_kernel<USAC_EST_HOMOGRAPHY>, (const void*)lo_batch_kernel<USAC_EST_FUNDAMENTAL>,
        (const void*)lo_batch_kernel<USAC_EST_ESSENTIAL>, (const void*)lo_batch_kernel<USAC_EST_LINE2D>,
        (const void*)lo_pool_batch_kernel<USAC_EST_HOMOGRAPHY>, (const void*)lo_pool_batch_kernel<USAC_EST_FUNDAMENTAL>,
        (const void*)lo_pool_batch_kernel<USAC_EST_ESSENTIAL>, (const void*)lo_pool_batch_kernel<USAC_EST_LINE2D>,
        (const void*)lo_wave_batch_kernel<USAC_EST_HOMOGRAPHY>, (const void*)lo_wave_batch_kernel<USAC_EST_FUNDAMENTAL>,
        (const void*)lo_wave_batch_kernel<USAC_EST_ESSENTIAL>, (const void*)lo_wave_batch_kernel<USAC_EST_LINE2D>,
        (const void*)nonminimal_cta_kernel<USAC_EST_LINE2D>, (const void*)nonminimal_cta_kernel<USAC_EST_HOMOGRAPHY>,
        (const void*)nonminimal_cta_kernel<USAC_EST_FUNDAMENTAL>, (const void*)nonminimal_cta_kernel<USAC_EST_ESSENTIAL>,
    };
    for (const void* k : kernels) {
        const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

static bool lo_seq_env() {                                        // USAC_GPU_LO_SEQ=1: one CTA per LO call, no speculative waves
    static const bool seq = getenv("USAC_GPU_LO_SEQ") && atoi(getenv("USAC_GPU_LO_SEQ")) != 0;
    return seq;
}
#define LO_WAVE_LIST_BYTES (256u << 20)   // cap on the waves' candidate lists (inner_iters x variants x n ids per call)

struct LoRunner {
    usac_gpu_ctx* c;
    int problem, kind, m, n, w, dim;
    int sample_limit = 14, inner_iters = 20, iter_iters = 4, mult = 10;   // model.hpp:26-29
    float theta, lo_thr, step;
    uint64_t seed, calls = 0;
    unsigned inner_done = 0, iterative_done = 0;

    // the parameters and the state that persists across the calls of one fit (no device work)
    void setup(usac_gpu_ctx* ctx, int problem_, const usac_fit_cfg* cfg) {
        const float threshold = cfg->threshold;
        c = ctx; problem = problem_; kind = cfg->lo; seed = cfg->sampler.seed;
        if (cfg->lo_sample_size) sample_limit = (int)cfg->lo_sample_size;            // Model::setLOParametres, model.hpp:26-29
        if (cfg->lo_inner_iterations) inner_iters = (int)cfg->lo_inner_iterations;
        if (cfg->lo_iterative_iterations) iter_iters = (int)cfg->lo_iterative_iterations;
        if (cfg->lo_threshold_multiplier) mult = (int)cfg->lo_threshold_multiplier;
        const ProblemDesc& d = c->h_prob[problem];
        n = d.n; m = usac_sample_size(c->est); w = c->est == USAC_EST_LINE2D ? 3 : 9; dim = usac_point_dim(c->est);
        theta = threshold; lo_thr = threshold;
        step = (threshold * (unsigned)mult - threshold) / (unsigned)iter_iters;        // iterative_local_optimization.hpp:43
    }
    // the device arguments of one call
    LoArgs args(LoIO* io, int* A, int* B) const {
        LoArgs a;
        a.aos = c->d_aos.p + (size_t)c->h_prob[problem].aos_off * dim; a.prob = c->d_prob.p; a.problem = problem; a.n = n; a.m = m; a.kind = kind;
        a.sample_limit = sample_limit; a.inner_iters = inner_iters; a.iter_iters = iter_iters; a.mult = mult; a.theta = theta; a.step = step;
        a.seed = seed; a.io = io; a.A = A; a.B = B;
        return a;
    }
    // the state sent with a call, and the state its result leaves
    LoIO io_in(int best_inl, float best_sum) const {
        LoIO io;
        memset(&io, 0, sizeof(io));
        io.inliers = best_inl; io.score = best_sum; io.lo_thr = lo_thr; io.calls = calls;
        return io;
    }
    void io_out(const LoIO& io, float* best_model, int& best_inl, float& best_sum) {
        for (int i = 0; i < w; i++) best_model[i] = io.model[i];
        best_inl = io.inliers; best_sum = io.score; lo_thr = io.lo_thr; calls = io.calls;
        inner_done += io.inner_done; iterative_done += io.iterative_done;
    }

    int init(usac_gpu_ctx* ctx, int problem_, const usac_fit_cfg* cfg) {
        setup(ctx, problem_, cfg);
        CUDA_TRY(c, c->d_lo_ids_a.ensure((size_t)n));
        CUDA_TRY(c, c->d_lo_ids_b.ensure((size_t)n));
        CUDA_TRY(c, c->d_lo_io.ensure(1));
        // speculative waves (lo.cuh) unless their candidate lists would not fit (inner_iters x variants x n ids) or USAC_GPU_LO_SEQ=1
        const size_t lists = (size_t)inner_iters * LO_WAVE_VARIANTS * (size_t)n;
        waves = !lo_seq_env() && lists * sizeof(int) <= LO_WAVE_LIST_BYTES;
        if (waves) {
            CUDA_TRY(c, c->d_lo_bwave.ensure(lists));
            CUDA_TRY(c, c->d_lo_spec.ensure((size_t)inner_iters * LO_WAVE_VARIANTS));
            CUDA_TRY(c, c->d_lo_ws.ensure(1));
            CUDA_TRY(c, c->h_lo_ws.ensure(1));
        }
        return USAC_OK;
    }
    bool waves = false;
    unsigned long long wave_count = 0, wave_calls = 0;           // diagnostics (USAC_GPU_TRACE)

    template <int EST>
    int run_waves(const LoWaveArgs& w) {
        const size_t smem = sizeof(LoShared);
        lo_pool_kernel<EST><<<1, LO_THREADS, smem, c->stream>>>(w);
        c->last_launches++;
        for (int guard = 0; guard <= inner_iters; guard++) {
            lo_wave_kernel<EST><<<dim3(inner_iters, LO_WAVE_VARIANTS), LO_THREADS, smem, c->stream>>>(w);
            lo_commit_kernel<<<1, LO_THREADS, 0, c->stream>>>(w);
            c->last_launches += 2;
            wave_count++;
            CUDA_TRY(c, cudaMemcpyAsync(c->h_lo_ws.p, c->d_lo_ws.p, sizeof(LoWaveState), cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            if (c->h_lo_ws.p->finished) return USAC_OK;
        }
        return fail(c, USAC_ERR_STATE, "local optimisation: the speculative waves did not finish");
    }

    // InnerLocalOptimization::GetModelScore: model / score updated in place. One launch (lo.cuh), one synchronisation.
    int get_model_score(float* best_model, int& best_inl, float& best_sum) {
        if (best_inl < 12) return USAC_OK;                                              // inner_local_optimization.hpp:76
        LoIO io = io_in(best_inl, best_sum);
        for (int i = 0; i < w; i++) io.model[i] = best_model[i];
        CUDA_TRY(c, cudaMemcpyAsync(c->d_lo_io.p, &io, sizeof(io), cudaMemcpyHostToDevice, c->stream));
        const LoArgs a = args(c->d_lo_io.p, c->d_lo_ids_a.p, c->d_lo_ids_b.p);
        if (waves) {
            LoWaveArgs wv;
            wv.a = a; wv.ws = c->d_lo_ws.p; wv.spec = c->d_lo_spec.p; wv.Bwave = c->d_lo_bwave.p;
            wave_calls++;
            int rc;
            switch (c->est) {
                case USAC_EST_LINE2D: rc = run_waves<USAC_EST_LINE2D>(wv); break;
                case USAC_EST_HOMOGRAPHY: rc = run_waves<USAC_EST_HOMOGRAPHY>(wv); break;
                case USAC_EST_FUNDAMENTAL: rc = run_waves<USAC_EST_FUNDAMENTAL>(wv); break;
                default: rc = run_waves<USAC_EST_ESSENTIAL>(wv); break;
            }
            if (rc) return rc;
        } else {
            switch (c->est) {
                case USAC_EST_LINE2D: lo_kernel<USAC_EST_LINE2D><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(a); break;
                case USAC_EST_HOMOGRAPHY: lo_kernel<USAC_EST_HOMOGRAPHY><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(a); break;
                case USAC_EST_FUNDAMENTAL: lo_kernel<USAC_EST_FUNDAMENTAL><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(a); break;
                default: lo_kernel<USAC_EST_ESSENTIAL><<<1, LO_THREADS, sizeof(LoShared), c->stream>>>(a); break;
            }
            c->last_launches++;
        }
        CUDA_TRY(c, cudaMemcpyAsync(&io, c->d_lo_io.p, sizeof(io), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        CUDA_TRY(c, cudaGetLastError());
        io_out(io, best_model, best_inl, best_sum);
        return USAC_OK;
    }
};

// A batched LO step: the pending calls of several problems of a round (one per problem), each on a model still on the device
// (models_raw at (slot, q)). With many calls pending, one CTA per call (lo_batch_kernel): the calls keep the GPU busy and the
// waves' 6 x 20 speculative iterations per call would be work for nothing. With few - a small batch, the tail of a large one -
// the speculative waves of every call side by side (DESIGN 4.7, "Batches": LO_WAVE_MAX_CALLS from tools/lo_batch_time.py).
#define LO_WAVE_MAX_CALLS 4
struct LoCall { int slot, q, inl; float score; };

template <int EST>
static int lo_batch_launch(usac_gpu_ctx* c, int ncalls, bool waves, int inner_iters, unsigned long long& nwaves) {
    const size_t smem = sizeof(LoShared);
    const LoWaveArgs* calls = c->d_lo_calls.p;
    if (!waves) {
        lo_batch_kernel<EST><<<ncalls, LO_THREADS, smem, c->stream>>>(calls);
        c->last_launches++;
        CUDA_TRY(c, cudaPeekAtLastError());
        return USAC_OK;
    }
    lo_pool_batch_kernel<EST><<<ncalls, LO_THREADS, smem, c->stream>>>(calls);
    c->last_launches++;
    for (int guard = 0; guard <= inner_iters; guard++) {
        lo_wave_batch_kernel<EST><<<dim3(inner_iters, LO_WAVE_VARIANTS, ncalls), LO_THREADS, smem, c->stream>>>(calls);
        lo_commit_batch_kernel<<<ncalls, LO_THREADS, 0, c->stream>>>(calls);
        c->last_launches += 2;
        nwaves++;
        CUDA_TRY(c, cudaMemcpyAsync(c->h_lo_ws.p, c->d_lo_ws.p, sizeof(LoWaveState) * ncalls, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        CUDA_TRY(c, cudaGetLastError());
        bool finished = true;
        for (int k = 0; k < ncalls; k++) finished = finished && c->h_lo_ws.p[k].finished;
        if (finished) return USAC_OK;
    }
    return fail(c, USAC_ERR_STATE, "local optimisation: the speculative waves did not finish");
}

// runs `calls` (slots of `active`) and leaves their results in c->h_lo_io; A / B lists are carved at each problem's point offset
static int lo_batch_step(usac_gpu_ctx* c, const std::vector<LoRunner>& lo, const std::vector<int>& active, const std::vector<LoCall>& calls,
                         int KS, unsigned long long& nwaves, int& wave_steps) {
    const int ncalls = (int)calls.size();
    const int inner_iters = lo[active[calls[0].slot]].inner_iters, w = c->est == USAC_EST_LINE2D ? 3 : 9;
    size_t lists = 0;
    for (const LoCall& k : calls) lists += (size_t)inner_iters * LO_WAVE_VARIANTS * (size_t)c->h_prob[active[k.slot]].n;
    const bool waves = !lo_seq_env() && ncalls <= LO_WAVE_MAX_CALLS && lists * sizeof(int) <= LO_WAVE_LIST_BYTES;
    CUDA_TRY(c, c->d_lo_calls.ensure((size_t)ncalls));
    CUDA_TRY(c, c->h_lo_calls.ensure((size_t)ncalls));
    CUDA_TRY(c, c->d_lo_io.ensure((size_t)ncalls));
    CUDA_TRY(c, c->h_lo_io.ensure((size_t)ncalls));
    CUDA_TRY(c, c->d_lo_src.ensure((size_t)ncalls));
    CUDA_TRY(c, c->h_lo_src.ensure((size_t)ncalls));
    if (waves) {
        CUDA_TRY(c, c->d_lo_bwave.ensure(lists));
        CUDA_TRY(c, c->d_lo_spec.ensure((size_t)ncalls * inner_iters * LO_WAVE_VARIANTS));
        CUDA_TRY(c, c->d_lo_ws.ensure((size_t)ncalls));
        CUDA_TRY(c, c->h_lo_ws.ensure((size_t)ncalls));
        wave_steps++;
    }
    size_t boff = 0;
    for (int k = 0; k < ncalls; k++) {
        const LoCall& call = calls[k];
        const LoRunner& r = lo[active[call.slot]];
        const long long off = c->h_prob[r.problem].aos_off;
        c->h_lo_io.p[k] = r.io_in(call.inl, call.score);
        c->h_lo_src.p[k] = (long long)call.slot * KS + call.q;
        LoWaveArgs& wa = c->h_lo_calls.p[k];
        wa.a = r.args(c->d_lo_io.p + k, c->d_lo_ids_a.p + off, c->d_lo_ids_b.p + off);
        wa.ws = nullptr; wa.spec = nullptr; wa.Bwave = nullptr;
        if (waves) {
            wa.ws = c->d_lo_ws.p + k; wa.spec = c->d_lo_spec.p + (size_t)k * inner_iters * LO_WAVE_VARIANTS; wa.Bwave = c->d_lo_bwave.p + boff;
            boff += (size_t)inner_iters * LO_WAVE_VARIANTS * (size_t)r.n;
        }
    }
    CUDA_TRY(c, cudaMemcpyAsync(c->d_lo_io.p, c->h_lo_io.p, sizeof(LoIO) * ncalls, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_lo_calls.p, c->h_lo_calls.p, sizeof(LoWaveArgs) * ncalls, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_lo_src.p, c->h_lo_src.p, sizeof(long long) * ncalls, cudaMemcpyHostToDevice, c->stream));
    lo_load_models_kernel<<<(ncalls * 9 + 255) / 256, 256, 0, c->stream>>>(c->d_models_raw.p, c->d_lo_src.p, ncalls, w, c->d_lo_io.p);
    c->last_launches++;
    int rc;
    switch (c->est) {
        case USAC_EST_LINE2D: rc = lo_batch_launch<USAC_EST_LINE2D>(c, ncalls, waves, inner_iters, nwaves); break;
        case USAC_EST_HOMOGRAPHY: rc = lo_batch_launch<USAC_EST_HOMOGRAPHY>(c, ncalls, waves, inner_iters, nwaves); break;
        case USAC_EST_FUNDAMENTAL: rc = lo_batch_launch<USAC_EST_FUNDAMENTAL>(c, ncalls, waves, inner_iters, nwaves); break;
        default: rc = lo_batch_launch<USAC_EST_ESSENTIAL>(c, ncalls, waves, inner_iters, nwaves); break;
    }
    if (rc) return rc;
    CUDA_TRY(c, cudaMemcpyAsync(c->h_lo_io.p, c->d_lo_io.p, sizeof(LoIO) * ncalls, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

// inlier mask of one model over the points in their given (quality-sorted) order: Quality::getInliers -> bytes
static int fetch_mask(usac_gpu_ctx* c, int problem, const float* model, float thr, std::vector<unsigned char>& mask, std::vector<int>& ids) {
    const ProblemDesc& d = c->h_prob[problem];
    const int dim = usac_point_dim(c->est);
    int rc = upload_one_record(c, problem, model, thr);
    if (rc) return rc;
    CUDA_TRY(c, c->d_q_ids.ensure((size_t)d.n + 1));
    const float* aos = c->d_aos.p + (size_t)d.aos_off * dim;
    int* cnt = c->d_q_ids.p + d.n;
    rc = launch_inliers(c, aos, d.n, c->d_q_recs.p, thr, c->d_q_ids.p, cnt);
    if (rc) return rc;
    c->last_launches++;
    ids.resize((size_t)d.n + 1);
    CUDA_TRY(c, cudaMemcpyAsync(ids.data(), c->d_q_ids.p, sizeof(int) * ((size_t)d.n + 1), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    mask.assign((size_t)d.n, 0);
    for (int i = 0; i < ids[d.n]; i++) mask[ids[i]] = 1;
    return USAC_OK;
}

template <int EST>
static void launch_solve(usac_gpu_ctx* c, const RoundArgs& a, int slots) {
    if (EST == USAC_EST_ESSENTIAL) {
        dim3 gw((a.K + E5_WARPS_PER_CTA - 1) / E5_WARPS_PER_CTA, slots);
        solve_kernel_e5_warp<<<gw, 32 * E5_WARPS_PER_CTA, 0, c->stream>>>(a);
    } else {
        dim3 gs((a.K + 63) / 64, slots);
        solve_kernel<EST><<<gs, 64, 0, c->stream>>>(a);
    }
    c->last_launches++;
}
// warps of the tail kernels: one per handed-over walk, at most 8 per SM (a walk is a latency chain, not a throughput problem)
static int sprt_tail_blocks(const usac_gpu_ctx* c, size_t walks) {
    return (int)std::max<size_t>(1, std::min<size_t>((walks + 3) / 4, (size_t)c->prop.multiProcessorCount * 2));
}
template <int EST>
static int launch_walk(usac_gpu_ctx* c, const RoundArgs& a, int slots) {
    const size_t walks = (size_t)slots * a.mstride;
    CUDA_TRY(c, c->d_sprt_carry.ensure(walks));
    CUDA_TRY(c, c->d_sprt_count.ensure(1));
    CUDA_TRY(c, cudaMemsetAsync(c->d_sprt_count.p, 0, sizeof(unsigned), c->stream));
    dim3 g((a.K * a.S + 63) / 64, slots);
    sprt_walk_kernel<EST><<<g, 64, 0, c->stream>>>(a, c->d_pool_pts.p, c->d_sprt_carry.p, c->d_sprt_count.p);
    sprt_tail_kernel<EST><<<sprt_tail_blocks(c, walks), 128, 0, c->stream>>>(a, c->d_pool_pts.p, c->d_sprt_carry.p, c->d_sprt_count.p);
    c->last_launches += 2;
    return USAC_OK;
}

extern "C" void usac_prosac_growth_function(unsigned n, unsigned sample_size, unsigned* out) {
    if (!out || n == 0) return;
    std::vector<unsigned> g;
    prosac_growth(n, sample_size, g);
    memcpy(out, g.data(), sizeof(unsigned) * n);
}

// LO settings of usac_gpu_fit / usac_gpu_lo_model_score: the kind, and an inlier subset size that lo_subset can draw (at most 16
// positions) and that over-determines the model (more than the minimal sample). nullptr when they are valid.
static const char* check_lo_cfg(int est, const usac_fit_cfg* cfg) {
    if (cfg->lo != 1 && cfg->lo != 2) return "lo must be 1 (InItLORsc) or 2 (InItFLORsc); GC / IRLS are not built";
    if (cfg->lo_sample_size && (cfg->lo_sample_size < (unsigned)usac_sample_size(est) + 1 || cfg->lo_sample_size > 16))
        return "lo_sample_size must be 0 or lie in [sample size + 1, 16]";
    return nullptr;
}

extern "C" int usac_gpu_lo_model_score(usac_gpu_ctx* c, int problem, const usac_fit_cfg* cfg, uint64_t* call_counter, float* lo_threshold, float* model, int* inliers,
                                       float* score, unsigned* inner_iters, unsigned* iterative_iters) {
    if (!c || !cfg || problem < 0 || problem >= c->P || !call_counter || !model || !inliers || !score) return fail(c, USAC_ERR_ARG, "lo_model_score: bad arguments");
    if (const char* why = check_lo_cfg(c->est, cfg)) return fail(c, USAC_ERR_ARG, why);
    if (!(cfg->threshold > 0.f)) return fail(c, USAC_ERR_ARG, "lo_model_score: threshold must be positive");
    cudaSetDevice(c->device);
    int rc = push_desc(c);
    if (rc) return rc;
    LoRunner lo;
    rc = lo.init(c, problem, cfg);
    if (rc) return rc;
    lo.calls = *call_counter;
    if (lo_threshold && *lo_threshold > 0.f) lo.lo_thr = *lo_threshold;
    rc = lo.get_model_score(model, *inliers, *score);
    *call_counter = lo.calls;
    if (lo_threshold) *lo_threshold = lo.lo_thr;
    if (inner_iters) *inner_iters += lo.inner_done;
    if (iterative_iters) *iterative_iters += lo.iterative_done;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return rc;
}

template <int EST>
static void launch_sprt_verify(usac_gpu_ctx* c, const float* recs, int M, const float* P, int n, const unsigned* start, const int* count_all,
                               double eps, double delta, double A, SprtModelResult* out) {
    sprt_verify_kernel<EST><<<(M + 63) / 64, 64, 0, c->stream>>>(recs, M, P, n, start, count_all, eps, delta, A, out, c->d_sprt_carry.p, c->d_sprt_count.p);
    sprt_verify_tail_kernel<EST><<<sprt_tail_blocks(c, (size_t)M), 128, 0, c->stream>>>(recs, P, n, eps, delta, A, out, c->d_sprt_carry.p, c->d_sprt_count.p);
}

extern "C" int usac_gpu_sprt_verify(usac_gpu_ctx* c, int problem, const float* models, int M, float threshold, double epsilon, double delta, double A,
                                    const unsigned* start, const int* count_all, usac_sprt_result* out) {
    if (!c || problem < 0 || problem >= c->P || !models || M <= 0 || !start || !out || !(threshold > 0.f)) return fail(c, USAC_ERR_ARG, "sprt_verify: bad arguments");
    if (!c->h_pool_set[problem]) return fail(c, USAC_ERR_STATE, "sprt_verify: usac_gpu_set_sprt_pool was not called for this problem");
    cudaSetDevice(c->device);
    int rc = push_desc(c);
    if (rc) return rc;
    const ProblemDesc& d = c->h_prob[problem];
    const int w = c->est == USAC_EST_LINE2D ? 3 : 9, dim = usac_point_dim(c->est);
    CUDA_TRY(c, c->d_q_models.ensure((size_t)M * w));
    CUDA_TRY(c, c->d_q_recs.ensure((size_t)M * USAC_REC_STRIDE));
    CUDA_TRY(c, c->d_sprt_res.ensure((size_t)M));
    CUDA_TRY(c, c->d_sprt_carry.ensure((size_t)M));
    CUDA_TRY(c, c->d_sprt_count.ensure(1));
    CUDA_TRY(c, cudaMemsetAsync(c->d_sprt_count.p, 0, sizeof(unsigned), c->stream));
    CUDA_TRY(c, c->d_q_ids.ensure((size_t)std::max(2 * M, d.n + 1)));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_q_models.p, models, sizeof(float) * w * M, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_q_ids.p, start, sizeof(unsigned) * M, cudaMemcpyHostToDevice, c->stream));
    if (count_all) CUDA_TRY(c, cudaMemcpyAsync(c->d_q_ids.p + M, count_all, sizeof(int) * M, cudaMemcpyHostToDevice, c->stream));
    prepare_models_kernel<<<(M + 127) / 128, 128, 0, c->stream>>>(c->est, c->d_q_models.p, M, w, threshold, c->d_prob.p, problem, c->d_q_recs.p);
    const float* P = c->d_pool_pts.p + (size_t)d.aos_off * dim;
    const unsigned* d_start = reinterpret_cast<const unsigned*>(c->d_q_ids.p);
    const int* d_all = count_all ? c->d_q_ids.p + M : nullptr;
    switch (c->est) {
        case USAC_EST_LINE2D: launch_sprt_verify<USAC_EST_LINE2D>(c, c->d_q_recs.p, M, P, d.n, d_start, d_all, epsilon, delta, A, c->d_sprt_res.p); break;
        case USAC_EST_HOMOGRAPHY: launch_sprt_verify<USAC_EST_HOMOGRAPHY>(c, c->d_q_recs.p, M, P, d.n, d_start, d_all, epsilon, delta, A, c->d_sprt_res.p); break;
        case USAC_EST_FUNDAMENTAL: launch_sprt_verify<USAC_EST_FUNDAMENTAL>(c, c->d_q_recs.p, M, P, d.n, d_start, d_all, epsilon, delta, A, c->d_sprt_res.p); break;
        default: launch_sprt_verify<USAC_EST_ESSENTIAL>(c, c->d_q_recs.p, M, P, d.n, d_start, d_all, epsilon, delta, A, c->d_sprt_res.p); break;
    }
    static_assert(sizeof(usac_sprt_result) == sizeof(SprtModelResult), "usac_sprt_result mirrors SprtModelResult");
    CUDA_TRY(c, cudaMemcpyAsync(out, c->d_sprt_res.p, sizeof(usac_sprt_result) * M, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    return USAC_OK;
}

// Rounds with SPRT and/or PROSAC termination (host_replay.hpp): device = sample, solve, verify/score; host = replay.
static void print_marks(usac_gpu_ctx* c) {
    if (c->marks_used < 2) return;
    std::map<std::string, double> tot;
    for (size_t i = 1; i < c->marks_used; i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, c->marks[i - 1].second, c->marks[i].second);
        tot[c->marks[i].first] += ms * 1e3;
    }
    std::string line = "usac_gpu_fit kernels (us, device time between launches):";
    for (auto& kv : tot) { char buf[96]; snprintf(buf, sizeof(buf), " %s=%.0f", kv.first.c_str(), kv.second); line += buf; }
    fprintf(stderr, "%s\n", line.c_str());
}

// models (slot, q) of a round -> packed [n][9] (the winners of the problems of a batched SPRT round)
__global__ void gather_models_kernel(const float* __restrict__ models_raw, const int2* __restrict__ picks, int n, int KS, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * 9) return;
    const int2 pk = picks[i / 9];
    out[i] = models_raw[((size_t)pk.x * KS + pk.y) * 9 + i % 9];
}

// One problem's replay of one round in hypothesis order (ransac.cpp:58-139), shared by fit_host_replay and fit_batch_replay.
// next() walks the hypotheses from the cursor - evaluation costs, SPRT bookkeeping, `iters` - and stops at the next one whose score
// beats the best (Score::bigger); the caller runs LO on it (ransac.cpp:108-110) and hands the result to accept(), which stores the
// best and its termination bound. A batch can so pause a problem at a new best, run the LO calls of many problems in one step and
// resume. finish() closes the round: one SPRT re-design (the test is frozen within a round), the counters.
struct RoundReplay {
    int K, S, m;
    unsigned n, before_sprt, max_iterations;
    float log_1_p;
    const SprtModelResult* res;          // SPRT: per-model results of the round (nullptr without SPRT)
    const int2* scores;                  // without SPRT: (count, sum bits) per model
    const int* nmodels;
    unsigned long long hyp0;
    unsigned iters_round_start;
    long long last_improving = -1;
    unsigned long long rej_inl = 0, rej_pts = 0, evals = 0, useful = 0;
    bool stopped = false, done = false;  // done: the fit ended inside this round
    int j = 0, i = 0;                    // cursor: model i of sample j is next

    RoundReplay(const FitState& hs, const usac_fit_cfg* cfg, unsigned n_, int K_, int S_, int m_, const SprtModelResult* res_,
                const int2* scores_, const int* nmodels_)
        : K(K_), S(S_), m(m_), n(n_), before_sprt(cfg->max_hypothesis_test_before_sprt ? cfg->max_hypothesis_test_before_sprt : 20u),   // model.hpp:39
          max_iterations(cfg->max_iterations), log_1_p((float)logf(1 - cfg->confidence)), res(res_), scores(scores_), nmodels(nmodels_),
          hyp0(hs.samples_drawn), iters_round_start(hs.iters) {}

    bool next(FitState& hs, int& q, int& inl, float& score) {
        for (; j < K; j++, i = 0) {
            if (i == 0 && !stopped && !(hs.iters < hs.max_iters)) { stopped = true; done = true; }
            for (; i < nmodels[j]; i++) {
                q = j * S + i;
                unsigned long long cost;
                if (res) cost = (unsigned long long)res[q].tested_pts + ((!res[q].good && hyp0 + j < before_sprt) ? (unsigned long long)(n - res[q].tested_pts) : 0ull);
                else cost = n;
                evals += cost;
                if (stopped) continue;
                useful += cost;
                if (res) {
                    const SprtModelResult& r = res[q];
                    if (r.good) { if (r.tested_inl > hs.best_cnt) last_improving = r.tested_inl; }
                    else { rej_inl += (unsigned long long)r.tested_inl; rej_pts += (unsigned long long)r.tested_pts; }
                    if (!r.good && hs.iters >= before_sprt) { hs.iters++; continue; }       // ransac.cpp:77-85
                    inl = r.full_inl; score = (float)inl;                           // sprt.hpp:240-241
                } else {
                    inl = scores[q].x; memcpy(&score, &scores[q].y, 4);
                }
                if (inl > hs.best_cnt || (inl == hs.best_cnt && score > hs.best_sum)) { i++; return true; }   // Score::bigger
            }
            if (!stopped) hs.iters++;
        }
        return false;
    }
    // the best of hypothesis q after LO; `model` = nullptr leaves hs.best_model to the caller. prosac_bound >= 0: PROSAC's bound
    void accept(FitState& hs, SprtHost* sprt, int q, int inl, float score, const float* model, int w, long long prosac_bound = -1) {
        hs.best_cnt = inl; hs.best_sum = score; hs.best_hyp = (long long)(hyp0 + q / S); hs.best_midx = q % S;
        if (model) for (int k = 0; k < w; k++) hs.best_model[k] = model[k];
        hs.max_iters = prosac_bound >= 0 ? (unsigned)prosac_bound : standard_termination_value((unsigned)inl, n, m, log_1_p, max_iterations);
        if (sprt) hs.max_iters = std::min(hs.max_iters, sprt->upper_bound(inl));   // ransac.cpp:129-133
    }
    void finish(FitState& hs, SprtHost* sprt) {
        if (sprt) {
            const SprtTestH t = sprt->current();
            double eps = t.epsilon, delta = t.delta;
            bool redesign = false;
            if (last_improving >= 0) { eps = (float)last_improving / n; redesign = true; }
            if (rej_pts > 0) {
                const float delta_estimated = (float)rej_inl / (unsigned)rej_pts;
                if (delta_estimated > 0 && std::fabs(t.delta - delta_estimated) / t.delta > 0.05) { delta = delta_estimated; redesign = true; }
            }
            if (redesign) sprt->push(eps, delta, (int)iters_round_start);
            sprt->cursor = (unsigned)(((unsigned long long)sprt->cursor + 32ull * (unsigned long long)K * S) % n);
            hs.sprt_ntests = (int)sprt->hist.size();
        }
        hs.samples_drawn += (unsigned)K;
        hs.rounds++;
        hs.evals += evals;
        hs.useful_evals += useful;
    }
};

static void fill_result(const FitState& hs, int w, usac_fit_result& r) {
    memset(&r, 0, sizeof(r));
    for (int i = 0; i < w; i++) r.model[i] = hs.best_model[i];
    r.inliers = hs.best_cnt; r.score = hs.best_sum; r.iterations = hs.iters; r.samples_drawn = hs.samples_drawn;
    r.best_hyp = hs.best_hyp; r.best_model_idx = hs.best_midx; r.rounds = hs.rounds; r.evals = hs.evals; r.useful_evals = hs.useful_evals;
}

// SPRT and / or LO rounds for SEVERAL problems in flight (uniform / NAPSAC samplers): one set of launches per round for every
// problem still searching (the SPRT walks, or the scoring kernel + per-model scores), one copy of the per-model results, then the
// host replays every problem's K hypotheses (RoundReplay, as fit_host_replay). A problem pauses at a new best that LO works on
// (>= 12 inliers, inner_local_optimization.hpp:76); the paused problems' calls run as one batched LO step (lo_batch_step) and their
// replays resume - one sync per round plus one per LO step. The models of new bests that LO did not touch come back through one
// gather. Rounds stay K (no growth) and without SPRT each problem's points are chunked as in a fit of its own, so every record is
// that of the problem fitted alone.
static int fit_batch_replay(usac_gpu_ctx* c, const usac_fit_cfg* cfg, usac_fit_result* results, int K) {
    const int P = c->P, m = usac_sample_size(c->est), S = fit_models_per_sample(c->est, cfg), w = c->est == USAC_EST_LINE2D ? 3 : 9;
    const bool is_sprt = cfg->sprt != 0, is_lo = cfg->lo != 0;
    const int KS = K * S;
    const int mblocks = (KS + USAC_SCORE_THREADS - 1) / USAC_SCORE_THREADS;
    // chunk plan of each problem as a fit of its own plans it (the error sums add the chunks' partial sums in order)
    std::vector<int2> plan(P);
    int max_chunks = 1;
    for (int p = 0; p < P; p++) {
        plan[p] = make_int2(c->h_prob[p].n_pairs, 1);
        if (!is_sprt) plan_chunks(c, 1, mblocks, c->h_prob[p].n_pairs, &plan[p].x, &plan[p].y);
        max_chunks = std::max(max_chunks, plan[p].y);
    }
    int rc = ensure_round_buffers(c, P, K, max_chunks, 1, S);
    if (rc) return rc;
    CUDA_TRY(c, c->h_rp_nmodels.ensure((size_t)P * K));
    if (is_sprt) CUDA_TRY(c, c->h_rp_res.ensure((size_t)P * KS));
    CUDA_TRY(c, c->h_rp_scores.ensure((size_t)P * KS + P));           // per-model scores, then the gather's (slot, q) picks
    CUDA_TRY(c, c->d_model_scores.ensure((size_t)P * KS + P));        // the same on the device
    CUDA_TRY(c, c->h_rp_models.ensure((size_t)P * 9));
    CUDA_TRY(c, c->d_q_models.ensure((size_t)P * 9));
    if (is_lo) {
        CUDA_TRY(c, c->d_lo_ids_a.ensure((size_t)c->total_points));
        CUDA_TRY(c, c->d_lo_ids_b.ensure((size_t)c->total_points));
    }
    std::vector<SprtHost> sprt(is_sprt ? P : 0);
    std::vector<LoRunner> lo(is_lo ? P : 0);
    std::vector<int> active(P);
    for (int p = 0; p < P; p++) {
        init_state(c->h_state[p], c->h_prob[p], c->est, cfg->max_iterations, 0);
        if (is_sprt) sprt[p].init(c->est, (unsigned)c->h_prob[p].n, (unsigned)m, cfg->max_iterations);
        if (is_lo) lo[p].setup(c, p, cfg);
        active[p] = p;
    }
    static const bool trace = getenv("USAC_GPU_TRACE") != nullptr;
    int n_rounds = 0, n_lo = 0, n_lo_steps = 0, wave_steps = 0;
    unsigned long long n_waves = 0;
    std::vector<RoundReplay> rr;
    std::vector<int> best_q, run, next;
    std::vector<LoCall> calls;
    while (!active.empty()) {
        // slots grouped by chunk plan: one scoring launch per plan
        if (!is_sprt) std::stable_sort(active.begin(), active.end(), [&](int x, int y) { return plan[x].x < plan[y].x; });
        const int slots = (int)active.size();
        for (int q = 0; q < slots; q++) {
            const int p = active[q];
            FitState& hs = c->h_state[p];
            if (is_sprt) { const SprtTestH& t = sprt[p].current(); hs.sprt_eps = t.epsilon; hs.sprt_delta = t.delta; hs.sprt_A = t.A; hs.sprt_cursor = sprt[p].cursor; }
            c->h_active[q] = p;
        }
        CUDA_TRY(c, cudaMemcpyAsync(c->d_state.p, c->h_state, sizeof(FitState) * P, cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_active.p, c->h_active, sizeof(int) * slots, cudaMemcpyHostToDevice, c->stream));
        RoundArgs a;
        fill_round_args(c, a, cfg->sampler, K, S);
        a.thr = cfg->threshold; a.confidence = cfg->confidence; a.max_iterations = cfg->max_iterations;
        a.table_rows = cfg->sample_table_rows; a.nchunks = 1; a.sprt = cfg->sprt; a.pool = c->d_pool.p; a.sprt_res = c->d_sprt_res.p;
        a.before_sprt = cfg->max_hypothesis_test_before_sprt ? cfg->max_hypothesis_test_before_sprt : 20u;
        launch_sampler(c, a, slots);
        switch (c->est) {
            case USAC_EST_LINE2D: launch_solve<USAC_EST_LINE2D>(c, a, slots); break;
            case USAC_EST_HOMOGRAPHY: launch_solve<USAC_EST_HOMOGRAPHY>(c, a, slots); break;
            case USAC_EST_FUNDAMENTAL: launch_solve<USAC_EST_FUNDAMENTAL>(c, a, slots); break;
            default: launch_solve<USAC_EST_ESSENTIAL>(c, a, slots); break;
        }
        prepare_kernel<<<slots, 256, 0, c->stream>>>(a);
        c->last_launches++;
        if (is_sprt) {
            switch (c->est) {
                case USAC_EST_LINE2D: rc = launch_walk<USAC_EST_LINE2D>(c, a, slots); break;
                case USAC_EST_HOMOGRAPHY: rc = launch_walk<USAC_EST_HOMOGRAPHY>(c, a, slots); break;
                case USAC_EST_FUNDAMENTAL: rc = launch_walk<USAC_EST_FUNDAMENTAL>(c, a, slots); break;
                default: rc = launch_walk<USAC_EST_ESSENTIAL>(c, a, slots); break;
            }
            if (rc) return rc;
            CUDA_TRY(c, c->h_rp_res.ensure((size_t)P * KS));
            CUDA_TRY(c, cudaMemcpyAsync(c->h_rp_res.p, c->d_sprt_res.p, sizeof(SprtModelResult) * (size_t)slots * KS, cudaMemcpyDeviceToHost, c->stream));
        } else {
            size_t part = 0;                                           // the groups' partial sums follow each other in d_part_*
            for (int g0 = 0, g1; g0 < slots; g0 = g1) {
                // one launch per chunk width; the group's chunk grid covers its longest problem (a shorter problem's chunks past its
                // end hold 0, and adding 0 leaves its sum as it was)
                int2 pl = plan[active[g0]];
                for (g1 = g0 + 1; g1 < slots && plan[active[g1]].x == pl.x; g1++) pl.y = std::max(pl.y, plan[active[g1]].y);
                ScoreArgs sa{};
                sa.pairs = c->d_pairs.p; sa.aos = c->d_aos.p; sa.prob = c->d_prob.p; sa.active = c->d_active.p + g0;
                sa.recs = c->d_recs.p + (size_t)g0 * KS * USAC_REC_STRIDE; sa.mvalid = c->d_mvalid.p + g0;
                sa.M = KS; sa.mstride = KS; sa.chunk_pairs = pl.x; sa.nchunks = pl.y;
                sa.part_cnt = c->d_part_cnt.p + part; sa.part_sum = c->d_part_sum.p + part;
                launch_score(c, sa, g1 - g0, mblocks);
                RoundArgs ga = a;
                ga.nmodels = a.nmodels + (size_t)g0 * K; ga.offsets = a.offsets + (size_t)g0 * K; ga.nchunks = pl.y;
                ga.part_cnt = sa.part_cnt; ga.part_sum = sa.part_sum;
                model_scores_kernel<<<dim3((KS + 127) / 128, g1 - g0), 128, 0, c->stream>>>(ga, c->d_model_scores.p + (size_t)g0 * KS);
                c->last_launches++;
                part += (size_t)(g1 - g0) * pl.y * KS;
            }
            CUDA_TRY(c, cudaMemcpyAsync(c->h_rp_scores.p, c->d_model_scores.p, sizeof(int2) * (size_t)slots * KS, cudaMemcpyDeviceToHost, c->stream));
        }
        CUDA_TRY(c, cudaMemcpyAsync(c->h_rp_nmodels.p, c->d_nmodels.p, sizeof(int) * (size_t)slots * K, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));              // the host sync of the round
        CUDA_TRY(c, cudaGetLastError());
        n_rounds++;

        rr.clear();
        best_q.assign(slots, -1);                                    // a new best whose model is still on the device (slot, q)
        run.resize(slots);
        for (int slot = 0; slot < slots; slot++) {
            const int p = active[slot];
            rr.emplace_back(c->h_state[p], cfg, (unsigned)c->h_prob[p].n, K, S, m, is_sprt ? c->h_rp_res.p + (size_t)slot * KS : nullptr,
                            c->h_rp_scores.p + (size_t)slot * KS, c->h_rp_nmodels.p + (size_t)slot * K);
            run[slot] = slot;
        }
        while (!run.empty()) {                                       // replay until every problem reaches the end of its round
            calls.clear();
            for (int slot : run) {
                const int p = active[slot];
                FitState& hs = c->h_state[p];
                int q, inl;
                float score;
                while (rr[slot].next(hs, q, inl, score)) {
                    if (is_lo && inl >= 12) { calls.push_back({slot, q, inl, score}); break; }   // pause: LO works on this one
                    rr[slot].accept(hs, is_sprt ? &sprt[p] : nullptr, q, inl, score, nullptr, w);
                    best_q[slot] = q;
                }
            }
            if (calls.empty()) break;
            rc = lo_batch_step(c, lo, active, calls, KS, n_waves, wave_steps);
            if (rc) return rc;
            n_lo += (int)calls.size(); n_lo_steps++;
            run.clear();
            for (size_t k = 0; k < calls.size(); k++) {
                const LoCall& call = calls[k];
                const int p = active[call.slot];
                float model[9] = {0};
                int inl = call.inl;
                float score = call.score;
                lo[p].io_out(c->h_lo_io.p[k], model, inl, score);
                rr[call.slot].accept(c->h_state[p], is_sprt ? &sprt[p] : nullptr, call.q, inl, score, model, w);
                best_q[call.slot] = -1;
                run.push_back(call.slot);
            }
        }
        int npicks = 0;
        int2* picks = c->h_rp_scores.p + (size_t)P * KS;
        std::vector<int> pick_problem;
        next.clear();
        for (int slot = 0; slot < slots; slot++) {
            const int p = active[slot];
            FitState& hs = c->h_state[p];
            rr[slot].finish(hs, is_sprt ? &sprt[p] : nullptr);
            if (best_q[slot] >= 0) { picks[npicks] = make_int2(slot, best_q[slot]); pick_problem.push_back(p); npicks++; }
            if (!rr[slot].done && hs.iters < hs.max_iters) next.push_back(p);
            else hs.done = 1;
        }
        if (npicks) {                                                // the models of this round's new bests that LO did not touch, one gather
            int2* d_picks = c->d_model_scores.p + (size_t)P * KS;
            CUDA_TRY(c, cudaMemcpyAsync(d_picks, picks, sizeof(int2) * npicks, cudaMemcpyHostToDevice, c->stream));
            gather_models_kernel<<<(npicks * 9 + 255) / 256, 256, 0, c->stream>>>(c->d_models_raw.p, d_picks, npicks, KS, c->d_q_models.p);
            c->last_launches++;
            CUDA_TRY(c, cudaMemcpyAsync(c->h_rp_models.p, c->d_q_models.p, sizeof(float) * 9 * npicks, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            for (int i = 0; i < npicks; i++) {
                FitState& hs = c->h_state[pick_problem[i]];
                for (int k = 0; k < 9; k++) hs.best_model[k] = 0.f;
                for (int k = 0; k < w; k++) hs.best_model[k] = c->h_rp_models.p[(size_t)i * 9 + k];
            }
        }
        active.swap(next);
    }
    for (int p = 0; p < P; p++) {
        const FitState& hs = c->h_state[p];
        usac_fit_result& r = results[p];
        fill_result(hs, w, r);
        if (is_lo) { r.lo_inner_iters = lo[p].inner_done; r.lo_iterative_iters = lo[p].iterative_done; }
        r.msac = is_sprt ? nanf("") : usac_msac_cost(c->h_prob[p].n, r.inliers, r.score, cfg->threshold);
    }
    if (trace)
        fprintf(stderr, "usac_gpu_fit[batch replay] P=%d K=%d rounds=%d: LO %d calls in %d steps (%d with waves, %llu waves)\n",
                P, K, n_rounds, n_lo, n_lo_steps, wave_steps, n_waves);
    return USAC_OK;
}

static int fit_host_replay(usac_gpu_ctx* c, const usac_fit_cfg* cfg, usac_fit_result* results, int K) {
    const int P = c->P, m = usac_sample_size(c->est), S = fit_models_per_sample(c->est, cfg), w = c->est == USAC_EST_LINE2D ? 3 : 9;
    const bool is_prosac = cfg->sampler.sampler == USAC_SAMPLER_PROSAC, is_sprt = cfg->sprt != 0;
    const int KS = K * S;
    const unsigned before_sprt = cfg->max_hypothesis_test_before_sprt ? cfg->max_hypothesis_test_before_sprt : 20u;   // model.hpp:39
    std::vector<int> ids;
    std::vector<unsigned char> mask;
    std::vector<unsigned> growth;
    // Solve-ahead: with the uniform sampler a sample depends on its hypothesis id only, so the minimal solver runs for G rounds of K
    // samples at once (the five-point solver is a latency chain of ~0.7 ms per warp: 512 warps leave the GPU empty) and each round
    // verifies its own K of them under its own frozen test - the semantics of rounds of K are untouched.
    int G = 1;
    if (is_sprt && !is_prosac && cfg->sampler.sampler == USAC_SAMPLER_UNIFORM) {
        const char* e = getenv("USAC_GPU_SOLVE_AHEAD");
        G = e ? std::max(1, atoi(e)) : (c->est == USAC_EST_ESSENTIAL ? 8 : 2);
        while (G > 1 && (size_t)K * G > 8192) G--;
    }
    const int KB = K * G;                                         // samples per solved block
    // ... and the NEXT block is solved on a second stream while this block's rounds run (walks, copies, the host replay): two sets of
    // sample / model / record buffers, used alternately
    const bool overlap = G > 1 && !(getenv("USAC_GPU_SOLVE_OVERLAP") && atoi(getenv("USAC_GPU_SOLVE_OVERLAP")) == 0);
    int rc = ensure_round_buffers(c, 1, overlap ? 2 * KB : KB, 1, 1, S);
    if (rc) return rc;
    if (overlap && !c->stream2) {
        CUDA_TRY(c, cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_block[i], cudaEventDisableTiming));
        CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_round, cudaEventDisableTiming));
    }
    CUDA_TRY(c, c->d_model_scores.ensure(KS));
    CUDA_TRY(c, c->h_rp_nmodels.ensure(K));
    CUDA_TRY(c, c->h_rp_res.ensure(KS));
    CUDA_TRY(c, c->h_rp_scores.ensure(KS));
    CUDA_TRY(c, c->h_rp_models.ensure((size_t)KS * 9));
    CUDA_TRY(c, c->h_rp_state.ensure(1));
    int* const h_nmodels = c->h_rp_nmodels.p;
    SprtModelResult* const h_res = c->h_rp_res.p;
    int2* const h_scores = c->h_rp_scores.p;
    float* const h_models = c->h_rp_models.p;
    // USAC_GPU_TRACE: host wall-clock split of the replay path on stderr (tables / enqueue / waiting for the round / replay / LO / mask)
    static const bool trace = getenv("USAC_GPU_TRACE") != nullptr;
    static const bool trace_kernels = trace && atoi(getenv("USAC_GPU_TRACE")) >= 2;
#define RK(name) do { if (trace_kernels && c->marks_used < 4096) c->mark(name); } while (0)
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::micro>(b - a).count(); };
    double t_tables = 0, t_enqueue = 0, t_wait = 0, t_replay = 0, t_lo = 0, t_mask = 0;
    int n_rounds = 0, n_lo = 0, n_mask = 0;
    unsigned long long n_waves = 0;

    for (int p = 0; p < P; p++) {
        const auto t_p0 = now();
        const ProblemDesc& pd = c->h_prob[p];
        const unsigned n = (unsigned)pd.n;
        FitState& hs = c->h_state[p];
        init_state(hs, pd, c->est, cfg->max_iterations, 0);
        SprtHost sprt;
        ProsacTermHost pterm;
        if (is_sprt) sprt.init(c->est, n, (unsigned)m, cfg->max_iterations);
        if (is_prosac) { prosac_growth(n, (unsigned)m, growth); pterm.init(growth, n, (unsigned)m, cfg->confidence, cfg->max_iterations); }
        LoRunner lo;
        if (cfg->lo) { rc = lo.init(c, p, cfg); if (rc) return rc; }
        bool done = false;
        int block_round = 0;                                       // rounds since the first solved block of this problem
        int prelaunched = -1;                                      // index of the block that has been solved ahead on stream2
        t_tables += us(t_p0, now());
        while (!done && hs.iters < hs.max_iters) {
            const auto t_r0 = now();
            n_rounds++;
            if (is_prosac) hs.prosac_term_len = pterm.termination_length;
            if (is_sprt) { const SprtTestH& t = sprt.current(); hs.sprt_eps = t.epsilon; hs.sprt_delta = t.delta; hs.sprt_A = t.A; hs.sprt_cursor = sprt.cursor; }
            CUDA_TRY(c, cudaMemcpyAsync(c->d_state.p + p, &hs, sizeof(FitState), cudaMemcpyHostToDevice, c->stream));
            c->h_active[0] = p;
            CUDA_TRY(c, cudaMemcpyAsync(c->d_active.p, c->h_active, sizeof(int), cudaMemcpyHostToDevice, c->stream));
            int chunk_pairs = pd.n_pairs, nchunks = 1;
            const int mblocks = (KS + USAC_SCORE_THREADS - 1) / USAC_SCORE_THREADS;
            if (!is_sprt) {
                plan_chunks(c, 1, mblocks, pd.n_pairs, &chunk_pairs, &nchunks);
                rc = ensure_round_buffers(c, 1, K, nchunks, 1, S);
                if (rc) return rc;
            }
            if (overlap) CUDA_TRY(c, cudaEventRecord(c->ev_round, c->stream));   // everything up to this round's state upload
            RK("start");
            // ---- sample + solve + records: once per block of G rounds ----
            const int g = block_round % G;                       // this round's position in the solved block
            const int blk = block_round / G, par = overlap ? (blk & 1) : 0;
            auto launch_block = [&](int parity, unsigned long long hyp_base_p1) {   // sample + solve + records of one block of G rounds
                RoundArgs b;
                fill_round_args(c, b, cfg->sampler, KB, S);
                b.thr = cfg->threshold; b.confidence = cfg->confidence; b.max_iterations = cfg->max_iterations;
                b.table_rows = cfg->sample_table_rows; b.nchunks = nchunks; b.sprt = cfg->sprt; b.pool = c->d_pool.p; b.sprt_res = c->d_sprt_res.p;
                b.before_sprt = before_sprt;
                b.hyp_base_p1 = hyp_base_p1;
                b.samples = c->d_samples.p + (size_t)parity * KB * m; b.nmodels = c->d_nmodels.p + (size_t)parity * KB;
                b.offsets = c->d_offsets.p + (size_t)parity * KB; b.models_raw = c->d_models_raw.p + (size_t)parity * KB * S * 9;
                b.recs = c->d_recs.p + (size_t)parity * KB * S * USAC_REC_STRIDE; b.mvalid = c->d_mvalid.p + parity;
                b.seeds = c->d_seeds.p + (size_t)parity * KB;
                launch_sampler(c, b, 1);
                RK("sample");
                switch (c->est) {
                    case USAC_EST_LINE2D: launch_solve<USAC_EST_LINE2D>(c, b, 1); break;
                    case USAC_EST_HOMOGRAPHY: launch_solve<USAC_EST_HOMOGRAPHY>(c, b, 1); break;
                    case USAC_EST_FUNDAMENTAL: launch_solve<USAC_EST_FUNDAMENTAL>(c, b, 1); break;
                    default: launch_solve<USAC_EST_ESSENTIAL>(c, b, 1); break;
                }
                RK("solve");
                prepare_kernel<<<1, KB >= 1024 ? 1024 : 256, 0, c->stream>>>(b);
                c->last_launches++;
                RK("prepare");
            };
            if (g == 0) {
                if (prelaunched == blk) CUDA_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_block[par], 0));   // solved beside the previous block's rounds
                else launch_block(par, 0);
                // the next block, on the second stream (its hypothesis ids are known: K per round) - unless this block will most likely end
                // the fit: iterations per sample so far (1 + rejected models, ransac.cpp:77-85) x the samples of one block
                const double per_sample = hs.samples_drawn ? (double)hs.iters / (double)hs.samples_drawn : 1.0;
                const bool likely_more = (double)(hs.max_iters - hs.iters) > 0.9 * per_sample * (double)KB;
                if (overlap && likely_more) {
                    // the second stream starts behind everything the main stream had been given when this round began (the descriptors, the
                    // active list, the SPRT pool of a first fit: a kernel of the block must not run ahead of those uploads)
                    CUDA_TRY(c, cudaStreamWaitEvent(c->stream2, c->ev_round, 0));
                    cudaStream_t main_stream = c->stream;
                    c->stream = c->stream2;
                    launch_block(par ^ 1, (unsigned long long)hs.samples_drawn + (unsigned long long)KB + 1ull);
                    c->stream = main_stream;
                    CUDA_TRY(c, cudaEventRecord(c->ev_block[par ^ 1], c->stream2));
                    prelaunched = blk + 1;
                }
            }
            block_round++;
            // this round's view of the block: samples [g K, (g + 1) K); record offsets stay relative to the block
            RoundArgs a;
            fill_round_args(c, a, cfg->sampler, K, S);
            a.thr = cfg->threshold; a.confidence = cfg->confidence; a.max_iterations = cfg->max_iterations;
            a.table_rows = cfg->sample_table_rows; a.nchunks = nchunks; a.sprt = cfg->sprt; a.pool = c->d_pool.p; a.sprt_res = c->d_sprt_res.p;
            a.before_sprt = before_sprt;
            a.nmodels = c->d_nmodels.p + (size_t)par * KB + (size_t)g * K; a.offsets = c->d_offsets.p + (size_t)par * KB + (size_t)g * K;
            a.models_raw = c->d_models_raw.p + ((size_t)par * KB * S + (size_t)g * KS) * 9;
            a.recs = c->d_recs.p + (size_t)par * KB * S * USAC_REC_STRIDE; a.mvalid = c->d_mvalid.p + par;
            if (is_sprt) {
                switch (c->est) {
                    case USAC_EST_LINE2D: rc = launch_walk<USAC_EST_LINE2D>(c, a, 1); break;
                    case USAC_EST_HOMOGRAPHY: rc = launch_walk<USAC_EST_HOMOGRAPHY>(c, a, 1); break;
                    case USAC_EST_FUNDAMENTAL: rc = launch_walk<USAC_EST_FUNDAMENTAL>(c, a, 1); break;
                    default: rc = launch_walk<USAC_EST_ESSENTIAL>(c, a, 1); break;
                }
                if (rc) return rc;
                CUDA_TRY(c, cudaMemcpyAsync(h_res, c->d_sprt_res.p, sizeof(SprtModelResult) * KS, cudaMemcpyDeviceToHost, c->stream));
            } else {
                ScoreArgs sa{};
                sa.pairs = c->d_pairs.p; sa.aos = c->d_aos.p; sa.prob = c->d_prob.p; sa.active = c->d_active.p; sa.recs = c->d_recs.p;
                sa.mvalid = c->d_mvalid.p; sa.M = KS; sa.mstride = KS; sa.chunk_pairs = chunk_pairs; sa.nchunks = nchunks;
                sa.part_cnt = c->d_part_cnt.p; sa.part_sum = c->d_part_sum.p;
                launch_score(c, sa, 1, mblocks);
                model_scores_kernel<<<dim3((KS + 127) / 128, 1), 128, 0, c->stream>>>(a, c->d_model_scores.p);
                c->last_launches++;
                CUDA_TRY(c, cudaMemcpyAsync(h_scores, c->d_model_scores.p, sizeof(int2) * KS, cudaMemcpyDeviceToHost, c->stream));
            }
            RK("walk_or_score");
            FitState& dev_state = *c->h_rp_state.p;
            CUDA_TRY(c, cudaMemcpyAsync(h_nmodels, a.nmodels, sizeof(int) * K, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(c, cudaMemcpyAsync(h_models, a.models_raw, sizeof(float) * KS * 9, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(c, cudaMemcpyAsync(&dev_state, c->d_state.p + p, sizeof(FitState), cudaMemcpyDeviceToHost, c->stream));
            RK("d2h");
            const auto t_r1 = now();
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));      // the host sync of the round
            CUDA_TRY(c, cudaGetLastError());
            const auto t_r2 = now();
            t_enqueue += us(t_r0, t_r1); t_wait += us(t_r1, t_r2);
            double t_lo_round = 0, t_mask_round = 0;

            // ---- replay the round in hypothesis order (ransac.cpp:58-139) ----
            RoundReplay rr(hs, cfg, n, K, S, m, is_sprt ? h_res : nullptr, h_scores, h_nmodels);
            int q, inl;
            float score;
            while (rr.next(hs, q, inl, score)) {
                float cand[9] = {0};
                for (int k = 0; k < w; k++) cand[k] = h_models[(size_t)q * 9 + k];
                if (cfg->lo) {                                                   // ransac.cpp:108-110
                    const auto t0 = now();
                    rc = lo.get_model_score(cand, inl, score);
                    if (rc) return rc;
                    t_lo_round += us(t0, now()); n_lo++;
                }
                long long prosac_bound = -1;
                if (is_prosac) {                                                 // ransac.cpp:123-125
                    const auto t0 = now();
                    rc = fetch_mask(c, p, cand, cfg->threshold, mask, ids);
                    if (rc) return rc;
                    prosac_bound = pterm.update(hs.iters, mask, dev_state.prosac_largest_next);
                    t_mask_round += us(t0, now()); n_mask++;
                }
                rr.accept(hs, is_sprt ? &sprt : nullptr, q, inl, score, cand, w, prosac_bound);
            }
            done = rr.done;
            hs.prosac_t = dev_state.prosac_t_next; hs.prosac_n = dev_state.prosac_n_next; hs.prosac_largest = dev_state.prosac_largest_next;
            hs.prosac_t_next = hs.prosac_t; hs.prosac_n_next = hs.prosac_n; hs.prosac_largest_next = hs.prosac_largest;
            rr.finish(hs, is_sprt ? &sprt : nullptr);
            t_lo += t_lo_round; t_mask += t_mask_round;
            t_replay += us(t_r2, now()) - t_lo_round - t_mask_round;
        }
        hs.done = 1;
        if (overlap && prelaunched > (block_round - 1) / G) CUDA_TRY(c, cudaStreamSynchronize(c->stream2));   // solved ahead and never used (rare: see likely_more): its buffers are free again
        usac_fit_result& r = results[p];
        fill_result(hs, w, r);
        if (cfg->lo) { r.lo_inner_iters = lo.inner_done; r.lo_iterative_iters = lo.iterative_done; n_waves += lo.wave_count; }
        r.msac = is_sprt ? nanf("") : usac_msac_cost(pd.n, r.inliers, r.score, cfg->threshold);
    }
#undef RK
    if (trace_kernels) print_marks(c);
    if (trace)
        fprintf(stderr, "usac_gpu_fit[replay] P=%d K=%d rounds=%d: tables %.0f us, enqueue %.0f us, wait %.0f us, replay %.0f us, LO %.0f us (%d calls), "
                "PROSAC mask+update %.0f us (%d); LO waves %llu\n", P, K, n_rounds, t_tables, t_enqueue, t_wait, t_replay, t_lo, n_lo, t_mask, n_mask, n_waves);
    return USAC_OK;
}

// The fit loop keeps the host->device copy engine out of its way (an upload of the next point sets by another context would
// otherwise delay every small copy of a running fit): initial states come from a device-resident template, the list of active
// problems is compacted on the device from the round's `done` flags (same order as the host's bookkeeping).
__global__ void copy_states_kernel(const FitState* __restrict__ src, FitState* __restrict__ dst, int P) {
    const size_t words = (size_t)P * (sizeof(FitState) / 4);
    const unsigned* s = reinterpret_cast<const unsigned*>(src);
    unsigned* d = reinterpret_cast<unsigned*>(dst);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < words; i += (size_t)gridDim.x * blockDim.x) d[i] = s[i];
}
__global__ void iota_kernel(int* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = i;
}
__global__ void __launch_bounds__(1024) compact_active_kernel(const int* __restrict__ active, const int* __restrict__ done, int slots,
                                                              int* __restrict__ next) {
    __shared__ int sm[33];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int q0 = 0; q0 < slots; q0 += blockDim.x) {
        const int q = q0 + threadIdx.x;
        const int keep = (q < slots && !done[q]) ? 1 : 0;
        int total;
        const int off = block_exclusive_scan(keep, &total, sm);
        if (keep) next[base + off] = active[q];
        __syncthreads();
        if (threadIdx.x == 0) base += total;
        __syncthreads();
    }
}

extern "C" int usac_gpu_fit(usac_gpu_ctx* c, const usac_fit_cfg* cfg, usac_fit_result* results) {
    if (!c || !cfg || !results) return fail(c, USAC_ERR_ARG, "fit: bad arguments");
    if (c->P <= 0) return fail(c, USAC_ERR_STATE, "fit: no points uploaded");
    if (!(cfg->threshold > 0.f) || cfg->max_iterations == 0) return fail(c, USAC_ERR_ARG, "fit: threshold and max_iterations must be positive");
    const int nranks = std::max(cfg->nranks, 1), rank = cfg->rank;
    if (rank < 0 || rank >= nranks) return fail(c, USAC_ERR_ARG, "fit: rank out of range");
    const bool peers_ready = c->peer_nranks == nranks && c->peer_rank == rank && c->peer_self;
    if (nranks > 1 && !c->allgather && !peers_ready)
        return fail(c, USAC_ERR_STATE, "fit: nranks > 1 needs usac_gpu_peer_attach, usac_gpu_nccl_init or usac_gpu_set_allgather");
    if (const char* why = check_sampler_cfg(cfg->sampler)) return fail(c, USAC_ERR_ARG, why);
    if (cfg->sampler.rng == USAC_RNG_TABLE && (!cfg->sample_table || cfg->sample_table_rows == 0)) return fail(c, USAC_ERR_ARG, "fit: empty sample table");
    if (cfg->lo) if (const char* why = check_lo_cfg(c->est, cfg)) return fail(c, USAC_ERR_ARG, why);
    if (cfg->essential_roots != USAC_E5_ROOTS_FIRST_VALID && cfg->essential_roots != USAC_E5_ROOTS_ALL_VALID)
        return fail(c, USAC_ERR_ARG, "fit: essential_roots must be USAC_E5_ROOTS_FIRST_VALID or USAC_E5_ROOTS_ALL_VALID");
    if (cfg->essential_roots && c->est != USAC_EST_ESSENTIAL) return fail(c, USAC_ERR_ARG, "fit: essential_roots applies to essential fits only");
    const bool host_replay = cfg->sprt || cfg->lo || cfg->sampler.sampler == USAC_SAMPLER_PROSAC;
    if (host_replay && nranks > 1) return fail(c, USAC_ERR_ARG, "fit: SPRT / PROSAC termination with hypothesis sharding is not supported");
    cudaSetDevice(c->device);
    // USAC_GPU_TRACE=1: host-side wall-clock split of one fit on stderr (setup / enqueue / waiting for the round's flags / read-back)
    static const bool trace = getenv("USAC_GPU_TRACE") != nullptr;
    static const bool trace_kernels = trace && atoi(getenv("USAC_GPU_TRACE")) >= 2;
    c->marks_used = 0;
#define TK(name) do { if (trace_kernels) c->mark(name); } while (0)
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::micro>(b - a).count(); };
    const auto t_begin = now();
    double t_enqueue = 0, t_wait = 0;
    int n_rounds = 0;
    const int P = c->P, m = usac_sample_size(c->est), S = fit_models_per_sample(c->est, cfg);
    int max_n = 0;
    for (int p = 0; p < P; p++) max_n = std::max(max_n, c->h_prob[p].n);
    if (S > 3 && max_n >= (1 << 28)) return fail(c, USAC_ERR_ARG, "fit: USAC_E5_ROOTS_ALL_VALID needs fewer than 2^28 points per problem");
    if (cfg->sprt) for (int p = 0; p < P; p++) if (!c->h_pool_set[p]) return fail(c, USAC_ERR_STATE, "fit: SPRT needs usac_gpu_set_sprt_pool for every problem");

    int K = cfg->round_size;
    if (K <= 0) K = max_n >= 100000 ? 2048 : 512;
    K = (int)std::min<unsigned>((unsigned)K, std::max(cfg->max_iterations, 1u));
    if (nranks > 1) K = ((K + nranks - 1) / nranks) * nranks;

    // termination tables (cached by n) and sampler side data
    {
        std::vector<long long> sig = {(long long)m, (long long)__builtin_bit_cast(unsigned, cfg->confidence), (long long)cfg->max_iterations};
        for (int p = 0; p < P; p++) sig.push_back(c->h_prob[p].n);
        bool offsets_set = true;
        for (int p = 0; p < P; p++) offsets_set = offsets_set && c->h_prob[p].term_off >= 0;
        if (sig != c->term_signature || !offsets_set) {              // same sizes and parameters as the last fit: d_term already holds the tables
            std::map<int, long long> by_n;
            std::vector<unsigned> all;
            if (c->term_cache.size() > 64) c->term_cache.clear();
            for (int p = 0; p < P; p++) {
                const int n = c->h_prob[p].n;
                auto it = by_n.find(n);
                if (it == by_n.end()) {
                    auto key = std::make_tuple(n, m, cfg->confidence, cfg->max_iterations);
                    auto ct = c->term_cache.find(key);
                    if (ct == c->term_cache.end()) {
                        std::vector<unsigned> t;
                        standard_termination_table((unsigned)n, m, cfg->confidence, cfg->max_iterations, t);
                        ct = c->term_cache.emplace(key, std::move(t)).first;
                    }
                    it = by_n.insert({n, (long long)all.size()}).first;
                    all.insert(all.end(), ct->second.begin(), ct->second.end());
                }
                c->h_prob[p].term_off = it->second;
            }
            CUDA_TRY(c, c->d_term.ensure(all.size()));
            CUDA_TRY(c, cudaMemcpyAsync(c->d_term.p, all.data(), sizeof(unsigned) * all.size(), cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            c->term_signature = sig;
        }
    }
    int rc = setup_sampler_side(c, cfg->sampler);
    if (rc) return rc;
    rc = push_desc(c);
    if (rc) return rc;
    if (cfg->sampler.rng == USAC_RNG_TABLE) {
        const int n0 = c->h_prob[0].n;
        for (size_t i = 0; i < (size_t)cfg->sample_table_rows * m; i++)
            if (cfg->sample_table[i] < 0 || cfg->sample_table[i] >= n0) return fail(c, USAC_ERR_ARG, "fit: sample table index out of range");
        CUDA_TRY(c, c->d_table.ensure((size_t)cfg->sample_table_rows * m));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_table.p, cfg->sample_table, sizeof(int) * (size_t)cfg->sample_table_rows * m, cudaMemcpyHostToDevice, c->stream));
    }
    if (host_replay) {
        c->score_events_used = 0; c->last_launches = 0; c->last_score_launches = 0;
        cudaEventRecord(c->ev0, c->stream);
        // USAC_GPU_SPRT_BATCH=0 (A/B knob): SPRT-only batches one problem at a time
        static const bool batch_off = getenv("USAC_GPU_SPRT_BATCH") && atoi(getenv("USAC_GPU_SPRT_BATCH")) == 0;
        const bool batch = c->P > 1 && (cfg->lo || (cfg->sprt && !batch_off)) && cfg->sampler.sampler != USAC_SAMPLER_PROSAC &&
                           cfg->sampler.rng != USAC_RNG_TABLE;
        rc = batch ? fit_batch_replay(c, cfg, results, K) : fit_host_replay(c, cfg, results, K);
        cudaEventRecord(c->ev1, c->stream);
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        collect_timing(c);
        return rc;
    }
    {
        std::vector<long long> sig = {(long long)c->est, (long long)cfg->max_iterations, (long long)P};
        for (int p = 0; p < P; p++) sig.push_back(c->h_prob[p].n);
        if (sig != c->state_init_sig) {
            for (int p = 0; p < P; p++) init_state(c->h_state[p], c->h_prob[p], c->est, cfg->max_iterations, 0);
            CUDA_TRY(c, cudaMemcpyAsync(c->d_state_init.p, c->h_state, sizeof(FitState) * P, cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            c->state_init_sig = sig;
        }
        copy_states_kernel<<<std::min(4 * c->prop.multiProcessorCount, (P * (int)(sizeof(FitState) / 4) + 255) / 256), 256, 0, c->stream>>>(
            c->d_state_init.p, c->d_state.p, P);
    }

    std::vector<int> active(P);
    for (int p = 0; p < P; p++) active[p] = p;
    int* act_cur = c->d_active.p;
    int* act_next = c->d_active2.p;
    iota_kernel<<<(P + 255) / 256, 256, 0, c->stream>>>(act_cur, P);
    int setup_launches = 2;                                      // copy_states_kernel + iota_kernel (counted below: the counters are reset next)
    c->score_events_used = 0; c->last_launches = setup_launches; c->last_score_launches = 0;
    cudaEventRecord(c->ev0, c->stream);

    // Without SPRT and PROSAC the result does not depend on the round size (prefix semantics of select_kernel), so the
    // round grows as problems finish: the tail of a batch then needs a few large rounds instead of many tiny ones.
    const char* growth_env = getenv("USAC_GPU_ROUND_GROWTH");      // tuning knob: 0 disables, N caps the growth factor
    const int growth_cap = growth_env ? atoi(growth_env) : 8;     // measured on C2 x 2368 (profiles/README.md): 8 is the sweet spot
    const bool k_free = growth_cap > 1 && !cfg->sprt && cfg->sampler.sampler != USAC_SAMPLER_PROSAC && cfg->sampler.rng != USAC_RNG_TABLE;
    const int K0 = K;
    const auto t_setup = now();
    while (!active.empty()) {
        const auto t_r0 = now();
        const int slots = (int)active.size();
        if (k_free && slots < P) {
            long long kr = std::min<long long>({2048LL, (long long)P * K0 / slots, (long long)K0 * growth_cap});
            kr = std::min<long long>(kr, std::max(cfg->max_iterations, 1u));
            kr = std::max<long long>(K0, kr / 128 * 128);
            if (nranks > 1) kr = (kr + nranks - 1) / nranks * nranks;
            K = (int)kr;
        }
        int max_pairs = 0;
        for (int p : active) max_pairs = std::max(max_pairs, c->h_prob[p].n_pairs);
        const int mblocks = (K * S + USAC_SCORE_THREADS - 1) / USAC_SCORE_THREADS;
        int chunk_pairs, nchunks;
        // chunks are planned for the model groups a round is EXPECTED to produce (the item list holds the real ones): one model
        // per sample for lines and homographies; about every second sample for the five-point solver (0 or 1 model) and for
        // the seven-point solver after the oriented-epipolar filter (0..3 models)
        const int expect_models = (c->est == USAC_EST_FUNDAMENTAL || c->est == USAC_EST_ESSENTIAL) ? (K + 1) / 2 : K;
        plan_chunks(c, slots, std::max(1, ((expect_models + USAC_SCORE_THREADS - 1) / USAC_SCORE_THREADS) / nranks), max_pairs, &chunk_pairs, &nchunks);
        rc = ensure_round_buffers(c, slots, K, nchunks, nranks, S);
        if (rc) return rc;
        RoundArgs a;
        fill_round_args(c, a, cfg->sampler, K, S);
        a.active = act_cur;
        a.thr = cfg->threshold; a.confidence = cfg->confidence; a.max_iterations = cfg->max_iterations;
        a.table_rows = cfg->sample_table_rows; a.rank = rank; a.nranks = nranks; a.nchunks = nchunks;
        a.sprt = cfg->sprt; a.pool = c->d_pool.p; a.sprt_res = c->d_sprt_res.p; a.done_out = c->d_done.p;
        a.limit_remaining = 1;
        a.items = c->d_items.p; a.item_count = c->d_item_count.p;
        // exchange: through the peer windows when they are attached and the round fits, else through the host's hook (NCCL)
        const bool use_peer = nranks > 1 && peers_ready && (size_t)nranks * slots * ((K + nranks - 1) / nranks) <= c->peer_cap;
        if (nranks > 1 && !use_peer && !c->allgather) return fail(c, USAC_ERR_STATE, "fit: the round does not fit the peer windows and no all-gather hook is installed");
        if (use_peer) {
            a.peer_win = c->d_peer_win.p; a.peer_self = c->peer_self; a.peer_cap = c->peer_cap;
            a.peer_counter = c->d_peer_counter.p; a.peer_error = c->d_peer_error.p;
        }
        // One large problem (a 1M-point fit is ~1 ms of scoring per round): several rounds are enqueued back to back and the host
        // synchronises once per batch instead of once per round - a round that starts after the fit has ended solves and scores
        // nothing (limit_remaining) and select_kernel / winner_kernel skip it. With many small problems the host needs the
        // `done` flags after every round to size the next one, and a wasted round would cost as much as a useful one.
        int rounds_ahead = 1;
        if (P == 1 && max_n >= 65536) rounds_ahead = (int)std::min<unsigned>(8u, (cfg->max_iterations + (unsigned)K - 1) / (unsigned)K);
        for (int ahead = 0; ahead < rounds_ahead; ahead++) {
            TK("round");
            CUDA_TRY(c, cudaMemsetAsync(c->d_item_count.p, 0, 2 * sizeof(unsigned), c->stream));

            launch_sampler(c, a, slots);
            TK("sampler");
            switch (c->est) {
                case USAC_EST_LINE2D: launch_round_est<USAC_EST_LINE2D>(c, a, slots, cfg->sprt); break;
                case USAC_EST_HOMOGRAPHY: launch_round_est<USAC_EST_HOMOGRAPHY>(c, a, slots, cfg->sprt); break;
                case USAC_EST_FUNDAMENTAL: launch_round_est<USAC_EST_FUNDAMENTAL>(c, a, slots, cfg->sprt); break;
                default: launch_round_est<USAC_EST_ESSENTIAL>(c, a, slots, cfg->sprt); break;
            }
            TK("solve");
            prepare_kernel<<<slots, (slots == 1 && K >= 1024) ? 1024 : 256, 0, c->stream>>>(a);   // one large problem: one CTA compacts the whole round
            c->last_launches++;
            {
                ScoreArgs sa{};
                sa.pairs = c->d_pairs.p; sa.aos = c->d_aos.p; sa.prob = c->d_prob.p; sa.active = act_cur; sa.recs = c->d_recs.p;
                sa.mvalid = c->d_mvalid.p; sa.M = K * S; sa.mstride = K * S; sa.chunk_pairs = chunk_pairs; sa.nchunks = nchunks;
                sa.part_cnt = c->d_part_cnt.p; sa.part_sum = c->d_part_sum.p;
                sa.items = c->d_items.p; sa.item_count = c->d_item_count.p;
                TK("prepare");
                launch_score(c, sa, slots, mblocks);
                TK("score");
                dim3 gr((K + 127) / 128, slots);
                if (use_peer) { a.peer_seq = ++c->peer_seq; c->peer_rounds++; }
                const dim3 grc_grid(((K + nranks - 1) / nranks + 31) / 32, slots);
                if (nchunks > 8 && S > 3) reduce_chunks_kernel<USAC_E5_MAX_ROOTS><<<grc_grid, 256, 0, c->stream>>>(a);
                else if (nchunks > 8) reduce_chunks_kernel<USAC_MAX_MODELS_PER_SAMPLE><<<grc_grid, 256, 0, c->stream>>>(a);
                else reduce_kernel<<<gr, 128, 0, c->stream>>>(a);
                c->last_launches++;
                const uint2* scores = c->d_scores.p;
                TK("reduce");
                if (nranks > 1 && !use_peer) {
                    const size_t bytes = (size_t)slots * (K / nranks) * sizeof(uint2);
                    int grc = c->allgather(c->allgather_user, c->d_scores.p, c->d_scores_all.p, bytes, (void*)c->stream);
                    if (grc) return fail(c, USAC_ERR_NCCL, "fit: all-gather failed");
                    scores = c->d_scores_all.p;
                }
                TK("allgather");
                select_kernel<<<slots, 256, 0, c->stream>>>(a, scores);
                c->last_launches++;
            }
            switch (c->est) {
                case USAC_EST_LINE2D: launch_winner_est<USAC_EST_LINE2D>(c, a, slots); break;
                case USAC_EST_HOMOGRAPHY: launch_winner_est<USAC_EST_HOMOGRAPHY>(c, a, slots); break;
                case USAC_EST_FUNDAMENTAL: launch_winner_est<USAC_EST_FUNDAMENTAL>(c, a, slots); break;
                default: launch_winner_est<USAC_EST_ESSENTIAL>(c, a, slots); break;
            }
            TK("select+winner");
        }
        compact_active_kernel<<<1, 1024, 0, c->stream>>>(act_cur, c->d_done.p, slots, act_next);
        c->last_launches++;
        std::swap(act_cur, act_next);
        // the one host sync of the round: one `done` flag per active problem
        CUDA_TRY(c, cudaMemcpyAsync(c->h_done, c->d_done.p, sizeof(int) * slots, cudaMemcpyDeviceToHost, c->stream));
        if (P == 1) {                                                // single problem: its final state rides on the same synchronisation
            CUDA_TRY(c, cudaMemcpyAsync(c->h_state, c->d_state.p, sizeof(FitState), cudaMemcpyDeviceToHost, c->stream));
            cudaEventRecord(c->ev1, c->stream);
        }
        if (use_peer) CUDA_TRY(c, cudaMemcpyAsync(c->h_peer_error, c->d_peer_error.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        const auto t_r1 = now();
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        CUDA_TRY(c, cudaGetLastError());
        if (use_peer && *c->h_peer_error) {
            cudaMemsetAsync(c->d_peer_error.p, 0, sizeof(int), c->stream);
            return fail(c, USAC_ERR_NCCL, "fit: a rank did not publish its scores within 2 s (peer exchange)");
        }
        t_enqueue += us(t_r0, t_r1); t_wait += us(t_r1, now()); n_rounds++;
        std::vector<int> next;
        for (int q = 0; q < slots; q++) if (!c->h_done[q]) next.push_back(active[q]);
        active.swap(next);
    }
    if (P != 1) {
        CUDA_TRY(c, cudaMemcpyAsync(c->h_state, c->d_state.p, sizeof(FitState) * P, cudaMemcpyDeviceToHost, c->stream));
        cudaEventRecord(c->ev1, c->stream);
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    collect_timing(c);
    const int w = c->est == USAC_EST_LINE2D ? 3 : 9;
    for (int p = 0; p < P; p++) {
        const FitState& s = c->h_state[p];
        usac_fit_result& r = results[p];
        memset(&r, 0, sizeof(r));
        for (int i = 0; i < w; i++) r.model[i] = s.best_model[i];
        r.inliers = s.best_cnt; r.score = s.best_sum; r.iterations = s.iters; r.samples_drawn = s.samples_drawn;
        r.best_hyp = s.best_hyp; r.best_model_idx = s.best_midx; r.rounds = s.rounds; r.evals = s.evals;
        r.useful_evals = s.useful_evals;
        r.msac = usac_msac_cost(c->h_prob[p].n, r.inliers, r.score, cfg->threshold);
    }
    if (trace_kernels) print_marks(c);
    if (trace)
        fprintf(stderr, "usac_gpu_fit trace: %d problems, %d rounds: setup %.0f us, enqueue %.0f us, wait %.0f us, total %.0f us (GPU events: %.0f us, scoring %.0f us)\n",
                P, n_rounds, us(t_begin, t_setup), t_enqueue, t_wait, us(t_begin, now()), c->last_total_ms * 1e3, c->last_score_ms * 1e3);
    return USAC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Exchange over peer memory: every rank owns a window in its HBM that all ranks can write (CUDA IPC across processes, plain
// pointers inside one process); the reduce kernels store the packed per-sample scores of a round straight into every window
// over NVLink and select_kernel waits for the flags - no collective call, no extra launch (pipeline.cuh: peer_store /
// peer_publish / peer_wait).
// ------------------------------------------------------------------------------------------------------------------
static int peer_make_window(usac_gpu_ctx* c) {
    if (c->peer_self) return USAC_OK;
    cudaSetDevice(c->device);
    const unsigned cap = 1u << 17;                                  // 131072 packed scores per parity (1 MiB): rounds of up to cap samples x problems
    const size_t bytes = USAC_PEER_HEADER_BYTES + 2ull * cap * sizeof(uint2);
    CUDA_TRY(c, cudaMalloc(&c->peer_self, bytes));
    CUDA_TRY(c, cudaMemset(c->peer_self, 0, bytes));
    CUDA_TRY(c, c->d_peer_counter.ensure(1));
    CUDA_TRY(c, c->d_peer_error.ensure(1));
    CUDA_TRY(c, cudaMemset(c->d_peer_counter.p, 0, sizeof(unsigned)));
    CUDA_TRY(c, cudaMemset(c->d_peer_error.p, 0, sizeof(int)));
    if (!c->h_peer_error) CUDA_TRY(c, cudaMallocHost(&c->h_peer_error, sizeof(int)));
    *c->h_peer_error = 0;
    c->peer_cap = cap;
    return USAC_OK;
}

extern "C" int usac_gpu_peer_export(usac_gpu_ctx* c, char handle_out[USAC_PEER_HANDLE_BYTES]) {
    if (!c || !handle_out) return fail(c, USAC_ERR_ARG, "peer_export: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == USAC_PEER_HANDLE_BYTES, "USAC_PEER_HANDLE_BYTES is the size of a CUDA IPC handle");
    int rc = peer_make_window(c);
    if (rc) return rc;
    cudaIpcMemHandle_t h;
    CUDA_TRY(c, cudaIpcGetMemHandle(&h, c->peer_self));
    memcpy(handle_out, &h, sizeof(h));
    return USAC_OK;
}

extern "C" int usac_gpu_peer_window(usac_gpu_ctx* c, void** window_out) {
    if (!c || !window_out) return fail(c, USAC_ERR_ARG, "peer_window: bad arguments");
    int rc = peer_make_window(c);
    if (rc) return rc;
    *window_out = c->peer_self;
    return USAC_OK;
}

static int peer_finish_attach(usac_gpu_ctx* c, const std::vector<void*>& wins, int rank, int nranks) {
    CUDA_TRY(c, c->d_peer_win.ensure((size_t)nranks));
    CUDA_TRY(c, cudaMemcpy(c->d_peer_win.p, wins.data(), sizeof(void*) * nranks, cudaMemcpyHostToDevice));
    c->peer_rank = rank; c->peer_nranks = nranks;
    return USAC_OK;
}

extern "C" int usac_gpu_peer_attach(usac_gpu_ctx* c, const char* handles, int rank, int nranks) {
    if (!c || !handles || rank < 0 || rank >= nranks || nranks > USAC_PEER_MAX_RANKS) return fail(c, USAC_ERR_ARG, "peer_attach: bad arguments");
    if (c->peer_nranks) return fail(c, USAC_ERR_STATE, "peer_attach: windows are already attached");
    int rc = peer_make_window(c);
    if (rc) return rc;
    std::vector<void*> wins(nranks);
    for (int r = 0; r < nranks; r++) {
        if (r == rank) { wins[r] = c->peer_self; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * USAC_PEER_HANDLE_BYTES, sizeof(h));
        void* w = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&w, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (void* o : c->peer_opened) cudaIpcCloseMemHandle(o);
            c->peer_opened.clear();
            c->err = std::string("peer_attach: cudaIpcOpenMemHandle failed: ") + cudaGetErrorString(e);
            return USAC_ERR_CUDA;
        }
        c->peer_opened.push_back(w);
        wins[r] = w;
    }
    return peer_finish_attach(c, wins, rank, nranks);
}

extern "C" int usac_gpu_peer_detach(usac_gpu_ctx* c) {
    if (!c) return USAC_ERR_ARG;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (void* w : c->peer_opened) cudaIpcCloseMemHandle(w);
    c->peer_opened.clear();
    c->peer_rank = -1; c->peer_nranks = 0;                           // the window itself stays (it may be exported again)
    return USAC_OK;
}

extern "C" int usac_gpu_peer_attach_ptrs(usac_gpu_ctx* c, void* const* windows, int rank, int nranks) {
    if (!c || !windows || rank < 0 || rank >= nranks || nranks > USAC_PEER_MAX_RANKS) return fail(c, USAC_ERR_ARG, "peer_attach_ptrs: bad arguments");
    if (c->peer_nranks) return fail(c, USAC_ERR_STATE, "peer_attach_ptrs: windows are already attached");
    int rc = peer_make_window(c);
    if (rc) return rc;
    if (windows[rank] != c->peer_self) return fail(c, USAC_ERR_ARG, "peer_attach_ptrs: windows[rank] must be this context's own window (usac_gpu_peer_window)");
    std::vector<void*> wins(windows, windows + nranks);
    return peer_finish_attach(c, wins, rank, nranks);
}

// ------------------------------------------------------------------------------------------------------------------
// NCCL binding (dlopen: libusac_gpu.so itself has no link-time dependency on NCCL)
// ------------------------------------------------------------------------------------------------------------------
struct NcclUniqueId { char internal[128]; };
typedef int (*nccl_get_id_fn)(NcclUniqueId*);
typedef int (*nccl_init_rank_fn)(void**, int, NcclUniqueId, int);
typedef int (*nccl_allgather_fn)(const void*, void*, size_t, int, void*, cudaStream_t);

static void* open_nccl() {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    return h;
}

extern "C" int usac_gpu_nccl_unique_id(char id_out[128]) {
    void* h = open_nccl();
    if (!h) { g_create_error = "libnccl.so.2 not found"; return USAC_ERR_NCCL; }
    nccl_get_id_fn f = (nccl_get_id_fn)dlsym(h, "ncclGetUniqueId");
    if (!f) return USAC_ERR_NCCL;
    NcclUniqueId id;
    if (f(&id) != 0) return USAC_ERR_NCCL;
    memcpy(id_out, id.internal, 128);
    return USAC_OK;
}

static int nccl_allgather_hook(void* user, const void* d_send, void* d_recv, size_t bytes, void* stream) {
    usac_gpu_ctx* c = (usac_gpu_ctx*)user;
    nccl_allgather_fn f = (nccl_allgather_fn)dlsym(c->nccl_lib, "ncclAllGather");
    if (!f) return 1;
    return f(d_send, d_recv, bytes, /*ncclUint8*/ 1, c->nccl_comm, (cudaStream_t)stream);
}

extern "C" int usac_gpu_nccl_init(usac_gpu_ctx* c, const char id[128], int rank, int nranks) {
    if (!c || !id || rank < 0 || rank >= nranks) return fail(c, USAC_ERR_ARG, "nccl_init: bad arguments");
    cudaSetDevice(c->device);
    c->nccl_lib = open_nccl();
    if (!c->nccl_lib) return fail(c, USAC_ERR_NCCL, "libnccl.so.2 not found");
    nccl_init_rank_fn f = (nccl_init_rank_fn)dlsym(c->nccl_lib, "ncclCommInitRank");
    if (!f) return fail(c, USAC_ERR_NCCL, "ncclCommInitRank not found");
    NcclUniqueId uid;
    memcpy(uid.internal, id, 128);
    if (f(&c->nccl_comm, nranks, uid, rank) != 0) return fail(c, USAC_ERR_NCCL, "ncclCommInitRank failed");
    c->allgather = nccl_allgather_hook;
    c->allgather_user = c;
    return USAC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// measurement helpers
// ------------------------------------------------------------------------------------------------------------------
extern "C" int usac_gpu_last_timing(const usac_gpu_ctx* c, float* total_ms, float* score_kernel_ms, int* launches, int* score_launches) {
    if (!c) return USAC_ERR_ARG;
    if (total_ms) *total_ms = c->last_total_ms;
    if (score_kernel_ms) *score_kernel_ms = c->last_score_ms;
    if (launches) *launches = c->last_launches;
    if (score_launches) *score_launches = c->last_score_launches;
    return USAC_OK;
}

__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters) {
    float a[8];
#pragma unroll
    for (int i = 0; i < 8; i++) a[i] = 1.0f + threadIdx.x * 1e-3f + i;
    const float b = 0.999f, cc = 1e-3f;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) a[i] = fmaf(a[i], b, cc);
    }
    float s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s += a[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" int usac_gpu_measure_fp32_peak(usac_gpu_ctx* c, double* tflops_out) {
    if (!c || !tflops_out) return USAC_ERR_ARG;
    cudaSetDevice(c->device);
    const int ctas = c->prop.multiProcessorCount * 8, iters = 1 << 14;
    DevBuf<float> out;
    CUDA_TRY(c, out.ensure((size_t)ctas * 256));
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(c->ev0, c->stream);
        fp32_peak_kernel<<<ctas, 256, 0, c->stream>>>(out.p, iters);
        cudaEventRecord(c->ev1, c->stream);
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        const double fl = 2.0 * 8 * iters * 256.0 * ctas;
        if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    out.release();
    *tflops_out = best;
    return USAC_OK;
}
