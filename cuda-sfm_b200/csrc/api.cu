// C ABI implementation (include/sfmb200.h).  Host orchestration only: every
// stage is a handful of kernel launches on the handle's stream into a
// pre-allocated arena (the reference does ~21 cudaMalloc + ~19 cudaFree + >=4
// device syncs per estimateE call, SfM/sfm.cu:94-236).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <new>

#include "../../include/sfmb200.h"
#include "internal.cuh"
#include "sampson.cuh"

using namespace sfmb200;

static thread_local char g_err[512] = "";

static int fail(int code, const char* msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}
static int fail_cuda(const char* what, cudaError_t e) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return SFMB200_ERR_CUDA;
}
#define CK(call)                                           \
    do {                                                   \
        cudaError_t e_ = (call);                           \
        if (e_ != cudaSuccess) return fail_cuda(#call, e_); \
    } while (0)
#define CKL()                                                        \
    do {                                                             \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) return fail_cuda("kernel launch", e_); \
    } while (0)

// What s.E holds.
enum class Held { nothing, essential, homography };

// Which results of earlier calls the handle holds (include/sfmb200.h, "handle state").  Entry points check their
// prerequisites with need() and change the record only through these transitions.
struct HandleState {
    bool points;        // correspondences are ingested
    Held E;
    bool candidates;    // the candidate arena holds hypotheses [h_begin, h_begin + H) of the last estimate, with counts
    bool pose;          // pose candidates of the current E
    bool chain;         // chain_views ran on the current reconstruction
    void new_points() { points = true; chain = false; }     // the chained reconstruction belonged to the old ones
    void lose_points() { points = false; }
    void estimate(Held model) { E = model; candidates = true; pose = chain = false; }
    void lose_candidates() { candidates = false; }
    void new_E() { E = Held::essential; pose = chain = false; }
    void lose_essential() { if (E == Held::essential) E = Held::nothing; }
    void poses() { pose = true; }
    void chained() { chain = true; }
};

struct sfmb200_handle {
    DeviceState s;
    RefitState refit;
    BAState ba;
    ChainState chain;
    void* chain_arena;     // lazily allocated by sfmb200_chain_views
    GbaState gba;
    void* gba_arena;       // lazily allocated by sfmb200_bundle_adjust_global
    float* gba_stats;      // device [8] statistics of the last global adjustment
    HandleState st;
    float* px_staging;     // lazily allocated: device copy of pageable host input
    float* pack_points;    // lazily allocated: device [B][4][n] compact copy of the triangulated points (run_host results)
    void* ba_arena;        // lazily allocated by sfmb200_bundle_adjust (6 floats + 1 byte per correspondence)
    MgPeers mg;            // multi-GPU peer exchange (mg.cu); mg.world == 0 until sfmb200_mg_init
    void* mg_local;        // this rank's exchange buffer (cudaMalloc, exported through CUDA IPC)
    bool mg_connected;
    long long mg_calls;
    int* mg_failed_host;   // sticky failure word of the exchange (pinned, mapped): calls that timed out; != 0 poisons it
    int* mg_failed_dev;    // device alias of the same word
    int mg_clock_khz;
    long long mg_timeout_cycles;
    cudaStream_t stream;
    bool own_stream;
    int device;
    int sms;               // SM count of the handle's device (cached at create)
    int compat;
    int score_variant;
    int tri_inliers_only;
    int hyp_solver;
    int small_path;        // SFMB200_OPT_SMALL_PATH: -1 auto, 0 never, 1 whenever eligible
    long long small_evals; // auto: use the fused single-launch path when n * H is at most this
    // state of the last estimate
    int H;            // hypotheses in the local slice
    int h_begin;
    float thr;
    ScorePlan plan;
    int64_t launches;
    int* filter_scratch;   // [n_max / 256 + 2] per-CTA counts / offsets of the filtered ingest
    float* pack_header;    // device [B][32]: E 9, selected P 16, pose index, inliers, best index (run_host results)
    float* host_header;    // pinned mirror of pack_header
    int* adapt;            // device [4]: adaptive termination flag, hypotheses used, pairs unsatisfied, spare
    void* arena;
    // correspondence counts of the current points (set by every ingest) and the smallest per-pair count
    PointCounts pc;
    int n_min;
    // per-pair-count mode: the counts table (RaggedTable), allocated by the first *_ragged ingest.  The pinned mirror is
    // filled on the host and uploaded with one copy; ragged_ev marks that copy, the next fill waits for it.
    void* ragged_host;
    void* ragged_dev;
    cudaEvent_t ragged_ev;
    // optional per-stage timing (SFMB200_OPT_PROFILE): ring of event sets, one set
    // per run_device / run_host call, 8 boundary marks -> 7 stage durations
    int profile;
    int prof_cur;                 // set being recorded
    long long prof_total;         // sets started since profiling was enabled
    cudaEvent_t (*prof_ev)[8];    // [PROF_RING][8]
    unsigned char* prof_mask;     // [PROF_RING] bit k = mark k recorded
};
static const int PROF_RING = 256;

// Counts table of a batch with per-pair counts, one block in the same layout on the host and on the device:
// grain_off [B + 1] (DeviceState::grain_off), n_pair [B] (DeviceState::n_pair), row_off [B + 1] (first packed row per pair).
struct RaggedTable {
    long long* grain_off;
    int* n_pair;
    int* row_off;
    static size_t bytes(int B) { return (size_t)(B + 1) * sizeof(long long) + (size_t)B * sizeof(int) + (size_t)(B + 1) * sizeof(int); }
    static RaggedTable at(void* base, int B) {
        RaggedTable r;
        r.grain_off = (long long*)base;
        r.n_pair = (int*)(r.grain_off + B + 1);
        r.row_off = r.n_pair + B;
        return r;
    }
};
static bool is_ragged(const sfmb200_handle* h) { return h->s.n_pair != nullptr; }
// Correspondences of pair b on the host side (getters, packed outputs).
static int host_pair_n(const sfmb200_handle* h, int b) {
    return is_ragged(h) ? RaggedTable::at(h->ragged_host, h->s.B).n_pair[b] : h->s.n;
}
// Stages that need the same number of correspondences in every pair refuse a handle in per-pair-count mode.
static int refuse_ragged(const sfmb200_handle* h, const char* stage) {
    if (!is_ragged(h)) return SFMB200_OK;
    char msg[256];
    snprintf(msg, sizeof(msg), "%s needs the same number of correspondences in every pair; the last ingest was *_ragged", stage);
    return fail(SFMB200_ERR_STATE, msg);
}
static inline void prof_mark(sfmb200_handle* h, int k) {
    if (!h->profile) return;
    cudaEventRecord(h->prof_ev[h->prof_cur][k], h->stream);
    h->prof_mask[h->prof_cur] |= (unsigned char)(1u << k);
}
static inline void prof_next(sfmb200_handle* h) {
    if (!h->profile) return;
    h->prof_cur = (int)(h->prof_total % PROF_RING);
    h->prof_total++;
    h->prof_mask[h->prof_cur] = 0;
}

// Every entry point runs with the handle's device current, whatever the caller's current device is (a process
// that drives several GPUs keeps one handle per GPU), and restores the caller's device on return.
struct DeviceScope {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceScope(const sfmb200_handle* h) {
        if (!h) return;
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != h->device) {
            err = cudaSetDevice(h->device);
            switched = err == cudaSuccess;
        }
    }
    ~DeviceScope() {
        if (switched) cudaSetDevice(prev);
    }
};
#define ENTER(h)        \
    DeviceScope scope_(h); \
    if (scope_.err != cudaSuccess) return fail_cuda("cannot make the handle's device current", scope_.err)
// ENTER for the entry points that refuse a null handle
#define ENTER_HANDLE(h) \
    ENTER(h);           \
    if (!h) return fail(SFMB200_ERR_ARG, "null handle")

// Prerequisites of an entry point: need() refuses the call with SFMB200_ERR_STATE and `msg` unless the handle holds all.
constexpr unsigned NEED_POINTS = 1;
constexpr unsigned NEED_ESSENTIAL = 2;      // s.E holds an essential matrix
constexpr unsigned NEED_MODEL = 4;          // s.E holds an essential matrix or a homography
constexpr unsigned NEED_POSE = 8;
constexpr unsigned NEED_CHAIN = 16;
constexpr unsigned NEED_CANDIDATES = 32;
static int need(const sfmb200_handle* h, unsigned what, const char* msg) {
    const HandleState& st = h->st;
    const unsigned held = (st.points ? NEED_POINTS : 0u) | (st.E == Held::essential ? NEED_ESSENTIAL : 0u) |
                          (st.E != Held::nothing ? NEED_MODEL : 0u) | (st.pose ? NEED_POSE : 0u) | (st.chain ? NEED_CHAIN : 0u) |
                          (st.candidates ? NEED_CANDIDATES : 0u);
    return (held & what) == what ? SFMB200_OK : fail(SFMB200_ERR_STATE, msg);
}

// Inlier threshold of the stages that follow an estimate: the last estimate's, or the reference's literal (sfm.cu:220)
// while none has set one.
static float stage_thr(const sfmb200_handle* h) { return h->thr > 0 ? h->thr : 1e-6f; }

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// An arena is written once, as a layout: a function that calls carve(&dst, count) for every buffer in it.  The layout
// runs twice, first to size the allocation (every buffer 256-byte aligned), then to point each dst into it.
struct Carver {
    char* base;       // nullptr while sizing
    size_t bytes;
    template <typename T>
    void operator()(T** dst, size_t count) {
        if (base) *dst = (T*)(base + bytes);
        bytes = align_up(bytes + count * sizeof(T), 256);
    }
};
template <typename Layout>
static cudaError_t alloc_arena(void** arena, size_t* bytes, Layout layout) {
    Carver size = {nullptr, 0};
    layout(size);
    cudaError_t e = cudaMalloc(arena, size.bytes);
    if (e != cudaSuccess) return e;
    Carver place = {(char*)*arena, 0};
    layout(place);
    *bytes = size.bytes;
    return cudaSuccess;
}
// Scratch that only some workflows need: allocated and zeroed (on the handle's stream) by the first call that uses it.
template <typename Layout>
static int lazy_arena(sfmb200_handle* h, void** arena, Layout layout) {
    if (*arena) return SFMB200_OK;
    size_t bytes = 0;
    CK(alloc_arena(arena, &bytes, layout));
    CK(cudaMemsetAsync(*arena, 0, bytes, h->stream));
    return SFMB200_OK;
}

// Frees whatever the handle holds: sfmb200_destroy, and sfmb200_create when it fails part-way.
static void release(sfmb200_handle* h) {
    if (h->own_stream) cudaStreamDestroy(h->stream);
    if (h->host_header) cudaFreeHost(h->host_header);
    if (h->ragged_host) cudaFreeHost(h->ragged_host);
    if (h->ragged_ev) cudaEventDestroy(h->ragged_ev);
    if (h->prof_ev) {
        for (int i = 0; i < PROF_RING; i++)
            for (int k = 0; k < 8; k++) cudaEventDestroy(h->prof_ev[i][k]);
        delete[] h->prof_ev;
        delete[] h->prof_mask;
    }
    for (void* p : {h->arena, h->chain_arena, h->gba_arena, h->ba_arena, (void*)h->px_staging, (void*)h->pack_points, h->ragged_dev})
        if (p) cudaFree(p);
    delete h;
}

extern "C" {

const char* sfmb200_last_error(void) { return g_err; }
int sfmb200_version(void) { return 100; }

int sfmb200_create(const float K[9], const float Kinv[9], int pairs, int max_points, int max_hyp, sfmb200_t** out) {
    if (!K || !Kinv || !out) return fail(SFMB200_ERR_ARG, "null argument");
    if (pairs < 1 || max_points < 8 || max_hyp < 1) return fail(SFMB200_ERR_ARG, "pairs >= 1, max_points >= 8, max_hypotheses >= 1 required");
    if (pairs > 65535) return fail(SFMB200_ERR_ARG, "at most 65535 pairs per handle (grid.y / grid.z limit)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(SFMB200_ERR_NODEVICE, "no CUDA device: sfmb200 has no CPU fallback");
    }
    sfmb200_handle* h = new (std::nothrow) sfmb200_handle();
    if (!h) return fail(SFMB200_ERR_ARG, "out of host memory");
    memset(h, 0, sizeof(*h));
    cudaError_t e = cudaGetDevice(&h->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, h->device);
    if (e != cudaSuccess) {
        release(h);
        return fail_cuda("create: device query", e);
    }
    DeviceState& s = h->s;
    s.B = pairs;
    s.n_max = max_points;
    s.h_max = max_hyp;
    s.n = 0;
    s.n_stride = (int)align_up(max_points, SCORE_CHUNK);
    s.h_stride = (int)align_up(max_hyp, 1024);
    s.tiles_max = s.h_stride / SCORE_MIN_TILE;
    memcpy(s.K, K, sizeof(float) * 9);
    memcpy(s.Kinv, Kinv, sizeof(float) * 9);
    s.pt_scale = make_thr_scale(1e-6f).ik;     // the reference's threshold literal (sfm.cu:220) until told otherwise
    const size_t B = pairs;
    RefitState& r = h->refit;
    r.max_blocks = 64;
    size_t bytes = 0;
    e = alloc_arena(&h->arena, &bytes, [&](Carver& carve) {
        carve(&s.corr, B * s.n_stride);
        carve(&s.corr_s, B * s.n_stride);
        carve(&s.Ecand, B * 9 * (size_t)s.h_stride);
        carve(&s.counts, B * (size_t)s.h_stride);
        carve(&s.tile_done, B * (size_t)s.tiles_max);
        carve(&s.best, B);
        carve(&s.E, B * 9);
        carve(&s.best_idx, B);
        carve(&s.best_count, B);
        carve(&s.P, B * 64);
        carve(&s.P_ind, B);
        carve(&s.points, B * 4 * (size_t)s.n_stride);
        carve(&s.tri_count, B);
        carve(&s.vote, B * 8);
        carve(&h->filter_scratch, (size_t)max_points / 256 + 2);
        carve(&h->pack_header, B * 32);
        carve(&h->adapt, 4);
        carve(&r.cand, B * 9);
        carve(&r.T, B * 8);
        carve(&r.flags, B * 4);
        carve(&r.iters_done, B);
        carve(&r.mom_part, B * r.max_blocks * 8);
        carve(&r.gram_part, B * r.max_blocks * 45);
    });
    if (e != cudaSuccess) {
        release(h);
        return fail_cuda("cudaMalloc(arena)", e);
    }
    h->ba.persistent = 1;      // the bundle-adjustment scratch itself is allocated on first use (ensure_ba_arena)
    e = cudaMemset(h->arena, 0, bytes);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        h->own_stream = true;
        e = cudaMallocHost((void**)&h->host_header, B * 32 * sizeof(float));
    }
    if (e != cudaSuccess) {
        release(h);
        return fail_cuda("create", e);
    }
    h->compat = 1;
    h->hyp_solver = 1;     // Cholesky projector: same parity as the Jacobi eigensolve, 3.5-4.4x faster (profiles/)
    h->score_variant = -1;
    h->tri_inliers_only = 0;
    h->small_path = -1;
    h->small_evals = 2500000;      // crossover with the five-launch path on B200: device time ~1.5e6, call latency ~2.5e6 (profiles/r02_small_path.md)
    *out = h;
    return SFMB200_OK;
}

int sfmb200_destroy(sfmb200_t* h) {
    ENTER(h);
    if (!h) return SFMB200_OK;
    cudaStreamSynchronize(h->stream);
    sfmb200_mg_close(h);          // unmaps the peers' exchange buffers; needs the stream, so before it goes
    release(h);
    return SFMB200_OK;
}

int sfmb200_set_option(sfmb200_t* h, int option, int value) {
    ENTER_HANDLE(h);
    switch (option) {
        case SFMB200_OPT_COMPAT: h->compat = value ? 1 : 0; break;
        case SFMB200_OPT_SCORE_VARIANT:
            if (value < -1 || value >= score_num_variants()) return fail(SFMB200_ERR_ARG, "score variant out of range");
            h->score_variant = value;
            break;
        case SFMB200_OPT_TRI_INLIERS_ONLY: h->tri_inliers_only = value ? 1 : 0; break;
        case SFMB200_OPT_HYP_SOLVER:
            if (value < 0 || value > 1) return fail(SFMB200_ERR_ARG, "hypothesis solver must be 0 (Jacobi) or 1 (Cholesky projector)");
            h->hyp_solver = value;
            break;
        case SFMB200_OPT_BA_PERSISTENT: h->ba.persistent = value ? 1 : 0; break;
        case SFMB200_OPT_SAMPLER:
            if (value < 0 || value > 1) return fail(SFMB200_ERR_ARG, "sampler must be 0 (independent subsets) or 1 (disjoint permutation)");
            h->s.sampler = value;
            break;
        case SFMB200_OPT_SCORE_METRIC:
            if (value < 0 || value > 1) return fail(SFMB200_ERR_ARG, "score metric must be 0 (Sampson error) or 1 (symmetric epipolar distance)");
            h->s.metric = value;
            break;
        case SFMB200_OPT_SMALL_PATH:
            if (value < -1 || value > 1) return fail(SFMB200_ERR_ARG, "small path must be -1 (auto), 0 (never) or 1 (whenever eligible)");
            h->small_path = value;
            break;
        case SFMB200_OPT_SMALL_PATH_EVALS:
            if (value < 0) return fail(SFMB200_ERR_ARG, "evaluation limit must be >= 0");
            h->small_evals = value;
            break;
        case SFMB200_OPT_PROFILE:
            if (value && !h->prof_ev) {
                h->prof_ev = new cudaEvent_t[PROF_RING][8];
                h->prof_mask = new unsigned char[PROF_RING]();
                for (int i = 0; i < PROF_RING; i++)
                    for (int k = 0; k < 8; k++) CK(cudaEventCreate(&h->prof_ev[i][k]));
            }
            h->profile = value ? 1 : 0;
            h->prof_total = 0;
            h->prof_cur = 0;
            if (h->prof_mask) memset(h->prof_mask, 0, PROF_RING);
            break;
        default: return fail(SFMB200_ERR_ARG, "unknown option");
    }
    return SFMB200_OK;
}

int sfmb200_set_stream(sfmb200_t* h, void* stream) {
    ENTER_HANDLE(h);
    if (h->own_stream) {
        cudaStreamSynchronize(h->stream);
        cudaStreamDestroy(h->stream);
        h->own_stream = false;
    }
    h->stream = (cudaStream_t)stream;
    return SFMB200_OK;
}

int sfmb200_synchronize(sfmb200_t* h) {
    ENTER_HANDLE(h);
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}

static int check_n(sfmb200_t* h, const void* p, int n) {
    if (!h || !p) return fail(SFMB200_ERR_ARG, "null argument");
    if (n < 8 || n > h->s.n_max) return fail(SFMB200_ERR_ARG, "n must be in [8, max_points]");
    return SFMB200_OK;
}
// Every uniform ingest commits its n through here, which also returns the handle to uniform mode.
static void set_uniform(sfmb200_handle* h, int n) {
    h->s.n = n;
    h->s.n_pair = nullptr;
    h->s.grain_off = nullptr;
    const long long B = h->s.B;
    h->pc = PointCounts{h->s.B, n, B * n, B * ((n + SCORE_GRAIN - 1) / SCORE_GRAIN), false};
    h->n_min = n;
}

int sfmb200_set_points_sift(sfmb200_t* h, const void* d_sift, int n) {
    ENTER(h);
    int rc = check_n(h, d_sift, n);
    if (rc) return rc;
    if (h->s.B != 1) return fail(SFMB200_ERR_ARG, "SiftPoint ingest needs pairs == 1");
    set_uniform(h, n);
    launch_ingest_sift(h->s, d_sift, n, h->stream);
    CKL();
    h->launches++;
    h->st.new_points();
    return SFMB200_OK;
}
int sfmb200_set_points_sift_filtered(sfmb200_t* h, const void* d_sift, int n, float min_score, float max_ambiguity,
                                     int32_t* d_kept_index, int32_t* h_kept) {
    ENTER(h);
    int rc = check_n(h, d_sift, n);
    if (rc) return rc;
    if (h->s.B != 1) return fail(SFMB200_ERR_ARG, "SiftPoint ingest needs pairs == 1");
    h->st.lose_points();
    launch_ingest_sift_filtered(h->s, d_sift, n, min_score, max_ambiguity, h->filter_scratch, d_kept_index, h->stream);
    CKL();
    h->launches += 3;
    int kept = 0;
    int blocks = (n + 255) / 256;
    // the survivor count sizes every later launch, so it has to come back to the host
    CK(cudaMemcpyAsync(&kept, h->filter_scratch + blocks, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h_kept) *h_kept = kept;
    if (kept < 8) return fail(SFMB200_ERR_STATE, "fewer than 8 correspondences survive the match filter");
    set_uniform(h, kept);
    h->st.new_points();
    return SFMB200_OK;
}
// `scale` > 0: the ingest also commits a new threshold scale for the scaled copies (run_device / run_host pass the
// scale of their threshold).  It is committed only once the arguments are validated, right before the launch that
// writes corr_s with it - a failed call leaves pt_scale describing what the buffers really hold.
static int ingest_xy(sfmb200_t* h, const float* d_px, int n, float scale) {
    int rc = check_n(h, d_px, n);
    if (rc) return rc;
    set_uniform(h, n);
    if (scale > 0.0f) h->s.pt_scale = scale;
    prof_mark(h, 0);
    launch_ingest_xy(h->s, d_px, n, h->stream);
    prof_mark(h, 1);
    CKL();
    h->launches++;
    h->st.new_points();
    return SFMB200_OK;
}
int sfmb200_set_points_xy(sfmb200_t* h, const float* d_px, int n) {
    ENTER(h);
    return ingest_xy(h, d_px, n, 0.0f);
}
// Device copy of host input that the kernels cannot reach directly (pageable, or larger than the zero-copy limit): the
// staging buffer is allocated on first use, so device-resident workflows (run_device, the batched configs) never pay for it.
// rows: correspondences in h_px, packed (at most pairs * max_points).
static int stage_input(sfmb200_handle* h, const float* h_px, long long rows) {
    if (!h->px_staging) CK(cudaMalloc(&h->px_staging, (size_t)h->s.B * h->s.n_stride * 4 * sizeof(float)));
    CK(cudaMemcpyAsync(h->px_staging, h_px, (size_t)rows * 4 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    return SFMB200_OK;
}
int sfmb200_set_points_xy_host(sfmb200_t* h, const float* h_px, int n) {
    ENTER(h);
    if (int rc = check_n(h, h_px, n)) return rc;
    if (int rc = stage_input(h, h_px, (long long)h->s.B * n)) return rc;
    return ingest_xy(h, h->px_staging, n, 0.0f);
}
int sfmb200_set_points_normalised(sfmb200_t* h, const float* d_x, int n) {
    ENTER(h);
    int rc = check_n(h, d_x, n);
    if (rc) return rc;
    set_uniform(h, n);
    launch_ingest_normalised(h->s, d_x, n, h->stream);
    CKL();
    h->launches++;
    h->st.new_points();
    return SFMB200_OK;
}

// ---- per-pair counts: packed rows, pair b owns rows [offs[b], offs[b + 1]) ----
static int check_ragged(sfmb200_t* h, const void* px, const int32_t* offs) {
    if (!h || !px || !offs) return fail(SFMB200_ERR_ARG, "null argument");
    if (offs[0] != 0) return fail(SFMB200_ERR_ARG, "offsets[0] must be 0");
    for (int b = 0; b < h->s.B; b++) {
        const long long c = (long long)offs[b + 1] - offs[b];
        if (c < 0) return fail(SFMB200_ERR_ARG, "offsets must not decrease");
        if (c < 8 || c > h->s.n_max) return fail(SFMB200_ERR_ARG, "every count offsets[b+1] - offsets[b] must be in [8, max_points]");
    }
    return SFMB200_OK;
}
// Validated offsets: fills the counts table, uploads it and launches the ingest.  `scale` as for ingest_xy.
static int ingest_ragged(sfmb200_t* h, const float* d_px, const int32_t* offs, float scale) {
    DeviceState& s = h->s;
    const int B = s.B;
    const size_t bytes = RaggedTable::bytes(B);
    if (!h->ragged_dev) CK(cudaMalloc(&h->ragged_dev, bytes));
    if (!h->ragged_host) CK(cudaMallocHost(&h->ragged_host, bytes));
    if (!h->ragged_ev) CK(cudaEventCreateWithFlags(&h->ragged_ev, cudaEventDisableTiming));
    CK(cudaEventSynchronize(h->ragged_ev));      // the previous upload has read the mirror
    const RaggedTable m = RaggedTable::at(h->ragged_host, B), d = RaggedTable::at(h->ragged_dev, B);
    long long grains = 0, sum = 0;
    int n_max = 0, n_min = s.n_max;
    m.grain_off[0] = 0;
    for (int b = 0; b < B; b++) {
        const int c = offs[b + 1] - offs[b];
        m.n_pair[b] = c;
        m.row_off[b] = offs[b];
        grains += (c + SCORE_GRAIN - 1) / SCORE_GRAIN;
        m.grain_off[b + 1] = grains;
        sum += c;
        n_max = c > n_max ? c : n_max;
        n_min = c < n_min ? c : n_min;
    }
    m.row_off[B] = offs[B];
    CK(cudaMemcpyAsync(h->ragged_dev, h->ragged_host, bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->ragged_ev, h->stream));
    s.n = n_max;
    s.n_pair = d.n_pair;
    s.grain_off = d.grain_off;
    h->pc = PointCounts{B, n_max, sum, grains, true};
    h->n_min = n_min;
    if (scale > 0.0f) s.pt_scale = scale;
    prof_mark(h, 0);
    launch_ingest_xy_ragged(s, d_px, d.row_off, h->stream);
    prof_mark(h, 1);
    CKL();
    h->launches++;
    h->st.new_points();
    return SFMB200_OK;
}
int sfmb200_set_points_xy_ragged(sfmb200_t* h, const float* d_px, const int32_t* h_offsets) {
    ENTER(h);
    if (int rc = check_ragged(h, d_px, h_offsets)) return rc;
    return ingest_ragged(h, d_px, h_offsets, 0.0f);
}
int sfmb200_get_point_counts(sfmb200_t* h, int32_t* h_counts) {
    ENTER(h);
    if (!h || !h_counts) return fail(SFMB200_ERR_ARG, "null argument");
    for (int b = 0; b < h->s.B; b++) h_counts[b] = host_pair_n(h, b);
    return SFMB200_OK;
}

// The scoring kernels read coordinates scaled by 1/sqrt(thr) (sampson.cuh).  The ingest kernels write them
// with the scale the handle currently holds; when an estimate asks for another one (a different threshold,
// or 1 for the homography model) the copies are re-materialised first.
static int ensure_scaled(sfmb200_handle* h, float scale) {
    if (h->s.pt_scale == scale) return SFMB200_OK;
    h->s.pt_scale = scale;
    launch_rescale_points(h->s, h->stream);
    CKL();
    h->launches++;
    return SFMB200_OK;
}

// Scoring launch of the essential-matrix model with the handle's metric: Sampson error (the tuned kernel family) or
// symmetric epipolar distance (same kernel, MODEL = 2, in the three tile sizes).  h->plan must be set.
static void score_essential(sfmb200_handle* h, const DeviceState& s, int H, int h_offset, float thr) {
    const int* h_n_pair = is_ragged(h) ? RaggedTable::at(h->ragged_host, s.B).n_pair : nullptr;
    if (s.metric == 0) launch_score(s, h->plan, H, h_offset, thr, h_n_pair, h->stream);
    else launch_score_symmetric(s, h->plan, H, h_offset, thr, h_n_pair, h->stream);
}
static ScorePlan plan_essential(const sfmb200_handle* h, int H) {
    return h->s.metric == 0 ? make_score_plan(h->pc, H, h->score_variant, h->sms) : make_score_plan_homography(h->pc, H, h->sms);
}

// The fused single-launch path (small.cu) serves essential-matrix estimates with the projector solver whose
// hypotheses fit one cluster's shared memory; `pose`: the call also runs the pose stage, which the fused kernel
// implements in reference (compat) semantics only.  Not used while per-stage events are being recorded.
constexpr int SMALL_PATH_MAX_PAIRS = 4;
// `ragged`: the points are (or are about to be) held with per-pair counts, which the fused kernel does not take.
static bool small_path_ok(const sfmb200_handle* h, int n, int H, bool pose, bool ragged) {
    if (ragged || h->small_path == 0 || h->profile || h->hyp_solver != 1 || h->s.skip != nullptr || h->s.metric != 0) return false;
    if (h->score_variant >= 0 && h->small_path != 1) return false;      // the caller asked for a specific scoring kernel
    if (pose && !h->compat) return false;
    if (H > small_path_max_hypotheses()) return false;
    if (h->small_path == 1) return true;
    // automatic: one 16-CTA cluster per pair fills a GPC, so beyond a handful of pairs the clusters queue up behind each other
    // while the general path's kernels spread every pair over the whole GPU (measured: 4 pairs 28.7 vs 30.7 us, 8 pairs 50 vs 35 us)
    if (h->s.B > SMALL_PATH_MAX_PAIRS) return false;
    return (long long)n * (long long)H <= h->small_evals;
}

int sfmb200_estimate_e_slice(sfmb200_t* h, const int32_t* d_idx, int H_total, int h_begin, int H, uint64_t seed,
                             float thr) {
    ENTER_HANDLE(h);
    if (int rc = need(h, NEED_POINTS, "estimate_e before set_points")) return rc;
    if (H < 1 || H > h->s.h_max || h_begin < 0 || (long long)h_begin + H > (long long)H_total)
        return fail(SFMB200_ERR_ARG, "hypothesis slice out of range / above max_hypotheses");
    if (!(thr > 0.0f)) return fail(SFMB200_ERR_ARG, "threshold must be positive");
    if (!d_idx && h->s.sampler == 1 && 8ll * H_total > (long long)h->n_min)
        return fail(SFMB200_ERR_ARG, "the disjoint-permutation sampler needs 8 * H_total <= n, in every pair (the reference uses H = N / 8)");
    h->H = H;
    h->h_begin = h_begin;
    h->thr = thr;
    if (int rc = ensure_scaled(h, make_thr_scale(thr).ik)) return rc;
    if (small_path_ok(h, h->s.n, H, false, is_ragged(h))) {
        // hypothesis generation + scoring + arg-max + selection in one cluster launch
        CK(launch_small_path(h->s, nullptr, d_idx, (long long)H_total * 8, H, h_begin, seed, thr, h->compat, 0, SMALL_ESTIMATE, h->stream));
        memset(&h->plan, 0, sizeof(h->plan));
        h->plan.variant = -2;      // reported by sfmb200_score_plan: the fused path
        h->launches += 1;
    } else {
        h->plan = plan_essential(h, H);
        launch_hypgen(h->s, d_idx, (long long)H_total * 8, H, h_begin, seed, h->hyp_solver, h->stream);
        prof_mark(h, 2);
        CKL();
        score_essential(h, h->s, H, h_begin, thr);
        prof_mark(h, 3);
        CKL();
        launch_select(h->s, h_begin, h->stream);
        prof_mark(h, 4);
        CKL();
        h->launches += 3;
    }
    h->st.estimate(Held::essential);
    return SFMB200_OK;
}

int sfmb200_find_homography(sfmb200_t* h, int loops, uint64_t seed, float thresh, float* h_H, int32_t* h_matches) {
    ENTER_HANDLE(h);
    if (int rc = refuse_ragged(h, "find_homography")) return rc;
    if (int rc = need(h, NEED_POINTS, "find_homography before set_points")) return rc;
    if (loops < 1 || loops > h->s.h_max) return fail(SFMB200_ERR_ARG, "loops out of range / above max_hypotheses");
    if (!(thresh > 0.0f)) return fail(SFMB200_ERR_ARG, "threshold must be positive");
    // `thresh` is in PIXELS like CudaSift's (matching.cu:953-996 runs on pixel coordinates), but the handle holds
    // K^-1-normalised coordinates.  For a camera with square pixels and no skew a pixel distance is exactly f times
    // a normalised one, so the test runs in normalised units with thresh / f and the result is mapped back with
    // H_px = K H K^-1.  Any other K would make the pixel metric anisotropic in normalised units: refused.
    const float* Kc = h->s.K;
    const float f = Kc[0];
    const bool isotropic = f > 0.0f && fabsf(Kc[4] - f) <= 1e-6f * f && Kc[1] == 0.0f && Kc[3] == 0.0f && Kc[6] == 0.0f &&
                           Kc[7] == 0.0f && Kc[8] == 1.0f;
    if (!isotropic)
        return fail(SFMB200_ERR_ARG, "find_homography needs K = [f 0 cx; 0 f cy; 0 0 1] (square pixels, no skew): the pixel threshold is applied as thresh / f");
    const float thresh_n = thresh / f;
    const float thr2 = thresh_n * thresh_n;
    if (int rc = ensure_scaled(h, 1.0f)) return rc;      // the transfer-error test works on the unscaled coordinates
    h->H = loops;
    h->h_begin = 0;
    h->thr = thr2;
    h->plan = make_score_plan_homography(h->pc, loops, h->sms);
    launch_hypgen(h->s, nullptr, (long long)loops * 8, loops, 0, seed, 2, h->stream);
    CKL();
    launch_score_homography(h->s, h->plan, loops, 0, thr2, h->stream);
    CKL();
    launch_select(h->s, 0, h->stream);
    CKL();
    h->launches += 3;
    h->st.estimate(Held::homography);      // the pose stages must not consume it
    if (h_H) CK(cudaMemcpyAsync(h_H, h->s.E, (size_t)h->s.B * 9 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_matches) CK(cudaMemcpyAsync(h_matches, h->s.best_count, (size_t)h->s.B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (h_H || h_matches) CK(cudaStreamSynchronize(h->stream));
    if (h_H) {
        // back to pixel coordinates, H_px = K H K^-1 (fp64 on the host: 2 x 27 multiply-adds per pair), then h8 = 1
        // like CudaSift (matching.cu:907-948 solves for 8 parameters) when h8 is not ~0
        for (int b = 0; b < h->s.B; b++) {
            float* Hm = h_H + 9 * b;
            double T[9], R[9];
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) {
                    double a = 0.0;
                    for (int k = 0; k < 3; k++) a += (double)Hm[3 * i + k] * (double)h->s.Kinv[3 * k + j];
                    T[3 * i + j] = a;
                }
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) {
                    double a = 0.0;
                    for (int k = 0; k < 3; k++) a += (double)h->s.K[3 * i + k] * T[3 * k + j];
                    R[3 * i + j] = a;
                }
            const double inv = fabs(R[8]) > 1e-12 ? 1.0 / R[8] : 1.0;
            for (int i = 0; i < 9; i++) Hm[i] = (float)(R[i] * inv);
        }
    }
    return SFMB200_OK;
}
int sfmb200_estimate_e(sfmb200_t* h, const int32_t* d_idx, int H, uint64_t seed, float thr) {
    ENTER(h);
    return sfmb200_estimate_e_slice(h, d_idx, H, 0, H, seed, thr);
}

// Rounds cover [0, first), [first, first*growth), ... up to H_max; everything is enqueued at
// once and the rounds after the termination test passes return immediately on the device
// (hypgen.cu: adaptive_decide_kernel), so there is no host round trip between rounds.
// The result equals sfmb200_estimate_e(h, d_idx, used, seed, thr) bit for bit when d_idx is NULL
// (counter-based sampler) or when d_idx rows are the same prefix.
int sfmb200_estimate_e_adaptive(sfmb200_t* h, const int32_t* d_idx, int H_max, int first_round, int growth,
                                uint64_t seed, float thr, float confidence, int32_t* h_used) {
    ENTER_HANDLE(h);
    if (int rc = need(h, NEED_POINTS, "estimate_e before set_points")) return rc;
    if (H_max < 1 || first_round < 1 || growth < 2) return fail(SFMB200_ERR_ARG, "H_max >= 1, first_round >= 1, growth >= 2 required");
    if (!(thr > 0.0f)) return fail(SFMB200_ERR_ARG, "threshold must be positive");
    if (!(confidence > 0.0f && confidence < 1.0f)) return fail(SFMB200_ERR_ARG, "confidence must be in (0, 1)");
    // every round must fit the candidate arena
    {
        long long lo = 0, hi = first_round;
        while (lo < H_max) {
            if (hi > H_max) hi = H_max;
            if (hi - lo > h->s.h_max) return fail(SFMB200_ERR_ARG, "a round exceeds max_hypotheses of the handle");
            lo = hi;
            hi *= growth;
        }
    }
    const double log1mp = log1p(-(double)confidence);
    if (int rc = ensure_scaled(h, make_thr_scale(thr).ik)) return rc;
    CK(cudaMemsetAsync(h->adapt, 0, 4 * sizeof(int), h->stream));
    DeviceState s = h->s;
    s.skip = h->adapt;
    long long lo = 0, hi = first_round;
    int rounds = 0;
    while (lo < H_max) {
        if (hi > H_max) hi = H_max;
        const int Hr = (int)(hi - lo);
        h->plan = plan_essential(h, Hr);
        launch_hypgen(s, d_idx, (long long)H_max * 8, Hr, (int)lo, seed, h->hyp_solver, h->stream, rounds > 0);
        CKL();
        score_essential(h, s, Hr, (int)lo, thr);
        CKL();
        launch_adaptive_decide(s, h->adapt, (int)lo, (int)hi, log1mp, hi >= H_max, h->stream);
        CKL();
        h->launches += 3;
        rounds++;
        h->H = Hr;
        h->h_begin = (int)lo;
        lo = hi;
        hi *= growth;
    }
    // the decide kernel of each round publishes the running winner (E, index, count) from that round's arena
    h->thr = thr;
    h->st.estimate(Held::essential);
    h->st.lose_candidates();      // the candidate arena holds whichever round ran last, not [0, used)
    if (h_used) {
        CK(cudaMemcpyAsync(h_used, h->adapt + 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return SFMB200_OK;
}

// ---- multi-GPU, hypothesis-sharded, peer-memory exchange (mg.cu) ----
// Opaque per-rank blob exchanged at set-up: the CUDA IPC handle of the exchange buffer + the UUID of the device
// that owns it (so a peer can check that it reaches that device with native P2P atomics).
struct MgBlob {
    cudaIpcMemHandle_t ipc;
    unsigned char uuid[16];
};
int sfmb200_mg_handle_bytes(void) { return (int)sizeof(MgBlob); }

int sfmb200_mg_init(sfmb200_t* h, int rank, int world, void* h_handle_out) {
    ENTER(h);
    if (!h || !h_handle_out) return fail(SFMB200_ERR_ARG, "null argument");
    if (world < 1 || world > MG_MAX_WORLD || rank < 0 || rank >= world) return fail(SFMB200_ERR_ARG, "bad rank / world (at most 16 ranks)");
    if (h->mg_local) return fail(SFMB200_ERR_STATE, "mg_init called twice");
    const size_t bytes = mg_buffer_bytes(h->s.B, world);
    CK(cudaMalloc(&h->mg_local, bytes));
    CK(cudaMemset(h->mg_local, 0, bytes));
    CK(cudaHostAlloc((void**)&h->mg_failed_host, sizeof(int), cudaHostAllocMapped));
    *h->mg_failed_host = 0;
    CK(cudaHostGetDevicePointer((void**)&h->mg_failed_dev, h->mg_failed_host, 0));
    MgBlob blob;
    memset(&blob, 0, sizeof(blob));
    CK(cudaIpcGetMemHandle(&blob.ipc, h->mg_local));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    memcpy(blob.uuid, prop.uuid.bytes, 16);
    memcpy(h_handle_out, &blob, sizeof(blob));
    memset(&h->mg, 0, sizeof(h->mg));
    h->mg.rank = rank;
    h->mg.world = world;
    h->mg.base[rank] = (unsigned long long*)h->mg_local;
    h->mg_connected = false;
    h->mg_calls = 0;
    int clock_khz = 0;
    cudaDeviceGetAttribute(&clock_khz, cudaDevAttrClockRate, h->device);      // slow query: once, not per call
    h->mg_clock_khz = clock_khz > 0 ? clock_khz : 1900000;
    h->mg_timeout_cycles = 2000LL * h->mg_clock_khz;                          // ~2 s of SM clock
    return SFMB200_OK;
}

int sfmb200_mg_set_timeout_ms(sfmb200_t* h, int ms) {
    ENTER(h);
    if (!h || ms < 1) return fail(SFMB200_ERR_ARG, "timeout must be >= 1 ms");
    if (!h->mg_local) return fail(SFMB200_ERR_STATE, "mg_set_timeout_ms before mg_init");
    h->mg_timeout_cycles = (long long)ms * h->mg_clock_khz;
    return SFMB200_OK;
}

int sfmb200_mg_connect(sfmb200_t* h, const void* h_handles) {
    ENTER(h);
    if (!h || !h_handles) return fail(SFMB200_ERR_ARG, "null argument");
    if (!h->mg_local) return fail(SFMB200_ERR_STATE, "mg_connect before mg_init");
    if (h->mg_connected) return fail(SFMB200_ERR_STATE, "mg_connect called twice");
    const MgBlob* all = (const MgBlob*)h_handles;
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    for (int r = 0; r < h->mg.world; r++) {
        if (r == h->mg.rank) continue;
        // the exchange relies on system-scope atomics over the peer mapping: they are only atomic when the two
        // devices support NATIVE P2P atomics (NVLink); refuse PCIe-only peers instead of racing silently
        int peer_dev = -1;
        for (int d = 0; d < ndev && peer_dev < 0; d++) {
            cudaDeviceProp prop;
            CK(cudaGetDeviceProperties(&prop, d));
            if (memcmp(prop.uuid.bytes, all[r].uuid, 16) == 0) peer_dev = d;
        }
        if (peer_dev < 0) return fail(SFMB200_ERR_ARG, "mg_connect: a peer's device is not visible to this process");
        if (peer_dev != h->device) {
            int native = 0;
            CK(cudaDeviceGetP2PAttribute(&native, cudaDevP2PAttrNativeAtomicSupported, h->device, peer_dev));
            if (!native) return fail(SFMB200_ERR_STATE, "mg_connect: no native P2P atomics between this device and a peer (not NVLink-connected)");
        }
        void* p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, all[r].ipc, cudaIpcMemLazyEnablePeerAccess));
        h->mg.base[r] = (unsigned long long*)p;
    }
    h->mg_connected = true;
    return SFMB200_OK;
}

int sfmb200_mg_close(sfmb200_t* h) {
    ENTER(h);
    if (!h) return SFMB200_OK;
    if (h->mg_local) {
        cudaStreamSynchronize(h->stream);
        for (int r = 0; r < h->mg.world; r++)
            if (r != h->mg.rank && h->mg.base[r]) cudaIpcCloseMemHandle(h->mg.base[r]);
        cudaFree(h->mg_local);
        cudaFreeHost(h->mg_failed_host);
        h->mg_local = nullptr;
        h->mg_failed_host = nullptr;
        h->mg_failed_dev = nullptr;
        h->mg_connected = false;
        memset(&h->mg, 0, sizeof(h->mg));
    }
    return SFMB200_OK;
}

// Every rank calls this with the same arguments on the same correspondences: scores its own slice of the
// H_total hypotheses, exchanges the packed winners through peer memory and takes the global winner's E.
int sfmb200_estimate_e_mg(sfmb200_t* h, const int32_t* d_idx, int H_total, uint64_t seed, float thr) {
    ENTER_HANDLE(h);
    if (int rc = refuse_ragged(h, "estimate_e_mg")) return rc;
    if (!h->mg_connected) return fail(SFMB200_ERR_STATE, "estimate_e_mg before mg_init / mg_connect");
    if (*(volatile int*)h->mg_failed_host != 0) {
        h->st.lose_essential();
        h->st.lose_candidates();
        return fail(SFMB200_ERR_STATE, "the peer exchange timed out earlier (a rank is lost or late): sfmb200_mg_close + mg_init + mg_connect on every rank");
    }
    const int world = h->mg.world, rank = h->mg.rank;
    if (H_total < world) return fail(SFMB200_ERR_ARG, "fewer hypotheses than ranks");
    const long long base = H_total / world, rem = H_total % world;
    const long long lo = rank * base + (rank < rem ? rank : rem), cnt = base + (rank < rem ? 1 : 0);
    int rc = sfmb200_estimate_e_slice(h, d_idx, H_total, (int)lo, (int)cnt, seed, thr);
    if (rc) return rc;
    launch_mg_exchange(h->s, h->mg, h->mg_calls, H_total, h->mg_timeout_cycles, h->mg_failed_dev, h->stream);
    CKL();
    h->mg_calls++;
    h->launches += 2;
    h->st.lose_candidates();           // the candidate arena holds this rank's slice only
    return SFMB200_OK;
}

// Calls of sfmb200_estimate_e_mg on this rank that timed out and produced no result (0 in a healthy job).  Any
// value != 0 is final until the exchange is reconnected.  Synchronises the stream so that every call enqueued so
// far is accounted for.
int sfmb200_mg_status(sfmb200_t* h, int32_t* h_timeouts) {
    ENTER(h);
    if (!h || !h_timeouts) return fail(SFMB200_ERR_ARG, "null argument");
    *h_timeouts = 0;
    if (!h->mg_failed_host) return SFMB200_OK;
    CK(cudaStreamSynchronize(h->stream));
    *h_timeouts = *(volatile int*)h->mg_failed_host;
    if (*h_timeouts != 0) h->st.lose_essential();
    return SFMB200_OK;
}

int sfmb200_best_buffer(sfmb200_t* h, uint64_t** d_best) {
    ENTER(h);
    if (!h || !d_best) return fail(SFMB200_ERR_ARG, "null argument");
    *d_best = (uint64_t*)h->s.best;
    return SFMB200_OK;
}
int sfmb200_adopt_best(sfmb200_t* h, const int32_t* d_idx, int H_total, uint64_t seed) {
    ENTER_HANDLE(h);
    if (int rc = refuse_ragged(h, "adopt_best")) return rc;
    if (int rc = need(h, NEED_POINTS, "adopt_best before set_points")) return rc;
    if (h->st.E == Held::homography || !(h->thr > 0.0f))
        return fail(SFMB200_ERR_STATE, "adopt_best follows an essential-matrix estimate (estimate_e / estimate_e_slice) on this handle");
    launch_regen_best(h->s, d_idx, (long long)H_total * 8, seed, h->hyp_solver, h->stream);
    CKL();
    h->launches++;
    h->st.new_E();         // an essential matrix scored at h->thr (set by the slice estimate that preceded)
    return SFMB200_OK;
}

int sfmb200_refine_e(sfmb200_t* h, int iterations) {
    ENTER_HANDLE(h);
    if (int rc = refuse_ragged(h, "refine_e")) return rc;
    if (iterations < 0 || iterations > 64) return fail(SFMB200_ERR_ARG, "iterations must be in [0, 64]");
    if (int rc = need(h, NEED_POINTS | NEED_ESSENTIAL, "refine_e before an essential matrix exists")) return rc;
    if (iterations == 0) return SFMB200_OK;
    h->launches += launch_refit(h->s, h->refit, stage_thr(h), iterations, h->stream);
    CKL();
    h->st.new_E();
    return SFMB200_OK;
}
// Scratch of the bundle adjustment: allocated on first use so that handles that never adjust (the batched
// configs: thousands of pairs) do not carry 25 bytes per correspondence for it.
static int ensure_ba_arena(sfmb200_handle* h) {
    const size_t B = h->s.B, n = h->s.n_stride;
    BAState& ba = h->ba;
    int ba_blocks = (592 + h->s.B - 1) / h->s.B;          // LM kernels: ~4 CTAs per SM over the whole batch
    ba.max_blocks = ba_blocks < 2 ? 2 : (ba_blocks > 296 ? 296 : ba_blocks);
    return lazy_arena(h, &h->ba_arena, [&](Carver& carve) {
        carve(&ba.pts, B * 2 * 3 * n);
        carve(&ba.active, B * n);
        carve(&ba.cam, B * 24);
        carve(&ba.dc, B * 6);
        carve(&ba.ctl_i, B * 8);
        carve(&ba.ctl_f, B * 8);
        carve(&ba.part, B * ba.max_blocks * 34);
        carve(&ba.part2, B * ba.max_blocks * 2);
        carve(&ba.stats, B * 8);
        carve(&ba.cand, B * 32);
        carve(&ba.base_count, B);
    });
}

// Bundle adjustment of the selected pose and the triangulated inliers with inlier re-selection
// (bundle.cu).  Each outer round: inliers of the current E -> LM iterations -> refined camera,
// E derived from it, cloud re-triangulated, inliers recounted.  h_stats (optional, host
// [pairs][8]): active points, cost at entry, cost at exit, accepted steps, lambda, gauge scale,
// inliers of the refined E, spare - of the LAST round.
int sfmb200_bundle_adjust(sfmb200_t* h, int outer_rounds, int iterations, float* h_stats) {
    ENTER_HANDLE(h);
    if (int rc = refuse_ragged(h, "bundle_adjust")) return rc;
    if (outer_rounds < 1 || outer_rounds > 64 || iterations < 1 || iterations > 256)
        return fail(SFMB200_ERR_ARG, "outer_rounds in [1, 64] and iterations in [1, 256] required");
    if (int rc = need(h, NEED_POINTS | NEED_ESSENTIAL | NEED_POSE, "bundle_adjust needs an essential matrix and a chosen pose"))
        return rc;
    if (int rc = ensure_ba_arena(h)) return rc;
    for (int r = 0; r < outer_rounds; r++) {
        h->launches += launch_bundle_adjust(h->s, h->ba, stage_thr(h), iterations, 1e-3f, h->tri_inliers_only, r == 0, h->ba.stats, h->stream);
        CKL();
    }
    if (h_stats) {
        CK(cudaMemcpyAsync(h_stats, h->ba.stats, (size_t)h->s.B * 8 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return SFMB200_OK;
}

// N-view chaining (chain.cu): pairs of the handle = consecutive view pairs over index-aligned tracks.
int sfmb200_chain_views(sfmb200_t* h, float* d_cloud, int32_t* d_count, float* h_cameras, float* h_scales, int32_t* h_used) {
    ENTER_HANDLE(h);
    if (int rc = refuse_ragged(h, "chain_views")) return rc;
    if (h->s.B > 256) return fail(SFMB200_ERR_ARG, "chain_views handles at most 256 pairs (257 views)");
    if (int rc = need(h, NEED_POINTS | NEED_ESSENTIAL | NEED_POSE,
                      "chain_views needs an essential matrix, a chosen pose and triangulated points per pair"))
        return rc;
    const size_t B = h->s.B;
    ChainState& c = h->chain;
    int rc = lazy_arena(h, &h->chain_arena, [&](Carver& carve) {
        carve(&c.hist, B * 2048);
        carve(&c.median_bin, B);
        carve(&c.used, B);
        carve(&c.bin_sum, B);
        carve(&c.bin_cnt, B);
        carve(&c.scales, B);
        carve(&c.cum_scales, B);
        carve(&c.cameras, (B + 1) * 12);
    });
    if (rc) return rc;
    h->launches += launch_chain(h->s, c, stage_thr(h), d_cloud, d_count, h->stream);
    CKL();
    if (h_cameras) CK(cudaMemcpyAsync(h_cameras, c.cameras, (B + 1) * 12 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_scales) CK(cudaMemcpyAsync(h_scales, c.scales, B * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_used) CK(cudaMemcpyAsync(h_used, c.used, B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (h_cameras || h_scales || h_used) CK(cudaStreamSynchronize(h->stream));
    h->st.chained();
    return SFMB200_OK;
}

// Global bundle adjustment of all cameras and all points of the chained reconstruction (chain.cu).
int sfmb200_bundle_adjust_global(sfmb200_t* h, float* d_cloud, const int32_t* d_count, int iterations, float* h_cameras,
                                 float* h_stats) {
    ENTER(h);
    if (!h || !d_cloud || !d_count) return fail(SFMB200_ERR_ARG, "null argument");
    if (int rc = refuse_ragged(h, "bundle_adjust_global")) return rc;
    if (iterations < 1 || iterations > 1000) return fail(SFMB200_ERR_ARG, "iterations must be in [1, 1000]");
    if (h->s.B > GBA_MAX_PAIRS) return fail(SFMB200_ERR_ARG, "bundle_adjust_global handles at most 16 pairs (17 views)");
    if (int rc = need(h, NEED_CHAIN | NEED_POINTS | NEED_ESSENTIAL | NEED_POSE,
                      "bundle_adjust_global follows chain_views (cloud and count from that call)"))
        return rc;
    const size_t B = h->s.B, V = B + 1, n = h->s.n_max;
    GbaState& g = h->gba;
    g.nb = 148;
    int rc = lazy_arena(h, &h->gba_arena, [&](Carver& carve) {
        carve(&g.cam, 2 * V * 12);
        carve(&g.pts, 2 * 3 * n);
        carve(&g.obs, n);
        carve(&g.lin, n * 9);
        carve(&g.part, gba_part_doubles(h->s.B, g.nb));
        carve(&g.part2, (size_t)g.nb * 2);
        carve(&g.dc, 6 * B);
        carve(&g.ctl_i, 8);
        carve(&g.ctl_f, 8);
        carve(&h->gba_stats, 8);
    });
    if (rc) return rc;
    h->launches += launch_global_ba(h->s, h->chain, g, stage_thr(h), iterations, d_cloud, d_count, h->gba_stats, h->stream);
    CKL();
    if (h_cameras) CK(cudaMemcpyAsync(h_cameras, h->chain.cameras, V * 12 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_stats) CK(cudaMemcpyAsync(h_stats, h->gba_stats, 8 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_cameras || h_stats) CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}

int sfmb200_get_refit_iterations(sfmb200_t* h, int32_t* h_iters) {
    ENTER(h);
    if (!h || !h_iters) return fail(SFMB200_ERR_ARG, "null argument");
    CK(cudaMemcpyAsync(h_iters, h->refit.iters_done, (size_t)h->s.B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}

int sfmb200_pose_candidates(sfmb200_t* h) {
    ENTER_HANDLE(h);
    if (int rc = need(h, NEED_ESSENTIAL, "pose_candidates before an essential matrix exists")) return rc;
    launch_pose_candidates(h->s, h->compat, h->stream);
    prof_mark(h, 5);
    CKL();
    h->launches++;
    h->st.poses();
    return SFMB200_OK;
}
int sfmb200_choose_pose(sfmb200_t* h) {
    ENTER_HANDLE(h);
    if (int rc = need(h, NEED_POSE | NEED_POINTS, "choose_pose before pose_candidates")) return rc;
    launch_choose_pose(h->s, h->compat, stage_thr(h), h->stream);
    prof_mark(h, 6);
    CKL();
    h->launches++;
    return SFMB200_OK;
}
int sfmb200_triangulate(sfmb200_t* h) {
    ENTER_HANDLE(h);
    if (int rc = need(h, NEED_POSE | NEED_POINTS, "triangulate before pose_candidates")) return rc;
    launch_triangulate(h->s, h->tri_inliers_only, stage_thr(h), h->stream);
    prof_mark(h, 7);
    CKL();
    h->launches++;
    return SFMB200_OK;
}

// Whole path in 5 launches: ingest (done by the caller), hypgen, score, the fused
// select + pose candidates + cheirality kernel, [inlier vote in non-compat mode],
// triangulation.  Stage marks 4..6 collapse onto the fused kernel.
static int run_stages(sfmb200_t* h, int H, uint64_t seed, float thr) {
    h->H = H;
    h->h_begin = 0;
    h->thr = thr;
    if (int rc = ensure_scaled(h, make_thr_scale(thr).ik)) return rc;     // no-op after run_device / run_host's own ingest
    h->plan = plan_essential(h, H);
    launch_hypgen(h->s, nullptr, (long long)H * 8, H, 0, seed, h->hyp_solver, h->stream);
    prof_mark(h, 2);
    CKL();
    score_essential(h, h->s, H, 0, thr);
    prof_mark(h, 3);
    CKL();
    launch_select_pose_choose(h->s, 0, h->compat, h->stream);
    prof_mark(h, 4);
    prof_mark(h, 5);
    CKL();
    h->launches += 3;
    if (!h->compat) {
        launch_choose_pose(h->s, 0, thr, h->stream);
        CKL();
        h->launches++;
    }
    prof_mark(h, 6);
    h->st.estimate(Held::essential);
    h->st.poses();
    return sfmb200_triangulate(h);
}

// Whole path in ONE launch (small.cu), for the problems small_path_ok admits.  d_px: device-readable pixel
// correspondences.
static int run_small(sfmb200_t* h, const float* d_px, int n, int H, uint64_t seed, float thr) {
    set_uniform(h, n);
    h->s.pt_scale = make_thr_scale(thr).ik;
    cudaError_t e = launch_small_path(h->s, d_px, nullptr, (long long)H * 8, H, 0, seed, thr, h->compat, h->tri_inliers_only,
                                      SMALL_INGEST | SMALL_ESTIMATE | SMALL_POSE | SMALL_TRI, h->stream);
    if (e != cudaSuccess) return fail_cuda("fused small-problem launch", e);
    h->H = H;
    h->h_begin = 0;
    h->thr = thr;
    memset(&h->plan, 0, sizeof(h->plan));
    h->plan.variant = -2;
    h->launches += 1;
    h->st.new_points();
    h->st.estimate(Held::essential);
    h->st.poses();
    return SFMB200_OK;
}

// Arguments of run_device / run_host and their *_ragged forms (offs != nullptr: n is not used).  All are checked before
// anything is enqueued, so a call that fails here leaves the handle as it was.
static int check_run(sfmb200_t* h, const void* px, int n, const int32_t* offs, int H, float thr) {
    if (!(thr > 0.0f)) return fail(SFMB200_ERR_ARG, "threshold must be positive");
    if (int rc = offs ? check_ragged(h, px, offs) : check_n(h, px, n)) return rc;
    if (H < 1 || H > h->s.h_max) return fail(SFMB200_ERR_ARG, "H out of range / above max_hypotheses");
    return SFMB200_OK;
}

// The whole path on validated arguments and device-readable pixel correspondences: the fused single launch when the
// problem is small, else the ingest followed by the five-launch path.
static int run_path(sfmb200_t* h, const float* d_px, int n, int H, uint64_t seed, float thr) {
    if (small_path_ok(h, n, H, true, false)) return run_small(h, d_px, n, H, seed, thr);
    if (int rc = ingest_xy(h, d_px, n, make_thr_scale(thr).ik)) return rc;     // writes the scaled copies for this threshold
    return run_stages(h, H, seed, thr);
}
static int run_path_ragged(sfmb200_t* h, const float* d_px, const int32_t* offs, int H, uint64_t seed, float thr) {
    if (int rc = ingest_ragged(h, d_px, offs, make_thr_scale(thr).ik)) return rc;
    return run_stages(h, H, seed, thr);
}

int sfmb200_run_device(sfmb200_t* h, const float* d_px, int n, int H, uint64_t seed, float thr) {
    ENTER_HANDLE(h);
    if (int rc = check_run(h, d_px, n, nullptr, H, thr)) return rc;
    prof_next(h);
    return run_path(h, d_px, n, H, seed, thr);
}
int sfmb200_run_device_ragged(sfmb200_t* h, const float* d_px, const int32_t* h_offsets, int H, uint64_t seed, float thr) {
    ENTER_HANDLE(h);
    if (int rc = check_run(h, d_px, 0, h_offsets, H, thr)) return rc;
    prof_next(h);
    return run_path_ragged(h, d_px, h_offsets, H, seed, thr);
}

// Results of the whole path packed for the host: one small header per pair and a
// compact [4][n] copy of the points, so run_host needs two DMA transfers instead
// of six (each small D2H copy costs ~5-10 us of latency on the critical path).
// row_off (per-pair counts): pair b's [4][n_b] block starts at float 4 * row_off[b]; nullptr: at b * 4 * n.
__global__ void pack_results_kernel(DeviceState s, float* header, float* points, const int* row_off, int want_points) {
    const int b = blockIdx.y;
    if (blockIdx.x == 0 && threadIdx.x < 32) {
        const int t = threadIdx.x;
        float v = 0.0f;
        if (t < 9) v = s.E[(size_t)b * 9 + t];
        else if (t < 25) v = s.P[(size_t)b * 64 + 16 * s.P_ind[b] + (t - 9)];
        else if (t == 25) v = __int_as_float(s.P_ind[b]);
        else if (t == 26) v = __int_as_float(s.best_count[b]);
        else if (t == 27) v = __int_as_float(s.best_idx[b]);
        header[(size_t)b * 32 + t] = v;
    }
    if (!want_points) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = pair_n(s, b);
    if (i >= n) return;
    const float* in = s.points + (size_t)b * 4 * s.n_stride;
    float* out = points + (row_off ? 4 * (size_t)row_off[b] : (size_t)b * 4 * n);
#pragma unroll
    for (int r = 0; r < 4; r++) out[(size_t)r * n + i] = in[(size_t)r * s.n_stride + i];
}

// Device-visible alias of a host pointer when it is page-locked (cudaHostAlloc / cudaHostRegister / torch
// pin_memory): kernels then read the input and write the results straight through it (zero copy), which takes
// the three DMA launches and their latencies off the critical path of a 0.4 ms call.  NULL for pageable memory.
static void* pinned_alias(const void* host) {
    if (!host) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

// zero copy pays where latency dominates (config-2-sized calls: 160 KB each way); bulk transfers (batched
// config 4: hundreds of MB) stay with the copy engines, which keep more PCIe requests in flight than a kernel
constexpr size_t ZERO_COPY_LIMIT = 4u << 20;

// Device-readable form of run_host*'s input of `rows` packed correspondences: a pinned alias, or the staging copy.
static int host_input(sfmb200_handle* h, const float* h_px, long long rows, const float** d_px) {
    *d_px = (size_t)rows * 4 * sizeof(float) <= ZERO_COPY_LIMIT ? (const float*)pinned_alias(h_px) : nullptr;
    if (!*d_px) {          // pageable, or too large for zero copy: one copy into the staging buffer
        if (int rc = stage_input(h, h_px, rows)) return rc;
        *d_px = h->px_staging;
    }
    return SFMB200_OK;
}

// Results of run_host* to the host after the path ran: `rows` points in all; row_off as for pack_results_kernel.
static int host_results(sfmb200_handle* h, long long rows, const int* row_off, float* h_E, float* h_P, int32_t* h_pose_index,
                        int32_t* h_inliers, float* h_points) {
    DeviceState& s = h->s;
    const size_t B = s.B, pts_bytes = (size_t)rows * 4 * sizeof(float);
    float* pts_alias = pts_bytes <= ZERO_COPY_LIMIT ? (float*)pinned_alias(h_points) : nullptr;
    if (h_points && !pts_alias && !h->pack_points) CK(cudaMalloc(&h->pack_points, B * 4 * (size_t)s.n_max * sizeof(float)));
    dim3 grid(h_points ? (s.n + 255) / 256 : 1, (unsigned)B);
    // header: always through the handle's own pinned buffer (device-visible under UVA); points: straight into the
    // caller's buffer when it is pinned, else into the device staging copy followed by one DMA
    pack_results_kernel<<<grid, 256, 0, h->stream>>>(s, h->host_header, pts_alias ? pts_alias : h->pack_points, row_off,
                                                     h_points ? 1 : 0);
    CKL();
    h->launches++;
    if (h_points && !pts_alias) CK(cudaMemcpyAsync(h_points, h->pack_points, pts_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (size_t b = 0; b < B; b++) {
        const float* hd = h->host_header + b * 32;
        if (h_E) memcpy(h_E + b * 9, hd, 9 * sizeof(float));
        if (h_P) memcpy(h_P + b * 16, hd + 9, 16 * sizeof(float));
        if (h_pose_index) memcpy(h_pose_index + b, hd + 25, sizeof(int32_t));
        if (h_inliers) memcpy(h_inliers + b, hd + 26, sizeof(int32_t));
    }
    return SFMB200_OK;
}

int sfmb200_run_host(sfmb200_t* h, const float* h_px, int n, int H, uint64_t seed, float thr, float* h_E, float* h_P,
                     int32_t* h_pose_index, int32_t* h_inliers, float* h_points) {
    ENTER_HANDLE(h);
    if (int rc = check_run(h, h_px, n, nullptr, H, thr)) return rc;
    prof_next(h);
    const long long rows = (long long)h->s.B * n;
    const float* d_px = nullptr;
    if (int rc = host_input(h, h_px, rows, &d_px)) return rc;
    if (int rc = run_path(h, d_px, n, H, seed, thr)) return rc;
    return host_results(h, rows, nullptr, h_E, h_P, h_pose_index, h_inliers, h_points);
}
int sfmb200_run_host_ragged(sfmb200_t* h, const float* h_px, const int32_t* h_offsets, int H, uint64_t seed, float thr,
                            float* h_E, float* h_P, int32_t* h_pose_index, int32_t* h_inliers, float* h_points) {
    ENTER_HANDLE(h);
    if (int rc = check_run(h, h_px, 0, h_offsets, H, thr)) return rc;
    prof_next(h);
    const long long rows = h_offsets[h->s.B];
    const float* d_px = nullptr;
    if (int rc = host_input(h, h_px, rows, &d_px)) return rc;
    if (int rc = run_path_ragged(h, d_px, h_offsets, H, seed, thr)) return rc;
    return host_results(h, rows, RaggedTable::at(h->ragged_dev, h->s.B).row_off, h_E, h_P, h_pose_index, h_inliers, h_points);
}

int sfmb200_copy_to_vbo(sfmb200_t* h, int pair, float* d_pos, float* d_col) {
    ENTER(h);
    if (!h || pair < 0 || pair >= h->s.B) return fail(SFMB200_ERR_ARG, "bad handle / pair");
    launch_vbo(h->s, pair, d_pos, d_col, 1.0f, h->stream);
    CKL();
    h->launches++;
    CK(cudaStreamSynchronize(h->stream));   // the reference ends with cudaDeviceSynchronize (sfm.cu:382)
    return SFMB200_OK;
}

int sfmb200_copy_to_vbo_coloured(sfmb200_t* h, int pair, float* d_pos, float* d_col, float scale, int mode, float z_near, float z_far) {
    ENTER(h);
    if (!h || pair < 0 || pair >= h->s.B) return fail(SFMB200_ERR_ARG, "bad handle / pair");
    if (mode < 0 || mode > 2) return fail(SFMB200_ERR_ARG, "colour mode must be 0 (ones), 1 (inlier / outlier) or 2 (depth ramp)");
    if (mode == 1) {
        if (int rc = need(h, NEED_ESSENTIAL, "inlier colouring needs an essential matrix")) return rc;
    }
    launch_vbo_colour(h->s, pair, d_pos, d_col, scale, mode, stage_thr(h), z_near, z_far, h->stream);
    CKL();
    h->launches++;
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}

int sfmb200_get_E(sfmb200_t* h, float* h_E) {
    ENTER(h);
    if (!h || !h_E) return fail(SFMB200_ERR_ARG, "null argument");
    CK(cudaMemcpyAsync(h_E, h->s.E, (size_t)h->s.B * 9 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}
int sfmb200_set_E(sfmb200_t* h, const float* h_E) {
    ENTER(h);
    if (!h || !h_E) return fail(SFMB200_ERR_ARG, "null argument");
    CK(cudaMemcpyAsync(h->s.E, h_E, (size_t)h->s.B * 9 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->st.new_E();
    if (!(h->thr > 0)) h->thr = 1e-6f;
    return SFMB200_OK;
}
int sfmb200_get_best(sfmb200_t* h, int32_t* h_index, int32_t* h_count) {
    ENTER(h);
    if (!h) return fail(SFMB200_ERR_ARG, "null argument");
    if (h_index) CK(cudaMemcpyAsync(h_index, h->s.best_idx, (size_t)h->s.B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (h_count) CK(cudaMemcpyAsync(h_count, h->s.best_count, (size_t)h->s.B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}
int sfmb200_get_poses(sfmb200_t* h, float* h_P) {
    ENTER(h);
    if (!h || !h_P) return fail(SFMB200_ERR_ARG, "null argument");
    CK(cudaMemcpyAsync(h_P, h->s.P, (size_t)h->s.B * 64 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}
int sfmb200_get_pose_index(sfmb200_t* h, int32_t* h_ind) {
    ENTER(h);
    if (!h || !h_ind) return fail(SFMB200_ERR_ARG, "null argument");
    CK(cudaMemcpyAsync(h_ind, h->s.P_ind, (size_t)h->s.B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}
static int check_pair(sfmb200_t* h, int pair, const void* p) {
    if (!h || !p) return fail(SFMB200_ERR_ARG, "null argument");
    if (pair < 0 || pair >= h->s.B) return fail(SFMB200_ERR_ARG, "pair out of range");
    return SFMB200_OK;
}
int sfmb200_get_points(sfmb200_t* h, int pair, float* d_points) {
    ENTER(h);
    int rc = check_pair(h, pair, d_points);
    if (rc) return rc;
    const DeviceState& s = h->s;
    const size_t n = host_pair_n(h, pair);
    CK(cudaMemcpy2DAsync(d_points, n * sizeof(float), s.points + (size_t)pair * 4 * s.n_stride,
                         (size_t)s.n_stride * sizeof(float), n * sizeof(float), 4, cudaMemcpyDeviceToDevice,
                         h->stream));
    return SFMB200_OK;
}
int sfmb200_get_points_host(sfmb200_t* h, int pair, float* h_points) {
    ENTER(h);
    int rc = check_pair(h, pair, h_points);
    if (rc) return rc;
    const DeviceState& s = h->s;
    const size_t n = host_pair_n(h, pair);
    CK(cudaMemcpy2DAsync(h_points, n * sizeof(float), s.points + (size_t)pair * 4 * s.n_stride,
                         (size_t)s.n_stride * sizeof(float), n * sizeof(float), 4, cudaMemcpyDeviceToHost,
                         h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return SFMB200_OK;
}
int sfmb200_get_inlier_counts(sfmb200_t* h, int pair, int32_t* d_counts) {
    ENTER(h);
    int rc = check_pair(h, pair, d_counts);
    if (rc) return rc;
    if ((rc = need(h, NEED_CANDIDATES, "no estimate yet"))) return rc;
    CK(cudaMemcpyAsync(d_counts, h->s.counts + (size_t)pair * h->s.h_stride, (size_t)h->H * sizeof(int),
                       cudaMemcpyDeviceToDevice, h->stream));
    return SFMB200_OK;
}
int sfmb200_get_E_candidates(sfmb200_t* h, int pair, float* d_E) {
    ENTER(h);
    int rc = check_pair(h, pair, d_E);
    if (rc) return rc;
    if ((rc = need(h, NEED_CANDIDATES, "no estimate yet"))) return rc;
    launch_export_ecand(h->s, pair, h->H, d_E, h->stream);
    CKL();
    h->launches++;
    return SFMB200_OK;
}
int sfmb200_get_X(sfmb200_t* h, int pair, int image, float* d_X) {
    ENTER(h);
    int rc = check_pair(h, pair, d_X);
    if (rc) return rc;
    if (image < 0 || image > 1) return fail(SFMB200_ERR_ARG, "image must be 0 or 1");
    if ((rc = need(h, NEED_POINTS, "no points yet"))) return rc;
    launch_export_X(h->s, pair, image, d_X, h->stream);
    CKL();
    h->launches++;
    return SFMB200_OK;
}
int sfmb200_get_inlier_mask(sfmb200_t* h, int pair, uint8_t* d_mask) {
    ENTER(h);
    int rc = check_pair(h, pair, d_mask);
    if (rc) return rc;
    if ((rc = need(h, NEED_MODEL | NEED_POINTS, "no model yet"))) return rc;
    launch_inlier_mask(h->s, pair, stage_thr(h), h->st.E == Held::homography ? 1 : 0, d_mask, h->stream);
    CKL();
    h->launches++;
    return SFMB200_OK;
}
int sfmb200_device_views(sfmb200_t* h, float** d_E, float** d_P, int32_t** d_pose_index, float** d_points,
                         int* point_stride) {
    ENTER_HANDLE(h);
    if (d_E) *d_E = h->s.E;
    if (d_P) *d_P = h->s.P;
    if (d_pose_index) *d_pose_index = h->s.P_ind;
    if (d_points) *d_points = h->s.points;
    if (point_stride) *point_stride = h->s.n_stride;
    return SFMB200_OK;
}
int sfmb200_score_plan(sfmb200_t* h, int32_t out[4]) {
    ENTER(h);
    if (!h || !out) return fail(SFMB200_ERR_ARG, "null argument");
    out[0] = h->plan.variant;
    out[1] = h->plan.tiles;
    out[2] = h->plan.ctas;
    out[3] = h->plan.hyp_per_cta;
    return SFMB200_OK;
}
int64_t sfmb200_launch_count(sfmb200_t* h) { return h ? h->launches : 0; }

int sfmb200_stage_times(sfmb200_t* h, int max_sets, float* ms, int* sets) {
    ENTER(h);
    if (!h || !ms || !sets) return fail(SFMB200_ERR_ARG, "null argument");
    *sets = 0;
    if (!h->prof_ev) return fail(SFMB200_ERR_STATE, "profiling was never enabled");
    CK(cudaStreamSynchronize(h->stream));
    long long have = h->prof_total < PROF_RING ? h->prof_total : PROF_RING;
    long long first = h->prof_total - have;
    for (long long t = first; t < h->prof_total && *sets < max_sets; t++) {
        int i = (int)(t % PROF_RING);
        if (h->prof_mask[i] != 0xFF) continue;
        for (int k = 0; k < 7; k++) CK(cudaEventElapsedTime(&ms[(size_t)(*sets) * 7 + k], h->prof_ev[i][k], h->prof_ev[i][k + 1]));
        (*sets)++;
    }
    return SFMB200_OK;
}

int sfmb200_small_path_debug(int64_t* d_stamps) {
    small_path_set_debug((long long*)d_stamps);
    return SFMB200_OK;
}

int sfmb200_fma_probe(int mode, int iters, double* fmas, float* ms) {
    if (!fmas || !ms || iters < 1 || mode < 0 || mode > 4) return fail(SFMB200_ERR_ARG, "bad argument");
    float* sink = nullptr;
    cudaEvent_t e0, e1;
    CK(cudaMalloc(&sink, 256));
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    launch_fma_probe(mode, 4, 0, sink);   // warm-up
    CK(cudaEventRecord(e0, 0));
    *fmas = launch_fma_probe(mode, iters, 0, sink);
    CK(cudaEventRecord(e1, 0));
    CK(cudaEventSynchronize(e1));
    CKL();
    CK(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    return SFMB200_OK;
}

}  // extern "C"
