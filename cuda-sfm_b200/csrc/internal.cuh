// Internal declarations shared by the kernels and the C ABI (api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sfmb200 {

// Launch parameters of the scoring kernel; chosen by the host per problem shape.
struct ScorePlan {
    int variant;        // index into the scoring kernel family (score.cu: kVariants)
    int hyp_per_cta;    // hypotheses per CTA (threads * hyp/thread)
    int tiles;          // ceil(H / hyp_per_cta), per pair
    int n_units;        // grains of SCORE_GRAIN points per tile
    long long total_units;   // pairs * tiles * n_units
    int ctas;           // persistent grid size (SMs x resident CTAs, capped by the work)
};

#ifndef SFMB200_SCORE_CHUNK
#define SFMB200_SCORE_CHUNK 512
#endif
constexpr int SCORE_CHUNK = SFMB200_SCORE_CHUNK;     // points per TMA stage
constexpr int SCORE_GRAIN = 64;      // work-partition granularity in points
constexpr int SCORE_MIN_TILE = 256;  // smallest hypothesis tile of any kernel variant

// Everything one handle owns on the device.  All per-pair arrays are laid out
// [pair][...] with fixed strides so a batch is one launch (blockIdx.y / z = pair).
// The struct is every kernel's first parameter, and the code nvcc schedules for the scoring kernels depends on where
// the fields sit in it: moving corr .. vote by 8 bytes made the flagship step 1.3 % slower (B200, 1000 W power
// limit).  Add fields at the end.
struct DeviceState {
    int B;              // pairs in the batch
    int sampler;        // device-drawn sample rows: 0 independent 8-subsets per hypothesis, 1 one permutation cut into disjoint
                        // groups of 8 (the reference's scheme, sfm.cu:95-104)
    int n_max;          // capacity: correspondences per pair
    int h_max;          // capacity: hypotheses per pair (local slice)
    int n;              // current correspondences per pair (per-pair-count mode: the largest count)
    int n_stride;       // points stride (n_max rounded up to SCORE_CHUNK)
    int h_stride;       // hypothesis stride (h_max rounded up to 1024)
    int tiles_max;
    float Kinv[9];
    float K[9];

    float pt_scale;     // 1/sqrt(thr) currently materialised in corr_s (sampson.cuh); 1 for the homography model
    float4* corr;       // [B][n_stride]   (x1,y1,x2,y2) normalised camera coords
    float4* corr_s;     // [B][n_stride]   corr * pt_scale: what the scalar scoring kernels stage
    const int* skip;    // adaptive termination: when non-null and *skip != 0 the hypgen / score kernels of
                        // the remaining rounds return at once (set by adaptive_decide_kernel); else nullptr
    float* Ecand;       // [B][9][h_stride] SoA essential-matrix candidates
    int* counts;        // [B][h_stride] inlier count per hypothesis
    int* tile_done;     // [B][tiles_max] split tickets per hypothesis tile
    unsigned long long* best;   // [B] packed (count << 32) | (0xFFFFFFFF - global index)
    float* E;           // [B][9] selected essential matrix
    int* best_idx;      // [B]
    int* best_count;    // [B]
    float* P;           // [B][4][16] pose candidates (row-major 4x4 each)
    int* P_ind;         // [B]
    float* points;      // [B][4][n_stride] SoA (x,y,z,1), the reference's d_final_points layout
    int* tri_count;     // [B] points triangulated in front of both cameras (diagnostic)
    int* vote;          // [B][8] cheirality votes of the four candidates + ticket (choose_pose_vote_kernel)
    int metric;         // inlier test of the essential-matrix model: 0 Sampson error (default), 1 symmetric epipolar distance
    // Per-pair-count mode (the last ingest was *_ragged): pair b holds n_pair[b] correspondences and n is the largest
    // of them (grid sizes).  nullptr on a uniform handle, where every pair holds n.  Kernels use pair_n().
    const int* n_pair;             // [B]
    const long long* grain_off;    // [B + 1] prefix sum of ceil(n_pair[b] / SCORE_GRAIN): the scoring work space
};

// Correspondences of pair b.
__device__ __forceinline__ int pair_n(const DeviceState& s, int b) { return s.n_pair ? s.n_pair[b] : s.n; }

// Correspondence counts of a batch as the score planner needs them: the largest (grains per tile of a uniform batch),
// the sum (evaluations per hypothesis), the sum of ceil(count / SCORE_GRAIN) (the work space in grains per tile) and
// whether the counts are per pair (which instantiation of the scoring kernel runs).
struct PointCounts {
    int B, n_max;
    long long n_sum, grains;
    bool ragged;
};

// Scratch of the local-optimisation (refit) stage, per pair.
struct RefitState {
    float* cand;        // [B][9]  next candidate E
    float* T;           // [B][8]  Hartley similarity of the incumbent's inliers: s1,c1x,c1y,s2,c2x,c2y
    int* flags;         // [B][4]  active, incumbent inlier count, eval ticket, solve ticket
    int* iters_done;    // [B]     accepted refits
    float* mom_part;    // [B][max_blocks][7]
    float* gram_part;   // [B][max_blocks][45]
    int max_blocks;
};
int launch_refit(const DeviceState& s, const RefitState& r, float thr, int iterations, cudaStream_t st);

// Scratch of the two-view bundle adjustment (bundle.cu), per pair.
struct BAState {
    float* pts;             // [B][2][3][n_stride] double-buffered 3-D points (SoA)
    unsigned char* active;  // [B][n_stride] 1 = takes part in the adjustment
    float* cam;             // [B][2][12] double-buffered camera 2: R row-major (9), t (3)
    double* dc;             // [B][6] camera step of the current iteration
    int* ctl_i;             // [B][8] see bundle.cu
    float* ctl_f;           // [B][8]
    double* part;           // [B][max_blocks][34] per-CTA partial sums of the normal equations
    double* part2;          // [B][max_blocks][2]  per-CTA candidate cost / bad-point count
    int persistent;         // 1: one cooperative launch per round when the grid is resident (default); 0: two launches per iteration
    float* stats;           // [B][8] device copy of the statistics of the last round
    int* base_count;        // [B] inliers of the model when sfmb200_bundle_adjust was called (commit guard)
    float* cand;            // [B][32] adjusted camera (16) + its essential matrix (9), before the commit decision
    int max_blocks;
};
// Peer exchange buffers of the hypothesis-sharded multi-GPU estimate (mg.cu): base[r] = rank r's buffer
// (keys[2][B] uint64, arrive uint64 (monotone), E[2][world][B][9] float), mapped into this process through CUDA IPC.
constexpr int MG_MAX_WORLD = 16;
struct MgPeers {
    unsigned long long* base[MG_MAX_WORLD];
    int rank, world;
};
void launch_mg_exchange(const DeviceState& s, const MgPeers& peers, long long call, int H_total, long long timeout_cycles,
                        int* d_failed, cudaStream_t st);
size_t mg_buffer_bytes(int B, int world);

// Scratch and results of the N-view chaining stage (chain.cu); allocated on first use.
struct ChainState {
    int* hist;                      // [B][2048] log-ratio histograms of the links
    int* median_bin;                // [B]
    int* used;                      // [B] tracks linking pair b-1 and b
    unsigned long long* bin_sum;    // [B] fixed-point sum of the log ratios in the median bin
    int* bin_cnt;                   // [B]
    float* scales;                  // [B] scale of pair b relative to pair b-1 (scale[0] = 1)
    float* cum_scales;              // [B]
    float* cameras;                 // [B+1][12] world (camera 0) -> camera k, row-major 3x4
};
int launch_chain(const DeviceState& s, const ChainState& c, float thr, float* d_cloud, int* d_count, cudaStream_t st);

// Scratch of the global bundle adjustment over the chained reconstruction (chain.cu); allocated on first use.
struct GbaState {
    float* cam;             // [2][pairs + 1][12] double-buffered cameras: R row-major (9), t (3)
    float* pts;             // [2][3][n] double-buffered points (SoA)
    unsigned int* obs;      // [n] bit k: view k observes the track; 0 = the track takes no part
    float* lin;             // [n][9] per track: inverse of the damped point block (6, packed) and its gradient (3)
    double* part;           // [nb][blocks + 1][42] per-CTA partial sums of the reduced camera system (+ the cost)
    double* part2;          // [nb][2] candidate cost / observations behind their camera
    double* dc;             // [6 pairs] camera step
    int* ctl_i;             // [8]
    float* ctl_f;           // [8]
    int nb;                 // CTAs of the accumulate / update kernels
};
constexpr int GBA_MAX_PAIRS = 16;
size_t gba_part_doubles(int pairs, int nb);
int launch_global_ba(const DeviceState& s, const ChainState& c, const GbaState& g, float thr, int iterations, float* d_cloud,
                     const int* d_count, float* d_stats, cudaStream_t st);

int launch_bundle_adjust(const DeviceState& s, const BAState& ba, float thr, int iterations, float lambda0,
                         int tri_inliers_only, int first_round, float* d_stats, cudaStream_t st);

void launch_ingest_sift(const DeviceState& s, const void* d_sift, int n, cudaStream_t st);
void launch_ingest_sift_filtered(const DeviceState& s, const void* d_sift, int n, float min_score, float max_ambiguity,
                                 int* d_scratch, int* d_kept_index, cudaStream_t st);
void launch_ingest_xy(const DeviceState& s, const float* d_px, int n, cudaStream_t st);
// packed rows: pair b's s.n_pair[b] rows start at row d_row_off[b] of d_px
void launch_ingest_xy_ragged(const DeviceState& s, const float* d_px, const int* d_row_off, cudaStream_t st);
void launch_ingest_normalised(const DeviceState& s, const float* d_x, int n, cudaStream_t st);
void launch_rescale_points(const DeviceState& s, cudaStream_t st);   // corr -> corr_s with s.pt_scale
void launch_hypgen(const DeviceState& s, const int32_t* d_idx, long long idx_pair_stride, int H, int h_offset,
                   unsigned long long seed, int solver, cudaStream_t st, int keep_best = 0);
void launch_adaptive_decide(const DeviceState& s, int* d_adapt, int round_begin, int done_after, double log1mp, int last,
                            cudaStream_t st);
ScorePlan make_score_plan(const PointCounts& c, int H, int variant_override, int sms);
int score_num_variants();
// h_n_pair: host copy of s.n_pair (nullptr on a uniform handle); the constant-bank variant sizes its launches with it
void launch_score(const DeviceState& s, const ScorePlan& plan, int H, int h_offset, float thr, const int* h_n_pair, cudaStream_t st);
void launch_score_homography(const DeviceState& s, ScorePlan& plan, int H, int h_offset, float thr2, cudaStream_t st);
void launch_score_symmetric(const DeviceState& s, ScorePlan& plan, int H, int h_offset, float thr, const int* h_n_pair, cudaStream_t st);
ScorePlan make_score_plan_homography(const PointCounts& c, int H, int sms);
void launch_select(const DeviceState& s, int h_offset, cudaStream_t st);
void launch_regen_best(const DeviceState& s, const int32_t* d_idx, long long idx_pair_stride,
                       unsigned long long seed, int solver, cudaStream_t st);
void launch_pose_candidates(const DeviceState& s, int compat, cudaStream_t st);
void launch_select_pose_choose(const DeviceState& s, int h_offset, int compat, cudaStream_t st);
void launch_choose_pose(const DeviceState& s, int compat, float thr, cudaStream_t st);
void launch_triangulate(const DeviceState& s, int inliers_only, float thr, cudaStream_t st);
void launch_vbo(const DeviceState& s, int pair, float* d_pos, float* d_col, float scale, cudaStream_t st);
void launch_vbo_colour(const DeviceState& s, int pair, float* d_pos, float* d_col, float scale, int mode, float thr, float z_near,
                       float z_far, cudaStream_t st);
void launch_export_ecand(const DeviceState& s, int pair, int H, float* d_out_Hx9, cudaStream_t st);
void launch_export_X(const DeviceState& s, int pair, int image, float* d_out_3xN, cudaStream_t st);
void launch_inlier_mask(const DeviceState& s, int pair, float thr, int model, unsigned char* d_mask, cudaStream_t st);

// Fused single-launch path for small problems (small.cu): one thread-block cluster per pair.
enum { SMALL_INGEST = 1, SMALL_ESTIMATE = 2, SMALL_POSE = 4, SMALL_TRI = 8 };
int small_path_max_hypotheses();
void small_path_set_debug(long long* d_stamps);      // measurement hook: phase time stamps of the fused kernel
cudaError_t launch_small_path(const DeviceState& s, const float* d_px, const int32_t* d_idx, long long idx_pair_stride, int H,
                              int h_offset, unsigned long long seed, float thr, int compat, int inliers_only, int mask,
                              cudaStream_t st);

// Programmatic dependent launch (sm_90+): a kernel launched with the attribute may become resident while its
// predecessor in the stream drains; it must execute pdl_wait() before touching anything the predecessor wrote
// (the wait returns once the predecessor grid has completed and its writes are visible).  pdl_trigger() lets the
// successor of THIS kernel start launching early.  Compiled in with -DSFMB200_PDL (A/B: profiles/r01_modes.md).
#ifdef SFMB200_PDL
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline void launch_dep(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#else
__device__ __forceinline__ void pdl_wait() {}
__device__ __forceinline__ void pdl_trigger() {}
template <typename... KArgs, typename... Args>
inline void launch_dep(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    kernel<<<grid, block, smem, st>>>(KArgs(args)...);
}
#endif

// FP32 pipe micro-benchmark (bench/roofline denominator): returns lane-FMAs issued.
double launch_fma_probe(int mode, int iters, cudaStream_t st, float* d_sink);

}  // namespace sfmb200
