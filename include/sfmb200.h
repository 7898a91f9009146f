/* sfmb200 - C ABI of the B200-native two-view SfM hot path.
 *
 * Drop-in boundary for the hot path of Black-Phoenix/CUDA-SfM: RANSAC
 * essential-matrix estimation -> 4 pose candidates -> cheirality selection ->
 * linear triangulation.  The reference has no FFI layer: its boundary is the
 * C++ class SfM::Image_pair (SfM/sfm.h:20-60) called from src/main.cpp:298-307.
 * Each entry point below names the reference interface it replaces; the
 * source-compatible C++ facade (cuda-sfm_b200/SfM/sfm.h, kernels.h, svd.h) and
 * the Python mirror (cuda-sfm_b200/image_pair.py) are thin layers over this
 * file.  See INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions
 *  - every function returns 0 on success or a negative sfmb200_status;
 *    sfmb200_last_error() gives the message.  Nothing here prints or exits
 *    (the reference's checkCUDAError prints and exit()s, SfM/common.cu:3-15).
 *  - pointers named d_* are DEVICE pointers, h_* are HOST pointers.
 *  - matrices are row-major float (access2/access3, SfM/common.h:19-20);
 *    point sets are SoA (3xN / 4xN) exactly as the reference stores them.
 *  - a handle owns one device (the current one at create time), one stream and
 *    a pre-sized arena; no allocation happens in any other call.  Handles are
 *    not thread-safe; different handles are independent.
 *  - a handle processes a BATCH of `pairs` image pairs with the same capacity
 *    (max_points correspondences each); SfM::Image_pair is the pairs == 1 case.
 *    The pairs hold the same number of correspondences n (set_points_*, run_host,
 *    run_device) or one count per pair (the *_ragged entry points below).
 *  - there is no CPU fallback: every compute entry point needs a CUDA device.
 */
#ifndef SFMB200_H
#define SFMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sfmb200_handle sfmb200_t;

typedef enum {
    SFMB200_OK = 0,
    SFMB200_ERR_ARG = -1,      /* bad argument (null, out of capacity, n < 8, ...) */
    SFMB200_ERR_CUDA = -2,     /* a CUDA runtime call failed */
    SFMB200_ERR_STATE = -3,    /* stage called before its prerequisite */
    SFMB200_ERR_NODEVICE = -4  /* no CUDA device */
} sfmb200_status;

/* Options (sfmb200_set_option).  Defaults reproduce the reference's literals. */
typedef enum {
    SFMB200_OPT_COMPAT = 1,        /* 1 (default): reference semantics for poses / cheirality / triangulation
                                      (SURVEY.md Appendix A); 0: textbook geometry with an inlier vote */
    SFMB200_OPT_SCORE_VARIANT = 2, /* -1 auto (default); >= 0: index into the scoring kernel family
                                      (0 scalar FFMA 2 hyp/thread, 1 packed FFMA2 4 hyp/thread, ... see score.cu) */
    SFMB200_OPT_TRI_INLIERS_ONLY = 3, /* 0 (default, reference: all N points, sfm.cu:309-336); 1: inliers of E only */
    SFMB200_OPT_HYP_SOLVER = 5,    /* null vector of the 8x9 design matrix: 0 register-resident 9x9 Jacobi eigensolve +
                                      design-row refinement; 1 (default) 8x8 Cholesky projector: same measured
                                      accuracy, 3.5-4.4x faster on B200 (see hyp_solver.cuh, DESIGN.md 3.2) */
    SFMB200_OPT_PROFILE = 4,       /* 1: record CUDA events between the stages of run_device / run_host
                                      (the reference's unused PerformanceTimer, common.h:48-132, done per stage) */
    SFMB200_OPT_BA_PERSISTENT = 6, /* bundle adjustment: 1 (default) all LM iterations of a round in one cooperative
                                      launch when the grid is resident; 0: two launches per iteration (same bits) */
    SFMB200_OPT_SMALL_PATH = 7,    /* fused single-launch path for small problems (one thread-block cluster per pair runs
                                      ingest, hypothesis generation, scoring + arg-max, poses, cheirality and
                                      triangulation; same bits as the five-launch path): -1 (default) when n * H is at most
                                      SFMB200_OPT_SMALL_PATH_EVALS, 0 never, 1 whenever eligible (projector solver,
                                      H <= 128 * cluster size, reference pose semantics, no per-stage profiling) */
    SFMB200_OPT_SMALL_PATH_EVALS = 8, /* the n * H limit of the automatic choice (default 2,500,000; the automatic choice also needs <= 4 pairs per handle) */
    SFMB200_OPT_SAMPLER = 10,      /* sample rows drawn on the device (d_idx == NULL): 0 (default) 8 distinct indices per hypothesis,
                                      independent between hypotheses; 1 the reference's scheme (sfm.cu:95-104): ONE
                                      permutation of the point indices cut into disjoint groups of 8, which needs
                                      8 * H_total <= n (H = N / 8 is the reference's own choice) */
    SFMB200_OPT_SCORE_METRIC = 9   /* inlier test of the essential-matrix model, used by scoring and by every later
                                      classifier (mask, refit, cheirality vote, bundle adjustment, chaining): 0 (default)
                                      Sampson error, what BASELINE's north_star mandates; 1 symmetric epipolar distance
                                      n^2 (1/|(E x2)_01|^2 + 1/|(E^T x1)_01|^2) < thr, what the reference's calculateInliers was
                                      written to compute (sfm.cu:155-221, SURVEY Q14) */
} sfmb200_option;

const char* sfmb200_last_error(void);
int sfmb200_version(void);
/* "src=<hash> nvcc_flags=<...>": hash of the sources this library was compiled from (cuda-sfm_b200/build.py: source_hash) */
const char* sfmb200_build_info(void);

/* ---- handle state ----
 * A handle remembers which stages have run: a stage called before its prerequisite returns SFMB200_ERR_STATE (triangulate
 * before the poses, poses before an estimate, chain / global bundle adjustment before chain_views ...).  What a call leaves:
 *   set_points_*            new correspondences; a previous E / pose stays usable (e.g. triangulate other matches with a known
 *                           pose), the chained reconstruction does not
 *   estimate_e* / run_*     an essential-matrix estimate (run_*: also poses, pose index, points); chained reconstruction dropped
 *   refine_e                a new E: pose_candidates / choose_pose / triangulate must run again before the stages that need a pose
 *   bundle_adjust           refined E, selected pose and points, consistent with each other (chain_views may follow directly)
 *   find_homography         a HOMOGRAPHY in place of E: the pose stages refuse it until the next estimate_e* / run_*
 * Whatever ran before, estimate_e* / run_* give the bits a fresh handle gives (tests/test_gpu_edge_8f.py). */

/* ---- lifetime: SfM::Image_pair::Image_pair / ~Image_pair (SfM/sfm.cu:28-78, 346-359) ---- */
/* K, Kinv: host 3x3 row-major, as src/main.cpp:292-297 builds them. */
int sfmb200_create(const float h_K[9], const float h_Kinv[9], int pairs, int max_points, int max_hypotheses,
                   sfmb200_t** out);
int sfmb200_destroy(sfmb200_t* h);
int sfmb200_set_option(sfmb200_t* h, int option, int value);
/* cudaStream_t to enqueue on (default: a private non-blocking stream). */
int sfmb200_set_stream(sfmb200_t* h, void* cuda_stream);
int sfmb200_synchronize(sfmb200_t* h);

/* ---- ingest: Image_pair::fillXU (SfM/sfm.cu:80-92; kernels::copy_point kernels.h:261-279) ---- */
/* d_sift: device array of n CudaSift SiftPoint structs (576 B each, CudaSift/cudaSift.h:6-22). pairs must be 1. */
int sfmb200_set_points_sift(sfmb200_t* h, const void* d_sift, int n);
/* Same with match filtering (not in the reference, which feeds every match unfiltered: main.cpp:298-299,
 * 283-290; SURVEY.md 8f rank 1): keeps SiftPoint i iff score > min_score && ambiguity < max_ambiguity (the
 * test of CudaSift's FindHomography, matching.cu:1035), compacted in original order.  d_kept_index (device
 * int32 [n], nullable) receives the original index of every kept correspondence; *h_kept their number.
 * SFMB200_ERR_STATE when fewer than 8 survive.  Synchronises (the count sizes the later launches). */
int sfmb200_set_points_sift_filtered(sfmb200_t* h, const void* d_sift, int n, float min_score, float max_ambiguity,
                                     int32_t* d_kept_index, int32_t* h_kept);
/* d_px: device [pairs][n][4] pixel coordinates (u1, v1, u2, v2). */
int sfmb200_set_points_xy(sfmb200_t* h, const float* d_px, int n);
/* same from host memory (pinned or pageable); copied on the handle's stream. */
int sfmb200_set_points_xy_host(sfmb200_t* h, const float* h_px, int n);
/* already normalised camera coordinates (x1, y1, x2, y2), device [pairs][n][4]. */
int sfmb200_set_points_normalised(sfmb200_t* h, const float* d_x, int n);

/* ---- batches with a different number of correspondences per pair ----
 * d_px / h_px: PACKED pixel rows (u1, v1, u2, v2), [offsets[pairs]][4]; pair b owns rows [offsets[b], offsets[b+1]).
 * h_offsets: HOST int32 [pairs + 1], offsets[0] == 0, every count offsets[b+1] - offsets[b] in [8, max_points].
 * Contract: pair b of a ragged batch gives the same bits as a one-pair handle holding only pair b's rows
 * (n = count_b) with the batch's per-pair seed, seed + 0x632BE59BD9B4E019 * b (mod 2^64): inlier counts, best index
 * and count, E, the four poses and the pose index, the points of its count_b rows and the inlier mask.
 * Mode: a handle whose last ingest was *_ragged is in per-pair-count mode whatever the counts are; any uniform ingest
 * (set_points_*, run_device, run_host) returns it to uniform mode.  In per-pair-count mode:
 *  - estimate_e / _slice / _adaptive, pose_candidates, choose_pose, triangulate, both score metrics, every scoring
 *    variant and every getter accept the points; the adaptive bound uses w = count / count_b;
 *  - caller-supplied sample rows keep the [pairs][H_total][8] layout; a row with an index >= count_b is degenerate
 *    (E = 0, count 0); the disjoint sampler (option 10 = 1) needs 8 * H_total <= the smallest count;
 *  - per-pair getters (get_points*, get_X, get_inlier_mask, copy_to_vbo*) return count_b entries for pair b;
 *    device_views keeps point_stride, and rows at or beyond count_b are unspecified there;
 *  - refine_e, bundle_adjust, chain_views, bundle_adjust_global, find_homography, estimate_e_mg and adopt_best return
 *    SFMB200_ERR_STATE; the fused small path (option 7) is never taken.
 * Every argument is checked before anything is enqueued; a refused call leaves the handle as it was.
 * run_host_ragged: host buffers as run_host; h_points is packed like the input: pair b's [4][count_b] block starts at
 * float 4 * offsets[b].  E, P, pose index and inliers are [pairs] arrays as in run_host. */
int sfmb200_set_points_xy_ragged(sfmb200_t* h, const float* d_px, const int32_t* h_offsets);
int sfmb200_run_device_ragged(sfmb200_t* h, const float* d_px, const int32_t* h_offsets, int H, uint64_t seed, float thr);
int sfmb200_run_host_ragged(sfmb200_t* h, const float* h_px, const int32_t* h_offsets, int H, uint64_t seed, float thr,
                            float* h_E, float* h_P, int32_t* h_pose_index, int32_t* h_inliers, float* h_points);
/* correspondences per pair of the current points (uniform mode: n for every pair) */
int sfmb200_get_point_counts(sfmb200_t* h, int32_t* h_counts /* [pairs] */);

/* ---- RANSAC: Image_pair::estimateE (SfM/sfm.cu:94-153) + calculateInliers (155-236) ----
 * H hypotheses per pair.  d_idx: device int32 [pairs][H_total][8] sample rows
 * (the reference's shuffled `indices`, sfm.cu:97-106, generalised), or NULL to
 * draw them on the device from `seed` (counter-based, reproducible on any GPU).
 * thr: Sampson threshold in normalised coordinates (reference literal 1e-6,
 * sfm.cu:220).  Hypotheses [h_begin, h_begin + H) of H_total are generated and
 * scored by this handle: h_begin > 0 is the multi-GPU hypothesis-slice case. */
int sfmb200_estimate_e(sfmb200_t* h, const int32_t* d_idx, int H, uint64_t seed, float thr);
int sfmb200_estimate_e_slice(sfmb200_t* h, const int32_t* d_idx, int H_total, int h_begin, int H, uint64_t seed,
                             float thr);
/* RANSAC with adaptive termination (SURVEY.md 8f rank 2; "limit on RANSAC iterations" is
 * listed as future work in the reference's README.md:65-69).  Hypotheses are tried in
 * rounds [0, first_round), [first_round, first_round*growth), ... up to H_max; after each
 * round the usual bound  needed = log(1 - confidence) / log(1 - w^8),  w = best inlier ratio,
 * is evaluated on the device for every pair, and once the hypotheses tried reach it for all
 * pairs the remaining rounds are skipped on the device (no host synchronisation between
 * rounds).  *h_used (optional; forces one stream synchronisation) = hypotheses tried.
 * The selected E, index and count are exactly those of sfmb200_estimate_e over the first
 * `used` hypotheses.  d_idx: NULL or int32 [pairs][H_max][8].  Afterwards the per-hypothesis
 * getters (get_inlier_counts, get_E_candidates) are not available. */
int sfmb200_estimate_e_adaptive(sfmb200_t* h, const int32_t* d_idx, int H_max, int first_round, int growth,
                                uint64_t seed, float thr, float confidence, int32_t* h_used);
/* ---- multi-GPU without a collective library on the data path (one process per GPU, one NVLink box) ----
 * The exchange step of the hypothesis-sharded estimate is one 8-byte key per pair.  Instead of an
 * all-reduce every rank pushes its key into every peer's exchange buffer with a system-scope atomicMax over
 * peer memory together with the E of its local winner, counts arrivals, and reads the global winner's E from
 * the slot of the rank that owns the winning index (nothing is regenerated, nothing returns to the host).  Set-up: every rank calls sfmb200_mg_init
 * (which returns an opaque handle of sfmb200_mg_handle_bytes() bytes: a CUDA IPC memory handle), the ranks
 * exchange those handles by any means (the Python mirror uses torch.distributed.all_gather, once), and every
 * rank calls sfmb200_mg_connect with the world x bytes table indexed by rank.  Then sfmb200_estimate_e_mg,
 * called by every rank with the same arguments on the same correspondences, equals sfmb200_estimate_e over
 * all H_total hypotheses bit for bit.  The devices must support native P2P atomics with each other (NVLink):
 * sfmb200_mg_connect checks cudaDevP2PAttrNativeAtomicSupported and refuses otherwise.  Waits are bounded (~2 s,
 * sfmb200_mg_set_timeout_ms).  A wait that times out (lost or late peer) POISONS the exchange on that rank: the call
 * publishes no result (inlier count 0, E = 0), the rank stops publishing (so its peers time out too), every later
 * sfmb200_estimate_e_mg returns SFMB200_ERR_STATE, and sfmb200_mg_status returns the number of calls that timed out
 * (0 in a healthy job) until every rank reconnects: sfmb200_mg_close + sfmb200_mg_init + sfmb200_mg_connect. */
int sfmb200_mg_handle_bytes(void);
int sfmb200_mg_init(sfmb200_t* h, int rank, int world, void* h_handle_out);
int sfmb200_mg_connect(sfmb200_t* h, const void* h_handles);
int sfmb200_estimate_e_mg(sfmb200_t* h, const int32_t* d_idx, int H_total, uint64_t seed, float thr);
int sfmb200_mg_status(sfmb200_t* h, int32_t* h_timeouts);
/* bound of the exchange wait (default ~2000 ms) */
int sfmb200_mg_set_timeout_ms(sfmb200_t* h, int ms);
int sfmb200_mg_close(sfmb200_t* h);
/* Device pointer to the per-pair packed winners, uint64 [pairs]:
 * (count << 32) | (0xFFFFFFFF - global hypothesis index).  Multi-GPU: all-reduce
 * this buffer with MAX over ranks (8 bytes per pair), then call
 * sfmb200_adopt_best, which regenerates the winning E from its index. */
int sfmb200_best_buffer(sfmb200_t* h, uint64_t** d_best);
int sfmb200_adopt_best(sfmb200_t* h, const int32_t* d_idx, int H_total, uint64_t seed);

/* ---- homography RANSAC (SURVEY.md 8f rank 3): CudaSift's FindHomography (CudaSift/cudaSift.h:43,
 * matching.cu:1000-1087; the outlier pre-filter the reference's main.cpp:283-290 has commented out) on the
 * same hypothesis / scoring skeleton.  `loops` 4-point hypotheses per pair (device-drawn from `seed`), one-sided
 * transfer error of image-1 -> image-2 points under H below `thresh` (same division-free test as
 * TestHomographies, matching.cu:953-996), first maximum wins.  `thresh` is in PIXELS and h_H maps image-1 PIXELS
 * to image-2 pixels, like CudaSift's, whatever K the handle was created with: the test runs on the handle's
 * normalised coordinates with thresh / f and the winner is returned as K H K^-1.  That is exact for
 * K = [f 0 cx; 0 f cy; 0 0 1] (square pixels, no skew - the reference's K, main.cpp:292-294, and K = I); any
 * other K returns SFMB200_ERR_ARG.  h_H: host [pairs][9] row-major with h8 = 1 like CudaSift; h_matches: inlier
 * counts.  Afterwards get_inlier_mask / get_inlier_counts / get_best refer to the homography. */
int sfmb200_find_homography(sfmb200_t* h, int loops, uint64_t seed, float thresh, float* h_H, int32_t* h_matches);

/* ---- local optimisation (not in the reference; its README.md:65-69 lists it as future work,
 * SURVEY.md 8f rank 2): up to `iterations` rounds of { normalised 8-point fit on ALL inliers of
 * the current E through the 9x9 Jacobi eigensolve, rank-2 projection, re-score }, each accepted
 * only if it has more inliers.  Updates E and the inlier count in place; call after estimate_e. */
int sfmb200_refine_e(sfmb200_t* h, int iterations);

/* Two-view bundle adjustment with inlier re-selection (SURVEY.md 8f rank 4; "bundle
 * adjustment" is future work in the reference's README.md:65-69).  Needs a chosen pose.
 * Refines the selected camera-2 matrix P[pose_index] (x1 ~ X, x2 ~ P X: the convention of
 * linear_triangulation, sfm.cu:309-336) and the 3-D points of the inliers by Levenberg-
 * Marquardt on the reprojection error in normalised coordinates; camera 1 stays [I|0], the
 * gauge is |t| = 1.  Each of the `outer_rounds` rounds: inliers of the current E (same test
 * and threshold as the estimate) that triangulate in front of both cameras -> `iterations`
 * LM steps (point blocks eliminated by a Schur complement, 6x6 camera system) -> the essential
 * matrix of the adjusted camera is scored; if it still explains at least 95 % of the correspondences
 * the model had when this function was called the camera replaces P[pose_index], its E replaces E, the inlier count
 * replaces the best count and the adjusted points replace the triangulated ones of the active
 * correspondences; in either case the whole cloud is re-triangulated under the camera in place.
 * Everything is enqueued on the handle's stream.  h_stats: NULL or host float [pairs][8] of the
 * LAST round (forces a synchronise): active points, cost at entry, cost at exit (sum of squared
 * residuals), accepted steps, lambda, gauge scale, inliers of the adjusted model, committed (1 / 0). */
int sfmb200_bundle_adjust(sfmb200_t* h, int outer_rounds, int iterations, float* h_stats);
/* N-view chaining (SURVEY.md 8f rank 4; the reference shapes Image_pair for image_count views,
 * sfm.h:23,30-31, but handles two).  The handle's pairs are CONSECUTIVE view pairs - pair b =
 * (view b, view b+1) - over index-aligned tracks: correspondence i is the same track in every
 * pair.  After every pair has an E, a chosen pose and triangulated points (and ideally
 * sfmb200_bundle_adjust), this puts them in one frame: relative scale of pair b against pair
 * b-1 = median-bin mean of the depth ratios of the tracks valid in both (valid = inlier of the
 * pair's E, point finite and in front of both cameras); cameras G_0 = [I|0],
 * G_{b+1} = [R_b | S_b t_b] G_b in units of the first baseline; cloud = per track the mean over
 * the pairs where it is valid of G_b^-1 (S_b X_b).  At most 256 pairs.
 * d_cloud: NULL or device float [4][n] SoA (x,y,z,1; zeros when no pair sees the track);
 * d_count: NULL or device int32 [n] pairs that saw the track; h_cameras: NULL or host float
 * [pairs+1][12] row-major 3x4; h_scales: NULL or host float [pairs]; h_used: NULL or host int32
 * [pairs] tracks that linked pair b-1 and b.  Host outputs force a synchronise. */
int sfmb200_chain_views(sfmb200_t* h, float* d_cloud, int32_t* d_count, float* h_cameras, float* h_scales, int32_t* h_used);
/* Global bundle adjustment over the chained reconstruction (SURVEY.md 8f rank 4; README.md:65-69 lists bundle adjustment and more
 * views as future work): Levenberg-Marquardt on the reprojection error of EVERY observation - track i in view k, for the views
 * of the pairs in which the track is valid - over all cameras but the first (rotation + translation; camera 0 stays [I|0]) and
 * one 3-D point per track seen by at least two views.  Point blocks are eliminated; the reduced camera system (6 x pairs
 * unknowns) is assembled per camera pair and solved on the device by a Cholesky factorisation; a step is accepted on strict
 * decrease with every observation still in front of its camera (lambda / 3, else 4 lambda); the gauge (|t_1|) is restored at
 * the end.  Call after sfmb200_chain_views with the d_cloud / d_count of that call: d_cloud (device [4][n]) is updated in place
 * for the adjusted tracks, the chain's cameras are replaced.  At most 16 pairs.  h_cameras: NULL or host float [pairs+1][12]
 * row-major 3x4; h_stats: NULL or host float [8]: cost at entry, cost at exit (sum of squared residuals, normalised
 * coordinates), accepted steps, lambda, gauge scale, iterations run.  Host outputs force a synchronise. */
int sfmb200_bundle_adjust_global(sfmb200_t* h, float* d_cloud, const int32_t* d_count, int iterations, float* h_cameras,
                                 float* h_stats);
int sfmb200_get_refit_iterations(sfmb200_t* h, int32_t* h_accepted /* [pairs] */);

/* ---- poses: computePosecandidates (sfm.cu:238-252), choosePose (254-307) ---- */
int sfmb200_pose_candidates(sfmb200_t* h);
int sfmb200_choose_pose(sfmb200_t* h);
/* ---- linear_triangulation (sfm.cu:309-344) ---- */
int sfmb200_triangulate(sfmb200_t* h);
/* Whole path for host callers: H2D of pixel correspondences, every stage, D2H
 * of E [pairs][9], P (selected pose) [pairs][16], pose index [pairs], inlier
 * count [pairs] and, if h_points != NULL, points [pairs][4][n].  One stream
 * synchronisation at the end. */
/* Page-locked h_px / h_points (cudaHostAlloc, cudaHostRegister, torch pin_memory) of up to 4 MB are read and
 * written by the kernels directly through their device-visible aliases (no staging copies: the call is
 * latency bound at those sizes); larger or pageable buffers go through the copy engines. */
int sfmb200_run_host(sfmb200_t* h, const float* h_px, int n, int H, uint64_t seed, float thr, float* h_E, float* h_P,
                     int32_t* h_pose_index, int32_t* h_inliers, float* h_points);
/* Same with device-resident input, no output copies (results stay on the device). */
int sfmb200_run_device(sfmb200_t* h, const float* d_px, int n, int H, uint64_t seed, float thr);

/* ---- egress: copyBoidsToVBO (sfm.cu:374-383) ---- */
/* pos / col: device [n][4]; either may be NULL.  Synchronises like the reference. */
int sfmb200_copy_to_vbo(sfmb200_t* h, int pair, float* d_pos, float* d_col);
/* Same with a position scale (kernCopyPositionsToVBO's s_scale, kernels.h:471) and per-point colours
 * (SURVEY.md 8f rank 4; the reference writes ones, kernels.h:485-495).  mode 0: ones; 1: inliers of the
 * selected E (0,1,0,1), others (1,0,0,1); 2: depth ramp (t,0,1-t,1), t = clamp((z - z_near) / (z_far - z_near)),
 * for points with z > 0, grey (0.5,0.5,0.5,1) otherwise. */
int sfmb200_copy_to_vbo_coloured(sfmb200_t* h, int pair, float* d_pos, float* d_col, float scale, int mode, float z_near,
                                 float z_far);

/* ---- getters (the reference keeps these members private, sfm.h:21-41) ---- */
int sfmb200_get_E(sfmb200_t* h, float* h_E /* [pairs][9] */);
int sfmb200_set_E(sfmb200_t* h, const float* h_E /* [pairs][9] */);   /* inject E (parity harness) */
int sfmb200_get_best(sfmb200_t* h, int32_t* h_index, int32_t* h_count /* [pairs] each */);
int sfmb200_get_poses(sfmb200_t* h, float* h_P /* [pairs][4][16] */);
int sfmb200_get_pose_index(sfmb200_t* h, int32_t* h_ind /* [pairs] */);
int sfmb200_get_points(sfmb200_t* h, int pair, float* d_points /* device [4][n] */);
int sfmb200_get_points_host(sfmb200_t* h, int pair, float* h_points /* [4][n] */);
int sfmb200_get_inlier_counts(sfmb200_t* h, int pair, int32_t* d_counts /* device [H] */);
int sfmb200_get_E_candidates(sfmb200_t* h, int pair, float* d_E /* device [H][9] */);
int sfmb200_get_X(sfmb200_t* h, int pair, int image, float* d_X /* device [3][n] */);
int sfmb200_get_inlier_mask(sfmb200_t* h, int pair, uint8_t* d_mask /* device [n] */);
/* Raw device views for zero-copy consumers (valid until destroy). */
int sfmb200_device_views(sfmb200_t* h, float** d_E, float** d_P, int32_t** d_pose_index, float** d_points,
                         int* point_stride);
/* how the last estimate was launched: kernel variant, hypothesis tiles per pair, persistent CTAs, hypotheses per CTA */
int sfmb200_score_plan(sfmb200_t* h, int32_t out[4]);
/* kernels launched by this handle since creation (bench.py's gpu_launches) */
int64_t sfmb200_launch_count(sfmb200_t* h);
/* SFMB200_OPT_PROFILE: device time of the 7 stages (ingest, hypgen, score, select,
 * pose candidates, choose pose, triangulate) of the most recent run_* calls, oldest
 * first, ms [sets][7]; synchronises the stream. */
int sfmb200_stage_times(sfmb200_t* h, int max_sets, float* h_ms, int* sets);

/* ---- measurement helpers ---- */
/* FP32-pipe probe: runs `iters` iterations of an FFMA (mode 0), FFMA2 (mode 1), FMUL2 (2), FADD2 (3) or FFMA2-with-a-negated-
 * register-operand (4) stream on all SMs; returns lane operations executed in *fmas and device time in *ms. */
int sfmb200_fma_probe(int mode, int iters, double* fmas, float* ms);

/* measurement hook for the fused small-problem kernel: device int64 [16] receiving clock64() of pair 0 / CTA 0 at its phase
 * boundaries (slots 0..5: start, ingest, hypgen, scoring, pose, triangulation) and inside the scoring / pose phases (8..14);
 * NULL switches it off */
int sfmb200_small_path_debug(int64_t* d_stamps);

/* ---- host-side small-matrix entry points (no GPU): svd.h facade + CPU tests ---- */
void sfmb200_host_svd3(const float a[9], float u[9], float s[9], float v[9]);
/* same decomposition with the one discrete freedom of the contract (the sign of v3, which orders the four pose
 * candidates) fixed the way the reference's own svd() (SfM/svd.h:311-335) fixes it; used by the compat pose stage */
void sfmb200_host_svd3_reference_orientation(const float a[9], float u[9], float s[9], float v[9]);
void sfmb200_host_solve_hypothesis(const float pts[32], float E[9]);            /* 9x9 Jacobi eigensolve */
void sfmb200_host_solve_hypothesis_projector(const float pts[32], float E[9]);  /* 8x8 Cholesky projector */
void sfmb200_host_null4(const float A[16], float x[4]);
/* inverse-iteration fast path of the same null vector; returns 1 when it did not converge (caller falls back) */
int sfmb200_host_null4_fast(const float A[16], float x[4]);
/* null vector of a two-view DLT matrix (rows 0, 1 = camera 1 = I4: (-1,0,x1,0), (0,-1,y1,0)) by the adjugate power
 * iteration the triangulation kernel uses; returns 1 when it did not converge (caller falls back to null4) */
int sfmb200_host_dlt_null(const float A[16], float x[4]);
/* the fixed four-step form the triangulation kernel uses (direction only, not normalised; zeros for degenerate input) */
void sfmb200_host_dlt_null_power4(const float A[16], float x[4]);
int sfmb200_host_inv4(const float m[16], float out[16]);
void sfmb200_host_sample_indices(uint64_t seed, uint64_t h, int n, int32_t idx[8]);
void sfmb200_host_sample_indices_disjoint(uint64_t seed, uint64_t h, int n, int32_t idx[8]);   /* SFMB200_OPT_SAMPLER = 1 */

#ifdef __cplusplus
}
#endif
#endif /* SFMB200_H */
