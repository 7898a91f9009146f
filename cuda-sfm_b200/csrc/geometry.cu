// Ingest (fillXU), pose candidates, cheirality pose selection, linear
// triangulation and egress.  Reference: SfM/sfm.cu:80-92, 238-344, 374-383 and
// SfM/kernels.h:261-279, 357-450, 471-495.
#include "geometry.cuh"

namespace sfmb200 {

// SiftPoint is 576 bytes (CudaSift/cudaSift.h:6-22); only xpos@0, ypos@4,
// match_xpos@36, match_ypos@40 are read (kernels.h:268-273).
constexpr int SIFT_STRIDE_F = 144;
__global__ void ingest_sift_kernel(DeviceState s, const float* __restrict__ sift, int n, Mat9 k) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = sift + (size_t)i * SIFT_STRIDE_F;
    float2 a = __ldg(reinterpret_cast<const float2*>(p));
    float u2 = __ldg(p + 9), v2 = __ldg(p + 10);
    normalise_store(s, 0, i, a.x, a.y, u2, v2, k);
}
__global__ void ingest_xy_kernel(DeviceState s, const float4* __restrict__ px, int n, Mat9 k) {
    pdl_trigger();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y;
    if (i >= n) return;
    float4 p = __ldg(px + (size_t)b * n + i);
    normalise_store(s, b, i, p.x, p.y, p.z, p.w, k);
}
// Packed rows: pair b's s.n_pair[b] rows start at row row_off[b].
__global__ void ingest_xy_ragged_kernel(DeviceState s, const float4* __restrict__ px, const int* __restrict__ row_off, Mat9 k) {
    pdl_trigger();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y;
    if (i >= s.n_pair[b]) return;
    float4 p = __ldg(px + (size_t)row_off[b] + i);
    normalise_store(s, b, i, p.x, p.y, p.z, p.w, k);
}
// ---------------------------------------------------------------------------
// Ingest with match filtering (SURVEY.md 8f rank 1).  The reference feeds every
// SIFT point of image 1 to the estimator unfiltered (main.cpp:298-299; its
// homography pre-filter is commented out, main.cpp:283-290).  This keeps a match
// iff score > min_score && ambiguity < max_ambiguity - the test CudaSift's own
// FindHomography applies (CudaSift/matching.cu:1035) - and compacts the
// survivors in their original order (deterministic): per-CTA counts, a
// single-CTA scan, then an ordered scatter fused with the K^-1 normalisation.
// SiftPoint: score @ float 6, ambiguity @ float 7 (CudaSift/cudaSift.h:6-22).
// ---------------------------------------------------------------------------
constexpr int FILTER_THREADS = 256;
__device__ __forceinline__ bool sift_keep(const float* p, float min_score, float max_ambiguity) {
    return __ldg(p + 6) > min_score && __ldg(p + 7) < max_ambiguity;
}
__global__ void __launch_bounds__(FILTER_THREADS)
sift_filter_count_kernel(const float* __restrict__ sift, int n, float min_score, float max_ambiguity, int* block_counts) {
    int i = blockIdx.x * FILTER_THREADS + threadIdx.x;
    bool keep = i < n && sift_keep(sift + (size_t)i * SIFT_STRIDE_F, min_score, max_ambiguity);
    int c = __syncthreads_count(keep);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = c;
}
// exclusive scan of nblocks counts in place; total -> counts[nblocks]
__global__ void sift_filter_scan_kernel(int* counts, int nblocks) {
    __shared__ int carry;
    __shared__ int warp_sums[32];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nblocks; base += 1024) {
        int i = base + threadIdx.x;
        int v = i < nblocks ? counts[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if ((threadIdx.x & 31) >= o) x += y;
        }
        if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = x;
        __syncthreads();
        if (threadIdx.x < 32) {
            int w = warp_sums[threadIdx.x], z = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xFFFFFFFFu, z, o);
                if (threadIdx.x >= o) z += y;
            }
            warp_sums[threadIdx.x] = z - w;          // exclusive warp offsets
        }
        __syncthreads();
        int excl = carry + warp_sums[threadIdx.x >> 5] + x - v;
        if (i < nblocks) counts[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) counts[nblocks] = carry;
}
__global__ void __launch_bounds__(FILTER_THREADS)
sift_filter_scatter_kernel(DeviceState s, const float* __restrict__ sift, int n, float min_score, float max_ambiguity,
                           const int* __restrict__ block_offsets, int* kept_index, Mat9 k) {
    __shared__ int warp_counts[FILTER_THREADS / 32];
    int i = blockIdx.x * FILTER_THREADS + threadIdx.x;
    const float* p = sift + (size_t)i * SIFT_STRIDE_F;
    bool keep = i < n && sift_keep(p, min_score, max_ambiguity);
    unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_counts[warp] = __popc(m);
    __syncthreads();
    int off = block_offsets[blockIdx.x];
    for (int w = 0; w < warp; w++) off += warp_counts[w];
    if (!keep) return;
    int dst = off + __popc(m & ((1u << lane) - 1u));
    float2 a = __ldg(reinterpret_cast<const float2*>(p));
    normalise_store(s, 0, dst, a.x, a.y, __ldg(p + 9), __ldg(p + 10), k);
    if (kept_index) kept_index[dst] = i;
}
// Re-materialise the scaled copies after the threshold (or the model) changed without a new ingest.
__global__ void rescale_points_kernel(DeviceState s) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pair_n(s, blockIdx.y)) return;
    size_t o = (size_t)blockIdx.y * s.n_stride + i;
    float4 p = s.corr[o];
    store_scaled(s, o, p.x, p.y, p.z, p.w);
}
void launch_rescale_points(const DeviceState& s, cudaStream_t st) {
    rescale_points_kernel<<<dim3((s.n + 255) / 256, s.B), 256, 0, st>>>(s);
}

void launch_ingest_sift_filtered(const DeviceState& s, const void* d_sift, int n, float min_score, float max_ambiguity,
                                 int* d_scratch, int* d_kept_index, cudaStream_t st) {
    Mat9 k;
    for (int i = 0; i < 9; i++) k.v[i] = s.Kinv[i];
    int blocks = (n + FILTER_THREADS - 1) / FILTER_THREADS;
    sift_filter_count_kernel<<<blocks, FILTER_THREADS, 0, st>>>((const float*)d_sift, n, min_score, max_ambiguity, d_scratch);
    sift_filter_scan_kernel<<<1, 1024, 0, st>>>(d_scratch, blocks);
    sift_filter_scatter_kernel<<<blocks, FILTER_THREADS, 0, st>>>(s, (const float*)d_sift, n, min_score, max_ambiguity, d_scratch,
                                                                   d_kept_index, k);
}

void launch_ingest_sift(const DeviceState& s, const void* d_sift, int n, cudaStream_t st) {
    Mat9 k;
    for (int i = 0; i < 9; i++) k.v[i] = s.Kinv[i];
    ingest_sift_kernel<<<(n + 255) / 256, 256, 0, st>>>(s, (const float*)d_sift, n, k);
}
void launch_ingest_xy(const DeviceState& s, const float* d_px, int n, cudaStream_t st) {
    Mat9 k;
    for (int i = 0; i < 9; i++) k.v[i] = s.Kinv[i];
    dim3 grid((n + 255) / 256, s.B);
    ingest_xy_kernel<<<grid, 256, 0, st>>>(s, (const float4*)d_px, n, k);
}
void launch_ingest_xy_ragged(const DeviceState& s, const float* d_px, const int* d_row_off, cudaStream_t st) {
    Mat9 k;
    for (int i = 0; i < 9; i++) k.v[i] = s.Kinv[i];
    dim3 grid((s.n + 255) / 256, s.B);
    ingest_xy_ragged_kernel<<<grid, 256, 0, st>>>(s, (const float4*)d_px, d_row_off, k);
}
void launch_ingest_normalised(const DeviceState& s, const float* d_x, int n, cudaStream_t st) {
    Mat9 k = {{1, 0, 0, 0, 1, 0, 0, 0, 1}};
    dim3 grid((n + 255) / 256, s.B);
    ingest_xy_kernel<<<grid, 256, 0, st>>>(s, (const float4*)d_x, n, k);
}

// one thread per (pair, candidate)
__global__ void pose_candidates_kernel(DeviceState s, int compat) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    int b = g >> 2, c = g & 3;
    if (b >= s.B) return;
    float E[9], P[16];
#pragma unroll
    for (int i = 0; i < 9; i++) E[i] = s.E[(size_t)b * 9 + i];
    pose_candidate(E, c, compat, P);
#pragma unroll
    for (int i = 0; i < 16; i++) s.P[(size_t)b * 64 + 16 * c + i] = P[i];
}
void launch_pose_candidates(const DeviceState& s, int compat, cudaStream_t st) {
    int threads = 4 * s.B;
    pose_candidates_kernel<<<(threads + 63) / 64, 64, 0, st>>>(s, compat);
}

// ---------------------------------------------------------------------------
// choosePose (sfm.cu:254-307).
// compat = 1: cheirality of correspondence 0 only; every candidate is inverted
//   in place; depth tested in both frames; the LAST passing index wins (default
//   0); afterwards P holds the inverses (Q17-Q19).  One thread per pair.
// compat = 0: every inlier of the selected E votes (z > 0 in both cameras,
//   X2 = P_i X); arg-max of votes, first on ties; P is left untouched.
//   One 256-thread CTA per pair.
// ---------------------------------------------------------------------------
// 4 lanes per pair (one per candidate); the pairs of a warp vote with one ballot.
__global__ void choose_pose_compat_kernel(DeviceState s) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    int b = g >> 2, c = g & 3;
    bool active = b < s.B;
    bool pass = false;
    if (active) {
        float4 c0 = s.corr[(size_t)b * s.n_stride];
        float M[16], Minv[16];
#pragma unroll
        for (int i = 0; i < 16; i++) M[i] = s.P[(size_t)b * 64 + 16 * c + i];
        pass = cheirality_compat(c0, M, Minv);
#pragma unroll
        for (int i = 0; i < 16; i++) s.P[(size_t)b * 64 + 16 * c + i] = Minv[i];
    }
    unsigned m = __ballot_sync(0xFFFFFFFFu, pass);
    if (active && c == 0) {
        unsigned mine = (m >> ((threadIdx.x & 31) & ~3)) & 0xFu;
        s.P_ind[b] = mine ? 31 - __clz(mine) : 0;      // last passing index, default 0 (sfm.cu:284-297)
    }
}

// Whole-path fusion of select + pose candidates + (compat) cheirality: the three
// are each a few microseconds of latency-bound work, so as separate launches the
// gaps cost more than the math.  A CTA of two warps serves SPC_PAIRS pairs: warp 0 holds 4 lanes per pair (one pose
// candidate each: 3x3 SVD of E, candidate, cheirality), warp 1 one lane per pair for the replay of the reference's SVD
// orientation (reference_null_direction: as long a dependent chain as the SVD and independent of it), handed over through
// shared memory - the two chains run side by side instead of one after the other (small.cu does the same).
constexpr int SPC_PAIRS = 8;
__global__ void __launch_bounds__(64) select_pose_choose_kernel(DeviceState s, int h_offset, int compat) {
    pdl_wait();
    pdl_trigger();
    __shared__ float sNull[SPC_PAIRS][3];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = warp == 0 ? lane >> 2 : lane;           // pair slot inside the CTA
    const int c = lane & 3;                                   // candidate (warp 0)
    const int b = blockIdx.x * SPC_PAIRS + slot;
    const bool worker = warp == 0 && b < s.B;
    const bool helper = warp == 1 && compat && lane < SPC_PAIRS && b < s.B;
    bool pass = false;
    float E[9], P[16], u[9], sg[9], v[9];
    if (worker || helper) {
        unsigned long long packed = s.best[b];
        unsigned int hg = 0xFFFFFFFFu - (unsigned int)(packed & 0xFFFFFFFFull);
        int local = (int)hg - h_offset;
        const float* Eb = s.Ecand + (size_t)b * 9 * s.h_stride;
#pragma unroll
        for (int k = 0; k < 9; k++) E[k] = (local >= 0 && local < s.h_stride) ? Eb[(size_t)k * s.h_stride + local] : 0.0f;
        if (worker && c == 0) {
            s.best_idx[b] = (int)hg;
            s.best_count[b] = (int)(packed >> 32);
#pragma unroll
            for (int k = 0; k < 9; k++) s.E[(size_t)b * 9 + k] = E[k];
        }
        if (helper) {
            float r[3];
            reference_null_direction(E, r);
            sNull[slot][0] = r[0]; sNull[slot][1] = r[1]; sNull[slot][2] = r[2];
        } else {
            svd3<5>(E, u, sg, v);
        }
    }
    __syncthreads();
    if (worker) {
        if (compat) {
            const float r[3] = {sNull[slot][0], sNull[slot][1], sNull[slot][2]};
            svd3_orient(r, u, sg, v);
        }
        pose_from_svd(u, v, c, compat, P);
        if (compat) {
            float4 c0 = s.corr[(size_t)b * s.n_stride];
            float Minv[16];
            pass = cheirality_compat(c0, P, Minv);
#pragma unroll
            for (int i = 0; i < 16; i++) P[i] = Minv[i];
        }
#pragma unroll
        for (int i = 0; i < 16; i++) s.P[(size_t)b * 64 + 16 * c + i] = P[i];
    }
    if (warp == 0) {
        unsigned m = __ballot_sync(0xFFFFFFFFu, pass);
        if (worker && c == 0 && compat) {
            unsigned mine = (m >> (lane & ~3)) & 0xFu;
            s.P_ind[b] = mine ? 31 - __clz(mine) : 0;
        }
    }
}
void launch_select_pose_choose(const DeviceState& s, int h_offset, int compat, cudaStream_t st) {
    launch_dep(select_pose_choose_kernel, dim3((s.B + SPC_PAIRS - 1) / SPC_PAIRS), dim3(64), 0, st, s, h_offset, compat);
}

// compat = 0: every inlier of the selected E votes for the candidates that put it in front of both cameras.
// Grid over the correspondences (one thread per point, null vector by inverse iteration like the triangulation),
// integer vote counters per pair, the last CTA of a pair picks the arg-max (first on ties) and clears the scratch.
__global__ void __launch_bounds__(256) choose_pose_vote_kernel(DeviceState s, float thr) {
    const int b = blockIdx.y;
    __shared__ float sP[64];
    __shared__ float sE[9];
    __shared__ int s_last;
    if (threadIdx.x < 64) sP[threadIdx.x] = s.P[(size_t)b * 64 + threadIdx.x];
    if (threadIdx.x < 9) sE[threadIdx.x] = s.E[(size_t)b * 9 + threadIdx.x];
    __syncthreads();
    int local[4] = {0, 0, 0, 0};
    const float4* corr = s.corr + (size_t)b * s.n_stride;
    const int n = pair_n(s, b);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 p = corr[i];
        if (epipolar_d(s.metric, sE, p.x, p.y, p.z, p.w, -thr) >= 0.0f) continue;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            float A[16], v[4];
            dlt_matrix(p.x, p.y, p.z, p.w, sP + 16 * c, A);
            if (!dlt_null_adjugate1(A, v)) null4<5>(A, v);
            float X, Y, Z;
            dehomogenise(v, X, Y, Z);
            const float* M = sP + 16 * c;
            float z2 = fmaf(M[8], X, fmaf(M[9], Y, fmaf(M[10], Z, M[11])));
            local[c] += (Z > 0.0f && z2 > 0.0f) ? 1 : 0;
        }
    }
    int* votes = s.vote + (size_t)b * 8;          // [0..3] votes, [4] ticket
#pragma unroll
    for (int c = 0; c < 4; c++) {
        int v = local[c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&votes[c], v);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&votes[4], 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    int best = 0, vb = __ldcg(&votes[0]);
    for (int c = 1; c < 4; c++) {
        int vc = __ldcg(&votes[c]);
        if (vc > vb) { vb = vc; best = c; }
    }
    s.P_ind[b] = best;
    for (int c = 0; c < 5; c++) votes[c] = 0;     // clean for the next call
}
void launch_choose_pose(const DeviceState& s, int compat, float thr, cudaStream_t st) {
    if (compat)
        choose_pose_compat_kernel<<<(4 * s.B + 63) / 64, 64, 0, st>>>(s);
    else
    {
        int nb = (s.n + 255) / 256;
        int cap = (1184 + s.B - 1) / s.B;                  // ~8 CTAs per SM over the whole batch
        if (nb > cap) nb = cap < 1 ? 1 : cap;
        choose_pose_vote_kernel<<<dim3(nb, s.B), 256, 0, st>>>(s, thr);
    }
}

// ---------------------------------------------------------------------------
// Linear triangulation (sfm.cu:309-344): 4x4 DLT null vector per correspondence in registers (replaces the
// batched 4x4 cusolver gesvdj that writes U, S and V for every point), de-homogenised into the reference's
// 4xN SoA.  HBM roofline: 16 B read + 16 B written per point.
// One thread solves PTS points that lie THREADS apart (every load / store is warp-coalesced); the null vector
// comes from four power-iteration steps on the adjugate (dlt_null_power4, smallmat.cuh), which exploits camera 1 = I4
// and needs no convergence bookkeeping; the pose and E are read through uniform __ldg (one L1 line for the whole
// CTA), so there is no shared memory and no barrier.  inliers_only: points failing the Sampson test of the selected E
// get (0,0,0,1).
// ---------------------------------------------------------------------------
#ifndef SFMB200_TRI_PTS
#define SFMB200_TRI_PTS 2
#endif
#ifndef SFMB200_TRI_THREADS
#define SFMB200_TRI_THREADS 128
#endif
constexpr int TRI_THREADS = SFMB200_TRI_THREADS;
#ifndef SFMB200_TRI_MINB
#define SFMB200_TRI_MINB 8      // resident CTAs per SM the kernel is compiled for (<= 64 registers at 128 threads)
#endif
// RAGGED: per-pair counts.  A compile-time case so that the uniform kernel keeps its bound in the constant bank: at the
// 64-register cap one more live register spills.
template <int PTS, bool INLIERS_ONLY, bool RAGGED>
__global__ void __launch_bounds__(TRI_THREADS, SFMB200_TRI_MINB) triangulate_kernel(DeviceState s, float thr) {
    static_assert(PTS == 1 || PTS == 2, "one point per thread, or two in packed f32x2 arithmetic");
    pdl_wait();
    const int b = blockIdx.y;
    // (Tried on the cold start - the selected pose sits behind its index, two dependent misses: requesting the first points
    //  before the pose: 135 vs 131 us at 16M points, no change at 1M; an L2 prefetch of the four candidates from every thread:
    //  600k requests for the same two lines serialise on one L2 slice, 26.6 us instead of 14.3 us at 1M points.)
#ifdef SFMB200_TRI_FIXED_POSE      // measurement build: candidate 0 without the dependent index load
    const float* Mg = s.P + (size_t)b * 64;
#else
    const float* Mg = s.P + (size_t)b * 64 + 16 * __ldg(s.P_ind + b);
#endif
    float M[12], e[9];
#pragma unroll
    for (int k = 0; k < 12; k++) M[k] = __ldg(Mg + k);
    if constexpr (INLIERS_ONLY) {
#pragma unroll
        for (int k = 0; k < 9; k++) e[k] = __ldg(s.E + (size_t)b * 9 + k);
    }
    // persistent over the pair's points: grid.x CTAs stride through them, the next points are in flight while the current
    // ones are solved (the loads are the only long-latency operation), the pose stays in registers
    constexpr int CHUNK = TRI_THREADS * PTS;
    const int step = gridDim.x * CHUNK, n = RAGGED ? s.n_pair[b] : s.n;
    const float4* corr = s.corr + (size_t)b * s.n_stride;
    float* out = s.points + (size_t)b * 4 * s.n_stride;
    const float4 zero4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float4 nxt[PTS];
    int i0 = blockIdx.x * CHUNK;
#pragma unroll
    for (int p = 0; p < PTS; p++) {
        const int i = i0 + p * TRI_THREADS + threadIdx.x;
        nxt[p] = i < n ? __ldg(corr + i) : zero4;
    }
    for (; i0 < n; i0 += step) {
        float4 pt[PTS];
#pragma unroll
        for (int p = 0; p < PTS; p++) {
            pt[p] = nxt[p];
            const int i = i0 + step + p * TRI_THREADS + threadIdx.x;
            nxt[p] = i < n ? __ldg(corr + i) : zero4;
        }
        float v[PTS][4];
        bool keep[PTS];
#pragma unroll
        for (int p = 0; p < PTS; p++) {
            keep[p] = true;
            if constexpr (INLIERS_ONLY) keep[p] = epipolar_d(s.metric, e, pt[p].x, pt[p].y, pt[p].z, pt[p].w, -thr) < 0.0f;
        }
        // rows 2, 3 of the DLT matrix (compute_linear_triangulation_A, kernels.h:387-431), then the null vector
        if constexpr (PTS == 2) {
            const float2 x1 = make_float2(pt[0].x, pt[1].x), y1 = make_float2(pt[0].y, pt[1].y);
            const float2 x2 = make_float2(pt[0].z, pt[1].z), y2 = make_float2(pt[0].w, pt[1].w);
            float2 a[4], bb[4], vv[4];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const float2 m2 = make_float2(M[8 + c], M[8 + c]);
                a[c] = __ffma2_rn(x2, m2, make_float2(-M[c], -M[c]));
                bb[c] = __ffma2_rn(y2, m2, make_float2(-M[4 + c], -M[4 + c]));
            }
#ifdef SFMB200_TRI_COPY_ONLY     // measurement build: the launch shape and the memory traffic without the solve (tools/tri_ab.py)
#pragma unroll
            for (int c = 0; c < 4; c++) vv[c] = __ffma2_rn(a[c], x1, __fmul2_rn(bb[c], y1));
#else
            dlt_null_power4_lanes<LaneF2>(x1, y1, a, bb, vv);
#endif
#pragma unroll
            for (int c = 0; c < 4; c++) { v[0][c] = vv[c].x; v[1][c] = vv[c].y; }
        } else {
            float a[4], bb[4];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                a[c] = fmaf(pt[0].z, M[8 + c], -M[c]);
                bb[c] = fmaf(pt[0].w, M[8 + c], -M[4 + c]);
            }
            dlt_null_power4_lanes<LaneF1>(pt[0].x, pt[0].y, a, bb, v[0]);
        }
#pragma unroll
        for (int p = 0; p < PTS; p++) {
            const int i = i0 + p * TRI_THREADS + threadIdx.x;
            if (i >= n) continue;
            float X = 0.0f, Y = 0.0f, Z = 0.0f;
            if (keep[p]) dehomogenise(v[p], X, Y, Z);
            out[i] = X;
            out[(size_t)s.n_stride + i] = Y;
            out[(size_t)2 * s.n_stride + i] = Z;
            out[(size_t)3 * s.n_stride + i] = 1.0f;
        }
    }
}
// Two ADJACENT points per thread (2j, 2j + 1) in packed f32x2: one pointer walks the correspondences, each output row
// takes one 8-byte store per thread, and the bounds live outside the loop (an odd last point goes to the scalar tail).
// Issue cost of a packed instruction on this part is two slots (tools/pipe_probe.py), so what the loop saves is its
// non-arithmetic half: addresses, predicates, operand moves.
template <bool INLIERS_ONLY>
__global__ void __launch_bounds__(TRI_THREADS, SFMB200_TRI_MINB) triangulate_pairs_kernel(DeviceState s, float thr) {
    pdl_wait();
    const int b = blockIdx.y;
    const int n = pair_n(s, b), pairs = (n + 1) >> 1;            // an odd last point rides alone in the last pair (its twin is a copy)
    const float4* corr = s.corr + (size_t)b * s.n_stride;
    float* out = s.points + (size_t)b * 4 * s.n_stride;
    int j = blockIdx.x * TRI_THREADS + threadIdx.x;
    const int jstep = gridDim.x * TRI_THREADS;
    // the first correspondences are in flight before anything waits for the pose
    const float4* src = corr + 2 * (size_t)j;
    const float4 zero4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float4 n0 = zero4, n1 = zero4;
    if (j < pairs) { n0 = __ldg(src); n1 = 2 * j + 1 < n ? __ldg(src + 1) : n0; }
    const float* Mg = s.P + (size_t)b * 64 + 16 * __ldg(s.P_ind + b);
    float M[12], e[9];
#pragma unroll
    for (int k = 0; k < 12; k++) M[k] = __ldg(Mg + k);
    if constexpr (INLIERS_ONLY) {
#pragma unroll
        for (int k = 0; k < 9; k++) e[k] = __ldg(s.E + (size_t)b * 9 + k);
    }
    const size_t row = (size_t)s.n_stride;
    float2* dst = reinterpret_cast<float2*>(out) + j;
    const float2 one2 = make_float2(1.0f, 1.0f);
    for (; j < pairs; j += jstep) {
        const float4 p0 = n0, p1 = n1;
        src += 2 * (size_t)jstep;
        const int jn = j + jstep;
        if (jn < pairs) { n0 = __ldg(src); n1 = 2 * jn + 1 < n ? __ldg(src + 1) : n0; }
        const float2 x1 = make_float2(p0.x, p1.x), y1 = make_float2(p0.y, p1.y);
        const float2 x2 = make_float2(p0.z, p1.z), y2 = make_float2(p0.w, p1.w);
        // rows 2, 3 of the DLT matrix (compute_linear_triangulation_A, kernels.h:387-431), then the null vector
        float2 a[4], bb[4], vv[4];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const float2 m2 = make_float2(M[8 + c], M[8 + c]);
            a[c] = __ffma2_rn(x2, m2, make_float2(-M[c], -M[c]));
            bb[c] = __ffma2_rn(y2, m2, make_float2(-M[4 + c], -M[4 + c]));
        }
#ifdef SFMB200_TRI_COPY_ONLY     // measurement build: the launch shape and the memory traffic without the solve (tools/tri_ab.py)
#pragma unroll
        for (int c = 0; c < 4; c++) vv[c] = __ffma2_rn(a[c], x1, __fmul2_rn(bb[c], y1));
#else
        dlt_null_power4_lanes<LaneF2>(x1, y1, a, bb, vv);
#endif
        float2 X, Y, Z;
        dehomogenise2(vv, X, Y, Z);
        if constexpr (INLIERS_ONLY) {
            if (!(epipolar_d(s.metric, e, p0.x, p0.y, p0.z, p0.w, -thr) < 0.0f)) { X.x = 0.0f; Y.x = 0.0f; Z.x = 0.0f; }
            if (!(epipolar_d(s.metric, e, p1.x, p1.y, p1.z, p1.w, -thr) < 0.0f)) { X.y = 0.0f; Y.y = 0.0f; Z.y = 0.0f; }
        }
        float* d = reinterpret_cast<float*>(dst);
        if (2 * j + 1 < n) {
            *reinterpret_cast<float2*>(d) = X;
            *reinterpret_cast<float2*>(d + row) = Y;
            *reinterpret_cast<float2*>(d + 2 * row) = Z;
            *reinterpret_cast<float2*>(d + 3 * row) = one2;
        } else {
            d[0] = X.x;
            d[row] = Y.x;
            d[2 * row] = Z.x;
            d[3 * row] = 1.0f;
        }
        dst += jstep;
    }
}
#ifndef SFMB200_TRI_CTAS_PER_SM
#define SFMB200_TRI_CTAS_PER_SM 16     // grid cap; 8 are resident at 64 registers x 128 threads, the rest start as CTAs retire (measured faster than 8)
#endif
#ifndef SFMB200_TRI_KERNEL
#define SFMB200_TRI_KERNEL 1           // 1: triangulate_kernel<SFMB200_TRI_PTS> (shipped), 2: triangulate_pairs_kernel (measured slower: profiles/r02_triangulation.md)
#endif
void launch_triangulate(const DeviceState& s, int inliers_only, float thr, cudaStream_t st) {
    int cap = (148 * SFMB200_TRI_CTAS_PER_SM + s.B - 1) / s.B;          // resident CTAs over the whole batch
    if (cap < 1) cap = 1;
#if SFMB200_TRI_KERNEL == 2
    int gx = ((s.n >> 1) + TRI_THREADS - 1) / TRI_THREADS;
    if (gx < 1) gx = 1;
    if (gx > cap) gx = cap;
    dim3 grid(gx, s.B);
    if (inliers_only)
        launch_dep(triangulate_pairs_kernel<true>, grid, dim3(TRI_THREADS), 0, st, s, thr);
    else
        launch_dep(triangulate_pairs_kernel<false>, grid, dim3(TRI_THREADS), 0, st, s, thr);
#else
    constexpr int CHUNK = TRI_THREADS * SFMB200_TRI_PTS;
    int gx = (s.n + CHUNK - 1) / CHUNK;
    if (gx > cap) gx = cap;      // (a grid of only-resident CTAs with equal shares was measured: 10.5 vs 9.8 us at 1M, 127 vs 121 us at 16M points)
    dim3 grid(gx, s.B);
    const bool ragged = s.n_pair != nullptr;
    if (inliers_only && ragged)
        launch_dep(triangulate_kernel<SFMB200_TRI_PTS, true, true>, grid, dim3(TRI_THREADS), 0, st, s, thr);
    else if (inliers_only)
        launch_dep(triangulate_kernel<SFMB200_TRI_PTS, true, false>, grid, dim3(TRI_THREADS), 0, st, s, thr);
    else if (ragged)
        launch_dep(triangulate_kernel<SFMB200_TRI_PTS, false, true>, grid, dim3(TRI_THREADS), 0, st, s, thr);
    else
        launch_dep(triangulate_kernel<SFMB200_TRI_PTS, false, false>, grid, dim3(TRI_THREADS), 0, st, s, thr);
#endif
}

// ---------------------------------------------------------------------------
// Egress and getters.
// ---------------------------------------------------------------------------
// copyBoidsToVBO (sfm.cu:374-383, kernels.h:471-495): 4xN SoA -> Nx4 AoS, colour = 1.
__global__ void vbo_kernel(DeviceState s, int pair, float4* pos, float4* col, float scale) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pair_n(s, pair)) return;
    const float* in = s.points + (size_t)pair * 4 * s.n_stride;
    if (pos) pos[i] = make_float4(in[i] * scale, in[(size_t)s.n_stride + i] * scale, in[(size_t)2 * s.n_stride + i] * scale, 1.0f);
    if (col) col[i] = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
}
// Egress with per-point colour (SURVEY 8f rank 4: "AoS VBO writer with colour"; the reference writes all
// ones, kernels.h:485-495).  mode 1: inliers of the selected E green, others red.  mode 2: depth ramp
// blue (z <= z_near) -> red (z >= z_far) for points in front of the camera, grey for the rest.
__global__ void vbo_colour_kernel(DeviceState s, int pair, float4* pos, float4* col, float scale, int mode, float thr,
                                  float z_near, float z_far) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pair_n(s, pair)) return;
    const float* in = s.points + (size_t)pair * 4 * s.n_stride;
    const float X = in[i], Y = in[(size_t)s.n_stride + i], Z = in[(size_t)2 * s.n_stride + i];
    if (pos) pos[i] = make_float4(X * scale, Y * scale, Z * scale, 1.0f);
    if (!col) return;
    float4 c = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
    if (mode == 1) {
        float e[9];
#pragma unroll
        for (int k = 0; k < 9; k++) e[k] = s.E[(size_t)pair * 9 + k];
        const float4 p = s.corr[(size_t)pair * s.n_stride + i];
        const bool inl = epipolar_d(s.metric, e, p.x, p.y, p.z, p.w, -thr) < 0.0f;
        c = inl ? make_float4(0.0f, 1.0f, 0.0f, 1.0f) : make_float4(1.0f, 0.0f, 0.0f, 1.0f);
    } else if (mode == 2) {
        if (Z > 0.0f && z_far > z_near) {
            const float t = fminf(fmaxf((Z - z_near) / (z_far - z_near), 0.0f), 1.0f);
            c = make_float4(t, 0.0f, 1.0f - t, 1.0f);
        } else {
            c = make_float4(0.5f, 0.5f, 0.5f, 1.0f);
        }
    }
    col[i] = c;
}
void launch_vbo_colour(const DeviceState& s, int pair, float* d_pos, float* d_col, float scale, int mode, float thr, float z_near,
                       float z_far, cudaStream_t st) {
    vbo_colour_kernel<<<(s.n + 255) / 256, 256, 0, st>>>(s, pair, (float4*)d_pos, (float4*)d_col, scale, mode, thr, z_near, z_far);
}
void launch_vbo(const DeviceState& s, int pair, float* d_pos, float* d_col, float scale, cudaStream_t st) {
    vbo_kernel<<<(s.n + 255) / 256, 256, 0, st>>>(s, pair, (float4*)d_pos, (float4*)d_col, scale);
}

// E candidates as the reference stores them: [H][3][3] row-major (d_E_candidate).
__global__ void export_ecand_kernel(DeviceState s, int pair, int H, float* out) {
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= H) return;
    const float* Eb = s.Ecand + (size_t)pair * 9 * s.h_stride;
#pragma unroll
    for (int k = 0; k < 9; k++) out[(size_t)h * 9 + k] = Eb[(size_t)k * s.h_stride + h];
}
void launch_export_ecand(const DeviceState& s, int pair, int H, float* d_out, cudaStream_t st) {
    export_ecand_kernel<<<(H + 255) / 256, 256, 0, st>>>(s, pair, H, d_out);
}

// X[image] as the reference stores it: 3xN row-major, rows x, y, 1 (sfm.cu:88-89).
__global__ void export_X_kernel(DeviceState s, int pair, int image, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = pair_n(s, pair);
    if (i >= n) return;
    float4 p = s.corr[(size_t)pair * s.n_stride + i];
    out[i] = image == 0 ? p.x : p.z;
    out[(size_t)n + i] = image == 0 ? p.y : p.w;
    out[(size_t)2 * n + i] = 1.0f;
}
void launch_export_X(const DeviceState& s, int pair, int image, float* d_out, cudaStream_t st) {
    export_X_kernel<<<(s.n + 255) / 256, 256, 0, st>>>(s, pair, image, d_out);
}

// model 0: Sampson test of the essential matrix in s.E; model 1: transfer-error test of the
// homography in s.E (thr = squared threshold)
__global__ void inlier_mask_kernel(DeviceState s, int pair, float thr, int model, unsigned char* mask) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pair_n(s, pair)) return;
    float e[9];
#pragma unroll
    for (int k = 0; k < 9; k++) e[k] = s.E[(size_t)pair * 9 + k];
    float4 p = s.corr[(size_t)pair * s.n_stride + i];
    float d = model == 0 ? epipolar_d(s.metric, e, p.x, p.y, p.z, p.w, -thr) : homography_d(e, p.x, p.y, p.z, p.w, -thr);
    mask[i] = d < 0.0f ? 1 : 0;
}
void launch_inlier_mask(const DeviceState& s, int pair, float thr, int model, unsigned char* d_mask, cudaStream_t st) {
    inlier_mask_kernel<<<(s.n + 255) / 256, 256, 0, st>>>(s, pair, thr, model, d_mask);
}

}  // namespace sfmb200
