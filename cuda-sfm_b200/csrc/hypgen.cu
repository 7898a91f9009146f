// Hypothesis generation: one thread = one minimal sample = one E candidate.
// See hyp_solver.cuh for the per-hypothesis math and the reference kernels it
// replaces (SfM/kernels.h:196-295, SfM/sfm.cu:107-129).
//
// Roofline: FP32 pipe / issue.  Default solver (8x8 Cholesky projector): ~3.6 k instructions per hypothesis (ncu: 7.42e6
// warp instructions for 65,536 hypotheses); the 9x9 Jacobi eigensolve: ~5 sweeps x 36 rotations x ~80 FP32 instructions
// plus Gram build / refinement / 3x3 SVD ~= 17 k.  Memory traffic is 8 gathered 16-byte correspondences (L2 hits) in and
// 36 B out.
#include "hyp_solver.cuh"
#include "internal.cuh"

#ifndef SFMB200_HYPGEN_MINB
#define SFMB200_HYPGEN_MINB 4       // resident CTAs per SM the projector kernel is compiled for (A/B: profiles/r01_variant_sweep.md;
                                    // round 2, 96 registers without spills at 5: 18.4 vs 17.8 us at config 2, 0.140 vs 0.145 ms on a config-4 slice)
#endif

namespace sfmb200 {


template <int THREADS, int MINB, int SYNC, int SOLVER>
__global__ void __launch_bounds__(THREADS, MINB)
hypgen_kernel(DeviceState s, const int32_t* __restrict__ d_idx, long long idx_pair_stride, int H, int h_offset,
              unsigned long long seed, int keep_best) {
    pdl_wait();
    pdl_trigger();
    if (s.skip != nullptr && *s.skip != 0) return;      // adaptive termination reached in an earlier round
    const int b = blockIdx.y;
    const int j = blockIdx.x * THREADS + threadIdx.x;   // local hypothesis slot
    // Reset the per-launch accumulators of this pair (scoring adds into them).
    if (j < s.tiles_max) s.tile_done[(size_t)b * s.tiles_max + j] = 0;
    if (j == 0 && !keep_best) s.best[b] = 0ull;
    const bool live = j < H;
    if (SYNC == 0 && !live) return;                     // with barriers every thread must stay
    const float4* corr = s.corr + (size_t)b * s.n_stride;
    const int32_t* rows = d_idx ? d_idx + (size_t)b * idx_pair_stride : nullptr;
    Corr pts[8];
    float E[9];
    bool ok = load_sample(corr, pair_n(s, b), rows, seed + 0x632BE59BD9B4E019ull * (unsigned long long)b,
                          (long long)h_offset + (live ? j : 0), pts, s.sampler);
    if (SOLVER == 0) solve_hypothesis<SYNC>(pts, E);
    else if (SOLVER == 1) solve_hypothesis_projector(pts, E);
    else solve_homography(pts, E);                      // first 4 of the 8 sampled correspondences
    if (!live) return;
    float* out = s.Ecand + (size_t)b * 9 * s.h_stride + j;
#pragma unroll
    for (int k = 0; k < 9; k++) out[(size_t)k * s.h_stride] = ok ? E[k] : 0.0f;
    s.counts[(size_t)b * s.h_stride + j] = 0;
}

// solver 0: 9x9 Jacobi eigensolve (255 registers, 2 CTAs of 128 threads per SM);
// solver 1: 8x8 Cholesky projector (see hyp_solver.cuh), 4 CTAs of 128 threads per SM;
// solver 2: 4-point homography through the same projector (find_homography).
void launch_hypgen(const DeviceState& s, const int32_t* d_idx, long long idx_pair_stride, int H, int h_offset,
                   unsigned long long seed, int solver, cudaStream_t st, int keep_best) {
    int need = H > s.tiles_max ? H : s.tiles_max;
    dim3 grid((need + 127) / 128, s.B);
    if (solver == 0)
        hypgen_kernel<128, 2, 0, 0><<<grid, 128, 0, st>>>(s, d_idx, idx_pair_stride, H, h_offset, seed, keep_best);
    else if (solver == 1)
        launch_dep(hypgen_kernel<128, SFMB200_HYPGEN_MINB, 0, 1>, grid, dim3(128), 0, st, s, d_idx, idx_pair_stride, H, h_offset, seed, keep_best);
    else
        hypgen_kernel<128, 4, 0, 2><<<grid, 128, 0, st>>>(s, d_idx, idx_pair_stride, H, h_offset, seed, keep_best);
}

// Multi-GPU single-pair case: after the (count, index) all-reduce every rank
// regenerates the winning hypothesis from its global index instead of
// broadcasting 36 bytes (SURVEY 5.8).  best[] already holds the reduced value.
__global__ void regen_best_kernel(DeviceState s, const int32_t* __restrict__ d_idx, long long idx_pair_stride,
                                  unsigned long long seed, int solver) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= s.B) return;
    unsigned long long packed = s.best[b];
    unsigned int hg = 0xFFFFFFFFu - (unsigned int)(packed & 0xFFFFFFFFull);
    int cnt = (int)(packed >> 32);
    const float4* corr = s.corr + (size_t)b * s.n_stride;
    const int32_t* rows = d_idx ? d_idx + (size_t)b * idx_pair_stride : nullptr;
    Corr pts[8];
    float E[9];
    bool ok = load_sample(corr, pair_n(s, b), rows, seed + 0x632BE59BD9B4E019ull * (unsigned long long)b, (long long)hg, pts,
                          s.sampler);
    if (solver == 0) solve_hypothesis<0>(pts, E);      // same code path as hypgen_kernel: bit-identical E
    else if (solver == 1) solve_hypothesis_projector(pts, E);
    else solve_homography(pts, E);
#pragma unroll
    for (int k = 0; k < 9; k++) s.E[(size_t)b * 9 + k] = ok ? E[k] : 0.0f;
    s.best_idx[b] = (int)hg;
    s.best_count[b] = cnt;
}

// Adaptive termination (SURVEY 8f rank 2; the reference lists "limit on RANSAC iterations" as
// future work, README.md:65-69).  After the round that brings the hypotheses tried to
// `done_after`, every pair's best inlier ratio w gives the standard bound
//   needed = log(1 - confidence) / log(1 - w^8);
// when done_after >= needed for ALL pairs of the batch (or this is the last round) the flag is
// raised, the remaining rounds' kernels return immediately and adapt[1] records the
// hypotheses actually used.  One block; the host never synchronises between rounds.
__global__ void adaptive_decide_kernel(DeviceState s, int* adapt, int round_begin, int done_after, double log1mp, int last) {
    if (adapt[0] != 0) return;
    __shared__ int unsatisfied;
    if (threadIdx.x == 0) unsatisfied = 0;
    __syncthreads();
    int mine = 0;
    for (int b = threadIdx.x; b < s.B; b += blockDim.x) {
        const unsigned long long packed = s.best[b];
        const int cnt = (int)(packed >> 32);
        // the running winner lives in this round's candidate arena iff its index falls in [round_begin, done_after):
        // publish it now, so no hypothesis has to be regenerated after the last round
        const unsigned int hg = 0xFFFFFFFFu - (unsigned int)(packed & 0xFFFFFFFFull);
        const int local = (int)hg - round_begin;
        if (packed != 0ull && local >= 0 && (int)hg < done_after) {
            const float* Eb = s.Ecand + (size_t)b * 9 * s.h_stride;
#pragma unroll
            for (int k = 0; k < 9; k++) s.E[(size_t)b * 9 + k] = Eb[(size_t)k * s.h_stride + local];
        }
        if (packed == 0ull && round_begin == 0) {
#pragma unroll
            for (int k = 0; k < 9; k++) s.E[(size_t)b * 9 + k] = 0.0f;
        }
        s.best_idx[b] = (int)hg;
        s.best_count[b] = cnt;
        double w = (double)cnt / (double)pair_n(s, b);
        double w2 = w * w, w4 = w2 * w2, w8 = w4 * w4;
        bool ok = w8 >= 1.0 || (w8 > 0.0 && (double)done_after >= log1mp / log1p(-w8));
        mine += ok ? 0 : 1;
    }
    if (mine) atomicAdd(&unsatisfied, mine);
    __syncthreads();
    if (threadIdx.x == 0 && (unsatisfied == 0 || last)) {
        adapt[1] = done_after;
        adapt[2] = unsatisfied;
        __threadfence();
        adapt[0] = 1;
    }
}
void launch_adaptive_decide(const DeviceState& s, int* d_adapt, int round_begin, int done_after, double log1mp, int last,
                            cudaStream_t st) {
    adaptive_decide_kernel<<<1, 128, 0, st>>>(s, d_adapt, round_begin, done_after, log1mp, last);
}

void launch_regen_best(const DeviceState& s, const int32_t* d_idx, long long idx_pair_stride, unsigned long long seed,
                       int solver, cudaStream_t st) {
    regen_best_kernel<<<(s.B + 31) / 32, 32, 0, st>>>(s, d_idx, idx_pair_stride, seed, solver);
}

}  // namespace sfmb200
