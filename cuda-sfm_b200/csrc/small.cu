// Whole hot path of a SMALL problem in ONE launch: ingest -> hypothesis generation -> scoring + arg-max -> pose
// candidates + cheirality -> triangulation, for pairs whose n x H is a few million evaluations or less - the
// reference's real operating point (BASELINE config 1: the dino pair, ~2k correspondences, H = N/8 ~ 270).  At that
// size the five stage kernels of the general path hold ~0.5 us of arithmetic and ~45 us of launch latency and
// dependent-launch gaps (profiles/r01_dino_pipeline.md).
//
// One thread-block CLUSTER per pair (8 CTAs portable, 16 when the device allows it), 512 threads per CTA; the
// stages are separated by hardware cluster barriers (barrier.cluster, sub-microsecond) instead of kernel
// boundaries, and the data between stages (correspondences, candidates, counts: tens of KB) stays in L1 / L2.
//   ingest    every thread normalises a strided share of the correspondences (same code as ingest_xy_kernel)
//   hypgen    one hypothesis per thread, 32 per warp, warp k of the cluster = warp (k / C) of CTA (k % C): the first
//             C warps sit on C different SMs, so at config-1 sizes every solve runs alone on its scheduler
//             (the solve is a ~2k-instruction dependent chain: latency, not throughput)
//   score     CTA r owns the hypotheses [r * Hc, (r + 1) * Hc); their scaled E sit in shared memory and are read as
//             broadcasts, threads stride over the correspondences; counts by warp REDUX + shared atomics, the
//             cluster's (count, ~index) key by one atomicMax per CTA
//   pose      4 lanes of CTA 0: select + candidates + cheirality (same code as select_pose_choose_kernel)
//   tri       every thread, strided (same solve as triangulate_kernel)
// Every stage calls the SAME device functions as the general path (hyp_solver.cuh, sampson.cuh, geometry.cuh,
// smallmat.cuh), so candidates, counts, winner, poses and points are bit-identical to it (tests/test_gpu_small.py).
#include <cooperative_groups.h>

#include "geometry.cuh"
#include "hyp_solver.cuh"

namespace cg = cooperative_groups;

namespace sfmb200 {

constexpr int SMALL_THREADS = 512;
constexpr int SMALL_HC_MAX = 128;        // hypotheses per CTA kept in shared memory
constexpr int SMALL_SMEM_PTS = 2560;     // correspondences per shared-memory tile while scoring (40 KB; larger n: several tiles)

struct SmallArgs {
    const float4* px;        // [B][n] pixel correspondences (SMALL_INGEST)
    Mat9 kinv;
    const int32_t* d_idx;    // sample rows or nullptr
    long long idx_pair_stride;
    unsigned long long seed;
    int H, h_offset;
    float thr;
    int compat, inliers_only, mask;
    long long* dbg;          // optional [16] clock64 stamps (0..5 phase boundaries, 8..14 inside scoring / pose) of CTA 0 thread 0 at the phase boundaries (tools/small_phases.py)
};

__global__ void __launch_bounds__(SMALL_THREADS, 1) small_path_kernel(DeviceState s, SmallArgs a) {
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = s.n, H = a.H;
    const int stride = C * SMALL_THREADS;
    __shared__ float2 sE2[SMALL_HC_MAX / 2][9];      // scaled E of the CTA's hypotheses, two per float2
    __shared__ int sCnt[SMALL_HC_MAX];
    __shared__ unsigned long long sKey;
    __shared__ __align__(16) float4 sPts[SMALL_SMEM_PTS];   // scaled correspondences of the current tile

    int stamp = 0;
    auto mark = [&]() {
        if (a.dbg != nullptr && rank == 0 && tid == 0 && b == 0) a.dbg[stamp] = clock64();
        stamp++;
    };
    auto sub = [&](int id) {            // finer stamps inside a phase (slots 8..15), same thread
        if (a.dbg != nullptr && rank == 0 && tid == 0 && b == 0) a.dbg[id] = clock64();
    };
    mark();

    // ---- ingest ----  (letting the generating warps normalise their own samples from the pixels instead of waiting for this
    //      phase was measured: the first miss on the pixels is the latency either way, 43.75k vs 43.80k cycles in total)
    if (a.mask & SMALL_INGEST) {
        for (int i = rank * SMALL_THREADS + tid; i < n; i += stride) {
            const float4 p = __ldg(a.px + (size_t)b * n + i);
            normalise_store(s, b, i, p.x, p.y, p.z, p.w, a.kinv);
        }
        cluster.sync();
    }
    mark();

    if (a.mask & SMALL_ESTIMATE) {
        // ---- hypothesis generation: block k of 32 hypotheses -> cluster warp k ----
        const float4* corr = s.corr + (size_t)b * s.n_stride;
        const int32_t* rows = a.d_idx ? a.d_idx + (size_t)b * a.idx_pair_stride : nullptr;
        const int cluster_warps = C * (SMALL_THREADS / 32);
        // warps of this CTA that generate: 0 .. gen_warps-1.  The others would idle until the barrier: they bring the first
        // tile of scaled correspondences (written before the ingest barrier) into shared memory for the scoring phase.
        const int blocks32 = (H + 31) >> 5;
        const int gen_warps = min(SMALL_THREADS / 32, max(0, (blocks32 - rank + C - 1) / C));
        const float4* cs = s.corr_s + (size_t)b * s.n_stride;
        const int tile0 = min(n, SMALL_SMEM_PTS);
        const bool preload = gen_warps < SMALL_THREADS / 32;
        if (preload && warp >= gen_warps) {
            const int loaders = SMALL_THREADS - 32 * gen_warps;
            for (int i = tid - 32 * gen_warps; i < tile0; i += loaders) sPts[i] = __ldcg(cs + i);
        }
        for (int k = warp * C + rank; k * 32 < H; k += cluster_warps) {
            const int j = k * 32 + lane;
            const bool live = j < H;
            Corr pts[8];
            float E[9];
            const bool ok = load_sample<true>(corr, n, rows, a.seed + 0x632BE59BD9B4E019ull * (unsigned long long)b,
                                              (long long)a.h_offset + (live ? j : 0), pts, s.sampler);
            solve_hypothesis_projector(pts, E);
            if (live) {
                float* out = s.Ecand + (size_t)b * 9 * s.h_stride + j;
#pragma unroll
                for (int q = 0; q < 9; q++) out[(size_t)q * s.h_stride] = ok ? E[q] : 0.0f;
            }
        }
        cluster.sync();
        mark();

        // ---- scoring: CTA `rank` owns hypotheses [h0, h1), scored two at a time in packed FFMA2 (same fma tree per lane
        //      as the scalar form: sampson.cuh) ----
        const int Hc = (H + C - 1) / C;
        const int h0 = rank * Hc, h1 = min(H, h0 + Hc);
        const int mine = max(h1 - h0, 0), mine_pairs = (mine + 1) >> 1;
        const ThrScale ts = make_thr_scale(a.thr);
        const float* Eb = s.Ecand + (size_t)b * 9 * s.h_stride;
        for (int t = tid; t < mine_pairs * 18; t += SMALL_THREADS) {
            const int hh = t / 9, q = t - 9 * hh;                         // hh < 2 * mine_pairs; the odd tail is a zero E
            float v = hh < mine ? __ldcg(Eb + (size_t)q * s.h_stride + h0 + hh) : 0.0f;   // written by another SM before the barrier
            if (q != 8) v *= thr_scale_factor(ts, q);                      // E~ = D E D (sampson.cuh), as score_kernel does
            reinterpret_cast<float*>(&sE2[hh >> 1][q])[hh & 1] = v;
        }
        for (int t = tid; t < SMALL_HC_MAX; t += SMALL_THREADS) sCnt[t] = 0;
        if (tid == 0) sKey = 0ull;
        __syncthreads();
        sub(8);
        // Thread layout: hypothesis pair p = tid / T, T = 512 / pairs threads per pair, each striding over the tile's points with
        // the pair's E in registers for the whole phase and the point as the broadcast operand of the FFMA2s - the loop of the
        // large-problem kernel (score.cu) at 2 hypotheses per thread: no per-group reload of E, no partial register slots.
        const int T = mine_pairs > 0 ? SMALL_THREADS / mine_pairs : SMALL_THREADS;
        const int my_pair = tid / T;
        const bool active = my_pair < mine_pairs;
        const int first = tid - my_pair * T;
        float2 e2[9];
#pragma unroll
        for (int q = 0; q < 9; q++) e2[q] = active ? sE2[my_pair][q] : make_float2(0.0f, 0.0f);
        unsigned int cnt0 = 0u, cnt1 = 0u;
        for (int c0 = 0; c0 < n; c0 += SMALL_SMEM_PTS) {
            const int nc = min(SMALL_SMEM_PTS, n - c0);
            if (c0 > 0 || !preload) {
                if (c0 > 0) __syncthreads();                               // the previous tile has been consumed
                for (int i = tid; i < nc; i += SMALL_THREADS) sPts[i] = __ldcg(cs + c0 + i);
                __syncthreads();
            }
            if (active) {
                int i = first;
                for (; i + 3 * T < nc; i += 4 * T) {
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const float4 p = sPts[i + u * T];
                        const float2 d = sampson_unit_d2(e2, make_float2(p.x, p.x), make_float2(p.y, p.y), make_float2(p.z, p.z),
                                                         make_float2(p.w, p.w));
                        cnt0 += __float_as_uint(d.x) >> 31;
                        cnt1 += __float_as_uint(d.y) >> 31;
                    }
                }
                for (; i < nc; i += T) {
                    const float4 p = sPts[i];
                    const float2 d = sampson_unit_d2(e2, make_float2(p.x, p.x), make_float2(p.y, p.y), make_float2(p.z, p.z),
                                                     make_float2(p.w, p.w));
                    cnt0 += __float_as_uint(d.x) >> 31;
                    cnt1 += __float_as_uint(d.y) >> 31;
                }
            }
        }
        {   // the T threads of a pair: lanes of a warp that share the pair add up by REDUX, one shared atomic per warp and pair
            const unsigned int grp = __match_any_sync(0xFFFFFFFFu, active ? my_pair : -1);
            const unsigned int w0 = __reduce_add_sync(grp, cnt0), w1 = __reduce_add_sync(grp, cnt1);
            if (active && lane == __ffs(grp) - 1) {
                if (w0) atomicAdd(&sCnt[2 * my_pair], (int)w0);
                if (w1 && 2 * my_pair + 1 < mine) atomicAdd(&sCnt[2 * my_pair + 1], (int)w1);
            }
        }
        sub(9);
        __syncthreads();
        sub(10);
        unsigned long long key = 0ull;
        int* counts = s.counts + (size_t)b * s.h_stride;
        for (int t = tid; t < mine; t += SMALL_THREADS) {
            const int c = sCnt[t];
            counts[h0 + t] = c;
            const unsigned long long kk = ((unsigned long long)(unsigned)c << 32) |
                                          (unsigned long long)(0xFFFFFFFFu - (unsigned)(a.h_offset + h0 + t));
            key = kk > key ? kk : key;
        }
        // the CTA's best key stays in ITS shared memory: CTA 0 reads the C of them over the cluster's distributed shared
        // memory after the barrier (no atomic round trip through L2)
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o);
            key = other > key ? other : key;
        }
        if (lane == 0 && key != 0ull) atomicMax(&sKey, key);
        sub(11);
        cluster.sync();
        mark();
    }

    // ---- select (+ pose candidates + cheirality) : CTA 0.  Lanes 0..3 of warp 0 take one candidate each; in compat mode
    //      the replay of the reference's SVD orientation (reference_null_direction: as long a chain as the SVD itself, and
    //      independent of it) runs on warp 1 at the same time and is handed over through shared memory ----
    if ((a.mask & (SMALL_ESTIMATE | SMALL_POSE)) && rank == 0) {
        __shared__ float sNull[3];
        const bool split = (a.mask & SMALL_POSE) && a.compat;           // uniform over the CTA
        const int c = lane;
        const bool worker = warp == 0 && c < 4, helper = split && warp == 1 && lane == 0;
        bool pass = false;
        float E[9], P[16], u[9], sg[9], v[9];
        // the cluster's best key: lane r of warps 0 and 1 reads CTA r's, a shuffle tree takes the maximum
        unsigned long long cluster_key = 0ull;
        if (warp < 2 && (a.mask & SMALL_ESTIMATE)) {
            if (lane < C) cluster_key = *cluster.map_shared_rank(&sKey, lane);
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, cluster_key, o);
                cluster_key = other > cluster_key ? other : cluster_key;
            }
        }
        if (worker || helper) {
            if (a.mask & SMALL_ESTIMATE) {
                const unsigned long long packed = cluster_key;
                const unsigned int hg = 0xFFFFFFFFu - (unsigned int)(packed & 0xFFFFFFFFull);
                const int local = (int)hg - a.h_offset;
                const float* Eb = s.Ecand + (size_t)b * 9 * s.h_stride;
#pragma unroll
                for (int k = 0; k < 9; k++) E[k] = (local >= 0 && local < s.h_stride) ? __ldcg(Eb + (size_t)k * s.h_stride + local) : 0.0f;
                if (worker && c == 0) {
                    s.best[b] = packed;
                    s.best_idx[b] = (int)hg;
                    s.best_count[b] = (int)(packed >> 32);
#pragma unroll
                    for (int k = 0; k < 9; k++) s.E[(size_t)b * 9 + k] = E[k];
                }
            } else {
#pragma unroll
                for (int k = 0; k < 9; k++) E[k] = s.E[(size_t)b * 9 + k];
            }
            sub(12);
            if (a.mask & SMALL_POSE) {
                if (helper) {
                    float r[3];
                    reference_null_direction(E, r);
                    sNull[0] = r[0]; sNull[1] = r[1]; sNull[2] = r[2];
                } else {
                    svd3<5>(E, u, sg, v);
                }
            }
        }
        if (split) __syncthreads();
        if (worker && (a.mask & SMALL_POSE)) {
            if (split) {
                const float r[3] = {sNull[0], sNull[1], sNull[2]};
                svd3_orient(r, u, sg, v);
            }
            pose_from_svd(u, v, c, a.compat, P);
            sub(13);
            if (a.compat) {
                const float4 c0 = __ldcg(s.corr + (size_t)b * s.n_stride);
                float Minv[16];
                pass = cheirality_compat(c0, P, Minv);
#pragma unroll
                for (int i = 0; i < 16; i++) P[i] = Minv[i];
            }
#pragma unroll
            for (int i = 0; i < 16; i++) s.P[(size_t)b * 64 + 16 * c + i] = P[i];
        }
        if (warp == 0) {
            const unsigned m = __ballot_sync(0xFFFFFFFFu, pass) & 0xFu;
            if (lane == 0 && (a.mask & SMALL_POSE) && a.compat) s.P_ind[b] = m ? 31 - __clz(m) : 0;      // last passing index (sfm.cu:284-297)
        }
    }
    sub(14);
    cluster.sync();                       // also: no CTA leaves while CTA 0 may still read its shared memory
    if (!(a.mask & SMALL_TRI)) return;
    mark();

    // ---- triangulation: same solve as triangulate_kernel ----
    {
        const float* Mg = s.P + (size_t)b * 64 + 16 * __ldcg(s.P_ind + b);
        float M[12], e[9];
#pragma unroll
        for (int k = 0; k < 12; k++) M[k] = __ldcg(Mg + k);
#pragma unroll
        for (int k = 0; k < 9; k++) e[k] = __ldcg(s.E + (size_t)b * 9 + k);
        const float4* corr = s.corr + (size_t)b * s.n_stride;
        float* out = s.points + (size_t)b * 4 * s.n_stride;
        const int rounds = (n + stride - 1) / stride;
        for (int r = 0; r < rounds; r++) {
            const int i = r * stride + rank * SMALL_THREADS + tid;
            const bool inside = i < n;
            const float4 pt = inside ? __ldcg(corr + i) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            bool keep[1] = {inside};
            if (a.inliers_only) keep[0] = keep[0] && epipolar_d(s.metric, e, pt.x, pt.y, pt.z, pt.w, -a.thr) < 0.0f;
            float x1[1] = {pt.x}, y1[1] = {pt.y}, aa[1][4], bb[1][4], v[1][4];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                aa[0][c] = fmaf(pt.z, M[8 + c], -M[c]);
                bb[0][c] = fmaf(pt.w, M[8 + c], -M[4 + c]);
            }
            dlt_null_power4_lanes<LaneF1>(x1[0], y1[0], aa[0], bb[0], v[0]);
            if (!inside) continue;
            float X = 0.0f, Y = 0.0f, Z = 0.0f;
            if (keep[0]) dehomogenise(v[0], X, Y, Z);
            out[i] = X;
            out[(size_t)s.n_stride + i] = Y;
            out[(size_t)2 * s.n_stride + i] = Z;
            out[(size_t)3 * s.n_stride + i] = 1.0f;
        }
    }
    mark();
}

static long long* g_small_dbg = nullptr;
void small_path_set_debug(long long* d_stamps) { g_small_dbg = d_stamps; }

// Largest cluster the device can co-schedule for this kernel: 16 (non-portable) or 8.
static int small_cluster_size() {
    static int cached = 0;
    if (cached) return cached;
    cached = 8;
    if (cudaFuncSetAttribute(small_path_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(16, 1, 1);
        cfg.blockDim = dim3(SMALL_THREADS, 1, 1);
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 16;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, small_path_kernel, &cfg) == cudaSuccess && clusters >= 1) cached = 16;
    }
    cudaGetLastError();
    return cached;
}

int small_path_max_hypotheses() { return SMALL_HC_MAX * small_cluster_size(); }

// mask: SMALL_INGEST | SMALL_ESTIMATE | SMALL_POSE | SMALL_TRI.  Returns cudaSuccess or the launch error.
cudaError_t launch_small_path(const DeviceState& s, const float* d_px, const int32_t* d_idx, long long idx_pair_stride, int H,
                              int h_offset, unsigned long long seed, float thr, int compat, int inliers_only, int mask,
                              cudaStream_t st) {
    SmallArgs a;
    a.dbg = g_small_dbg;
    a.px = (const float4*)d_px;
    for (int i = 0; i < 9; i++) a.kinv.v[i] = s.Kinv[i];
    a.d_idx = d_idx;
    a.idx_pair_stride = idx_pair_stride;
    a.seed = seed;
    a.H = H;
    a.h_offset = h_offset;
    a.thr = thr;
    a.compat = compat;
    a.inliers_only = inliers_only;
    a.mask = mask;
    const int C = small_cluster_size();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C, s.B, 1);
    cfg.blockDim = dim3(SMALL_THREADS, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, small_path_kernel, s, a);
}

}  // namespace sfmb200
