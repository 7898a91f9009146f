// Inlier scoring: hypotheses x correspondences Sampson test with a fused
// (count, index) arg-max.  Replaces the reference's calculateInliers
// (SfM/sfm.cu:155-236: six cublasSgemmStridedBatched + element-wise kernels +
// vecnorm + threshold_count over 88*N*H bytes of temporaries) and the
// thrust::max_element selection (sfm.cu:135-137).
//
// Mapping.  A CTA works on a tile of hypotheses (threads own 2, 4 or 8
// hypotheses: E lives in registers) and a contiguous range of points; the
// (pair, tile, point) space is cut into equal shares, one per resident CTA
// (persistent grid, see ChunkWalk), so every SM finishes at the same time.
// Points stream through shared memory in 512-point stages filled by 1-D TMA
// bulk copies (cp.async.bulk + mbarrier complete_tx, double buffered); every
// thread reads the same point per step, so the LDS is a broadcast.  Inlier
// counts stay in per-thread registers: the sign bit of
//     d = fma(den, -thr, num*num)        (d < 0  <=>  num^2 < thr*den)
// is added with one integer instruction, so there is no ballot/popc per step.
// Per evaluation: 16 FFMA + 2 FMUL (FP32 pipe) + 1 integer add.
//
// Two code paths with bit-identical results (same fma tree per lane):
//   scalar : FFMA, 2 hypotheses per thread;
//   packed : FFMA2 (fma.rn.f32x2, new on sm_100) on hypothesis pairs,
//            4 hypotheses per thread, points staged as (x1,x1,y1,y1),(x2,x2,y2,y2).
//
// Epilogue.  A CTA that saw every point of a tile writes counts directly and
// reduces from registers.  Otherwise partial counts are atomically added to
// counts[] and a per-tile counter of points processed tells which CTA completed
// the tile; that CTA reads the totals and does the tile's arg-max.  Either way one atomicMax per tile on the packed
// key (count << 32) | (0xFFFFFFFF - global index): highest count, lowest index
// on ties = thrust::max_element semantics.  No separate arg-max kernel.
//
// Roofline: FP32 pipe; algorithmic work 34 FLOP per evaluation (SURVEY 8d).
#include <math.h>

#include <mutex>
#include <type_traits>

#include "internal.cuh"
#include "sampson.cuh"

#ifndef SFMB200_SCORE_UNROLL
#define SFMB200_SCORE_UNROLL 2      // points per unrolled step of the packed inner loop.  With the pre-duplicated tile: 4 (profiles/
                                    // r01_variant_sweep.md); with the broadcast-operand tile 1 / 2 / 3 / 4 / 8 -> 0.408 / 0.381 / 0.382 / 0.385 / 0.387 ms at config 2
#endif

namespace sfmb200 {

constexpr int kScoreUnroll = SFMB200_SCORE_UNROLL;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier.
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long w = __shfl_xor_sync(0xFFFFFFFFu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// Walks the chunks (<= SCORE_CHUNK points) of this CTA's share of the work.
// Work space = (pair, hypothesis tile, point) linearised in grains of
// SCORE_GRAIN points; CTA c owns grains [c*U/G, (c+1)*U/G): every CTA gets the
// same amount of work to within one grain whatever the problem shape
// ("stream-K" decomposition along the point axis), so there is no tail wave.
// A CTA's share is a sequence of segments, each a contiguous point range of one
// (pair, tile); segments are streamed chunk by chunk.
// Per-pair counts (RAGGED): pair b owns units [T * goff[b], T * goff[b + 1]), tile-major inside; with equal counts that
// is the uniform layout.  Shares cross pair boundaries like tile boundaries, so one large pair among small ones splits
// over every CTA.  The pair of the first unit is found by a binary search over goff; after that a segment starts in the
// same pair or the next one.  The uniform walk is the RAGGED = false case: it reads nothing but kernel parameters.
struct RaggedCursor {
    const long long* goff; // grain prefix (DeviceState::grain_off) and counts (DeviceState::n_pair)
    const int* n_pair;
    long long pair_lo, pair_hi;   // units of the current pair
};
struct UniformCursor {};
template <bool RAGGED>
struct ChunkWalk : std::conditional_t<RAGGED, RaggedCursor, UniformCursor> {
    long long u, end;      // grain cursor / end of this CTA's share
    int n_units, n, T;     // grains per tile, points of the current pair, tiles per pair
    int b, t, p0, cnt;     // current chunk: pair, tile, first point, points
    int seg_p0, seg_pts;   // current segment: first point, total points
    int left;              // points of the segment not yet handed out
    bool seg_first, seg_last;
    __device__ __forceinline__ void set_pair(int b_) {
        b = b_;
        this->pair_lo = (long long)T * this->goff[b];
        this->pair_hi = (long long)T * this->goff[b + 1];
        n_units = (int)(this->goff[b + 1] - this->goff[b]);
        n = this->n_pair[b];
    }
    __device__ __forceinline__ void init(long long u0, long long u1, int n_units_, int n_, int T_, int B,
                                         const long long* goff_, const int* n_pair_) {
        u = u0; end = u1; n_units = n_units_; n = n_; T = T_;
        left = 0; cnt = 0; p0 = 0;
        if constexpr (RAGGED) {
            this->goff = goff_;
            this->n_pair = n_pair_;
            if (u0 < u1) {
                int lo = 0, hi = B - 1;          // the last pair whose first unit is <= u0
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if ((long long)T * goff_[mid] <= u0) lo = mid; else hi = mid - 1;
                }
                set_pair(lo);
            }
        }
    }
    __device__ __forceinline__ bool next() {
        if (left == 0) {
            if (u >= end) return false;
            long long bt = 0;
            int pu;
            if constexpr (RAGGED) {
                while (u >= this->pair_hi) set_pair(b + 1);
                const long long rel = u - this->pair_lo;
                t = (int)(rel / n_units);
                pu = (int)(rel - (long long)t * n_units);
            } else {
                bt = u / n_units;
                pu = (int)(u - bt * n_units);
            }
            long long seg_units = end - u;
            if (seg_units > n_units - pu) seg_units = n_units - pu;
            if constexpr (!RAGGED) {
                b = (int)(bt / T);
                t = (int)(bt - (long long)b * T);
            }
            seg_p0 = pu * SCORE_GRAIN;
            int p1 = (pu + (int)seg_units) * SCORE_GRAIN;
            if (p1 > n) p1 = n;
            seg_pts = p1 - seg_p0;
            left = seg_pts;
            u += seg_units;
            p0 = seg_p0;
            seg_first = true;
        } else {
            p0 += cnt;
            seg_first = false;
        }
        cnt = left < SCORE_CHUNK ? left : SCORE_CHUNK;
        left -= cnt;
        seg_last = (left == 0);
        return true;
    }
};

// End of a segment (a contiguous point range of one (pair, tile) handled by one CTA): publish
// the counts and take part in the fused arg-max.  A CTA that saw every point of the tile writes
// counts directly and reduces from registers.  Otherwise partial counts are atomically added and
// a per-tile counter of points processed (it persists across launches of the same estimate)
// tells which CTA completed the tile; that CTA reads the totals and reduces them.  One atomicMax
// per tile on the packed key (count << 32) | (0xFFFFFFFF - global index).  Must be called by
// every thread of the CTA.
// `full`: this CTA saw every point of the tile.  Otherwise the tile's ticket counter advances by
// `inc` and the CTA that brings it to `total` completes the tile (TMA path: points processed out
// of the pair's count; constant-bank path: CTA arrivals out of the number the host scheduled for the tile).
template <int HPT, int THREADS>
__device__ __forceinline__ void segment_epilogue(const DeviceState& s, int b, int t, int H, int h_offset,
                                                 const unsigned int* cnt, bool full, int inc, int total,
                                                 unsigned long long* red, int* s_last) {
    constexpr int HPC = HPT * THREADS;
    const int tid = threadIdx.x;
    int* counts = s.counts + (size_t)b * s.h_stride;
    unsigned long long key = 0ull;
    bool do_argmax;
    if (full) {                          // this CTA saw every point of the tile
#pragma unroll
        for (int j = 0; j < HPT; j++) {
            int h = t * HPC + j * THREADS + tid;
            if (h < H) {
                counts[h] = (int)cnt[j];
                unsigned long long kk = ((unsigned long long)cnt[j] << 32) |
                                        (unsigned long long)(0xFFFFFFFFu - (unsigned)(h_offset + h));
                key = kk > key ? kk : key;
            }
        }
        do_argmax = true;
    } else {                             // partial: add, the CTA completing the tile reduces it
#pragma unroll
        for (int j = 0; j < HPT; j++) {
            int h = t * HPC + j * THREADS + tid;
            if (h < H && cnt[j] != 0u) atomicAdd(&counts[h], (int)cnt[j]);
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) {
            int before = atomicAdd(&s.tile_done[(size_t)b * s.tiles_max + t], inc);
            *s_last = (before + inc == total);
        }
        __syncthreads();
        do_argmax = *s_last != 0;
        if (do_argmax) {
            __threadfence();
#pragma unroll
            for (int j = 0; j < HPT; j++) {
                int h = t * HPC + j * THREADS + tid;
                if (h < H) {
                    unsigned int total = (unsigned int)__ldcg(&counts[h]);
                    unsigned long long kk = ((unsigned long long)total << 32) |
                                            (unsigned long long)(0xFFFFFFFFu - (unsigned)(h_offset + h));
                    key = kk > key ? kk : key;
                }
            }
        }
    }
    if (do_argmax) {                     // uniform across the CTA
        key = warp_max_u64(key);
        if ((tid & 31) == 0) red[tid >> 5] = key;
        __syncthreads();
        if (tid < 32) {
            unsigned long long v = tid < THREADS / 32 ? red[tid] : 0ull;
            v = warp_max_u64(v);
            if (tid == 0 && v != 0ull) atomicMax(&s.best[b], v);
        }
        __syncthreads();                 // red[] is reused by the next segment
    }
}

// Chunk descriptor handed from the producer thread to the consumers through
// shared memory (published by the mbarrier the chunk's TMA completes on).
struct ChunkDesc {
    int b, t;          // pair, hypothesis tile
    int cnt_flags;     // points in the chunk | seg_first << 30 | seg_last << 31; 0 = no more work
    int seg_pts;       // points of the whole segment (valid when seg_last)
};

template <int HPT, bool PACKED, int THREADS, int MINB, int MODEL, bool RAGGED = false>
__global__ void __launch_bounds__(THREADS, MINB)
score_kernel(DeviceState s, int H, int h_offset, int T, long long total_units, int n_units, float thr) {
    constexpr int HPC = HPT * THREADS;
    // One (x1, y1, x2, y2) per point for the scalar AND the packed form: FFMA2 takes a 32-bit register as an operand that it
    // broadcasts to both halves (SASS `R.F32`), so the point does not have to be staged pre-duplicated - half the shared
    // memory, half the LDS and TMA bytes, five register reads per FFMA2 instead of six (measured: config 2 0.3850 vs 0.3899 ms).
    __shared__ __align__(128) float4 buf[2][SCORE_CHUNK];
    __shared__ __align__(8) uint64_t full[2];
    __shared__ __align__(16) ChunkDesc desc[2];
    __shared__ ChunkWalk<RAGGED> walk;  // producer state lives here, not in loop-carried registers:
                                        // the FFMA stream needs every register for operand reuse
    __shared__ int desc_n[2];           // RAGGED: points of the pair of desc[]
    __shared__ unsigned long long red[THREADS / 32];
    __shared__ int s_last;

    pdl_wait();
    pdl_trigger();
    if (s.skip != nullptr && *s.skip != 0) return;      // adaptive termination reached in an earlier round
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        ChunkWalk<RAGGED> w;
        w.init(total_units * blockIdx.x / gridDim.x, total_units * (blockIdx.x + 1) / gridDim.x, n_units, s.n, T, s.B,
               s.grain_off, s.n_pair);
        walk = w;
    }
    __syncthreads();

    // Producer step (thread 0): advance the walk, publish the descriptor of the
    // next chunk and start its TMA; an empty descriptor + plain arrive ends the loop.
    auto produce = [&](int stage) {
        ChunkWalk<RAGGED> w = walk;
        bool more = w.next();
        walk = w;
        ChunkDesc d;
        d.b = w.b; d.t = w.t; d.seg_pts = w.seg_pts;
        if constexpr (RAGGED) desc_n[stage] = w.n;
        d.cnt_flags = more ? (w.cnt | (w.seg_first ? (1 << 30) : 0) | (w.seg_last ? (1 << 31) : 0)) : 0;
        desc[stage] = d;
        if (more) {
            const float4* src = s.corr_s + (size_t)w.b * s.n_stride + w.p0;
            uint32_t bytes = (uint32_t)w.cnt * 16u;
            mbar_expect_tx(&full[stage], bytes);
            tma_load_1d(&buf[stage][0], src, bytes, &full[stage]);
        } else {
            mbar_expect_tx(&full[stage], 0);
        }
    };
    if (tid == 0) produce(0);

    float e[PACKED ? 1 : HPT][9];               // scalar path: one E per hypothesis
    float2 e2[PACKED ? HPT / 2 : 1][9];         // packed path: E of a hypothesis pair per float2
    unsigned int cnt[HPT];
    const float nthr = -thr;
    const float2 nthr2 = make_float2(nthr, nthr);
    const ThrScale ts = make_thr_scale(thr);
    (void)e; (void)e2; (void)nthr2; (void)ts;

    for (int k = 0;; k++) {
        if (tid == 0) produce((k + 1) & 1);     // safe: stage (k+1)&1 was released by the barrier ending iteration k-1
        mbar_wait(&full[k & 1], (k >> 1) & 1);
        const ChunkDesc d = desc[k & 1];
        if (d.cnt_flags == 0) break;
        const int n_here = d.cnt_flags & 0x3FFFFFFF;
        if (d.cnt_flags & (1 << 30)) {
            // first chunk of a segment: this thread's essential matrices -> registers
            const float* Eb = s.Ecand + (size_t)d.b * 9 * s.h_stride;
#pragma unroll
            for (int j = 0; j < HPT; j++) {
                int h = d.t * HPC + j * THREADS + tid;
                bool valid = h < H;
#pragma unroll
                for (int q = 0; q < 9; q++) {
                    float v = valid ? __ldg(Eb + (size_t)q * s.h_stride + h) : 0.0f;
                    if (MODEL != 1 && q != 8) v *= thr_scale_factor(ts, q);      // E~ = D E D (sampson.cuh)
                    if constexpr (PACKED) {
                        if (j & 1) e2[j / 2][q].y = v; else e2[j / 2][q].x = v;
                    } else {
                        e[j][q] = v;
                    }
                }
                cnt[j] = 0u;
            }
        }
        const float4* pb = buf[k & 1];
        if constexpr (PACKED) {
#pragma unroll kScoreUnroll
            for (int i = 0; i < n_here; i++) {
                const float4 p = pb[i];
                const float2 x1 = make_float2(p.x, p.x), y1 = make_float2(p.y, p.y);      // splats: the compiler emits the
                const float2 x2 = make_float2(p.z, p.z), y2 = make_float2(p.w, p.w);      // broadcast operand form, no MOVs
#pragma unroll
                for (int j = 0; j < HPT / 2; j++) {
                    float2 dd = model_d2<MODEL>(e2[j], x1, y1, x2, y2, nthr2);
                    cnt[2 * j] += __float_as_uint(dd.x) >> 31;
                    cnt[2 * j + 1] += __float_as_uint(dd.y) >> 31;
                }
            }
        } else {
#pragma unroll 4
            for (int i = 0; i < n_here; i++) {
                float4 p = pb[i];
#pragma unroll
                for (int j = 0; j < HPT; j++) {
                    float dd = model_d<MODEL>(e[j], p.x, p.y, p.z, p.w, nthr);
                    cnt[j] += __float_as_uint(dd) >> 31;
                }
            }
        }
        __syncthreads();   // buf / desc [k & 1] are free for the chunk produced at the top of iteration k + 1
        if (d.cnt_flags >= 0) continue;   // bit 31 clear: segment continues

        // ---- end of a segment: counts + fused arg-max for (pair b, tile t) ----
        // (read here, not with d: the pair's count need not stay in a register across the point loop; the producer
        // rewrites desc_n[k & 1] only after the barrier inside the epilogue)
        const int n_b = RAGGED ? desc_n[k & 1] : s.n;
        segment_epilogue<HPT, THREADS>(s, d.b, d.t, H, h_offset, cnt, d.seg_pts == n_b, d.seg_pts, n_b, red, &s_last);
    }
}

// ---------------------------------------------------------------------------
// Constant-bank path.  ncu shows what bounds the kernels above (profiles/
// r01_ncu_score_variants.md): every FFMA reads three general registers and the
// register-bank conflicts surface as dispatch stalls (scalar) or the packed pipe
// saturates at ~80 %.  The point coordinates are the same for every thread, so
// they do not have to be general registers at all: staged in __constant__
// memory they are fetched by uniform loads (LDCU) into UNIFORM registers and
// each FFMA reads two general registers + one uniform one.  No shared memory,
// no reuse-cache dependence, 1.8e12 evals/s for any hypotheses-per-thread.
// The price: 64 KB of constant bank = 4,000 points per launch, so a pair is
// scored in ceil(n / 4000) launches whose partial counts meet in counts[] (one
// atomic per hypothesis per CTA) and in the per-tile arrival counter.
// MEASURED OUTCOME (B200, profiles/r01_const_bank.md): a stand-alone prototype
// with 1.2M hypotheses per launch reaches 1.80e12 evals/s (+8 % over the TMA /
// FFMA2 kernel), but in the product the refill + launch + wave tail per 4,000
// points and above all the H atomics per launch eat the gain: config 2 0.429 ms
// vs 0.404, config 3 665 ms vs 654.  It is therefore selectable
// (SFMB200_OPT_SCORE_VARIANT = 10, tested for parity) but never chosen
// automatically; the TMA-staged kernels remain the product path.
// ---------------------------------------------------------------------------
constexpr int CONST_PTS = 4000;
__constant__ float4 c_pts[CONST_PTS];

// Work split of one launch: grid (tiles, splits); CTA (t, y) scores tile t against points
// [y * chunk, y * chunk + np) of the batch, np = chunk except for the last split.  The loop
// counter runs from 0 to a bound that is a plain select between two kernel parameters and the
// base is c_pts + blockIdx.y * chunk: with anything more elaborate (min, shifts, a work-stealing
// walk) nvcc 12.9 moves the index to vector registers and the loads become LDC into general
// registers - exactly the operand traffic this kernel exists to avoid.
template <int HPT, int THREADS, int MINB, int MODEL>
__global__ void __launch_bounds__(THREADS, MINB)
score_const_kernel(DeviceState s, int b, int chunk, int last_np, int arrivals, int H, int h_offset, float thr) {
    constexpr int HPC = HPT * THREADS;
    __shared__ unsigned long long red[THREADS / 32];
    __shared__ int s_last;
    if (s.skip != nullptr && *s.skip != 0) return;      // adaptive termination reached in an earlier round
    const int tid = threadIdx.x;
    const int t = blockIdx.x;
    const float4* base = c_pts + blockIdx.y * chunk;
    const int np = (blockIdx.y == gridDim.y - 1) ? last_np : chunk;
    const float nthr = -thr;
    const ThrScale ts = make_thr_scale(thr);
    (void)ts;
    const float* Eb = s.Ecand + (size_t)b * 9 * s.h_stride;
    float e[HPT][9];
    unsigned int cnt[HPT];
#pragma unroll
    for (int j = 0; j < HPT; j++) {
        int h = t * HPC + j * THREADS + tid;
        bool valid = h < H;
#pragma unroll
        for (int k = 0; k < 9; k++) {
            float v = valid ? __ldg(Eb + (size_t)k * s.h_stride + h) : 0.0f;
            if (MODEL != 1 && k != 8) v *= thr_scale_factor(ts, k);      // E~ = D E D (sampson.cuh)
            e[j][k] = v;
        }
        cnt[j] = 0u;
    }
#pragma unroll 4
    for (int i = 0; i < np; i++) {
        const float4 p = base[i];                       // uniform address -> LDCU -> uniform registers
#pragma unroll
        for (int j = 0; j < HPT; j++) {
            float dd = model_d<MODEL>(e[j], p.x, p.y, p.z, p.w, nthr);
            cnt[j] += __float_as_uint(dd) >> 31;
        }
    }
    // Tile completion is counted in CTA arrivals, not points: feeding the loop bound `np` into the
    // per-thread epilogue code would pull it (and with it the whole point loop) off the uniform datapath.
    segment_epilogue<HPT, THREADS>(s, b, t, H, h_offset, cnt, arrivals == 1, 1, arrivals, red, &s_last);
}

// Number of point splits per tile for one launch: the grid tiles x splits should fill whole
// waves of `slots` resident CTAs (all CTAs of a launch take the same time), with at least
// `min_chunk` points per CTA to amortise loading its essential matrices.
static int const_splits(int tiles, int batch, long long slots, int min_chunk = 64) {
    int max_s = batch / min_chunk;
    if (max_s < 1) max_s = 1;
    if (max_s > 512) max_s = 512;
    int best_s = 1;
    double best_eff = -1.0;
    for (int sp = 1; sp <= max_s; sp++) {
        double waves = (double)tiles * sp / (double)slots;
        double eff = waves / ceil(waves);
        // prefer fewer splits on near-ties (fewer atomics, better amortisation)
        if (eff > best_eff + 0.02) { best_eff = eff; best_s = sp; }
        if (eff > 0.985 && waves >= 2.0) break;
    }
    return best_s;
}

constexpr int CONST_HPT = 8, CONST_THREADS = 128, CONST_MINB = 4;

// The __constant__ bank is one per device and process, not per handle or stream: refills are
// serialised with a mutex and every refill waits for the last kernel that read the previous
// contents, whichever stream it ran on.
struct ConstBankGuard {
    std::mutex mu;
    cudaEvent_t last_use[64] = {};
};
static ConstBankGuard g_const;

template <int MODEL>
static void launch_score_const(const DeviceState& s, const ScorePlan& plan, int H, int h_offset, float thr, const int* h_n_pair,
                               cudaStream_t st) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    std::lock_guard<std::mutex> lock(g_const.mu);
    if (!g_const.last_use[dev]) cudaEventCreateWithFlags(&g_const.last_use[dev], cudaEventDisableTiming);
    int n = -1, per = 0, arrivals = 0;
    for (int b = 0; b < s.B; b++) {
        const int nb = h_n_pair ? h_n_pair[b] : s.n;
        if (nb != n) {      // a new count: batches of the pair and the CTA arrivals each of its tiles will see in total
            n = nb;
            const int batches = (n + CONST_PTS - 1) / CONST_PTS;
            per = ((n + batches - 1) / batches + 15) / 16 * 16;      // even batches
            arrivals = 0;
            for (int off = 0; off < n; off += per) {
                const int cnt = n - off < per ? n - off : per;
                const int splits = const_splits(plan.tiles, cnt, plan.ctas);        // plan.ctas = resident CTA slots
                const int chunk = (cnt + splits - 1) / splits;
                arrivals += (cnt + chunk - 1) / chunk;
            }
        }
        for (int off = 0; off < n; off += per) {
            const int cnt = n - off < per ? n - off : per;
            const int splits = const_splits(plan.tiles, cnt, plan.ctas);
            const int chunk = (cnt + splits - 1) / splits;
            const int real_splits = (cnt + chunk - 1) / chunk;
            const int last_np = cnt - (real_splits - 1) * chunk;
            cudaStreamWaitEvent(st, g_const.last_use[dev], 0);
            cudaMemcpyToSymbolAsync(c_pts, s.corr_s + (size_t)b * s.n_stride + off, (size_t)cnt * sizeof(float4), 0,
                                    cudaMemcpyDeviceToDevice, st);
            score_const_kernel<CONST_HPT, CONST_THREADS, CONST_MINB, MODEL>
                <<<dim3(plan.tiles, real_splits), CONST_THREADS, 0, st>>>(s, b, chunk, last_np, arrivals, H, h_offset, thr);
            cudaEventRecord(g_const.last_use[dev], st);
        }
    }
}

// Kernel family.  Register-bank bandwidth is what bounds the FP32 pipe here: an
// FFMA reads three registers (an FFMA2 three register PAIRS) per issue and the
// only operand the operand-reuse cache can supply is the point coordinate
// shared by the HPT hypotheses of a thread, so more hypotheses per thread =
// more reuse, at the price of registers (occupancy) and coarser tiles.
// Measured on B200 (profiles/): scalar FFMA with 8 hypotheses per thread is the
// fastest at scale; the small-tile kernels serve small hypothesis counts.
#ifndef SFMB200_V4_MINB
#define SFMB200_V4_MINB 1      // resident CTAs per SM the default packed variant is compiled for (2 = 128-register cap: measured slower)
#endif
#ifndef SFMB200_V8_MINB
#define SFMB200_V8_MINB 2
#endif
struct ScoreVariant { int hpt; int packed; int threads; int minb; };
static const ScoreVariant kVariants[] = {
    {2, 0, 256, 1}, {4, 1, 256, 1}, {4, 0, 256, 1}, {8, 0, 256, 2}, {8, 1, 256, SFMB200_V4_MINB},
    {4, 0, 128, 1}, {4, 1, 128, 1}, {8, 0, 128, 4}, {8, 1, 128, SFMB200_V8_MINB}, {2, 0, 128, 1},
    {CONST_HPT, 0, CONST_THREADS, CONST_MINB},      // 10: constant-bank path (score_const_kernel)
    {8, 1, 128, 3},                                 // 11: packed, three 128-thread CTAs per SM = 3 warps per scheduler (<= 168 registers)
};
constexpr int kConstVariant = 10;
// Also measured on B200 and dropped (profiles/r01_variant_sweep.md): 12 / 16 hypotheses per
// thread, scalar or packed (fewer resident warps than the reuse gain pays for); packed with a
// 128-register cap for 16 warps/SM (less ILP: -8 %); 192 / 320 / 384-thread CTAs (warps not a
// multiple of the 4 schedulers, or 12 warps/SM: -5 .. -30 %: operand reuse needs back-to-back
// issue from the same warp, so fewer warps with more independent work each win).
constexpr int kNumVariants = sizeof(kVariants) / sizeof(kVariants[0]);

template <int HPT, bool PACKED, int THREADS, int MINB>
static void launch_one(const DeviceState& s, int ctas, int H, int h_offset, int T, long long units, int n_units, float thr,
                       cudaStream_t st) {
    if (s.n_pair)
        launch_dep(score_kernel<HPT, PACKED, THREADS, MINB, 0, true>, dim3(ctas), dim3(THREADS), 0, st, s, H, h_offset, T, units, n_units, thr);
    else
        launch_dep(score_kernel<HPT, PACKED, THREADS, MINB, 0>, dim3(ctas), dim3(THREADS), 0, st, s, H, h_offset, T, units, n_units, thr);
}
template <int HPT, bool PACKED, int THREADS, int MINB>
static int occupancy_one(bool ragged) {
    int n = 0;
    if (ragged) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, score_kernel<HPT, PACKED, THREADS, MINB, 0, true>, THREADS, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, score_kernel<HPT, PACKED, THREADS, MINB, 0>, THREADS, 0);
    return n > 0 ? n : 1;
}
#define SFM_FOR_VARIANT(v, CALL)                     \
    switch (v) {                                     \
        case 0: CALL(2, false, 256, 1); break;       \
        case 1: CALL(4, true, 256, 1); break;        \
        case 2: CALL(4, false, 256, 1); break;       \
        case 3: CALL(8, false, 256, 2); break;       \
        case 4: CALL(8, true, 256, SFMB200_V4_MINB); break;        \
        case 5: CALL(4, false, 128, 1); break;       \
        case 6: CALL(4, true, 128, 1); break;        \
        case 7: CALL(8, false, 128, 4); break;       \
        case 8: CALL(8, true, 128, SFMB200_V8_MINB); break;        \
        case 11: CALL(8, true, 128, 3); break;       \
        default: CALL(2, false, 128, 1); break;      \
    }

static int variant_occupancy(int v, bool ragged) {
    static int cache[2][kNumVariants] = {};
    int& c = cache[ragged ? 1 : 0][v];
    if (c == 0 && v == kConstVariant) {
        int n = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, score_const_kernel<CONST_HPT, CONST_THREADS, CONST_MINB, 0>, CONST_THREADS, 0);
        c = n > 0 ? n : 1;
    }
    if (c == 0) {
#define SFM_OCC(h, p, t, m) c = occupancy_one<h, p, t, m>(ragged)
        SFM_FOR_VARIANT(v, SFM_OCC)
#undef SFM_OCC
    }
    return c;
}

int score_num_variants() { return kNumVariants; }

ScorePlan make_score_plan(const PointCounts& c, int H, int variant_override, int sms) {
    ScorePlan p;
    if (variant_override >= 0 && variant_override < kNumVariants) {
        p.variant = variant_override;
    } else {
        // Measured on B200 (profiles/r02_score_variants.md, tools/score_plan_sweep.py): packed FFMA2 with 8 hypotheses per
        // thread and one 256-thread CTA per SM (4) is the fastest at every large shape; below ~1e8 evaluations per launch the
        // kernel is latency- rather than throughput-bound and the 512-hypothesis tile (6), below ~3e7 the 256-hypothesis
        // scalar tile (9) win by up to 24 %.  The constant-bank kernel (variant 10) is never chosen automatically: see the
        // note above score_const_kernel.
        const double W = (double)c.n_sum * (double)H;       // evaluations per launch
        if (H >= 1536) p.variant = W >= 1.2e8 ? 4 : 6;
        else if (H >= 768) p.variant = W >= 2e8 ? 1 : (W >= 3e7 ? 6 : 9);
        else p.variant = W >= 3e7 ? 6 : 9;
    }
    const ScoreVariant& v = kVariants[p.variant];
    p.hyp_per_cta = v.hpt * v.threads;
    p.tiles = (H + p.hyp_per_cta - 1) / p.hyp_per_cta;
    if (p.tiles < 1) p.tiles = 1;
    if (sms < 1) sms = 148;          // the handle caches the SM count of ITS device at create (api.cu)
    p.n_units = (c.n_max + SCORE_GRAIN - 1) / SCORE_GRAIN;      // used by the uniform walk only
    p.total_units = (long long)p.tiles * c.grains;
    long long ctas = (long long)sms * variant_occupancy(p.variant, c.ragged);   // persistent: all CTAs co-resident
    if (p.variant != kConstVariant && ctas > p.total_units) ctas = p.total_units;   // const path: ctas = resident slots
    if (ctas < 1) ctas = 1;
    p.ctas = (int)ctas;
    return p;
}

// Homography model: the same kernel with the transfer-error test; three tile sizes are enough
// (thr here is the SQUARED pixel / coordinate threshold).
ScorePlan make_score_plan_homography(const PointCounts& c, int H, int sms) {
#ifdef SFMB200_HOMOG_PLAN_BY_H      // the rule before the sweep (A/B)
    return make_score_plan(c, H, H >= 1536 ? 4 : (H >= 384 ? 6 : 9), sms);     // tiles of 2048 / 512 / 256 hypotheses
#else
    const double W = (double)c.n_sum * (double)H;      // same reading as make_score_plan: small launches are latency-bound
    return make_score_plan(c, H, H >= 1536 ? (W >= 1.2e8 ? 4 : 6) : (W >= 3e7 ? 6 : 9), sms);
#endif
}
// The other two models (homography transfer error; symmetric epipolar distance) in the three tile sizes of
// make_score_plan_homography.
template <int MODEL>
static void launch_score_model(const DeviceState& s, ScorePlan& plan, int H, int h_offset, float thr, const int* h_n_pair,
                               cudaStream_t st) {
    const int v = plan.variant;
    if (v == kConstVariant) {
        launch_score_const<MODEL>(s, plan, H, h_offset, thr, h_n_pair, st);
        return;
    }
    const bool big = kVariants[v].hpt * kVariants[v].threads >= 2048, mid = kVariants[v].hpt * kVariants[v].threads >= 512;
    if (s.n_pair) {
        if (big) score_kernel<8, true, 256, 1, MODEL, true><<<plan.ctas, 256, 0, st>>>(s, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr);
        else if (mid) score_kernel<4, true, 128, 1, MODEL, true><<<plan.ctas, 128, 0, st>>>(s, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr);
        else score_kernel<2, false, 128, 1, MODEL, true><<<plan.ctas, 128, 0, st>>>(s, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr);
    } else if (big) {
        score_kernel<8, true, 256, 1, MODEL><<<plan.ctas, 256, 0, st>>>(s, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr);
    } else if (mid) {
        score_kernel<4, true, 128, 1, MODEL><<<plan.ctas, 128, 0, st>>>(s, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr);
    } else {
        score_kernel<2, false, 128, 1, MODEL><<<plan.ctas, 128, 0, st>>>(s, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr);
    }
}
void launch_score_homography(const DeviceState& s, ScorePlan& plan, int H, int h_offset, float thr2, cudaStream_t st) {
    launch_score_model<1>(s, plan, H, h_offset, thr2, nullptr, st);
}
void launch_score_symmetric(const DeviceState& s, ScorePlan& plan, int H, int h_offset, float thr, const int* h_n_pair,
                            cudaStream_t st) {
    launch_score_model<2>(s, plan, H, h_offset, thr, h_n_pair, st);
}

void launch_score(const DeviceState& s, const ScorePlan& plan, int H, int h_offset, float thr, const int* h_n_pair,
                  cudaStream_t st) {
    if (plan.variant == kConstVariant) {
        launch_score_const<0>(s, plan, H, h_offset, thr, h_n_pair, st);
        return;
    }
#define SFM_LAUNCH(h, p, t, m) launch_one<h, p, t, m>(s, plan.ctas, H, h_offset, plan.tiles, plan.total_units, plan.n_units, thr, st)
    SFM_FOR_VARIANT(plan.variant, SFM_LAUNCH)
#undef SFM_LAUNCH
}

// Selected hypothesis -> E, index, count (per pair).
__global__ void select_kernel(DeviceState s, int h_offset) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= s.B) return;
    unsigned long long packed = s.best[b];
    unsigned int hg = 0xFFFFFFFFu - (unsigned int)(packed & 0xFFFFFFFFull);
    int local = (int)hg - h_offset;
    s.best_idx[b] = (int)hg;
    s.best_count[b] = (int)(packed >> 32);
    const float* Eb = s.Ecand + (size_t)b * 9 * s.h_stride;
#pragma unroll
    for (int k = 0; k < 9; k++)
        s.E[(size_t)b * 9 + k] = (local >= 0 && local < s.h_stride) ? Eb[(size_t)k * s.h_stride + local] : 0.0f;
}

void launch_select(const DeviceState& s, int h_offset, cudaStream_t st) {
    select_kernel<<<(s.B + 127) / 128, 128, 0, st>>>(s, h_offset);
}

// ---------------------------------------------------------------------------
// FP32-pipe probe: the roofline denominator for hypothesis generation and
// scoring is not in MEASURED_PEAKS.json (it has HBM and bf16 only), so bench.py
// measures it live: dependent-chain-free FFMA / FFMA2 streams, all SMs busy.
// mode 0: scalar FFMA with three distinct register operands
// mode 1: packed FFMA2
// ---------------------------------------------------------------------------
constexpr int PROBE_THREADS = 256;
constexpr int PROBE_CHAINS = 16;
constexpr int PROBE_INNER = 64;

template <int MODE>
__global__ void __launch_bounds__(PROBE_THREADS) fma_probe_kernel(int iters, float* sink, float a0, float b0) {
    if constexpr (MODE == 0) {
        float acc[PROBE_CHAINS];
        float a = a0 + threadIdx.x * 1e-9f, b = b0;
#pragma unroll
        for (int i = 0; i < PROBE_CHAINS; i++) acc[i] = (float)i;
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int r = 0; r < PROBE_INNER; r++)
#pragma unroll
                for (int i = 0; i < PROBE_CHAINS; i++) acc[i] = fmaf(acc[i], a, b);
        }
        float t = 0.0f;
#pragma unroll
        for (int i = 0; i < PROBE_CHAINS; i++) t += acc[i];
        if (t == 123.456f) sink[0] = t;
    } else {
        float2 acc[PROBE_CHAINS];
        float2 a = make_float2(a0 + threadIdx.x * 1e-9f, a0), b = make_float2(b0, b0 * 0.5f);
#pragma unroll
        for (int i = 0; i < PROBE_CHAINS; i++) acc[i] = make_float2((float)i, (float)-i);
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int r = 0; r < PROBE_INNER; r++)
#pragma unroll
                for (int i = 0; i < PROBE_CHAINS; i++) {
                    if constexpr (MODE == 1) acc[i] = __ffma2_rn(acc[i], a, b);
                    else if constexpr (MODE == 2) acc[i] = __fmul2_rn(acc[i], a);                                   // FMUL2
                    else if constexpr (MODE == 3) acc[i] = __fadd2_rn(acc[i], b);                                   // FADD2
                    else acc[i] = __ffma2_rn(acc[i], a, make_float2(-acc[(i + 1) % PROBE_CHAINS].x, -acc[(i + 1) % PROBE_CHAINS].y));   // negated register operand
                }
        }
        float t = 0.0f;
#pragma unroll
        for (int i = 0; i < PROBE_CHAINS; i++) t += acc[i].x + acc[i].y;
        if (t == 123.456f) sink[0] = t;
    }
}

double launch_fma_probe(int mode, int iters, cudaStream_t st, float* d_sink) {
    const int ctas = 148 * 8;
    if (mode == 0)
        fma_probe_kernel<0><<<ctas, PROBE_THREADS, 0, st>>>(iters, d_sink, 0.999f, 0.001f);
    else if (mode == 1)
        fma_probe_kernel<1><<<ctas, PROBE_THREADS, 0, st>>>(iters, d_sink, 0.999f, 0.001f);
    else if (mode == 2)
        fma_probe_kernel<2><<<ctas, PROBE_THREADS, 0, st>>>(iters, d_sink, 0.999f, 0.001f);
    else if (mode == 3)
        fma_probe_kernel<3><<<ctas, PROBE_THREADS, 0, st>>>(iters, d_sink, 0.999f, 0.001f);
    else
        fma_probe_kernel<4><<<ctas, PROBE_THREADS, 0, st>>>(iters, d_sink, 0.999f, 0.001f);
    double per_thread = (double)iters * PROBE_INNER * PROBE_CHAINS * (mode == 0 ? 1.0 : 2.0);
    return per_thread * PROBE_THREADS * ctas;
}

}  // namespace sfmb200
