// pgi_kernels.cuh — batched sm_100a kernels of the hypothesis-verification path (SURVEY §2.3 K0-K8).
//
//   K0 build_correspondences   a1  createCorrespondenceMatrix          pose_graph_builder.h:864-938
//   K1 score_hypotheses        a2-a6  test + getInliers fused          graph_traversal.h:136-168, :194-233
//   K2 fivept_first_solution   a7  cv::findEssentialMat(RANSAC, thr=inf)  pose_graph_builder.h:1013-1020
//   K4 fallback_solve          a8  minimal five-point solves of the robust loop   pose_graph_builder.h:1037-1044
//   K5 fallback_score          a8  scoring / LO refit / termination of the robust loop
//   K3 decompose_vote          a9-a11 + verdict packing (K8)           pose_utils.h:144-252, pose_graph_builder.h:1069-1075
//
// Data layout in HBM: correspondences are one contiguous FP64 array of [x1 y1 x2 y2] rows (32 B per
// correspondence, 16-B aligned => one LDG.128 pair per row), pair k owning rows corr_offset[k]..corr_offset[k+1].
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/pgi.h"
#include "pgi_math.cuh"

namespace pgi {

constexpr int kCtaThreads = 256;
constexpr int kK1Rows = 4;            // rows per thread and tile in K1 (8 x 32 B of loads in flight per thread)
constexpr int kFbChunk = 125;         // fallback iterations solved per K4 launch
constexpr int kLoRounds = 4;
constexpr int kLoMinInliers = 9;
constexpr int kDkMaxSweeps = 200;
constexpr double kDkTolSq = 1e-22;
constexpr double kLegacyDkTolSq = 1e-22;  // K2: Durand-Kerner stops at convergence instead of cv::solvePoly's fixed 1000 sweeps

enum : uint32_t {
    ST_HAVE_HYP = 1u,       // pair had >= 1 hypothesis in this wave
    ST_TEST_PASSED = 2u,    // last hypothesis passed InTraversalPoseTester::test
    ST_NEED_5PT = 4u,       // path branch continues into the five-point solve
    ST_PATH_OK = 8u,        // path branch succeeded (inlierNumber >= minInliers)
    ST_NEED_FB = 16u,       // fallback must run
    ST_FB_ACTIVE = 32u,     // fallback loop still iterating
    ST_FB_RAN = 64u,
    ST_HAVE_E = 128u,       // state.E is valid and must be decomposed
    ST_5PT_NOMODEL = 256u
};

// Per-wave-slot working state (device only).
struct SlotState {
    double E[9];
    unsigned long long bestCost;  // fixed-point MSAC cost of the best model so far (~0ull: none)
    double bestE[9];
    uint32_t flags;
    uint32_t testCount;
    uint32_t pathInliers;
    uint32_t inlierCount;
    int32_t bestInl;
    int32_t maxIters;
    int32_t it;
    uint32_t models;
    uint32_t tableIdx;
    uint32_t pad;
};

struct WaveArgs {
    // registered pairs
    const double *corr;        // sum N x 4
    const uint64_t *offset;    // n_pairs + 1
    const double *thr;         // n_pairs
    const uint32_t *pairTable; // n_pairs: sampler/iters table index of the pair's N
    // sampler tables
    const uint32_t *samplerTab;   // tables x maxIters x 5
    const uint16_t *itersTab;     // concatenated (N+1) tables
    const uint64_t *itersTabOff;  // tables
    // wave
    uint32_t n;
    const uint32_t *pairId;     // n
    const uint32_t *hypOffset;  // n + 1
    const double *hyp;          // sum H x 7
    SlotState *state;           // n
    uint32_t *bits;             // n x bitsStride words: inlier bit mask of the path branch
    uint32_t bitsStride;
    uint8_t *masks;             // optional: concatenated byte masks
    const uint64_t *maskOffset; // n + 1 (rows, wave-local)
    pgi_verdict *verdicts;      // n
    uint32_t flags;
    uint32_t minInliers;
    uint32_t testMinInliers;
    uint32_t fbMaxIters;
    double thrMultiplier;
    double thrOverride;        // the tester threshold of every pair when hasThrOverride (pgi_test_pose), whatever its value
    uint32_t hasThrOverride;   // 0: the tester threshold is thrMultiplier * thr[pair]
    // fallback scratch
    double *fbSols;     // n x kFbChunk x 90
    float4 *fbSolsF;    // n x kFbChunk x 10 models x 3 float4 (FP32 copy for the certificate)
    uint8_t *fbCounts;  // n x kFbChunk
    unsigned long long *counters;  // [0] corr evals, [1] fallback pairs, [2] fallback models
    uint32_t *k3Scratch;  // n x 8: votes[4], arrival ticket of the K3 point-range CTAs (all zero between launches)
    uint32_t *dkList;     // n x kFbChunk: (pair, iteration) slots of the chunk whose degree-10 polynomial awaits its roots
    uint32_t *dkCtl;      // [0] entries in dkList, [1] next entry to hand out (zeroed before every chunk)
};

// ---------------------------------------------------------------------------------------------
// K0: createCorrespondenceMatrix on the device from the compact layout (SURVEY §8f-1).
// One thread per correspondence; keypoint gathers hit L2 (<= 64 KB per view).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k0_build_correspondences(
    const double *__restrict__ focal, const double *__restrict__ sizeWH, const uint64_t *__restrict__ kpOffset,
    const float2 *__restrict__ kp, uint64_t nPairs, const uint2 *__restrict__ pairViews,
    const uint64_t *__restrict__ mOffset, const uint2 *__restrict__ matches, double thrPx, double4 *__restrict__ corr,
    double *__restrict__ thrNorm)
{
    const uint64_t p = blockIdx.y + (uint64_t)blockIdx.z * gridDim.y;
    if (p >= nPairs) return;
    const uint2 v = pairViews[p];
    const double f = focal[v.x];  // K = [f 0 w/2; 0 f h/2; 0 0 1]  pose_graph_builder.h:284-286
    const double cx = sizeWH[2 * v.x] / 2.0, cy = sizeWH[2 * v.x + 1] / 2.0;
    const uint64_t m0 = mOffset[p], m1 = mOffset[p + 1];
    const float2 *ks = kp + kpOffset[v.x];
    const float2 *kd = kp + kpOffset[v.y];
    for (uint64_t i = m0 + blockIdx.x * blockDim.x + threadIdx.x; i < m1; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint2 m = matches[i];
        const float2 a = ks[m.x], b = kd[m.y];
        // destination points are normalised with the SOURCE intrinsics (pose_graph_builder.h:908-912)
        corr[i] = make_double4(((double)a.x - cx) / f, ((double)a.y - cy) / f, ((double)b.x - cx) / f, ((double)b.y - cy) / f);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) thrNorm[p] = thrPx / ((f + f + f + f) / 4.0);  // :934-937
}

// ---------------------------------------------------------------------------------------------
// K1: one CTA per wave pair.  For every hypothesis: E = [t]x R, squared Sampson residual of every
// correspondence (one LDG.128 x2 per row, coalesced 32 B/thread), count under the squared (test) and
// un-squared (getInliers, GT:164) thresholds with warp ballots; the last passing hypothesis' inlier
// bits are kept for the sampler of K2.  HBM-bound: 32 B / correspondence, read once per hypothesis.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kCtaThreads, 3) k1_score_hypotheses(WaveArgs a)
{
    const uint32_t w = blockIdx.x;
    if (w >= a.n) return;
    const uint32_t pid = a.pairId[w];
    const uint64_t r0 = a.offset[pid];
    const uint32_t N = (uint32_t)(a.offset[pid + 1] - r0);
    const double4 *rows = reinterpret_cast<const double4 *>(a.corr) + r0;
    const double thrT = a.hasThrOverride ? a.thrOverride : a.thrMultiplier * a.thr[pid];  // 1.5 * thr_norm  (PGB:800, :964)
    const double thrTsq = thrT * thrT;                 // GT:184
    // two bit buffers per slot: the one being written and the one of the last hypothesis that reached
    // estimatePose (so a later failing hypothesis cannot clobber the sampler's input)
    uint32_t *bitsBase = a.bits + (size_t)w * a.bitsStride * 2;
    uint8_t *mask = (a.flags & PGI_WAVE_MASKS) ? a.masks + a.maskOffset[w] : nullptr;
    const bool noTest = (a.flags & PGI_WAVE_NO_TEST) != 0;

    __shared__ uint32_t sCnt[2][kCtaThreads / 32];
    __shared__ uint32_t sDecision, sValidSel;
    if (threadIdx.x == 0) sValidSel = 0;
    const uint32_t h0 = a.hypOffset[w], h1 = a.hypOffset[w + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    if (mask)
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) mask[i] = 0;

    uint32_t flags = 0, testCount = 0, pathInliers = 0;
    for (uint32_t h = h0; h < h1; ++h) {
        __syncthreads();  // sValidSel of the previous hypothesis is final
        // every thread derives E = [t]x R itself (identical operations, broadcast loads): no serial section
        double E[9];
        {
            double qt[7];
#pragma unroll
            for (int k = 0; k < 7; k++) qt[k] = a.hyp[7 * (size_t)h + k];
            essentialFromPose(qt, E);
        }
        const uint32_t cur = 1u - sValidSel;
        uint32_t *bits = bitsBase + (size_t)cur * a.bitsStride;
        uint32_t cTest = 0, cInl = 0;
        // Tiles of kK1Rows rows per thread: all loads of a tile are issued before any arithmetic (8 x 32 B in flight
        // per thread), then the residuals are classified.  The FP64 division of graph_traversal.h:114 is only
        // executed when the comparison is not already decided by  r^2  vs  thr * denom  with a 2^-50 guard band
        // (fl(r2/den) < T  is implied by  r2 < T den (1 - 2^-50)  and excluded by  r2 > T den (1 + 2^-50)), so the
        // result is bit-identical to dividing every time.
        const uint32_t tileRows = kK1Rows * kCtaThreads;
        for (uint32_t base = 0; base < N; base += tileRows) {
            double4 c[kK1Rows];
#pragma unroll
            for (int u = 0; u < kK1Rows; u++) {
                const uint32_t i = base + u * kCtaThreads + threadIdx.x;
                c[u] = i < N ? rows[i] : make_double4(0.0, 0.0, 0.0, 0.0);
            }
#pragma unroll
            for (int u = 0; u < kK1Rows; u++) {
                const uint32_t i = base + u * kCtaThreads + threadIdx.x;
                if (base + u * kCtaThreads >= N) break;  // warp-uniform: whole row group past the end
                bool t = false, in = false;
                if (i < N) {
                    const double x1 = c[u].x, y1 = c[u].y, x2 = c[u].z, y2 = c[u].w;
                    const double rxc = E[0] * x2 + E[3] * y2 + E[6];
                    const double ryc = E[1] * x2 + E[4] * y2 + E[7];
                    const double rwc = E[2] * x2 + E[5] * y2 + E[8];
                    const double r = (x1 * rxc + y1 * ryc + rwc);
                    const double rx = E[0] * x1 + E[1] * y1 + E[2];
                    const double ry = E[3] * x1 + E[4] * y1 + E[5];
                    const double r2 = r * r;
                    const double den = rxc * rxc + ryc * ryc + rx * rx + ry * ry;
                    const double q1 = thrTsq * den, q2 = thrT * den;
                    const double lo = 1.0 - 8.8817841970012523e-16, hi = 1.0 + 8.8817841970012523e-16;  // 1 -+ 2^-50
                    const bool sure1 = q1 > 1e-290 && (r2 < q1 * lo || r2 > q1 * hi);
                    const bool sure2 = q2 > 1e-290 && (r2 < q2 * lo || r2 > q2 * hi);
                    if (sure1 && sure2) {
                        t = r2 < q1;
                        in = r2 < q2;
                    } else {
                        const double sres = r2 / den;  // the reference's expression, evaluated only near a boundary
                        t = sres < thrTsq;             // GT:214
                        in = sres < thrT;              // GT:164 (un-squared threshold, reproduced)
                    }
                }
                const uint32_t bt = __ballot_sync(0xffffffffu, t);
                const uint32_t bi = __ballot_sync(0xffffffffu, in);
                if (lane == 0) {
                    cTest += __popc(bt);
                    cInl += __popc(bi);
                    // only words below ceil(N/32) exist for this pair (a row group past N would spill into the next
                    // bit buffer / slot); lane 0's i is the first row of the 32-row group
                    if (i < N) bits[i >> 5] = bi;
                }
            }
        }
        if (lane == 0) { sCnt[0][warp] = cTest; sCnt[1][warp] = cInl; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0, in = 0;
            for (int k = 0; k < kCtaThreads / 32; k++) { t += sCnt[0][k]; in += sCnt[1][k]; }
            const bool passed = noTest || (t >= a.testMinInliers);  // GT:221
            testCount = t < a.testMinInliers ? t : a.testMinInliers;  // early exit leaves inlierNumber_ at the minimum
            // the loop of PGB:974-1029 lets the LAST guess decide; guesses are the hypotheses that passed
            if (passed) {
                flags = ST_HAVE_HYP | ST_TEST_PASSED;
                pathInliers = in;
            } else
                flags |= ST_HAVE_HYP;
            sDecision = passed ? 1u : 0u;
            atomicAdd(a.counters + 0, (unsigned long long)N);
        }
        __syncthreads();
        // PGB:1000-1009: the mask accumulates the inliers of every guess that reached estimatePose
        if (mask && sDecision)
            for (uint32_t i = threadIdx.x; i < N; i += blockDim.x)
                if ((bits[i >> 5] >> (i & 31)) & 1u) mask[i] = 1;
        __syncthreads();
        if (threadIdx.x == 0 && sDecision) sValidSel = cur;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        SlotState &s = a.state[w];
        s.testCount = testCount;
        s.pathInliers = (flags & ST_TEST_PASSED) ? pathInliers : 0u;
        s.inlierCount = 0;
        s.tableIdx = a.pairTable[pid];
        s.pad = sValidSel;  // which bit buffer K2 samples from
        s.models = 0;
        s.it = 0;
        if ((flags & ST_TEST_PASSED) && pathInliers >= 5) flags |= ST_NEED_5PT;  // ptsetreg: count < modelPoints -> fail
        s.flags = flags;
    }
}

// ---------------------------------------------------------------------------------------------
// K1, streaming form (the default on full waves): persistent CTAs, the correspondences travel HBM -> shared memory as
// 1-D bulk async copies (cp.async.bulk, the TMA engine without a tensor map: a pair's rows are one contiguous run of 32 B
// records) through a ring of kK1Stages x kK1TileRows-row tiles armed on mbarriers, so kK1Stages - 1 tiles (128 KB) are in
// flight per SM while the warps score the tile that has landed.  Same arithmetic, same ballots, same per-slot
// bookkeeping as k1_score_hypotheses; waves that ask for byte masks keep the direct-load kernel.
// ---------------------------------------------------------------------------------------------
// Tile shape.  The first version scored one row per thread and tile (1 024 threads, 1 024-row tiles): ncu counted 237
// thread instructions per scored row, three quarters of them the per-tile bookkeeping (barrier, cursor, ballots) — the
// kernel was issue-bound at 0.34 of the HBM rate.  A tile now holds a whole 2 000-row pair (64 KB) and every thread
// scores kK1RowsPerThread rows of it, so the bookkeeping is paid once per 4 rows and the rows give the FP64 pipe
// independent work.
#ifndef PGI_K1_TILE_ROWS
#define PGI_K1_TILE_ROWS 2048
#endif
#ifndef PGI_K1_THREADS
#define PGI_K1_THREADS 512
#endif
#ifndef PGI_K1_STAGES
#define PGI_K1_STAGES 3
#endif
constexpr int kK1Stages = PGI_K1_STAGES;
constexpr int kK1TileRows = PGI_K1_TILE_ROWS;   // 64 KB per stage
constexpr int kK1TmaThreads = PGI_K1_THREADS;
constexpr int kK1RowsPerThread = kK1TileRows / kK1TmaThreads;
static_assert(kK1TileRows % kK1TmaThreads == 0 && kK1TmaThreads % 32 == 0, "tile rows must be a multiple of the CTA size");

__device__ __forceinline__ uint32_t smemAddr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbarInit(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smemAddr(bar)), "r"(count));
}
__device__ __forceinline__ void mbarExpectTx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smemAddr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarWait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smemAddr(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulkLoad(void *dstSmem, const void *srcGlobal, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smemAddr(dstSmem)),
                 "l"(srcGlobal), "r"(bytes), "r"(smemAddr(bar))
                 : "memory");
}

// Work of one CTA: the wave slots blockIdx.x, blockIdx.x + gridDim.x, ...  Their descriptors (row range, hypothesis
// range, threshold, E of the first hypothesis) are fetched kK1MetaSlots at a time by as many threads in parallel and kept
// in shared memory, so the streaming loop below never waits on a chain of dependent global loads (pair id -> offsets ->
// threshold / hypothesis) between two tiles.
constexpr int kK1MetaSlots = 128;
struct K1Meta {
    uint64_t r0[kK1MetaSlots];
    double thr[kK1MetaSlots];
    double E[kK1MetaSlots][9];
    uint32_t N[kK1MetaSlots], h0[kK1MetaSlots], h1[kK1MetaSlots], table[kK1MetaSlots];
};
struct K1Cursor {  // walks the (slot, hypothesis, tile) items of the descriptors in shared memory
    uint32_t k, h, row0;
};
__device__ __forceinline__ bool k1Next(const K1Meta &m, uint32_t nSlots, K1Cursor &c)
{
    if (c.h < m.h1[c.k] && c.row0 + kK1TileRows < m.N[c.k]) { c.row0 += kK1TileRows; return true; }
    if (c.h + 1 < m.h1[c.k]) { ++c.h; c.row0 = 0; return true; }
    if (++c.k >= nSlots) return false;
    c.h = m.h0[c.k];
    c.row0 = 0;
    return true;
}

__global__ void __launch_bounds__(kK1TmaThreads, 1) k1_score_hypotheses_tma(WaveArgs a)
{
    extern __shared__ __align__(128) unsigned char k1Smem[];
    double4 *tiles = reinterpret_cast<double4 *>(k1Smem);
    K1Meta &meta = *reinterpret_cast<K1Meta *>(k1Smem + (size_t)kK1Stages * kK1TileRows * 32);
    __shared__ __align__(8) uint64_t sFull[kK1Stages];
    __shared__ uint32_t sCnt[2][kK1TmaThreads / 32];
    __shared__ uint32_t sValidSel;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kK1Stages; s++) mbarInit(&sFull[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        sValidSel = 0;
    }
    __syncthreads();
    const bool noTest = (a.flags & PGI_WAVE_NO_TEST) != 0;
    uint32_t issued = 0, consumed = 0;  // items whose copy was started (thread 0) / that were scored (all threads)

    for (uint32_t slotBase = 0; blockIdx.x + (uint64_t)slotBase * gridDim.x < a.n; slotBase += kK1MetaSlots) {
        // ---- descriptors of the next kK1MetaSlots slots, one thread per slot
        const uint32_t remaining = (uint32_t)((a.n - blockIdx.x - (uint64_t)slotBase * gridDim.x + gridDim.x - 1) / gridDim.x);
        const uint32_t nSlots = remaining < (uint32_t)kK1MetaSlots ? remaining : (uint32_t)kK1MetaSlots;
        if (threadIdx.x < nSlots) {
            const uint32_t t = threadIdx.x, w = blockIdx.x + (slotBase + t) * gridDim.x;
            const uint32_t pid = a.pairId[w];
            const uint64_t r0 = a.offset[pid];
            meta.r0[t] = r0;
            meta.N[t] = (uint32_t)(a.offset[pid + 1] - r0);
            meta.h0[t] = a.hypOffset[w];
            meta.h1[t] = a.hypOffset[w + 1];
            meta.thr[t] = a.hasThrOverride ? a.thrOverride : a.thrMultiplier * a.thr[pid];  // 1.5 * thr_norm  (PGB:800, :964)
            meta.table[t] = a.pairTable[pid];
            if (meta.h1[t] > meta.h0[t]) {
                double qt[7], E[9];
#pragma unroll
                for (int k = 0; k < 7; k++) qt[k] = a.hyp[7 * (size_t)meta.h0[t] + k];
                essentialFromPose(qt, E);
#pragma unroll
                for (int k = 0; k < 9; k++) meta.E[t][k] = E[k];
            }
        }
        __syncthreads();

        K1Cursor prod{0, meta.h0[0], 0}, cons{0, meta.h0[0], 0};
        bool prodLive = true, consLive = true;
        auto issue = [&]() {  // thread 0: arm the stage and start the copy of the producer cursor's tile
            const uint32_t N = meta.N[prod.k];
            const uint32_t rows = prod.h < meta.h1[prod.k] && prod.row0 < N ? min((uint32_t)kK1TileRows, N - prod.row0) : 0u;
            const int st = issued % kK1Stages;
            if (rows) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // earlier generic reads of the stage precede the async write
                mbarExpectTx(&sFull[st], rows * 32u);
                bulkLoad(tiles + (size_t)st * kK1TileRows, reinterpret_cast<const double4 *>(a.corr) + meta.r0[prod.k] + prod.row0, rows * 32u,
                         &sFull[st]);
            } else
                mbarExpectTx(&sFull[st], 0u);  // empty item (no hypothesis / no rows): the phase still completes
            ++issued;
            prodLive = k1Next(meta, nSlots, prod);
        };
        if (threadIdx.x == 0)
            for (int k = 0; k < kK1Stages - 1 && prodLive; k++) issue();

        uint32_t flags = 0, testCount = 0, pathInliers = 0, cTest = 0, cInl = 0;  // per slot (thread 0) / per hypothesis (lane 0)
        double E[9];
        double thrT = 0.0, thrTsq = 0.0;
        bool slotStart = true, hypStart = true;
        while (consLive) {
            const uint32_t k = cons.k, N = meta.N[k];
            const uint32_t w = blockIdx.x + (slotBase + k) * gridDim.x;
            if (slotStart) {
                thrT = meta.thr[k];
                thrTsq = thrT * thrT;  // GT:184
                flags = testCount = pathInliers = 0;
                slotStart = false;
            }
            const bool haveHyp = cons.h < meta.h1[k];
            if (haveHyp && hypStart) {
                if (cons.h == meta.h0[k]) {
#pragma unroll
                    for (int q = 0; q < 9; q++) E[q] = meta.E[k][q];
                } else {
                    double qt[7];
#pragma unroll
                    for (int q = 0; q < 7; q++) qt[q] = a.hyp[7 * (size_t)cons.h + q];
                    essentialFromPose(qt, E);
                }
                cTest = cInl = 0;
                hypStart = false;
            }
            if (threadIdx.x == 0 && prodLive) issue();  // refills the stage consumed in the previous iteration
            const int st = consumed % kK1Stages;
            mbarWait(&sFull[st], (consumed / kK1Stages) & 1u);
            ++consumed;
            const uint32_t rows = haveHyp && cons.row0 < N ? min((uint32_t)kK1TileRows, N - cons.row0) : 0u;
            if (rows) {
                const double4 *tile = tiles + (size_t)st * kK1TileRows;
                uint32_t *bits = a.bits + ((size_t)w * 2 + (1u - sValidSel)) * a.bitsStride;
#pragma unroll
                for (int rr = 0; rr < kK1RowsPerThread; rr++) {
                const uint32_t li = threadIdx.x + (uint32_t)rr * kK1TmaThreads;  // rows li of the tile: one 32-row group per warp and rr
                if ((li & ~31u) < rows) {          // warp-uniform: the warp's 32-row group starts inside the tile
                    bool t = false, in = false;
                    if (li < rows) {
                        const double4 c = tile[li];
                        const double x1 = c.x, y1 = c.y, x2 = c.z, y2 = c.w;
                        const double rxc = E[0] * x2 + E[3] * y2 + E[6];
                        const double ryc = E[1] * x2 + E[4] * y2 + E[7];
                        const double rwc = E[2] * x2 + E[5] * y2 + E[8];
                        const double r = (x1 * rxc + y1 * ryc + rwc);
                        const double rx = E[0] * x1 + E[1] * y1 + E[2];
                        const double ry = E[3] * x1 + E[4] * y1 + E[5];
                        const double r2 = r * r;
                        const double den = rxc * rxc + ryc * ryc + rx * rx + ry * ry;
                        const double q1 = thrTsq * den, q2 = thrT * den;
                        const double lo = 1.0 - 8.8817841970012523e-16, hi = 1.0 + 8.8817841970012523e-16;  // 1 -+ 2^-50 (see k1_score_hypotheses)
                        const bool sure1 = q1 > 1e-290 && (r2 < q1 * lo || r2 > q1 * hi);
                        const bool sure2 = q2 > 1e-290 && (r2 < q2 * lo || r2 > q2 * hi);
                        if (sure1 && sure2) {
                            t = r2 < q1;
                            in = r2 < q2;
                        } else {
                            const double sres = r2 / den;
                            t = sres < thrTsq;  // GT:214
                            in = sres < thrT;   // GT:164 (un-squared threshold, reproduced)
                        }
                    }
                    const uint32_t bt = __ballot_sync(0xffffffffu, t);
                    const uint32_t bi = __ballot_sync(0xffffffffu, in);
                    if (lane == 0) {
                        cTest += __popc(bt);
                        cInl += __popc(bi);
                        bits[(cons.row0 + li) >> 5] = bi;
                    }
                }
                }
            }
            const bool hypEnd = haveHyp && cons.row0 + kK1TileRows >= N;
            const bool slotEnd = !haveHyp || (hypEnd && cons.h + 1 >= meta.h1[k]);
            if (hypEnd) {
                if (lane == 0) { sCnt[0][warp] = cTest; sCnt[1][warp] = cInl; }
                __syncthreads();
                if (threadIdx.x == 0) {
                    uint32_t t = 0, in = 0;
                    for (int q = 0; q < kK1TmaThreads / 32; q++) { t += sCnt[0][q]; in += sCnt[1][q]; }
                    const bool passed = noTest || (t >= a.testMinInliers);    // GT:221
                    testCount = t < a.testMinInliers ? t : a.testMinInliers;  // early exit leaves inlierNumber_ at the minimum
                    if (passed) {
                        flags = ST_HAVE_HYP | ST_TEST_PASSED;
                        pathInliers = in;
                        sValidSel = 1u - sValidSel;  // the buffer just written becomes the sampler's input
                    } else
                        flags |= ST_HAVE_HYP;
                    atomicAdd(a.counters + 0, (unsigned long long)N);
                }
                hypStart = true;
            }
            if (slotEnd && threadIdx.x == 0) {
                SlotState &s = a.state[w];
                s.testCount = testCount;
                s.pathInliers = (flags & ST_TEST_PASSED) ? pathInliers : 0u;
                s.inlierCount = 0;
                s.tableIdx = meta.table[k];
                s.pad = sValidSel;  // which bit buffer K2 samples from
                s.models = 0;
                s.it = 0;
                uint32_t f = flags;
                if ((f & ST_TEST_PASSED) && pathInliers >= 5) f |= ST_NEED_5PT;  // ptsetreg: count < modelPoints -> fail
                s.flags = f;
                sValidSel = 0;
            }
            if (slotEnd) slotStart = true;
            __syncthreads();  // every thread is done with the stage (and sees sValidSel) before it is refilled / reused
            consLive = k1Next(meta, nSlots, cons);
        }
        // all items of this round were issued and consumed; the descriptors may be overwritten
    }
}

// r-th set bit (0-based) of a bit mask.
__device__ inline uint32_t selectRank(const uint32_t *bits, uint32_t nWords, uint32_t r)
{
    uint32_t acc = 0;
    for (uint32_t wI = 0; wI < nWords; ++wI) {
        const uint32_t c = __popc(bits[wI]);
        if (acc + c > r) {
            uint32_t word = bits[wI];
            for (uint32_t k = r - acc; k > 0; --k) word &= word - 1;
            return wI * 32 + (__ffs(word) - 1);
        }
        acc += c;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// K2: legacy cv::findEssentialMat(RANSAC, threshold = DBL_MAX) on the inliers of the hypothesis:
// MWC RNG(2^64-1) draws 5 distinct ranks in [0,k); the first solution of the first sample that yields
// a model wins and every point is its inlier (SURVEY App. B.2).  One thread per wave pair (a warp of its own on
// small waves, where the kernel is a latency chain).  The Durand-Kerner
// root solve stops at convergence (kLegacyDkTolSq) rather than burning cv::solvePoly's 1000 fixed sweeps; polynomials
// whose sweeps fall into an exact floating-point cycle jump to the state sweep 1000 would produce (Brent's cycle
// detection on the bitwise root state, dkSolveFixed<., true>: identical to running every sweep).  The few % that neither
// converge nor cycle run all 1000 sweeps (3 us each) and set the latency of the wave round they are in — same
// trajectory, same root order, values equal to cv2's to ~1e-13 (the oracle does the same and is pinned to cv2).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k2_fivept_first_solution(WaveArgs a, int onePairPerWarp)
{
    __shared__ double sWs[kFivePointWs];  // work arrays of the lone lane (onePairPerWarp)
    if (onePairPerWarp && threadIdx.x != 0) return;
    const uint32_t w = onePairPerWarp ? blockIdx.x : blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= a.n) return;
    SlotState &s = a.state[w];
    uint32_t flags = s.flags;
    if (flags & ST_NEED_5PT) {
        const uint32_t pid = a.pairId[w];
        const uint64_t r0 = a.offset[pid];
        const uint32_t N = (uint32_t)(a.offset[pid + 1] - r0);
        const double4 *rows = reinterpret_cast<const double4 *>(a.corr) + r0;
        const uint32_t *bits = a.bits + ((size_t)w * 2 + s.pad) * a.bitsStride;
        const uint32_t nWords = (N + 31) / 32;
        const int k = (int)s.pathInliers;
        double x1[10], x2[10], E[9];
        bool found = false;
        if ((uint32_t)k < a.minInliers) {
            // PGB:1028 fails whatever the kernel returns; E is overwritten by the fallback (PGB:1037).  The
            // 1000-sweep solve is skipped and inlierNumber_ reported as k (what a successful solve gives).
            s.inlierCount = (uint32_t)k;
            flags &= ~ST_NEED_5PT;
        } else if (k == 5) {
            for (int i = 0; i < 5; i++) {
                const double4 c = rows[selectRank(bits, nWords, i)];
                x1[2 * i] = c.x; x1[2 * i + 1] = c.y; x2[2 * i] = c.z; x2[2 * i + 1] = c.w;
            }
            found = (onePairPerWarp ? fivePoint<true, true>(x1, x2, E, 1, 1000, kLegacyDkTolSq, sWs)
                                    : fivePoint<true>(x1, x2, E, 1, 1000, kLegacyDkTolSq)) > 0;
        } else {
            CvRng rng((uint64_t)-1);
            for (int iter = 0; iter < 1000 && !found; iter++) {
                int idx[5];
                for (int i = 0; i < 5; ++i) {
                    int idx_i;
                    for (;;) {
                        idx_i = rng.uniform(0, k);
                        bool dup = false;
                        for (int j = 0; j < i; j++) dup |= (idx[j] == idx_i);
                        if (!dup) break;
                    }
                    idx[i] = idx_i;
                    const double4 c = rows[selectRank(bits, nWords, (uint32_t)idx_i)];
                    x1[2 * i] = c.x; x1[2 * i + 1] = c.y; x2[2 * i] = c.z; x2[2 * i + 1] = c.w;
                }
                // the RANSAC loop keeps the first solution that has inliers at all, i.e. the first finite one
                found = (onePairPerWarp ? fivePoint<true, true>(x1, x2, E, 1, 1000, kLegacyDkTolSq, sWs, true)
                                        : fivePoint<true>(x1, x2, E, 1, 1000, kLegacyDkTolSq, nullptr, true)) > 0;
            }
        }
        if (!(flags & ST_NEED_5PT)) {
        } else if (found) {
            for (int q = 0; q < 9; q++) s.E[q] = E[q];
            s.inlierCount = (uint32_t)k;  // threshold^2 = inf: every point is an inlier  (PGB:1022)
            if ((uint32_t)k >= a.minInliers) flags |= ST_PATH_OK | ST_HAVE_E;  // PGB:1028
        } else {
            flags |= ST_5PT_NOMODEL;
            s.inlierCount = 0;
        }
    }
    if (!(flags & ST_PATH_OK) && (a.flags & PGI_WAVE_FALLBACK)) {
        const uint32_t pid = a.pairId[w];
        const uint32_t N = (uint32_t)(a.offset[pid + 1] - a.offset[pid]);
        flags |= ST_NEED_FB | ST_FB_RAN;
        if (N >= 5) flags |= ST_FB_ACTIVE;
        s.bestCost = ~0ull;
        s.bestInl = 0;
        s.maxIters = (int)a.fbMaxIters;
        s.it = 0;
        s.models = 0;
        for (int q = 0; q < 9; q++) s.bestE[q] = 0.0;
        atomicAdd(a.counters + 1, 1ull);
    }
    s.flags = flags;
}

// ---------------------------------------------------------------------------------------------
// K4: minimal solves of the fallback, one per (wave pair, iteration of the current chunk).
// The uniform sampler's sequence depends on N only (persistent-pool partial Fisher-Yates driven by
// cv::RNG(0), SURVEY App. B.5), so the samples come from a per-N table built at registration.
// The Durand-Kerner root solve is ~45 % of a minimal solve and its sweep count differs from polynomial to
// polynomial, so with one thread per solve a warp runs as long as its slowest lane (17 of 32 lanes active in the
// sweeps, measured).  K4 is therefore three kernels:
//   K4a  one thread per (pair, iteration): sample -> null space -> elimination -> polynomial; parks EE (36), b (39),
//        c (11) and the degree in the slot's 90-double solution record and appends the slot to a work list;
//   K4b  persistent lanes: every lane pulls the next polynomial from the list the moment its current one has
//        converged (register-resident roots, the same dkSweep sequence per polynomial) -> roots into the slot's
//        FP32-record area (20 doubles);
//   K4c  one thread per (pair, iteration): roots -> essential matrices, overwriting the parked data with the
//        solutions (9 doubles each, as fivePoint() returns them) and their FP32 copies for K5.
// Per polynomial the arithmetic is the same sequence of operations as fivePoint(): bit-identical solutions.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool k4SlotActive(const WaveArgs &a, int chunk, uint32_t g, uint32_t &w, uint32_t &j)
{
    w = g / kFbChunk;
    j = g % kFbChunk;
    if (w >= a.n) return false;
    const SlotState &s = a.state[w];
    if (!(s.flags & ST_FB_ACTIVE)) return false;
    return chunk * kFbChunk + (int)j < s.maxIters;
}

__global__ void __launch_bounds__(128, 4) k4a_polynomial(WaveArgs a, int chunk)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t w, j;
    if (!k4SlotActive(a, chunk, g, w, j)) return;
    const SlotState &s = a.state[w];
    const int it = chunk * kFbChunk + (int)j;
    const uint32_t pid = a.pairId[w];
    const double4 *rows = reinterpret_cast<const double4 *>(a.corr) + a.offset[pid];
    const uint32_t *smp = a.samplerTab + ((size_t)s.tableIdx * a.fbMaxIters + it) * 5;
    double x1[10], x2[10];
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const double4 c = rows[smp[i]];
        x1[2 * i] = c.x; x1[2 * i + 1] = c.y; x2[2 * i] = c.z; x2[2 * i + 1] = c.w;
    }
    double Vt[81], A[200], A1[100], inv[100], b[39], R6[60], c[11];
    const int n = fivePointFront<false>(x1, x2, Vt, A, A1, inv, b, R6, c);
    const size_t slot = (size_t)w * kFbChunk + j;
    double *park = a.fbSols + slot * 90;
    for (int k = 0; k < 36; k++) park[k] = Vt[45 + k];
    for (int k = 0; k < 39; k++) park[36 + k] = b[k];
    for (int k = 0; k < 11; k++) park[75 + k] = c[k];
    park[86] = (double)n;
    if (n == 10) {
        a.dkList[atomicAdd(a.dkCtl, 1u)] = (uint32_t)slot;
    } else {  // vanishing leading coefficients (rare): generic-degree solve in place
        Cx roots[10];
        dkSolveGeneric(c, n, roots, kDkMaxSweeps, kDkTolSq);
        double *r = reinterpret_cast<double *>(a.fbSolsF + slot * 30);
        for (int k = 0; k < n; k++) { r[2 * k] = roots[k].re; r[2 * k + 1] = roots[k].im; }
    }
}

__global__ void __launch_bounds__(128, 4) k4b_roots(WaveArgs a)
{
    // ~2 % of the polynomials never reach the tolerance: their sweeps fall into a short floating-point cycle and would
    // hold a lane (and the end of the kernel) for all kDkMaxSweeps sweeps.  Brent's cycle detection on the bitwise root
    // state (snapshot in shared memory, one column per lane) jumps to the state sweep kDkMaxSweeps would produce:
    // identical to running every sweep (dkSolveFixed<., true>, checked against the plain loop in the parity tests).
    __shared__ double sSnap[20][128];
    const uint32_t total = a.dkCtl[0];
    Cx roots[10];
    double co[11];
    uint32_t slot = 0;
    int sweeps = 0, power = 1, lam = 0, drain = -1;  // drain >= 0: sweeps left after a detected cycle, no more checks
    bool have = false, exhausted = false;
    for (;;) {
        if (!have && !exhausted) {
            const uint32_t e = atomicAdd(a.dkCtl + 1, 1u);
            if (e < total) {
                slot = a.dkList[e];
                const double *c = a.fbSols + (size_t)slot * 90 + 75;
#pragma unroll
                for (int i = 0; i <= 10; i++) co[i] = c[i];
                Cx p{1, 0};
                const Cx r{1, 1};
#pragma unroll
                for (int i = 0; i < 10; i++) {  // cv::solvePoly's start vector (dkSolveFixed)
                    roots[i] = p;
                    p = cmul(p, r);
                    sSnap[2 * i][threadIdx.x] = roots[i].re;
                    sSnap[2 * i + 1][threadIdx.x] = roots[i].im;
                }
                sweeps = 0; power = 1; lam = 0; drain = -1;
                have = true;
            } else
                exhausted = true;
        }
        if (!__any_sync(0xffffffffu, have)) break;
        if (have) {
            bool finished = false;
            if (drain == 0) {
                finished = true;
            } else {
                const double md = dkSweep<10>(co, roots);
                ++sweeps; ++lam;
                if (drain > 0) {
                    finished = --drain == 0;
                } else if (md <= kDkTolSq || sweeps >= kDkMaxSweeps) {
                    finished = true;
                } else {
                    bool same = true;
#pragma unroll
                    for (int i = 0; i < 10; i++)
                        same &= (__double_as_longlong(roots[i].re) == __double_as_longlong(sSnap[2 * i][threadIdx.x])) &&
                                (__double_as_longlong(roots[i].im) == __double_as_longlong(sSnap[2 * i + 1][threadIdx.x]));
                    if (same) {  // period lam: state(kDkMaxSweeps) == state(sweeps + (kDkMaxSweeps - sweeps) % lam)
                        drain = (kDkMaxSweeps - sweeps) % lam;
                        finished = drain == 0;
                    } else if (power == lam) {
#pragma unroll
                        for (int i = 0; i < 10; i++) {
                            sSnap[2 * i][threadIdx.x] = roots[i].re;
                            sSnap[2 * i + 1][threadIdx.x] = roots[i].im;
                        }
                        power *= 2;
                        lam = 0;
                    }
                }
            }
            if (finished) {
                double *r = reinterpret_cast<double *>(a.fbSolsF + (size_t)slot * 30);
#pragma unroll
                for (int i = 0; i < 10; i++) {
                    r[2 * i] = roots[i].re;
                    r[2 * i + 1] = fabs(roots[i].im) < 1e-100 ? 0.0 : roots[i].im;
                }
                have = false;
            }
        }
    }
}

__global__ void __launch_bounds__(128, 4) k4c_solutions(WaveArgs a, int chunk)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t w, j;
    if (!k4SlotActive(a, chunk, g, w, j)) return;
    const size_t slot = (size_t)w * kFbChunk + j;
    double *out = a.fbSols + slot * 90;
    float4 *outF = a.fbSolsF + slot * 30;
    double EE[36], b[39];
    Cx roots[10];
    for (int k = 0; k < 36; k++) EE[k] = out[k];
    for (int k = 0; k < 39; k++) b[k] = out[36 + k];
    const int n = (int)out[86];
    {
        const double *r = reinterpret_cast<const double *>(outF);
        for (int k = 0; k < n; k++) roots[k] = Cx{r[2 * k], r[2 * k + 1]};
    }
    double E[90];
    const int cnt = fivePointFinish(EE, b, roots, n, E, 10);
    a.fbCounts[slot] = (uint8_t)cnt;
    for (int q = 0; q < cnt; q++) {
        const double *e = E + q * 9;
        for (int k = 0; k < 9; k++) out[q * 9 + k] = e[k];
        outF[q * 3 + 0] = make_float4((float)e[0], (float)e[1], (float)e[2], (float)e[3]);
        outF[q * 3 + 1] = make_float4((float)e[4], (float)e[5], (float)e[6], (float)e[7]);
        outF[q * 3 + 2] = make_float4((float)e[8], 0.f, 0.f, 0.f);
    }
}

// ---------------------------------------------------------------------------------------------
// K5 building blocks.  Every reduction over correspondences is an exact 64-bit fixed-point sum (see
// oracle/pgo_fallback.hpp): terms are produced by IEEE FP64 operations, converted to integers once and
// added with integer arithmetic, so warps/CTAs may reduce in any order (shuffles, shared-memory atomics).
// ---------------------------------------------------------------------------------------------
#ifndef PGI_K5_BATCH
#define PGI_K5_BATCH 16
#endif
#ifndef PGI_K5_SLICES
#define PGI_K5_SLICES 1
#endif
#ifndef PGI_K5_QUEUE
#define PGI_K5_QUEUE 2048
#endif
constexpr uint32_t kK5QueuePts = PGI_K5_QUEUE;  // points per scoring block = entries of a warp's compaction queue (<= 2048: 64 mask bits per lane)
constexpr int kSlices = PGI_K5_SLICES;         // a scoring pass covers 1/kSlices of the pair's points (fixed-point sums: any split is exact)
constexpr int kBatch = PGI_K5_BATCH;                    // fallback iterations scored between two decision points of K5
constexpr double kCostOne = 4294967296.0;     // fixed-point MSAC cost of an outlier (2^32)
constexpr double kLsScale = 1099511627776.0;  // 2^40: fixed-point scale of the normal-equation products

__device__ __forceinline__ unsigned long long warpSumU64(unsigned long long v)
{
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) v += __shfl_down_sync(0xffffffffu, v, s);
    return v;  // valid in lane 0
}

__device__ __forceinline__ uint32_t blockSumU32(uint32_t v, uint32_t *sWarp /*8*/)
{
    v = __reduce_add_sync(0xffffffffu, v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sWarp[warp] = v;
    __syncthreads();
    uint32_t r = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) r += sWarp[k];
    return r;  // valid in all threads
}

// FP32 certificate constants (see scoreModelWarp).
struct F32Consts {
    float rOut;  // |r_f32| above this certifies "outside the truncation band" (see scoreModelWarp)
};

__device__ __forceinline__ void exactTerm(const double4 *rows, uint32_t i, const double *Eg, double thrSq, double truncSq,
                                          double invT, unsigned long long &cost, uint32_t &inl)
{
    double Ed[9];
#pragma unroll
    for (int k = 0; k < 9; k++) Ed[k] = Eg[k];
    const double4 c = rows[i];
    const double rr = sampsonSq(c.x, c.y, c.z, c.w, Ed);
    cost += (rr < truncSq) ? (unsigned long long)(rr * invT * kCostOne) : (unsigned long long)kCostOne;
    inl += (rr < thrSq) ? 1u : 0u;
}

// Score up to two models in one pass over the pair: thread t handles the points t, t + 256, ...
// FP32 (FMA, shared-memory float4 copy) only CERTIFIES that a correspondence is far outside the truncation band
// — then its term is exactly 2^32 and it is no inlier.  With r = x2h^T E x1h the Sampson numerator and
// denom = |(E^T x2h)_xy|^2 + |(E x1h)_xy|^2 <= ||E||_F^2 (|x1h|^2 + |x2h|^2) = D  (models have unit Frobenius norm):
//     |r_f32 - r| <= 4.2e-7 B < eAbs := 1e-6 max_i B_i,  B = (|x1|+|y1|+1)(|x2|+|y2|+1)   (input + 8 FMA roundings)
//  => |r_f32| > rOut := sqrt(truncSq max_i D_i)(1 + 2^-10) + eAbs   implies   r^2 / denom > truncSq.
// Hot loop: one LDS.128, an 8-FMA chain and one compare per (model, correspondence); the uncertain ones only set a
// bit in a per-thread mask.  Afterwards each warp compacts its masks into a shared-memory queue (one prefix scan)
// and the exact FP64 path runs DENSELY, 32 queued correspondences at a time, so the FP64 pipe only sees the few
// percent of evaluations that can matter.  Returns the warp's partial (cost, inliers) per model in lane 0.
__device__ __forceinline__ void exactQueue(const double4 *rows, const double *Eg, unsigned long long mask, uint32_t base,
                                           uint16_t *queue, double thrSq, double truncSq, double invT,
                                           unsigned long long &cost, uint32_t &inl)
{
    // bit j of `mask` = correspondence  base + lane + 32 j  of this lane is uncertain
    const int lane = threadIdx.x & 31;
    const uint32_t mine = (uint32_t)__popcll(mask);
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) return;  // warp-uniform
    uint32_t pos = incl - mine;
    while (mask) {
        const int j = __ffsll((long long)mask) - 1;
        mask &= mask - 1;
        queue[pos++] = (uint16_t)(base + lane + 32 * j);
    }
    __syncwarp();
    for (uint32_t b0 = 0; b0 < total; b0 += 32)
        if (b0 + lane < total) exactTerm(rows, queue[b0 + lane], Eg, thrSq, truncSq, invT, cost, inl);
    __syncwarp();
}

template <bool USE_F32>
__device__ __forceinline__ void scoreModelsWarp(const double4 *rows, const float4 *pts, uint32_t N, const double *Eg0,
                                                const double *Eg1 /*null: one model*/, const float4 *Ef /*3 float4 per model*/,
                                                double thrSq, double truncSq, double invT, float rOut, uint16_t *queue /*2048*/,
                                                unsigned long long costOut[2], uint32_t inlOut[2])
{
    // ONE warp scores the model(s) over all N correspondences (lane l: points l, l + 32, ...), in blocks of kK5QueuePts
    // points so that a lane's uncertainty mask fits 64 bits.  No cross-warp reduction is needed.
    const uint32_t lane = threadIdx.x & 31;
    unsigned long long cost0 = 0, cost1 = 0;
    uint32_t inl0 = 0, inl1 = 0;
    const bool two = Eg1 != nullptr;
    if (USE_F32) {
        const float4 a0 = Ef[0], a1 = Ef[1], a2 = Ef[2];  // e0..e8 of model 0
        float4 b0 = a0, b1 = a1, b2 = a2;
        if (two) { b0 = Ef[3]; b1 = Ef[4]; b2 = Ef[5]; }
        for (uint32_t blk = 0; blk < N; blk += kK5QueuePts) {
            unsigned long long m0 = 0, m1 = 0;
            const uint32_t end = N - blk < kK5QueuePts ? N - blk : kK5QueuePts;  // points in this block
            uint32_t j = 0;
#pragma unroll 4
            for (uint32_t o = lane; o < end; o += 32, ++j) {
                const float4 p = pts[blk + o];
                // model 0: E = [a0.x a0.y a0.z; a0.w a1.x a1.y; a1.z a1.w a2.x]
                const float rxc0 = fmaf(a0.x, p.z, fmaf(a0.w, p.w, a1.z));
                const float ryc0 = fmaf(a0.y, p.z, fmaf(a1.x, p.w, a1.w));
                const float rwc0 = fmaf(a0.z, p.z, fmaf(a1.y, p.w, a2.x));
                const float r0 = fmaf(p.x, rxc0, fmaf(p.y, ryc0, rwc0));
                const float rxc1 = fmaf(b0.x, p.z, fmaf(b0.w, p.w, b1.z));
                const float ryc1 = fmaf(b0.y, p.z, fmaf(b1.x, p.w, b1.w));
                const float rwc1 = fmaf(b0.z, p.z, fmaf(b1.y, p.w, b2.x));
                const float r1 = fmaf(p.x, rxc1, fmaf(p.y, ryc1, rwc1));
                m0 |= (unsigned long long)(!(fabsf(r0) > rOut)) << j;  // NaN stays uncertain
                m1 |= (unsigned long long)(!(fabsf(r1) > rOut)) << j;
            }
            const uint32_t nPts = end > lane ? (end - lane + 31) / 32 : 0u;
            cost0 += (unsigned long long)(nPts - (uint32_t)__popcll(m0)) << 32;
            exactQueue(rows, Eg0, m0, blk, queue, thrSq, truncSq, invT, cost0, inl0);
            if (two) {
                cost1 += (unsigned long long)(nPts - (uint32_t)__popcll(m1)) << 32;
                exactQueue(rows, Eg1, m1, blk, queue, thrSq, truncSq, invT, cost1, inl1);
            }
        }
    } else {
        for (uint32_t i = lane; i < N; i += 32) {
            exactTerm(rows, i, Eg0, thrSq, truncSq, invT, cost0, inl0);
            if (two) exactTerm(rows, i, Eg1, thrSq, truncSq, invT, cost1, inl1);
        }
    }
    costOut[0] = warpSumU64(cost0);
    inlOut[0] = __reduce_add_sync(0xffffffffu, inl0);
    if (two) {
        costOut[1] = warpSumU64(cost1);
        inlOut[1] = __reduce_add_sync(0xffffffffu, inl1);
    }
}

// Symmetric 9x9 cyclic Jacobi, eigenvector of the smallest eigenvalue.  Same rotation sequence and the same
// per-element operations as the oracle's sequential loops; the 9 independent element updates of each phase are
// spread over lanes 0..8 of the calling warp (A, V in shared memory, __syncwarp between phases).  A one-thread
// version of this solve (dependent shared-memory round trips) dominated K5 before.
__device__ inline void smallestEigvec9Warp(double *A /*81 shared*/, double *V /*81 shared*/, double *vOut /*9 shared*/)
{
    const int k = threadIdx.x & 31;
    if (k < 9)
        for (int j = 0; j < 9; j++) V[k * 9 + j] = k == j ? 1.0 : 0.0;
    __syncwarp();
    for (int sweep = 0; sweep < 30; sweep++) {
        double off = 0.0, diag = 0.0;  // every lane evaluates the same sums in the oracle's order
        for (int i = 0; i < 9; i++) {
            diag += A[i * 9 + i] * A[i * 9 + i];
            for (int j = i + 1; j < 9; j++) off += A[i * 9 + j] * A[i * 9 + j];
        }
        if (off <= 1e-30 * diag) break;
        for (int p = 0; p < 8; p++)
            for (int q = p + 1; q < 9; q++) {
                const double apq = A[p * 9 + q];
                if (apq == 0.0) continue;  // warp-uniform
                const double app = A[p * 9 + p], aqq = A[q * 9 + q];
                const double tau = (aqq - app) / (2.0 * apq);
                const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                const double c = 1.0 / sqrt(1.0 + t * t), s = t * c;
                __syncwarp();
                if (k < 9) {  // columns p, q
                    const double akp = A[k * 9 + p], akq = A[k * 9 + q];
                    A[k * 9 + p] = c * akp - s * akq;
                    A[k * 9 + q] = s * akp + c * akq;
                }
                __syncwarp();
                if (k < 9) {  // rows p, q, and the eigenvector accumulation
                    const double apk = A[p * 9 + k], aqk = A[q * 9 + k];
                    A[p * 9 + k] = c * apk - s * aqk;
                    A[q * 9 + k] = s * apk + c * aqk;
                    const double vkp = V[k * 9 + p], vkq = V[k * 9 + q];
                    V[k * 9 + p] = c * vkp - s * vkq;
                    V[k * 9 + q] = s * vkp + c * vkq;
                }
                __syncwarp();
            }
    }
    int m = 0;
    for (int i = 1; i < 9; i++)
        if (A[i * 9 + i] < A[m * 9 + m]) m = i;
    if (k < 9) vOut[k] = V[k * 9 + m];
    __syncwarp();
}

// Least-squares refit on the inliers of Ecur (8-point normal equations in 2^-40 fixed point, essential projection).
// Whole CTA cooperates; result in shared sEls / *sOk (valid after the trailing __syncthreads).
// Pass A marks the inliers once (FP32 certificate first: a point certified outside the truncation band is outside the
// tighter inlier band too; exact FP64 residual otherwise) into a shared bit mask; the accumulation passes only visit
// marked points.
template <bool USE_F32>
__device__ inline void lsRefitBlock(const double4 *rows, const float4 *pts, uint32_t N, const double Ecur[9], double thrSq,
                                    float rOut, uint32_t *sInlBits /*ceil(N/32)*/, long long *sAcc /*45*/, double *sM /*81*/,
                                    double *sV /*81*/, uint32_t *sWarpU, double *sEls /*9*/, int *sOk)
{
    if (threadIdx.x < 45) sAcc[threadIdx.x] = 0;
    uint32_t cntLocal = 0;
    {
        float Ef[9];
#pragma unroll
        for (int k = 0; k < 9; k++) Ef[k] = (float)Ecur[k];
        const uint32_t nRound = (N + 31u) & ~31u;
        for (uint32_t i = threadIdx.x; i < nRound; i += kCtaThreads) {
            bool in = false;
            if (i < N) {
                bool maybe = true;
                if (USE_F32) {
                    const float4 p = pts[i];
                    const float rxc = fmaf(Ef[0], p.z, fmaf(Ef[3], p.w, Ef[6]));
                    const float ryc = fmaf(Ef[1], p.z, fmaf(Ef[4], p.w, Ef[7]));
                    const float rwc = fmaf(Ef[2], p.z, fmaf(Ef[5], p.w, Ef[8]));
                    const float r = fmaf(p.x, rxc, fmaf(p.y, ryc, rwc));
                    maybe = !(fabsf(r) > rOut);
                }
                if (maybe) {
                    const double4 c = rows[i];
                    in = sampsonSq(c.x, c.y, c.z, c.w, Ecur) < thrSq;
                }
            }
            const uint32_t word = __ballot_sync(0xffffffffu, in);
            if ((threadIdx.x & 31) == 0) sInlBits[i >> 5] = word;
            cntLocal += in ? 1u : 0u;
        }
    }
    __syncthreads();
    // 3 sub-passes x 15 upper-triangular entries keep the accumulators in registers
#pragma unroll 1
    for (int sp = 0; sp < 3; sp++) {
        long long acc[15];
#pragma unroll
        for (int e = 0; e < 15; e++) acc[e] = 0;
        for (uint32_t i = threadIdx.x; i < N; i += kCtaThreads) {
            if (!((sInlBits[i >> 5] >> (i & 31)) & 1u)) continue;
            const double4 c = rows[i];
            const double av[9] = {c.z * c.x, c.z * c.y, c.z, c.w * c.x, c.w * c.y, c.w, c.x, c.y, 1.0};
            // entries e = 15 sp .. 15 sp + 14 of the row-major upper triangle (r <= q)
            int e = 0;
#pragma unroll
            for (int r = 0; r < 9; r++)
#pragma unroll
                for (int q = r; q < 9; q++, e++)
                    if (e / 15 == sp) acc[e % 15] += __double2ll_rn(av[r] * av[q] * kLsScale);
        }
#pragma unroll
        for (int e = 0; e < 15; e++) {
            const unsigned long long v = warpSumU64((unsigned long long)acc[e]);
            if ((threadIdx.x & 31) == 0) atomicAdd((unsigned long long *)&sAcc[sp * 15 + e], v);
        }
    }
    const uint32_t cnt = blockSumU32(cntLocal, sWarpU);  // also orders the atomics before the reads below
    if (threadIdx.x < 32 && cnt >= (uint32_t)kLoMinInliers) {  // warp 0
        if (threadIdx.x == 0) {
            int e = 0;
            for (int r = 0; r < 9; r++)
                for (int q = r; q < 9; q++, e++) {
                    const double v = (double)sAcc[e] / kLsScale;
                    sM[r * 9 + q] = v;
                    sM[q * 9 + r] = v;
                }
        }
        __syncwarp();
        smallestEigvec9Warp(sM, sV, sEls);
    }
    if (threadIdx.x == 0) {
        int ok = 0;
        if (cnt >= (uint32_t)kLoMinInliers) {
            double ev[9];
            for (int k = 0; k < 9; k++) ev[k] = sEls[k];
            double U[9], V[9], S[3];
            eigenJacobiSvd<3, true, true>(ev, U, V, S);
            if (S[1] > 0.0) {
                double nrm = 0.0, Eo[9];
                for (int i = 0; i < 3; i++)
                    for (int j = 0; j < 3; j++) {
                        const double x = U[i * 3 + 0] * V[j * 3 + 0] + U[i * 3 + 1] * V[j * 3 + 1];
                        Eo[i * 3 + j] = x;
                        nrm += x * x;
                    }
                nrm = sqrt(nrm);
                ok = 1;
                for (int k = 0; k < 9; k++) {
                    Eo[k] = Eo[k] / nrm;
                    if (Eo[k] != Eo[k]) ok = 0;
                    sEls[k] = Eo[k];
                }
            }
        }
        *sOk = ok;
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// K5: one CTA per wave pair; walks the chunk's iterations IN ORDER (best-so-far / LO / termination semantics of a
// sequential RANSAC).  All models of an iteration are scored by the whole CTA (FP32-certified, exact FP64 where it
// matters), their fixed-point costs land in shared memory through atomics, one barrier, then thread 0 decides.
// ---------------------------------------------------------------------------------------------
template <bool USE_F32>
__device__ __forceinline__ void k5Body(const WaveArgs &a, int chunk, int lastChunk, uint32_t w, float4 *sPts, uint16_t *sQueueAll,
                                       uint32_t queueStride, uint32_t *sInlBits)
{
    SlotState &st = a.state[w];
    const uint32_t flags0 = st.flags;
    const uint32_t pid = a.pairId[w];
    const uint64_t r0 = a.offset[pid];
    const uint32_t N = (uint32_t)(a.offset[pid + 1] - r0);
    const double4 *rows = reinterpret_cast<const double4 *>(a.corr) + r0;
    const double thr = a.thr[pid];
    const double thrSq = thr * thr;
    const double trunc = 1.5 * thr;
    const double truncSq = trunc * trunc;
    const double invT = 1.0 / truncSq;

    __shared__ uint32_t sWarpU[8];
    __shared__ float4 sElsF[3];
    __shared__ unsigned long long sCost[kBatch][10], sLoCost;
    __shared__ uint32_t sInl[kBatch][10], sLoInl, sModels;
    __shared__ int sNextB, sNextPass, sPassStart[kBatch + 1];
    __shared__ uint8_t sCnt[kFbChunk];  // models per iteration of this chunk (written by K4)
    __shared__ float sMaxB[8], sMaxD[8];
    __shared__ long long sAcc[45];
    __shared__ double sM[81], sV[81], sEls[9], sBestE[9];
    __shared__ unsigned long long sBestCost;
    __shared__ int sBestInl, sMaxIters, sOk, sUpdated, sHave;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *sQueue = sQueueAll + (size_t)warp * queueStride;  // this warp's compaction queue (32 x points-per-thread)
    if (threadIdx.x == 0) {
        sBestCost = st.bestCost;
        sBestInl = st.bestInl;
        sMaxIters = st.maxIters;
        sHave = st.bestCost != ~0ull ? 1 : 0;
        for (int k = 0; k < 9; k++) sBestE[k] = st.bestE[k];
    }
    for (int t = threadIdx.x; t < kBatch * 10; t += kCtaThreads) { sCost[t / 10][t % 10] = 0; sInl[t / 10][t % 10] = 0; }
    if (threadIdx.x == 0) sModels = 0;
    if (threadIdx.x < kFbChunk) sCnt[threadIdx.x] = a.fbCounts[(size_t)w * kFbChunk + threadIdx.x];
    const bool active = (flags0 & ST_FB_ACTIVE) != 0;
    const int nSlices = N >= 512u * kSlices ? kSlices : 1;
    const uint32_t slicePer = ((N + nSlices - 1) / nSlices + 31) & ~31u;
    F32Consts fc{3.0e38f};
    if (USE_F32 && active) {
        float maxB = 0.f, maxD = 0.f;
        for (uint32_t i = threadIdx.x; i < N; i += kCtaThreads) {
            const double4 c = rows[i];
            const float4 p = make_float4((float)c.x, (float)c.y, (float)c.z, (float)c.w);
            sPts[i] = p;
            const float B = (fabsf(p.x) + fabsf(p.y) + 1.0f) * (fabsf(p.z) + fabsf(p.w) + 1.0f);
            const float D = (p.x * p.x + p.y * p.y + 1.0f) + (p.z * p.z + p.w * p.w + 1.0f);
            maxB = fmaxf(maxB, B == B ? B : 3.0e38f);  // NaN coordinates: make the certificate unreachable
            maxD = fmaxf(maxD, D == D ? D : 3.0e38f);
        }
#pragma unroll
        for (int sh = 16; sh >= 1; sh >>= 1) {
            maxB = fmaxf(maxB, __shfl_xor_sync(0xffffffffu, maxB, sh));
            maxD = fmaxf(maxD, __shfl_xor_sync(0xffffffffu, maxD, sh));
        }
        if (lane == 0) { sMaxB[warp] = maxB; sMaxD[warp] = maxD; }
    }
    __syncthreads();
    if (USE_F32 && active) {
        float maxB = 0.f, maxD = 0.f;
#pragma unroll
        for (int k = 0; k < 8; k++) { maxB = fmaxf(maxB, sMaxB[k]); maxD = fmaxf(maxD, sMaxD[k]); }
        // computed in FP64 and rounded up: sqrt(truncSq * Dmax (1 + 2^-20)) (1 + 2^-10) + 1e-6 Bmax
        const double rOut = sqrt(truncSq * ((double)maxD * (1.0 + 9.5367431640625e-7))) * (1.0 + 9.765625e-4) + 1e-6 * (double)maxB;
        fc.rOut = (rOut < 1e30 && rOut == rOut) ? (float)(rOut * (1.0 + 1.1920928955078125e-7)) : 3.0e38f;
    }
    uint32_t models = 0;
    int it = st.it;
    if (active) {
        const uint16_t *itTab = a.itersTab + a.itersTabOff[st.tableIdx];
        const int itEnd = (chunk + 1) * kFbChunk;
        while (it < itEnd && it < sMaxIters) {
            // ---- phase 1: score every model of the next kBatch iterations (pure functions of the models) ----------
            int nb = itEnd - it < kBatch ? itEnd - it : kBatch;
            nb = sMaxIters - it < nb ? sMaxIters - it : nb;
            // (iteration, model pair) passes of the batch are handed to the warps dynamically (shared counter): models
            // with many near-inliers take longer in the exact path, a static split left warps idle at the barrier
            if (threadIdx.x == 0) {
                int acc = 0;
                for (int bI = 0; bI < nb; bI++) {
                    sPassStart[bI] = acc;
                    acc += ((sCnt[it + bI - chunk * kFbChunk] + 1) / 2) * nSlices;
                }
                sPassStart[nb] = acc;
                sNextPass = 0;
            }
            __syncthreads();
            for (;;) {
                int pass = 0;
                if (lane == 0) pass = atomicAdd(&sNextPass, 1);
                pass = __shfl_sync(0xffffffffu, pass, 0);
                if (pass >= sPassStart[nb]) break;
                int bI = 0;
                while (pass >= sPassStart[bI + 1]) ++bI;
                const int rel = pass - sPassStart[bI];
                const int q = 2 * (rel / nSlices);
                const uint32_t lo = min((uint32_t)(rel % nSlices) * slicePer, N);
                const uint32_t hi = min(lo + slicePer, N);
                const int j = it + bI - chunk * kFbChunk;
                const int ns = sCnt[j];
                const double *sols = a.fbSols + ((size_t)w * kFbChunk + j) * 90;
                const float4 *solsF = a.fbSolsF + ((size_t)w * kFbChunk + j) * 30;
                unsigned long long c[2];
                uint32_t n[2];
                const bool two = q + 1 < ns;
                scoreModelsWarp<USE_F32>(rows + lo, sPts + lo, hi - lo, sols + q * 9, two ? sols + (q + 1) * 9 : nullptr, solsF + q * 3,
                                         thrSq, truncSq, invT, fc.rOut, sQueue, c, n);
                if (lane == 0) {
                    atomicAdd(&sCost[bI][q], c[0]);
                    atomicAdd(&sInl[bI][q], n[0]);
                    if (two) {
                        atomicAdd(&sCost[bI][q + 1], c[1]);
                        atomicAdd(&sInl[bI][q + 1], n[1]);
                    }
                }
            }
            __syncthreads();
            // ---- phase 2: the sequential best-so-far walk, LO refits interleaved exactly where a sequential
            //      RANSAC would run them; iterations beyond a shrunken maxIters are discarded unscored-in-effect ----
            if (threadIdx.x == 0) sNextB = 0;
            for (;;) {
                if (threadIdx.x == 0) {
                    int bI = sNextB, upd = 0;
                    for (; bI < nb && it + bI < sMaxIters && !upd; ++bI) {
                        const int j = it + bI - chunk * kFbChunk;
                        const int ns = sCnt[j];
                        const double *sols = a.fbSols + ((size_t)w * kFbChunk + j) * 90;
                        for (int q = 0; q < ns; q++)
                            if (sCost[bI][q] < sBestCost) {
                                sBestCost = sCost[bI][q];
                                sBestInl = (int)sInl[bI][q];
                                for (int k = 0; k < 9; k++) sBestE[k] = sols[q * 9 + k];
                                upd = 1;
                                sHave = 1;
                            }
                        sModels += ns;
                    }
                    sNextB = bI;
                    sUpdated = upd;
                }
                __syncthreads();
                if (!sUpdated) break;
                for (int r = 0; r < kLoRounds; r++) {
                    double Eb[9];
#pragma unroll
                    for (int k = 0; k < 9; k++) Eb[k] = sBestE[k];
                    lsRefitBlock<USE_F32>(rows, sPts, N, Eb, thrSq, fc.rOut, sInlBits, sAcc, sM, sV, sWarpU, sEls, &sOk);
                    if (!sOk) break;
                    if (threadIdx.x == 0) {
                        sElsF[0] = make_float4((float)sEls[0], (float)sEls[1], (float)sEls[2], (float)sEls[3]);
                        sElsF[1] = make_float4((float)sEls[4], (float)sEls[5], (float)sEls[6], (float)sEls[7]);
                        sElsF[2] = make_float4((float)sEls[8], 0.f, 0.f, 0.f);
                        sLoCost = 0;
                        sLoInl = 0;
                    }
                    __syncthreads();
                    // the refit model is scored by the 8 warps on disjoint 1/8 slices of the points (fixed-point sums)
                    {
                        const uint32_t per = ((N + 7) / 8 + 31) & ~31u;
                        const uint32_t lo = warp * per < N ? warp * per : N;
                        const uint32_t hi = lo + per < N ? lo + per : N;
                        unsigned long long c[2];
                        uint32_t n[2];
                        scoreModelsWarp<USE_F32>(rows + lo, sPts + lo, hi - lo, sEls, nullptr, sElsF, thrSq, truncSq, invT, fc.rOut,
                                                 sQueue, c, n);
                        if (lane == 0) {
                            atomicAdd(&sLoCost, c[0]);
                            atomicAdd(&sLoInl, n[0]);
                        }
                    }
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        sModels += 1;
                        if (sLoCost < sBestCost) {
                            sBestCost = sLoCost;
                            sBestInl = (int)sLoInl;
                            for (int k = 0; k < 9; k++) sBestE[k] = sEls[k];
                            sOk = 1;
                        } else
                            sOk = 0;
                    }
                    __syncthreads();
                    if (!sOk) break;
                }
                if (threadIdx.x == 0) {
                    const int lim = (int)itTab[sBestInl];
                    sMaxIters = sMaxIters < lim ? sMaxIters : lim;
                }
                __syncthreads();
            }
            // consumed iterations: sNextB (all nb unless maxIters shrank below it + nb)
            it += sNextB;
            __syncthreads();
            for (int t = threadIdx.x; t < kBatch * 10; t += kCtaThreads) { sCost[t / 10][t % 10] = 0; sInl[t / 10][t % 10] = 0; }
            __syncthreads();
            if (sNextB < nb) break;  // maxIters reached inside the batch
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) models = sModels;
    const bool done = !active || it >= sMaxIters || lastChunk;
    // finalise: mask == sampson^2(E_final) < thr^2 and its count (SURVEY App. B.5)
    uint32_t finalInl = 0;
    if (done) {
        uint8_t *mask = (a.flags & PGI_WAVE_MASKS) ? a.masks + a.maskOffset[w] : nullptr;
        double E[9];
#pragma unroll
        for (int k = 0; k < 9; k++) E[k] = sBestE[k];
        uint32_t cnt = 0;
        for (uint32_t i = threadIdx.x; i < N; i += kCtaThreads) {
            uint32_t in = 0;
            if (sHave) {
                const double4 c = rows[i];
                in = sampsonSq(c.x, c.y, c.z, c.w, E) < thrSq ? 1u : 0u;
            }
            if (mask) mask[i] = (uint8_t)in;
            cnt += in;
        }
        finalInl = blockSumU32(cnt, sWarpU);
    }
    if (threadIdx.x == 0) {
        st.bestCost = sBestCost;
        st.bestInl = sBestInl;
        st.maxIters = sMaxIters;
        st.it = it;
        st.models += models;
        for (int k = 0; k < 9; k++) st.bestE[k] = sBestE[k];
        uint32_t f = flags0;
        if (done) {
            f &= ~ST_FB_ACTIVE;
            f &= ~ST_NEED_FB;
            st.inlierCount = finalInl;  // PGB:1047-1048
            if (sHave && finalInl >= a.minInliers) {  // PGB:1053
                f |= ST_HAVE_E;
                for (int k = 0; k < 9; k++) st.E[k] = sBestE[k];
            }
            atomicAdd(a.counters + 2, (unsigned long long)st.models);
        }
        st.flags = f;
    }
}

__global__ void __launch_bounds__(kCtaThreads, 3) k5_fallback_score(WaveArgs a, int chunk, int lastChunk, uint32_t smemPts)
{
    extern __shared__ float4 sPts[];  // smemPts float4 slots (FP32 copy of the pair's correspondences)
    const uint32_t w = blockIdx.x;
    if (w >= a.n) return;
    if (!(a.state[w].flags & ST_NEED_FB)) return;
    const uint32_t pid = a.pairId[w];
    const uint32_t N = (uint32_t)(a.offset[pid + 1] - a.offset[pid]);
    // dynamic shared memory: smemPts float4 points, then 8 per-warp queues of min(smemPts, 2048) uint16 indices
    const uint32_t queueStride = smemPts < kK5QueuePts ? ((smemPts + 31u) & ~31u) : kK5QueuePts;
    uint16_t *sQueueAll = reinterpret_cast<uint16_t *>(sPts + smemPts);
    // inlier bit mask of the LO refit: after the queues (staged pairs) or in global scratch-free form for huge pairs
    uint32_t *sInlBits = reinterpret_cast<uint32_t *>(sQueueAll + 8 * (size_t)queueStride);
    if (N <= smemPts)
        k5Body<true>(a, chunk, lastChunk, w, sPts, sQueueAll, queueStride, sInlBits);
    else
        k5Body<false>(a, chunk, lastChunk, w, sPts, sQueueAll, queueStride, a.bits + (size_t)w * 2 * a.bitsStride);  // pair too large to stage: exact FP64 for every point; the (unused) path bit buffers hold the mask
}

// Whole-CTA E -> candidates -> triangulation vote (pose_utils.h:172-240).  Results in shared memory.
__device__ inline void decomposeVoteBlock(const double E[9], const double4 *rows, uint32_t N, double (*sR)[9], double *sT,
                                          uint32_t *sVotes)
{
    if (threadIdx.x == 0) {
        double R1[9], R2[9], t[3];
        decomposeEssential(E, R1, R2, t);
        for (int k = 0; k < 9; k++) { sR[0][k] = R1[k]; sR[1][k] = R2[k]; }
        for (int k = 0; k < 3; k++) sT[k] = t[k];
    }
    if (threadIdx.x < 4) sVotes[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) {
        const double4 c = rows[i];
        double best = DBL_MAX;
        int bestPose = 5;
#pragma unroll 1
        for (int cand = 0; cand < 4; cand++) {
            const double sgn = (cand & 1) ? -1.0 : 1.0;
            const double *R = sR[cand >> 1];
            double P2[12];
#pragma unroll
            for (int r = 0; r < 3; r++) {
                P2[r * 4 + 0] = R[r * 3 + 0];
                P2[r * 4 + 1] = R[r * 3 + 1];
                P2[r * 4 + 2] = R[r * 3 + 2];
                P2[r * 4 + 3] = sgn * sT[r];
            }
            double err;
            if (!triangulateAndScore(P2, c.x, c.y, c.z, c.w, err)) continue;
            if (err < best) {
                best = err;
                bestPose = cand;
            }
        }
        if (bestPose < 5) atomicAdd(&sVotes[bestPose], 1u);
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// K3 (+K8): E -> (R1,R2,+-t) by the Eigen-faithful 3x3 Jacobi SVD, then the triangulation vote over
// ALL correspondences: 4 candidates x N 4x4 Jacobi SVDs, register resident, one thread per
// correspondence (looping the 4 candidates so the strict-< winner logic of pose_utils.h:226-230 is
// local).  FP64-pipe bound.  A pair is covered by `split` CTAs, each voting over a contiguous range of its
// points (small waves are latency bound: the host picks split so that the grid fills the GPU); the votes are
// integer counts, so merging them through global atomics is exact.  The last CTA of a pair to arrive picks the
// first maximum, converts to a unit quaternion and packs the 160-byte verdict.
// ---------------------------------------------------------------------------------------------
#ifndef PGI_K3_THREADS
#define PGI_K3_THREADS 256
#endif
constexpr int kK3Threads = PGI_K3_THREADS;
__global__ void __launch_bounds__(kK3Threads, 2) k3_decompose_vote(WaveArgs a, uint32_t split)
{
    const uint32_t w = blockIdx.x / split, part = blockIdx.x % split;
    if (w >= a.n) return;
    const SlotState &st = a.state[w];
    const uint32_t pid = a.pairId[w];
    const uint64_t r0 = a.offset[pid];
    const uint32_t N = (uint32_t)(a.offset[pid + 1] - r0);
    const uint32_t flags = st.flags;

    __shared__ double sR[2][9], sT[3];
    __shared__ uint32_t sVotes[4];
    if (flags & ST_HAVE_E) {
        double E[9];
        for (int k = 0; k < 9; k++) E[k] = st.E[k];
        const uint32_t per = (N + split - 1) / split;
        const uint32_t lo = min(part * per, N), hi = min(lo + per, N);
        decomposeVoteBlock(E, reinterpret_cast<const double4 *>(a.corr) + r0 + lo, hi - lo, sR, sT, sVotes);
    }
    if (threadIdx.x == 0 && split > 1) {
        uint32_t *g = a.k3Scratch + (size_t)w * 8;
        if (flags & ST_HAVE_E)
            for (int c = 0; c < 4; c++)
                if (sVotes[c]) atomicAdd(&g[c], sVotes[c]);
        __threadfence();
        if (atomicAdd(&g[4], 1u) != split - 1) return;  // not the last range of this pair
        __threadfence();
        for (int c = 0; c < 4; c++) sVotes[c] = atomicExch(&g[c], 0u);  // collect the totals and leave the scratch zeroed
        atomicExch(&g[4], 0u);
    }
    if (threadIdx.x == 0) {
        pgi_verdict v;
        v.pair_id = pid;
        v.n_corr = N;
        v.n_hypotheses = (uint8_t)min(255u, a.hypOffset[w + 1] - a.hypOffset[w]);
        v.test_passed = (flags & ST_TEST_PASSED) ? 1 : 0;
        v.test_count = st.testCount;
        v.path_inliers = st.pathInliers;
        v.inlier_count = st.inlierCount;
        v.iters = (flags & ST_FB_RAN) ? (uint32_t)st.it : 0u;
        v.status = ((flags & ST_FB_RAN) ? 1u : 0u) | ((flags & ST_5PT_NOMODEL) ? 2u : 0u);
        v.branch = 0;
        v.accepted = 0;
        for (int k = 0; k < 9; k++) v.E[k] = 0.0;
        v.q[0] = v.q[1] = v.q[2] = 0.0; v.q[3] = 1.0;
        v.t[0] = v.t[1] = v.t[2] = 0.0;
        if (flags & ST_HAVE_E) {
            for (int k = 0; k < 9; k++) v.E[k] = st.E[k];
            int maxIdx = 0;
            for (int i = 1; i < 4; i++)
                if (sVotes[i] > sVotes[maxIdx]) maxIdx = i;  // std::max_element: first maximum (PU:243-246)
            double R[9], t[3];
            const double sgn = (maxIdx & 1) ? -1.0 : 1.0;
            for (int k = 0; k < 9; k++) R[k] = sR[maxIdx >> 1][k];
            for (int k = 0; k < 3; k++) t[k] = sgn * sT[k];
            bool nan = false;
            for (int k = 0; k < 9; k++) nan |= (R[k] != R[k]);
            for (int k = 0; k < 3; k++) nan |= (t[k] != t[k]);
            if (nan) {  // PGB:1069-1070
                v.status |= 4u;
            } else {
                rotationToUnitQuat(R, v.q);
                v.t[0] = t[0]; v.t[1] = t[1]; v.t[2] = t[2];
                v.accepted = 1;
                v.branch = (flags & ST_PATH_OK) ? 1 : 2;
            }
        }
        a.verdicts[w] = v;
    }
}

// Stand-alone E -> (R, t, votes) for the parity tests (pgi_dbg_pose_from_essential).
__global__ void __launch_bounds__(kCtaThreads) kdbg_pose_from_essential(const double *E9, const double4 *rows, uint32_t N,
                                                                       double *Rout, double *tout, unsigned long long *votes)
{
    __shared__ double sR[2][9], sT[3];
    __shared__ uint32_t sVotes[4];
    double E[9];
    for (int k = 0; k < 9; k++) E[k] = E9[k];
    decomposeVoteBlock(E, rows, N, sR, sT, sVotes);
    if (threadIdx.x == 0) {
        int maxIdx = 0;
        for (int i = 1; i < 4; i++)
            if (sVotes[i] > sVotes[maxIdx]) maxIdx = i;
        const double sgn = (maxIdx & 1) ? -1.0 : 1.0;
        for (int k = 0; k < 9; k++) Rout[k] = sR[maxIdx >> 1][k];
        for (int k = 0; k < 3; k++) tout[k] = sgn * sT[k];
        for (int k = 0; k < 4; k++) votes[k] = sVotes[k];
    }
}

// FP64 non-fused peak probe (DMUL+DADD chain) / fused (DFMA) — roofline denominator for K2-K5 (SURVEY §8d).
__global__ void k_fp64_peak(double *out, int iters, int fused)
{
    double a0 = threadIdx.x * 1e-3 + 1.0, a1 = a0 + 0.1, a2 = a0 + 0.2, a3 = a0 + 0.3;
    double a4 = a0 + 0.4, a5 = a0 + 0.5, a6 = a0 + 0.6, a7 = a0 + 0.7;
    const double m = 1.0000001, c = 1e-9;
    if (fused) {
        for (int i = 0; i < iters; i++) {
            a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
            a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
        }
    } else {
        for (int i = 0; i < iters; i++) {
            a0 = __dadd_rn(__dmul_rn(a0, m), c); a1 = __dadd_rn(__dmul_rn(a1, m), c);
            a2 = __dadd_rn(__dmul_rn(a2, m), c); a3 = __dadd_rn(__dmul_rn(a3, m), c);
            a4 = __dadd_rn(__dmul_rn(a4, m), c); a5 = __dadd_rn(__dmul_rn(a5, m), c);
            a6 = __dadd_rn(__dmul_rn(a6, m), c); a7 = __dadd_rn(__dmul_rn(a7, m), c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

}  // namespace pgi
