// pgi_guided_batch.cuh — K10: guided matching (HashingBasedMatcherWithPose<false, 45>::match, matcher.h:199-405, and
// guidedMatching's selection, pose_graph_builder.h:760-782) for a chunk of (view pair, pose) cases of the registered scene,
// spread over the whole GPU.  Every pair's rows are bit-identical to the reference's: the arithmetic is the shared
// device functions of pgi_matcher.cuh, applied in the reference's order; only the split of the work differs.
//
//   k10_prepare       one thread per pair: guidedPrepare (F, epipole, angular range, bin count);
//   k10_bin_count     CTA (block of kK10DstBlock destination keypoints, pair): each keypoint's bin, per-block bin histogram;
//   k10_bin_offsets   one CTA per pair: bin starts, and where each block's run of each bin begins;
//   k10_bin_scatter   CTA (block, pair): the bins as index lists in keypoint order (the order decides ties between equal
//                     descriptor distances): a keypoint's slot is its block's start in the bin plus the keypoints of that
//                     bin before it in the block (earlier warps' counts, then __match_any_sync peers of lower lanes);
//   k10_match         CTA (block of kK10SrcPerCta source keypoints, pair), one warp per source keypoint: the lanes take 32
//                     consecutive entries of the keypoint's bin at a time, each computes the gate and, for a candidate, the
//                     descriptor distance on its own, and the lanes' states merge in list order (pgi_guided_nn.h);
//   k10_select        one CTA per pair: accepted matches compacted in source order, then with max_points > 0 the selection:
//                     above max_points matches a bitonic sort of (value, source index) in shared memory keeps the
//                     max_points smallest, else every match with the first match's value;
//   k9_offsets, k10_scatter: the chunk's rows packed back to back (only they are copied to the host).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "pgi_guided_nn.h"
#include "pgi_matcher.cuh"

namespace pgi {

constexpr int kK10Threads = 256;
constexpr int kK10DstBlock = 256;                    // destination keypoints per CTA of the bin kernels
constexpr int kK10Warps = kK10Threads / 32;
constexpr int kK10SrcPerCta = 4 * kK10Warps;         // source keypoints per CTA of k10_match (4 per warp)
constexpr int kK10SelectThreads = 1024;
constexpr uint32_t kK10MaxKp = 16384;                // keypoints per view (source indices fit the sort's 16-bit field)

// one case of the batch, as the host builds it (E of the pose, K of each view, the views' keypoint ranges)
struct GuidedPairIn {
    double E[9], Ks[9], Kd[9];
    uint64_t kS0, kD0;  // first keypoint of the source / destination view in the scene's arrays
    uint32_t nS, nD;
    int wS, hS, wD, hD, binNumber, pad;
};

// per-pair device state of a chunk
struct GuidedPairDev {
    GuidedPrep p;
    uint32_t binStart[kMatchMaxBins + 1];
};

// Per-pair scratch of a chunk: each array has `stride*` entries per pair (the batch's largest view).
struct GuidedScratch {
    const GuidedPairIn *in;
    GuidedPairDev *dev;
    uint8_t *binOfD;       // strideD
    uint32_t *binList;     // strideD
    uint32_t *blockOff;    // dstBlocks x kMatchMaxBins: block histogram, then the block's start in each bin
    uint32_t *cand;        // strideS: best destination index, 0xffffffff: none
    double *candRatio;     // strideS
    uint2 *stageM;         // strideS: the pair's final rows
    double *stageV;        // strideS
    uint32_t *counts;      // 1
    uint32_t strideS, strideD, dstBlocks;
};

__global__ void k10_prepare(GuidedScratch g, uint32_t cp)
{
    const uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x;
    if (pl >= cp) return;
    const GuidedPairIn &in = g.in[pl];
    GuidedPrep p;
    guidedPrepare(in.E, in.Ks, in.Kd, in.wS, in.hS, in.wD, in.hD, in.binNumber, p);
    if (in.nS == 0 || in.nD == 0) p.bins = 0;  // nothing to match
    g.dev[pl].p = p;
}

__global__ void __launch_bounds__(kK10DstBlock) k10_bin_count(GuidedScratch g, const float2 *__restrict__ kp)
{
    __shared__ uint32_t sHist[kMatchMaxBins];
    const uint32_t pl = blockIdx.y, blk = blockIdx.x;
    const GuidedPairIn &in = g.in[pl];
    const GuidedPrep &P = g.dev[pl].p;
    const int bins = P.bins;
    if (bins <= 0 || blk * kK10DstBlock >= in.nD) return;
    for (int b = threadIdx.x; b < bins; b += blockDim.x) sHist[b] = 0;
    __syncthreads();
    double F[9];
    for (int k = 0; k < 9; k++) F[k] = P.F[k];
    const uint32_t i = blk * kK10DstBlock + threadIdx.x;
    if (i < in.nD) {
        const float2 q = kp[in.kD0 + i];
        const int b = guidedDestinationBin(F, q.x, q.y, P.minAngle, P.range, bins);
        g.binOfD[(size_t)pl * g.strideD + i] = (uint8_t)b;
        atomicAdd(&sHist[b], 1u);
    }
    __syncthreads();
    uint32_t *h = g.blockOff + ((size_t)pl * g.dstBlocks + blk) * kMatchMaxBins;
    for (int b = threadIdx.x; b < bins; b += blockDim.x) h[b] = sHist[b];
}

__global__ void __launch_bounds__(kMatchMaxBins) k10_bin_offsets(GuidedScratch g)
{
    __shared__ uint32_t sTotal[kMatchMaxBins];
    const uint32_t pl = blockIdx.x;
    const int bins = g.dev[pl].p.bins;
    if (bins <= 0) return;
    const uint32_t nBlk = (g.in[pl].nD + kK10DstBlock - 1) / kK10DstBlock;
    uint32_t *off = g.blockOff + (size_t)pl * g.dstBlocks * kMatchMaxBins;
    const int b = threadIdx.x;
    uint32_t run = 0;
    if (b < bins)
        for (uint32_t j = 0; j < nBlk; j++) {  // exclusive scan over blocks, in place
            const uint32_t c = off[j * kMatchMaxBins + b];
            off[j * kMatchMaxBins + b] = run;
            run += c;
        }
    sTotal[b] = run;
    __syncthreads();
    uint32_t *start = g.dev[pl].binStart;
    if (threadIdx.x == 0) {
        uint32_t acc = 0;
        for (int k = 0; k < bins; k++) {
            const uint32_t t = sTotal[k];
            sTotal[k] = acc;
            start[k] = acc;
            acc += t;
        }
        start[bins] = acc;
    }
    __syncthreads();
    if (b < bins)
        for (uint32_t j = 0; j < nBlk; j++) off[j * kMatchMaxBins + b] += sTotal[b];
}

__global__ void __launch_bounds__(kK10DstBlock) k10_bin_scatter(GuidedScratch g)
{
    __shared__ uint32_t sWarpCount[kK10DstBlock / 32][kMatchMaxBins];
    const uint32_t pl = blockIdx.y, blk = blockIdx.x;
    const uint32_t nD = g.in[pl].nD;
    const int bins = g.dev[pl].p.bins;
    if (bins <= 0 || blk * kK10DstBlock >= nD) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = lane; b < bins; b += 32) sWarpCount[warp][b] = 0;
    __syncwarp();
    const uint32_t i = blk * kK10DstBlock + threadIdx.x;
    const bool in = i < nD;
    const int b = in ? g.binOfD[(size_t)pl * g.strideD + i] : kMatchMaxBins;  // out-of-range lanes form their own group
    const uint32_t peers = __match_any_sync(0xffffffffu, b);
    const uint32_t before = __popc(peers & ((1u << lane) - 1u));
    if (in && before == 0) sWarpCount[warp][b] = __popc(peers);
    __syncthreads();
    if (!in) return;
    uint32_t pos = g.blockOff[((size_t)pl * g.dstBlocks + blk) * kMatchMaxBins + b] + before;
    for (int w = 0; w < warp; w++) pos += sWarpCount[w][b];
    g.binList[(size_t)pl * g.strideD + pos] = i;
}

template <int DIM>
__global__ void __launch_bounds__(kK10Threads) k10_match(GuidedScratch g, const float2 *__restrict__ kp, const float *__restrict__ desc,
                                                         unsigned long long *__restrict__ distEvals)
{
    __shared__ __align__(16) float sDs[kK10Warps][DIM];
    __shared__ uint32_t sEvals;
    const uint32_t pl = blockIdx.y;
    const GuidedPairIn &in = g.in[pl];
    const GuidedPairDev &D = g.dev[pl];
    const int bins = D.p.bins;
    const uint32_t i0 = blockIdx.x * kK10SrcPerCta;
    if (i0 >= in.nS) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) sEvals = 0;
    __syncthreads();
    double F[9];
    for (int k = 0; k < 9; k++) F[k] = D.p.F[k];
    const double ex = D.p.ex, ey = D.p.ey, minAngle = D.p.minAngle, range = D.p.range;
    const float2 *kpD = kp + in.kD0;
    const float *dD = desc + in.kD0 * DIM;
    const uint32_t *list = g.binList + (size_t)pl * g.strideD;
    uint32_t evals = 0;
    for (uint32_t i = i0 + warp; i < in.nS && i < i0 + kK10SrcPerCta; i += kK10Warps) {
        GuidedNn s = guidedEmpty();
        if (bins > 0) {
            const float2 p = kp[in.kS0 + i];
            const double x1 = p.x, y1 = p.y;
            const int bin = guidedSourceBin(x1, y1, ex, ey, minAngle, range, bins);
            const float *ds = desc + (in.kS0 + i) * DIM;
            for (int m = lane * 4; m < DIM; m += 128)
                *reinterpret_cast<float4 *>(&sDs[warp][m]) = *reinterpret_cast<const float4 *>(ds + m);
            __syncwarp();
            const uint32_t k0 = D.binStart[bin], k1 = D.binStart[bin + 1];
            for (uint32_t base = k0; base < k1; base += 32) {
                const uint32_t k = base + lane;
                GuidedNn t = guidedEmpty();
                bool isCand = false;
                if (k < k1) {
                    const uint32_t nb = list[k];
                    const float2 q = kpD[nb];
                    isCand = guidedIsCandidate(guidedEpipolarSq(F, x1, y1, q.x, q.y));
                    if (isCand) {
                        guidedPush(t, guidedDescriptorSq(sDs[warp], dD + (size_t)nb * DIM, DIM), (int32_t)nb);
                        evals++;
                    }
                }
                if (__ballot_sync(0xffffffffu, isCand) == 0) continue;
                // lanes hold runs of one entry in list order: merge neighbours, then pairs of pairs, ... into lane 0
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    GuidedNn o;
                    o.best = __shfl_down_sync(0xffffffffu, t.best, off);
                    o.second = __shfl_down_sync(0xffffffffu, t.second, off);
                    o.bestIndex = __shfl_down_sync(0xffffffffu, t.bestIndex, off);
                    o.count = __shfl_down_sync(0xffffffffu, t.count, off);
                    if ((lane & (2 * off - 1)) == 0) t = guidedMerge(t, o);  // lane + off < 32 here
                }
                if (lane == 0) s = guidedMerge(s, t);
            }
            __syncwarp();
        }
        if (lane == 0) {
            const double adapted = guidedAdaptedRatio(s);
            g.cand[(size_t)pl * g.strideS + i] = guidedAccepted(s, adapted) ? (uint32_t)s.bestIndex : 0xffffffffu;
            g.candRatio[(size_t)pl * g.strideS + i] = adapted;
        }
    }
    for (int off = 16; off > 0; off >>= 1) evals += __shfl_down_sync(0xffffffffu, evals, off);
    if (lane == 0 && evals) atomicAdd(&sEvals, evals);
    __syncthreads();
    if (threadIdx.x == 0 && sEvals) atomicAdd(distEvals, (unsigned long long)sEvals);
}

// (value, source index) order of two selection keys: values as doubles, ties to the smaller index
__device__ __forceinline__ bool guidedKeyLess(double va, uint32_t ia, double vb, uint32_t ib)
{
    return va != vb ? va < vb : ia < ib;
}

// Dynamic shared memory: sortCap doubles + sortCap uint16 (sortCap = 0 when max_points == 0).
__global__ void __launch_bounds__(kK10SelectThreads) k10_select(GuidedScratch g, uint32_t maxPoints, uint32_t sortCap)
{
    extern __shared__ __align__(16) unsigned char k10Smem[];
    double *sVal = reinterpret_cast<double *>(k10Smem);
    uint16_t *sIdx = reinterpret_cast<uint16_t *>(sVal + sortCap);
    __shared__ uint32_t sScan[kK10SelectThreads / 32], sTotal;
    __shared__ double sFirst;
    const uint32_t pl = blockIdx.x;
    const uint32_t nS = g.in[pl].nS;
    const uint32_t *cand = g.cand + (size_t)pl * g.strideS;
    const double *ratio = g.candRatio + (size_t)pl * g.strideS;
    uint2 *outM = g.stageM + (size_t)pl * g.strideS;
    double *outV = g.stageV + (size_t)pl * g.strideS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t base = 0;
    if (g.dev[pl].p.bins > 0)
        for (uint32_t i0 = 0; i0 < nS; i0 += kK10SelectThreads) {  // compaction in source order
            const uint32_t i = i0 + threadIdx.x;
            const bool ok = i < nS && cand[i] != 0xffffffffu;
            const uint32_t m = __ballot_sync(0xffffffffu, ok);
            if (lane == 0) sScan[warp] = __popc(m);
            __syncthreads();
            uint32_t off = base;
            for (int w = 0; w < warp; w++) off += sScan[w];
            if (ok) {
                const uint32_t o = off + __popc(m & ((1u << lane) - 1u));
                outM[o] = make_uint2(i, cand[i]);
                outV[o] = ratio[i];
                if (maxPoints) { sVal[o] = ratio[i]; sIdx[o] = (uint16_t)i; }
            }
            if (threadIdx.x == 0) {
                uint32_t t = 0;
                for (int w = 0; w < kK10SelectThreads / 32; w++) t += sScan[w];
                sTotal = t;
            }
            __syncthreads();
            base += sTotal;
        }
    const uint32_t n = base;
    if (maxPoints == 0 || n == 0) {
        if (threadIdx.x == 0) g.counts[pl] = n;
        return;
    }
    if (n <= maxPoints) {  // every match, each carrying the first match's value (pose_graph_builder.h:777-779)
        if (threadIdx.x == 0) sFirst = outV[0];
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) outV[t] = sFirst;
        if (threadIdx.x == 0) g.counts[pl] = n;
        return;
    }
    // the maxPoints smallest (value, index) entries in ascending order (:760-776): the match list is in source order, so
    // the source index orders ties as the position in the list does
    uint32_t np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (uint32_t t = n + threadIdx.x; t < np2; t += blockDim.x) { sVal[t] = __longlong_as_double(0x7ff0000000000000ll); sIdx[t] = 0xffff; }
    __syncthreads();
    for (uint32_t k = 2; k <= np2; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < np2; t += blockDim.x) {
                const uint32_t u = t ^ j;
                if (u > t) {
                    const double va = sVal[t], vb = sVal[u];
                    const uint16_t ia = sIdx[t], ib = sIdx[u];
                    // padding (+inf, 0xffff) sorts after every match: match values are finite
                    if (guidedKeyLess(vb, ib, va, ia) == ((t & k) == 0)) { sVal[t] = vb; sVal[u] = va; sIdx[t] = ib; sIdx[u] = ia; }
                }
            }
            __syncthreads();
        }
    for (uint32_t t = threadIdx.x; t < maxPoints; t += blockDim.x) {
        const uint32_t i = sIdx[t];
        outM[t] = make_uint2(i, cand[i]);
        outV[t] = sVal[t];
    }
    if (threadIdx.x == 0) g.counts[pl] = maxPoints;
}

// the chunk's rows back to back: pair pl's at offset[pl] (k9_offsets over the counts, offset[0] = 0)
__global__ void k10_scatter(GuidedScratch g, const uint64_t *__restrict__ offset, uint2 *__restrict__ rowsM, double *__restrict__ rowsV)
{
    const uint32_t pl = blockIdx.x, n = g.counts[pl];
    const uint64_t o = offset[pl];
    for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) {
        rowsM[o + t] = g.stageM[(size_t)pl * g.strideS + t];
        rowsV[o + t] = g.stageV[(size_t)pl * g.strideS + t];
    }
}

}  // namespace pgi
