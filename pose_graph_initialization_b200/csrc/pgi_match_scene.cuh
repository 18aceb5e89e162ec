// pgi_match_scene.cuh — K9: matchFeatures (feature_utils.h:103-210) for every pair of a scene in one device call, with
// the result left on the device for K0 (createCorrespondenceMatrix).  Bit-identical to oracle.match_features.
//
// k9_knn2_tile: one CTA per (pair, block of kK9Rows source keypoints); it walks the destination keypoints in blocks of
//   kK9Cols.  Each 128 x 128 distance tile is computed ONCE in FP32, dimension order, multiply then add, never fused
//   (__fsub_rn / __fmul_rn / __fadd_rn) — fl(b - a) == -fl(a - b), so the tile is also the destination -> source
//   distance matrix bit for bit — and feeds both directions:
//     forward  (source query): per row, merged across the 16 lanes of the row and over the destination blocks, kept in
//              shared memory for the CTA's lifetime -> fwd[pair][src];
//     backward (destination query): per column, merged across the CTA's rows -> one partial per (source block, column)
//              in bpart, merged over the source blocks by k9_finish.
//   Both reductions use pgi_nn2.h's exact merge, so the result is the sequential scan's whatever the grouping.
// k9_finish: one CTA per pair: backward partials merged, ratio test in double (`d1 < 0.90 * d2`), mutual check,
//   survivors keyed (ratio bits << 32 | query) and bitonic-sorted in shared memory, written in PROSAC order to a
//   per-chunk staging area with the pair's count.
// k9_offsets: scan of a chunk's counts into m_offset (continuing from the previous chunk's last offset).
// k9_scatter: the chunk's sorted rows into the scene's compacted match list at their offsets.
#pragma once
#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

#include "pgi_nn2.h"

namespace pgi {

constexpr int kK9Threads = 256;
constexpr int kK9Rows = 128;   // source keypoints per CTA (16 row groups x 8)
constexpr int kK9Cols = 128;   // destination keypoints per tile (16 lanes x 2 x 4)
constexpr int kK9Dims = 16;    // dimensions per shared-memory stage
constexpr uint32_t kK9MaxKp = 16384;  // keypoints per view: k9_finish sorts up to this many keys in shared memory
constexpr int kK9FinishThreads = 1024;

__device__ __forceinline__ Nn2 nn2Shfl(const Nn2 &s, int lane)
{
    return Nn2{__shfl_xor_sync(0xffffffffu, s.d1, lane), __shfl_xor_sync(0xffffffffu, s.d2, lane),
               __shfl_xor_sync(0xffffffffu, s.i1, lane)};
}

// stage rows [r0, r0 + 128) x dims [k0, k0 + 16) of a row-major [n][DIM] block into s[16][128] (transposed); rows >= n are 0
template <int DIM>
__device__ __forceinline__ void k9Stage(float (*s)[kK9Rows], const float *__restrict__ g, uint32_t r0, uint32_t n, int k0)
{
    const int r = threadIdx.x & (kK9Rows - 1), h = threadIdx.x >> 7;  // 2 threads per row, 8 dims each
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f), w = u;
    if (r0 + r < n) {
        const float4 *p = reinterpret_cast<const float4 *>(g + (size_t)(r0 + r) * DIM + k0 + h * 8);
        u = __ldg(p);
        w = __ldg(p + 1);
    }
    float *c = &s[h * 8][r];
    c[0 * kK9Rows] = u.x; c[1 * kK9Rows] = u.y; c[2 * kK9Rows] = u.z; c[3 * kK9Rows] = u.w;
    c[4 * kK9Rows] = w.x; c[5 * kK9Rows] = w.y; c[6 * kK9Rows] = w.z; c[7 * kK9Rows] = w.w;
}

template <int DIM>
__global__ void __launch_bounds__(kK9Threads, 2)
k9_knn2_tile(const float *__restrict__ desc, const uint64_t *__restrict__ kpOff, const uint2 *__restrict__ pv, uint64_t pair0,
             uint32_t stride /*max keypoints per view*/, uint32_t maxSB, Nn2 *__restrict__ fwd, Nn2 *__restrict__ bpart)
{
    __shared__ __align__(16) float sA[kK9Dims][kK9Rows];
    __shared__ __align__(16) float sB[kK9Dims][kK9Cols];
    __shared__ Nn2 sRed[kK9Threads / 32][kK9Cols];
    __shared__ Nn2 sF[kK9Rows];  // forward state of the CTA's rows (row ty * 8 + i belongs to lane tx == 0 of group ty)
    const uint32_t pl = blockIdx.y;
    const uint2 v = pv[pair0 + pl];
    const uint64_t oS = kpOff[v.x], oD = kpOff[v.y];
    const uint32_t nS = (uint32_t)(kpOff[v.x + 1] - oS), nD = (uint32_t)(kpOff[v.y + 1] - oD);
    const uint32_t s0 = blockIdx.x * kK9Rows;
    if (s0 >= nS) return;
    const float *A = desc + oS * DIM, *B = desc + oD * DIM;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < kK9Rows) sF[threadIdx.x] = nn2Empty();
    for (uint32_t t0 = 0; t0 < nD; t0 += kK9Cols) {
        float acc[8][8];
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int j = 0; j < 8; j++) acc[i][j] = 0.0f;
        for (int k0 = 0; k0 < DIM; k0 += kK9Dims) {
            __syncthreads();
            k9Stage<DIM>(sA, A, s0, nS, k0);
            k9Stage<DIM>(sB, B, t0, nD, k0);
            __syncthreads();
#pragma unroll
            for (int k = 0; k < kK9Dims; k++) {
                float a[8], b[8];
                *reinterpret_cast<float4 *>(a) = *reinterpret_cast<const float4 *>(&sA[k][ty * 8]);
                *reinterpret_cast<float4 *>(a + 4) = *reinterpret_cast<const float4 *>(&sA[k][ty * 8 + 4]);
                *reinterpret_cast<float4 *>(b) = *reinterpret_cast<const float4 *>(&sB[k][tx * 4]);
                *reinterpret_cast<float4 *>(b + 4) = *reinterpret_cast<const float4 *>(&sB[k][64 + tx * 4]);
#pragma unroll
                for (int i = 0; i < 8; i++)
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float d = __fsub_rn(a[i], b[j]);
                        acc[i][j] = __fadd_rn(acc[i][j], __fmul_rn(d, d));
                    }
            }
        }
        // column j of this thread is t0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + j - 4): ascending in j
        uint32_t col[8];
#pragma unroll
        for (int j = 0; j < 8; j++) col[j] = t0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
        // forward: row s0 + ty * 8 + i over this tile's columns
#pragma unroll
        for (int i = 0; i < 8; i++) {
            Nn2 s = nn2Empty();
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (col[j] < nD) nn2Push(s, acc[i][j], col[j]);
#pragma unroll
            for (int m = 1; m < 16; m <<= 1) s = nn2Merge(s, nn2Shfl(s, m));
            if (tx == 0) sF[ty * 8 + i] = nn2Merge(sF[ty * 8 + i], s);
        }
        // backward: column col[j] over this CTA's rows (ascending row within the thread, then merged across ty)
#pragma unroll
        for (int j = 0; j < 8; j++) {
            Nn2 s = nn2Empty();
#pragma unroll
            for (int i = 0; i < 8; i++)
                if (s0 + ty * 8 + i < nS) nn2Push(s, acc[i][j], s0 + ty * 8 + i);
            s = nn2Merge(s, nn2Shfl(s, 16));
            if (lane < 16) sRed[warp][col[j] - t0] = s;
        }
        __syncthreads();
        if (threadIdx.x < kK9Cols && t0 + threadIdx.x < nD) {
            Nn2 s = sRed[0][threadIdx.x];
#pragma unroll
            for (int w = 1; w < kK9Threads / 32; w++) s = nn2Merge(s, sRed[w][threadIdx.x]);
            bpart[((size_t)pl * maxSB + blockIdx.x) * stride + t0 + threadIdx.x] = s;
        }
    }
    __syncthreads();
    if (threadIdx.x < kK9Rows && s0 + threadIdx.x < nS) fwd[(size_t)pl * stride + s0 + threadIdx.x] = sF[threadIdx.x];
}

// dynamic shared memory: pow2ceil(stride) keys (8 B) + stride backward winners (4 B)
__global__ void __launch_bounds__(kK9FinishThreads)
k9_finish(const uint64_t *__restrict__ kpOff, const uint2 *__restrict__ pv, uint64_t pair0, uint32_t stride, uint32_t keyCap,
          uint32_t maxSB, const Nn2 *__restrict__ fwd, const Nn2 *__restrict__ bpart, uint32_t *__restrict__ counts,
          uint2 *__restrict__ stageM, float *__restrict__ stageR)
{
    extern __shared__ __align__(16) unsigned char k9Smem[];
    unsigned long long *sKey = reinterpret_cast<unsigned long long *>(k9Smem);
    uint32_t *sBwd = reinterpret_cast<uint32_t *>(sKey + keyCap);
    __shared__ uint32_t sN;
    const uint32_t pl = blockIdx.x;
    const uint2 v = pv[pair0 + pl];
    const uint32_t nS = (uint32_t)(kpOff[v.x + 1] - kpOff[v.x]), nD = (uint32_t)(kpOff[v.y + 1] - kpOff[v.y]);
    const uint32_t nSB = (nS + kK9Rows - 1) / kK9Rows;
    if (threadIdx.x == 0) sN = 0;
    for (uint32_t j = threadIdx.x; j < nD; j += blockDim.x) {
        Nn2 s = nn2Empty();
        for (uint32_t b = 0; b < nSB; b++) s = nn2Merge(s, bpart[((size_t)pl * maxSB + b) * stride + j]);
        sBwd[j] = s.i1;
    }
    __syncthreads();
    // feature_utils.h:172-184: both directions need 2 neighbours (:174-176), ratio test and mutual check (:178-179);
    // a query without any finite neighbour (i1 == none) never survives
    if (nS >= 2 && nD >= 2)
        for (uint32_t i = threadIdx.x; i < nS; i += blockDim.x) {
            const Nn2 q = fwd[(size_t)pl * stride + i];
            if (q.i1 != kNn2None && (double)q.d1 < 0.90 * (double)q.d2 && sBwd[q.i1] == i)
                sKey[atomicAdd(&sN, 1u)] = matchKey(__fdiv_rn(q.d1, q.d2), i);  // :182 float / float
        }
    __syncthreads();
    const uint32_t n = sN;
    uint32_t np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (uint32_t t = n + threadIdx.x; t < np2; t += blockDim.x) sKey[t] = ~0ull;
    __syncthreads();
    for (uint32_t k = 2; k <= np2; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < np2; t += blockDim.x) {
                const uint32_t u = t ^ j;
                if (u > t) {
                    const unsigned long long a = sKey[t], b = sKey[u];
                    if ((a > b) == ((t & k) == 0)) { sKey[t] = b; sKey[u] = a; }
                }
            }
            __syncthreads();
        }
    if (threadIdx.x == 0) counts[pl] = n;
    for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) {
        const unsigned long long key = sKey[t];
        const uint32_t i = (uint32_t)key;
        stageM[(size_t)pl * stride + t] = make_uint2(i, fwd[(size_t)pl * stride + i].i1);
        stageR[(size_t)pl * stride + t] = __uint_as_float((uint32_t)(key >> 32));
    }
}

// offset[pair0 + 1 + p] = offset[pair0] + counts[0] + ... + counts[p], p < n (one CTA of 1024 threads)
__global__ void __launch_bounds__(1024) k9_offsets(const uint32_t *__restrict__ counts, uint32_t n, uint64_t *__restrict__ offset,
                                                   uint64_t pair0)
{
    __shared__ uint64_t sWarp[32];
    __shared__ uint64_t sCarry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) sCarry = offset[pair0];
    __syncthreads();
    for (uint32_t b = 0; b < n; b += 1024) {
        const uint32_t p = b + threadIdx.x;
        uint64_t x = p < n ? counts[p] : 0;
#pragma unroll
        for (int m = 1; m < 32; m <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, x, m);
            if (lane >= m) x += y;
        }
        if (lane == 31) sWarp[warp] = x;
        __syncthreads();
        uint64_t add = sCarry;
        for (int w = 0; w < warp; w++) add += sWarp[w];
        if (p < n) offset[pair0 + 1 + p] = add + x;
        __syncthreads();
        if (threadIdx.x == 1023) sCarry = add + x;
        __syncthreads();
    }
}

__global__ void k9_scatter(const uint64_t *__restrict__ offset, uint64_t pair0, uint32_t stride, const uint32_t *__restrict__ counts,
                           const uint2 *__restrict__ stageM, const float *__restrict__ stageR, uint2 *__restrict__ matches,
                           float *__restrict__ ratios)
{
    const uint32_t pl = blockIdx.x, n = counts[pl];
    const uint64_t o = offset[pair0 + pl];
    for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) {
        matches[o + t] = stageM[(size_t)pl * stride + t];
        ratios[o + t] = stageR[(size_t)pl * stride + t];
    }
}

// flag = 1 if any of the n values is not finite
__global__ void k9_check_finite(const float *__restrict__ x, uint64_t n, uint32_t *__restrict__ flag)
{
    bool bad = false;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        bad |= !isfinite(x[i]);
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(flag, 1u);
}

}  // namespace pgi
