// pgi_astar.cuh — K6: the reference's A* path search, batched on the device (one warp per search).
//
//   AStarTraversal<ImageSimilarityHeuristics>::getPath     graph_traversal.h:679-870
//   CostComparator (max-heap on the combined cost)           graph_traversal.h:656-677
//   ImageSimilarityHeuristics                                graph_traversal.h:569-596
//
// The search decides WHICH hypothesis is verified, and its pop order among equal costs is whatever
// std::priority_queue's binary heap does (SURVEY App. A.3), so the kernel replays libstdc++'s
// std::push_heap / std::pop_heap move for move on a heap that lives in HBM:
//   * one warp owns one search; its heap (16-B items) and its arena of expanded nodes are private slabs;
//   * an expansion scores 32 edge-list entries per step (coalesced 16-B loads, FP64 without FMA — the same
//     `weight * min(...) + (1 - weight) * max(...)` as graph_traversal.h:843-852), compacts the admissible children
//     with a ballot, appends them at the heap's tail in list order and then replays the sift-ups;
//   * sift-ups: a sequential std::push_heap of child k touches only ancestors of its slot.  Ancestors that were in the
//     heap before the batch can only GROW during the batch (a sift-up moves a larger value up), so a child that is not
//     larger than its parent when the batch starts stays where it is; the others take their turn in list order and
//     re-read memory, i.e. exactly the sequential result.  (Batches whose slots are parents of later slots of the same
//     batch — heaps smaller than 32 — are replayed child by child.)
//   * pop: libstdc++'s __adjust_heap walk (larger child, ties to the right child) + __push_heap of the former last
//     item.  The warp looks four levels ahead per memory round trip (30 descendants of the hole, one per lane) and
//     resolves the walk with shuffles, so a 15-level heap costs 4 dependent loads instead of 15.
// Children are lazy as on the host (pgb_host.cpp): an item is (f, parent arena node, entry | next vertex); cost tuples
// are re-derived from the same operands when (and only when) the item is popped.
//
// Graph layout in HBM: per-vertex edge lists of fixed capacity `cap` (16-B entries: score, other endpoint, tag),
// committed entries first (insertion order, pose_graph.h:219-220), then the open wave's predicted entries in wave
// position order with tag = position + 1; a search at wave position k sees tags <= k.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/pgi.h"

namespace pgi {

struct AdjDev {
    double score;
    uint32_t next;
    uint32_t tag;  // 0: committed; p + 1: predicted by wave position p
};
struct HeapItemDev {
    double f;
    uint32_t parent;  // arena index of the node that pushed this child (kNoNode: the start node)
    uint32_t en;      // entry index in the parent's edge list << 16 | child vertex
};
struct ArenaNodeDev {
    double c0, c1;    // (min edge score, max similarity to the destination) along the path  :843-848
    uint32_t vertex, parent, depth, pad;
};
constexpr uint32_t kNoNode = 0xffffffffu;
constexpr int kAstarWarps = 4;  // warps (searches in flight) per CTA

enum : uint8_t {  // pgi_search_result.status
    SEARCH_OK = 0,
    SEARCH_HEAP_OVERFLOW = 1,   // the heap slab is too small: the caller repeats the search on the host
    SEARCH_ARENA_OVERFLOW = 2,
    SEARCH_STALE_LIST = 3,      // an expanded vertex without edge list (pose_graph.h:145-146 quirk): host repeats it
    SEARCH_BUDGET = 4           // more nodes pushed than the query's budget: the caller repeats it (a device round lasts as
                                // long as its longest search, so the host keeps the rare very long ones for its thread pool)
};

struct SearchArgs {
    const AdjDev *adj;
    uint32_t cap;
    const uint32_t *ccnt, *cnt;  // committed / total entries per vertex
    const double *simT;          // V x V, transposed and clamped: simT[to * V + next]
    uint32_t V, words;
    uint32_t n;
    const pgi_query *queries;
    uint32_t maxDepth;
    double weight, oneMinusWeight;
    HeapItemDev *heaps;
    uint32_t heapCap;
    ArenaNodeDev *arenas;
    uint32_t arenaCap;
    pgi_search_result *results;
    uint32_t *expandedBits;  // n x words
    uint32_t *nextQuery;     // work counter (zeroed before the launch)
};

__device__ __forceinline__ HeapItemDev ldItem(const HeapItemDev *p)
{
    const uint4 v = *reinterpret_cast<const uint4 *>(p);
    HeapItemDev it;
    it.f = __hiloint2double((int)v.y, (int)v.x);
    it.parent = v.z;
    it.en = v.w;
    return it;
}
__device__ __forceinline__ void stItem(HeapItemDev *p, const HeapItemDev &it)
{
    uint4 v;
    v.x = (uint32_t)__double2loint(it.f);
    v.y = (uint32_t)__double2hiint(it.f);
    v.z = it.parent;
    v.w = it.en;
    *reinterpret_cast<uint4 *>(p) = v;
}

// Bring the cache line of *p into L1 (a real load: prefetch hints may be dropped).
__device__ __forceinline__ void touchL1(const HeapItemDev *p)
{
    unsigned long long sink;
    asm volatile("ld.global.ca.u64 %0, [%1];" : "=l"(sink) : "l"(p) : "memory");
    (void)sink;
}

// std::__push_heap(first, hole, 0, value, less-on-f) (libstdc++ bits/stl_heap.h) by the whole warp, in one memory
// round trip whatever the depth.  The path from a slot to the root is non-decreasing in f (heap property), so the
// ancestors smaller than `value` are the first L of the path: lane j loads the j-th ancestor, a ballot yields L,
// ancestors 1..L each move one level down (lane j stores what it loaded) and `value` lands on level L — exactly the
// moves of libstdc++'s sequential loop.  (A child that out-ranks most of a
// 10^5-entry heap climbs ~15 levels; one lane walking them costs 15 dependent loads.)  All lanes pass the same
// arguments; the caller separates consecutive calls with __syncwarp().
__device__ __forceinline__ void siftUpWarp(HeapItemDev *H, uint32_t hole, const HeapItemDev &value, int lane)
{
    const uint32_t q = (hole + 1) >> lane;  // 1-based index of the lane-th ancestor (lane 0: the hole itself)
    const bool have = lane >= 1 && q >= 1;
    HeapItemDev anc;
    anc.f = 0.0; anc.parent = 0; anc.en = 0;
    if (have) anc = ldItem(H + q - 1);
    const uint32_t smaller = __ballot_sync(0xffffffffu, have && anc.f < value.f);
    const uint32_t L = (uint32_t)__ffs((int)~(smaller >> 1)) - 1u;  // consecutive set bits from bit 1 on
    if (have && (uint32_t)lane <= L) stItem(H + (((hole + 1) >> (lane - 1)) - 1), anc);
    if (lane == 0) stItem(H + (((hole + 1) >> L) - 1), value);
}
__device__ __forceinline__ HeapItemDev shflItem(const HeapItemDev &it, int src)
{
    HeapItemDev r;
    r.f = __shfl_sync(0xffffffffu, it.f, src);
    r.parent = __shfl_sync(0xffffffffu, it.parent, src);
    r.en = __shfl_sync(0xffffffffu, it.en, src);
    return r;
}

// std::pop_heap(H, H + hs) (__pop_heap -> __adjust_heap -> __push_heap) by the whole warp.  Per step the hole's
// 2 + 4 + 8 + 16 descendants of the next four levels are loaded by lanes 0..29 (lane (2^j - 2) + i holds descendant i
// of level j), the walk "larger child, ties to the right" is resolved with shuffles, and the chosen items are stored
// one level up — the moves __adjust_heap makes, four levels at a time.
__device__ inline void popHeapWarp(HeapItemDev *H, uint32_t hs, int lane)
{
    if (hs <= 1) return;
    const uint32_t len = hs - 1;
    const uint32_t limit = (len - 1) / 2;  // loop while second < limit
    HeapItemDev value;
    value.f = 0.0; value.parent = 0; value.en = 0;
    if (lane == 0) value = ldItem(H + len);
    uint32_t hole = 0;  // == `second` of __adjust_heap between iterations
    // lane's level j in 1..4 and index i within the level
    int j = 0, i = 0;
    if (lane < 2) { j = 1; i = lane; }
    else if (lane < 6) { j = 2; i = lane - 2; }
    else if (lane < 14) { j = 3; i = lane - 6; }
    else if (lane < 30) { j = 4; i = lane - 14; }
    while (hole < limit) {
        // descendant i of level j below `hole`: ((hole + 1) << j) - 1 + i
        HeapItemDev mine;
        mine.f = 0.0; mine.parent = 0; mine.en = 0;
        uint32_t pos = 0;
        bool have = false;
        if (j > 0) {
            const uint64_t p64 = (((uint64_t)hole + 1) << j) - 1 + (uint64_t)i;
            // an item at p is needed only if the walk can reach it: its parent q must satisfy q < limit, and then
            // both children 2q+1, 2q+2 exist (2q+2 <= 2(limit-1)+2 = 2 limit <= len - 1)
            if (p64 < len) {
                pos = (uint32_t)p64;
                const uint32_t q = (pos - 1) >> 1;
                if (q < limit) { mine = ldItem(H + pos); have = true; }
            }
        }
        // walk up to four levels
        uint32_t cur = hole;      // current hole
        int curLaneIdx = 0;       // index of `cur` within its level relative to the step's root (level 0: 0)
        uint32_t steps = 0;
        int chosenLane[4];
#pragma unroll
        for (int lv = 1; lv <= 4; lv++) {
            chosenLane[lv - 1] = -1;
            if (cur < limit) {  // warp-uniform
                const int base = (1 << lv) - 2;
                const int li = base + 2 * curLaneIdx, ri = li + 1;
                const double lf = __shfl_sync(0xffffffffu, mine.f, li);
                const double rf = __shfl_sync(0xffffffffu, mine.f, ri);
                const bool takeLeft = rf < lf;  // comp(first + secondChild, first + secondChild - 1) -> secondChild--
                const int c = takeLeft ? li : ri;
                chosenLane[lv - 1] = c;
                curLaneIdx = 2 * curLaneIdx + (takeLeft ? 0 : 1);
                cur = 2 * cur + (takeLeft ? 1 : 2);
                ++steps;
            }
        }
        // moves: the item chosen at level lv goes to the position of the hole at level lv - 1
        // (level 0 position = `hole`; level lv - 1 position = position of the item chosen at lv - 1)
        {
            uint32_t dst = hole;
#pragma unroll
            for (int lv = 1; lv <= 4; lv++) {
                const int c = chosenLane[lv - 1];
                if (c >= 0) {  // warp-uniform
                    const uint32_t cpos = __shfl_sync(0xffffffffu, pos, c);
                    if (lane == c && have) stItem(H + dst, mine);
                    dst = cpos;
                }
            }
        }
        hole = cur;
        (void)steps;
    }
    __syncwarp();
    uint32_t h = hole;
    if ((len & 1u) == 0 && hole == (len - 2) / 2) {  // warp-uniform
        const uint32_t second = 2 * (hole + 1);
        if (lane == 0) stItem(H + h, ldItem(H + second - 1));
        h = second - 1;
        __syncwarp();
    }
    siftUpWarp(H, h, shflItem(value, 0), lane);
}

// ---- one batch of 32 edge-list entries, replayed directly on the heap in HBM ---------------------------------------------
// Returns false if the heap slab is full.  `hidden` reports that the batch met an entry predicted by a later wave position
// (everything behind it is hidden too).
__device__ __forceinline__ bool pushBatchGlobal(const SearchArgs &a, HeapItemDev *H, uint32_t &hs, uint32_t &pushes,
                                                const AdjDev *list, uint32_t total, uint32_t nc, uint32_t cutoff,
                                                const uint32_t *bits, const double *simTo, double c0, double c1, uint32_t ni,
                                                uint32_t base, int lane, bool &hiddenOut)
{
    const uint32_t ltMask = (1u << lane) - 1u;
    const uint32_t idx = base + lane;
    bool valid = false, hidden = false;
    double f = 0.0;
    uint32_t next = 0;
    if (idx < total) {
        const AdjDev e = list[idx];
        if (idx >= nc && e.tag > cutoff)
            hidden = true;  // predicted by a later wave position: not part of this search's graph
        else if (!(e.score < 0.0)) {  // kMinimumInlierRatio is `const bool` receiving 0.0 (:613, :839)
            next = e.next;
            if (!((bits[next >> 5] >> (next & 31)) & 1u)) {  // nodeStates.find(next) == end  :855-856
                const double edgeCost = c0 > e.score ? e.score : c0;  // MIN :843
                const double h = simTo[next];
                const double ntd = c1 < h ? h : c1;  // MAX :847
                f = a.weight * edgeCost + a.oneMinusWeight * ntd;  // :851-852
                valid = true;
            }
        }
    }
    const uint32_t m = __ballot_sync(0xffffffffu, valid);
    hiddenOut = __ballot_sync(0xffffffffu, hidden) != 0;
    const uint32_t cntv = __popc(m);
    if (cntv) {
        if (hs + cntv > a.heapCap) return false;
        const uint32_t pos = hs + __popc(m & ltMask);
        HeapItemDev it;
        it.f = f; it.parent = ni; it.en = (idx << 16) | next;
        if (valid) stItem(H + pos, it);
        __syncwarp();
        bool flag = false;
        if (valid) flag = hs < 32u ? true : (ldItem(H + ((pos - 1) >> 1)).f < f);
        uint32_t fm = __ballot_sync(0xffffffffu, flag);
        while (fm) {
            const int l = __ffs((int)fm) - 1;
            fm &= fm - 1;
            siftUpWarp(H, __shfl_sync(0xffffffffu, pos, l), shflItem(it, l), lane);
            __syncwarp();
        }
        hs += cntv;
        pushes += cntv;
    }
    return true;
}

// ---- staged expansion -------------------------------------------------------------------------------------------
// A search of the benchmark scenes keeps 10^4..10^5 entries in its heap — GBs over the searches in flight, far beyond L2 —
// and every std::push_heap that moves touches the slot's ancestors, one child after the other: on the heap in HBM each
// moving child costs a memory round trip of its own (measured: 27 % of the kernel's stall samples on that one load, ~700
// cycles per child).  So an expansion is replayed in shared memory, kChunk edge-list entries at a time:
//   * the chunk's admissible children are appended to a staging buffer (slots hs .. hs + C - 1 of the heap);
//   * ALL ancestors of those slots — for level j the contiguous window ((hs+1) >> j) - 1 .. ((hs+kChunk) >> j) - 1, up to
//     the root — are loaded next to them in ONE parallel round trip (the addresses depend on hs only);
//   * children not larger than their parent stay where they are (see the header); the others are replayed in list order
//     on the staged copy with the warp-cooperative sift-up (lane j reads the j-th ancestor, ballot, shift), at
//     shared-memory latency;
//   * new slots and the touched windows are written back in parallel.
// Chunks whose slots straddle two tree levels (the windows of different levels would then alias) or whose parents are
// new slots themselves (heaps below kChunk entries) take the batch path above; both are rare.
constexpr int kChunk = 128;
constexpr int kStageItems = 320;  // kChunk + (66 + 34 + 18 + 10 + 6 + 4) + 3 per level from the 7th on (heaps < 2^21 slots)
__device__ __forceinline__ int coneOff(int j)  // staging index of level j's window (level 0 = the new slots at index 0)
{
    // window sizes kChunk/2^j + 2 for j <= 6 (66, 34, 18, 10, 6, 4), 3 above
    return j <= 6 ? 2 * kChunk - (kChunk >> (j - 1)) + 2 * (j - 1) : 266 + 3 * (j - 7);
}
__device__ __forceinline__ uint32_t coneStart(uint32_t hs, int j) { return ((hs + 1) >> j) - 1; }  // level-j ancestor of slot hs

__device__ inline bool expandStaged(const SearchArgs &a, HeapItemDev *H, uint32_t &hs, uint32_t &pushes, const AdjDev *list,
                                    uint32_t total, uint32_t nc, uint32_t cutoff, const uint32_t *bits, const double *simTo,
                                    double c0, double c1, uint32_t ni, HeapItemDev *sStage, uint16_t *sList, int lane)
{
    const uint32_t ltMask = (1u << lane) - 1u;
    for (uint32_t base = 0; base < total; base += kChunk) {
        const int depth = 31 - __clz((int)(hs + 1));  // ancestors of slot hs (root = level `depth`)
        const bool stageable = hs >= (uint32_t)kChunk && depth == 31 - __clz((int)(hs + kChunk));
        if (!stageable) {
            bool hidden = false;
            for (uint32_t b0 = base; b0 < total && b0 < base + kChunk && !hidden; b0 += 32)
                if (!pushBatchGlobal(a, H, hs, pushes, list, total, nc, cutoff, bits, simTo, c0, c1, ni, b0, lane, hidden)) return false;
            __syncwarp();
            if (hidden) break;
            continue;
        }
        // ---- loads: 4 list entries per lane + every ancestor window (all independent of each other)
        AdjDev e[4];
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const uint32_t idx = base + 32u * b + lane;
            if (idx < total) e[b] = list[idx];
            else { e[b].score = 0.0; e[b].next = 0; e[b].tag = 0; }
        }
        for (int j = 1; j <= depth; j++) {
            const uint32_t count = ((hs + kChunk) >> j) - ((hs + 1) >> j) + 1;
            const int off = coneOff(j);
            for (uint32_t k = lane; k < count; k += 32) stItem(sStage + off + k, ldItem(H + coneStart(hs, j) + k));
        }
        // ---- evaluate the children (graph_traversal.h:830-862)
        bool valid[4];
        double f[4];
        uint32_t next[4], m[4];
        uint32_t hiddenAny = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const uint32_t idx = base + 32u * b + lane;
            valid[b] = false;
            f[b] = 0.0;
            next[b] = 0;
            bool hidden = false;
            if (idx < total) {
                if (idx >= nc && e[b].tag > cutoff)
                    hidden = true;  // predicted by a later wave position: not part of this search's graph
                else if (!(e[b].score < 0.0)) {  // kMinimumInlierRatio is `const bool` receiving 0.0 (:613, :839)
                    next[b] = e[b].next;
                    if (!((bits[next[b] >> 5] >> (next[b] & 31)) & 1u)) {  // nodeStates.find(next) == end  :855-856
                        const double edgeCost = c0 > e[b].score ? e[b].score : c0;  // MIN :843
                        const double h = simTo[next[b]];
                        const double ntd = c1 < h ? h : c1;  // MAX :847
                        f[b] = a.weight * edgeCost + a.oneMinusWeight * ntd;  // :851-852
                        valid[b] = true;
                    }
                }
            }
            m[b] = __ballot_sync(0xffffffffu, valid[b]);
            hiddenAny |= __ballot_sync(0xffffffffu, hidden);
        }
        const uint32_t C = __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
        if (C) {
            if (hs + C > a.heapCap) return false;
            uint32_t cIdx[4];
            {
                uint32_t acc = 0;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    cIdx[b] = acc + __popc(m[b] & ltMask);
                    acc += __popc(m[b]);
                }
            }
#pragma unroll
            for (int b = 0; b < 4; b++)
                if (valid[b]) {
                    HeapItemDev it;
                    it.f = f[b]; it.parent = ni; it.en = ((base + 32u * b + lane) << 16) | next[b];
                    stItem(sStage + cIdx[b], it);
                }
            __syncwarp();
            // ---- which children move at all (ordered list of their indices)
            uint32_t nf = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                bool flag = false;
                if (valid[b]) {
                    const uint32_t pp = (hs + cIdx[b] - 1) >> 1;
                    flag = ldItem(sStage + coneOff(1) + (pp - coneStart(hs, 1))).f < f[b];
                }
                const uint32_t bal = __ballot_sync(0xffffffffu, flag);
                if (flag) sList[nf + __popc(bal & ltMask)] = (uint16_t)cIdx[b];
                nf += __popc(bal);
            }
            __syncwarp();
            // ---- replay std::push_heap for those children, in list order, on the staged copy (siftUpWarp on shared memory)
            uint32_t maxLev = 0;
            for (uint32_t i = 0; i < nf; i++) {
                const uint32_t c = sList[i];
                const uint32_t p1 = hs + c + 1;  // 1-based slot
                const HeapItemDev value = ldItem(sStage + c);
                const bool have = lane >= 1 && lane <= depth;
                HeapItemDev anc;
                anc.f = 0.0; anc.parent = 0; anc.en = 0;
                if (have) anc = ldItem(sStage + coneOff(lane) + ((p1 >> lane) - 1 - coneStart(hs, lane)));
                const uint32_t smaller = __ballot_sync(0xffffffffu, have && anc.f < value.f);
                const uint32_t L = (uint32_t)__ffs((int)~(smaller >> 1)) - 1u;  // the ancestors below `value` are the first L
                if (have && (uint32_t)lane <= L) {
                    HeapItemDev *dst = lane == 1 ? sStage + c
                                                 : sStage + coneOff(lane - 1) + ((p1 >> (lane - 1)) - 1 - coneStart(hs, lane - 1));
                    stItem(dst, anc);
                }
                if (lane == 0 && L > 0) stItem(sStage + coneOff((int)L) + ((p1 >> L) - 1 - coneStart(hs, (int)L)), value);
                maxLev = maxLev < L ? L : maxLev;
                __syncwarp();
            }
            // ---- write back
            for (uint32_t c = lane; c < C; c += 32) stItem(H + hs + c, ldItem(sStage + c));
            for (int j = 1; j <= (int)maxLev; j++) {
                const uint32_t count = ((hs + kChunk) >> j) - ((hs + 1) >> j) + 1;
                const int off = coneOff(j);
                for (uint32_t k = lane; k < count; k += 32) stItem(H + coneStart(hs, j) + k, ldItem(sStage + off + k));
            }
            hs += C;
            pushes += C;
        }
        __syncwarp();
        if (hiddenAny) break;  // predicted entries are in position order: everything behind is hidden too
    }
    return true;
}

__global__ void __launch_bounds__(kAstarWarps * 32) k6_astar_search(SearchArgs a)
{
    extern __shared__ uint4 sDyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // per-warp shared memory: staging buffer of the expansion (kStageItems heap items), list of moving children, bit sets
    HeapItemDev *sStage = reinterpret_cast<HeapItemDev *>(sDyn) + (size_t)warp * kStageItems;
    uint16_t *sList = reinterpret_cast<uint16_t *>(reinterpret_cast<HeapItemDev *>(sDyn) + (size_t)kAstarWarps * kStageItems) + (size_t)warp * kChunk;
    uint32_t *sBitsAll = reinterpret_cast<uint32_t *>(reinterpret_cast<uint16_t *>(reinterpret_cast<HeapItemDev *>(sDyn) + (size_t)kAstarWarps * kStageItems) + (size_t)kAstarWarps * kChunk);
    uint32_t *bits = sBitsAll + (size_t)warp * 2 * a.words;  // expanded (blocks pushes)
    uint32_t *rbits = bits + a.words;                         // expanded below the maximum depth: lists that were read
    const uint32_t slot = blockIdx.x * kAstarWarps + warp;
    HeapItemDev *H = a.heaps + (size_t)slot * a.heapCap;
    ArenaNodeDev *A = a.arenas + (size_t)slot * a.arenaCap;
    for (;;) {
        uint32_t qi = 0;
        if (lane == 0) qi = atomicAdd(a.nextQuery, 1u);
        qi = __shfl_sync(0xffffffffu, qi, 0);
        if (qi >= a.n) break;
        const long long tStart = clock64();
        const pgi_query q = a.queries[qi];
        const uint32_t from = q.src, to = q.dst, cutoff = q.cutoff, budget = q.budget;
        for (uint32_t wI = lane; wI < 2 * a.words; wI += 32) bits[wI] = 0;
        const double *simTo = a.simT + (size_t)to * a.V;
        uint32_t hs = 1, na = 0, touched = 0, pushes = 0, status = SEARCH_OK, found = 0, pathLen = 0;
        uint32_t path[8];
        if (lane == 0) {
            HeapItemDev s;
            s.f = 0.0; s.parent = kNoNode; s.en = 0;  // start node, cost (1, 0, 0)  :721
            stItem(H, s);
        }
        __syncwarp();
        while (hs > 0) {
            const HeapItemDev top = ldItem(H);
            ++touched;  // :750
            __syncwarp();
            popHeapWarp(H, hs, lane);
            --hs;
            __syncwarp();
            uint32_t v, depth;
            double c0, c1;
            if (top.parent == kNoNode) {
                v = from; depth = 0; c0 = 1.0; c1 = 0.0;
            } else {
                const ArenaNodeDev pn = A[top.parent];
                v = top.en & 0xffffu;
                const double sc = a.adj[(size_t)pn.vertex * a.cap + (top.en >> 16)].score;
                const double h = simTo[v];
                c0 = pn.c0 > sc ? sc : pn.c0;  // MIN :843
                c1 = pn.c1 < h ? h : pn.c1;    // MAX :847
                depth = pn.depth + 1;
            }
            if (depth > a.maxDepth) continue;  // :755
            if (v == to) {                     // :766
                pathLen = 0;
                path[pathLen++] = v;
                for (uint32_t k = top.parent; k != kNoNode && pathLen < 8; k = A[k].parent) path[pathLen++] = A[k].vertex;
                found = 1;
                break;  // exactly one path is tested (:792-800 with kMaximumPathNumber = 1)
            }
            if (lane == 0) {
                bits[v >> 5] |= 1u << (v & 31);  // nodeStates[v] = Open  :814
                if (depth < a.maxDepth) rbits[v >> 5] |= 1u << (v & 31);  // edge list iterated below (:820)
            }
            if (na >= a.arenaCap) { status = SEARCH_ARENA_OVERFLOW; break; }
            const uint32_t ni = na++;
            if (lane == 0) {
                ArenaNodeDev nn;
                nn.c0 = c0; nn.c1 = c1; nn.vertex = v; nn.parent = top.parent; nn.depth = depth; nn.pad = 0;
                A[ni] = nn;
            }
            __syncwarp();
            const uint32_t total = a.cnt[v], nc = a.ccnt[v];
            if (total == 0) { status = SEARCH_STALE_LIST; break; }
            if (depth < a.maxDepth) {  // :820
                const AdjDev *list = a.adj + (size_t)v * a.cap;
                if (!expandStaged(a, H, hs, pushes, list, total, nc, cutoff, bits, simTo, c0, c1, ni, sStage, sList, lane)) {
                    status = SEARCH_HEAP_OVERFLOW;
                    break;
                }
                if (budget && pushes > budget) { status = SEARCH_BUDGET; break; }
            }
        }
        __syncwarp();
        if (lane == 0) {
            pgi_search_result r;
            r.touched = touched;
            r.pushes = pushes;
            for (int k = 0; k < 6; k++) r.path[k] = 0;
            // path[] holds destination .. source; emit source .. destination
            const uint32_t L = pathLen > 6 ? 6 : pathLen;
            for (uint32_t k = 0; k < L; k++) r.path[k] = (uint16_t)path[pathLen - 1 - k];
            r.found = (uint8_t)found;
            r.path_len = (uint8_t)pathLen;
            r.status = (uint8_t)status;
            r.pad = 0;
            r.kcycles = (uint32_t)((clock64() - tStart) >> 10);
            a.results[qi] = r;
        }
        for (uint32_t wI = lane; wI < a.words; wI += 32) a.expandedBits[(size_t)qi * a.words + wI] = rbits[wI];
        __syncwarp();
    }
}

// Scatter edge-list entries into the device graph (committed edges at commit time, the predicted overlay per round).
struct ApplyEntry {
    uint32_t vertex, index, next, tag;
    double score;
};
__global__ void k6_graph_apply(AdjDev *adj, uint32_t cap, const ApplyEntry *e, uint32_t n)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ApplyEntry x = e[i];
    AdjDev d;
    d.score = x.score; d.next = x.next; d.tag = x.tag;
    adj[(size_t)x.vertex * cap + x.index] = d;
}

}  // namespace pgi
