// pgb_host.cpp — host side of the B200 path (include/pgb.h): similarity queue, pose graph, visibility
// table, A* and the sequential commit of the reference, reorganised as speculative waves.
//
// Wave scheme (exact; SURVEY §7 hard part 3).  A wave is the next W pairs of the queue, positions 0..W-1.
//   * Every position k carries a PREDICTED verdict pv_k (initially the pair's hypothesis-independent fallback
//     verdict, which is prefetched).  The accepted predictions form an OVERLAY on the committed graph: an
//     append-only per-vertex edge list tagged with the position that adds the edge, plus a sequentially
//     simulated visibility table.  The search of position k sees the committed graph plus overlay entries of
//     positions < k — i.e. exactly the graph the sequential reference would have IF the predictions hold.
//   * All positions are searched in parallel (thread pool), the engine verifies the (pair, hypothesis) tuples,
//     the actual verdicts a_k replace the predictions where they differ (a path hypothesis was accepted), and
//     only the positions whose search READ something that changed are searched again: the only graph reads of
//     AStarTraversal::getPath are getEdgesByVertex(v) for every EXPANDED vertex v (graph_traversal.h:817) and
//     the edges of the found path (graph_traversal.h:323-328), so position m is stale iff an expanded vertex of
//     m is an endpoint of a changed position k < m, or its hasLink answer changed.
//   * Position 0 depends on nothing in the wave, so by induction the iteration reaches the fixed point
//     "h_k == A*(graph after the actual verdicts of positions < k) for every k", which IS the sequential
//     semantics; the whole wave is then committed in order.  (pair, hypothesis) -> verdict is a pure function and
//     is cached, so a re-searched position only costs engine work when its hypothesis really changed.
//
// Data structures are flat (arena A* nodes, bit-matrix visibility, per-vertex edge index vectors) but the
// heap is driven by the same std::push_heap/std::pop_heap calls std::priority_queue makes, so ties break
// exactly as in the reference (SURVEY App. A.3).
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <queue>
#include <thread>
#include <tuple>
#include <unordered_map>
#include <vector>

#include "../../include/pgb.h"
#include "pgi_nvtx.h"
// Tracklets share this translation unit with the hashing loop that drives them (pgb_run_hashing), so that the host
// compiles and links as one file.
#include "pgb_tracklets.cpp"

#if defined(__x86_64__) && defined(__GNUC__)
#include <immintrin.h>
#define PGB_HAVE_AVX2_PATH 1
#endif

namespace {

// ---- pose algebra (Sophus/Eigen semantics; scalar evaluation order as documented in DESIGN.md) --------
struct SE3 {
    double q[4];  // x y z w
    double t[3];
};
inline SE3 se3Identity() { return SE3{{0, 0, 0, 1}, {0, 0, 0}}; }
inline void cross3(const double a[3], const double b[3], double o[3])
{
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}
inline void quatRotate(const double q[4], const double p[3], double o[3])
{
    double uv[3], c2[3];
    cross3(q, p, uv);
    uv[0] += uv[0]; uv[1] += uv[1]; uv[2] += uv[2];
    cross3(q, uv, c2);
    o[0] = (p[0] + q[3] * uv[0]) + c2[0];
    o[1] = (p[1] + q[3] * uv[1]) + c2[1];
    o[2] = (p[2] + q[3] * uv[2]) + c2[2];
}
inline SE3 se3Mul(const SE3 &a, const SE3 &b)  // graph_traversal.h:341-344
{
    SE3 r;
    const double *A = a.q, *B = b.q;
    double w = A[3] * B[3] - A[0] * B[0] - A[1] * B[1] - A[2] * B[2];
    double x = A[3] * B[0] + A[0] * B[3] + A[1] * B[2] - A[2] * B[1];
    double y = A[3] * B[1] + A[1] * B[3] + A[2] * B[0] - A[0] * B[2];
    double z = A[3] * B[2] + A[2] * B[3] + A[0] * B[1] - A[1] * B[0];
    const double n = std::sqrt((x * x + y * y) + (z * z + w * w));
    r.q[0] = x / n; r.q[1] = y / n; r.q[2] = z / n; r.q[3] = w / n;
    double rt[3];
    quatRotate(a.q, b.t, rt);
    r.t[0] = a.t[0] + rt[0]; r.t[1] = a.t[1] + rt[1]; r.t[2] = a.t[2] + rt[2];
    return r;
}
inline SE3 se3Inverse(const SE3 &a)
{
    SE3 r;
    r.q[0] = -a.q[0]; r.q[1] = -a.q[1]; r.q[2] = -a.q[2]; r.q[3] = a.q[3];
    const double nt[3] = {a.t[0] * -1.0, a.t[1] * -1.0, a.t[2] * -1.0};
    quatRotate(r.q, nt, r.t);
    return r;
}

struct Edge {
    uint32_t src, dst;
    SE3 T;
    double score;
    uint32_t inlierNumber, nCorr;
    uint8_t branch;
};

inline uint64_t edgeKey(uint32_t s, uint32_t d) { return ((uint64_t)s << 32) | d; }

struct Adj {  // one entry of a vertex' edge list, flattened for the A* inner loop
    uint32_t next;   // the other endpoint (graph_traversal.h:838-840)
    uint32_t edge;
    double score;
};
struct Graph {
    std::vector<Edge> edges;                       // commit order (= PoseGraph::edges_ids)
    std::vector<std::vector<Adj>> byVertex;        // per-vertex edge list in insertion order (pose_graph.h:219-220)
    std::unordered_map<uint64_t, uint32_t> lookup; // (src,dst) -> edge index
    bool hasEdge(uint32_t s, uint32_t d) const { return lookup.find(edgeKey(s, d)) != lookup.end(); }
    const Edge *find(uint32_t s, uint32_t d) const
    {
        auto it = lookup.find(edgeKey(s, d));
        return it == lookup.end() ? nullptr : &edges[it->second];
    }
};

// visibility_table.h:45-171 with the map as a bit matrix and the neighbour std::sets as sorted bit rows
// (ascending iteration == std::set order).  pair2 = (third,third) entries (:101) can never be queried by
// hasLink (from == to returns early, :152), so they are not materialised; `!hasPair1 || !hasPair1` (:108)
// is kept as is.
struct Visibility {
    uint32_t V = 0, words = 0;
    uint64_t nLinks = 0;  // set bits of `link`; V(V-1)/2 = every pair linked: the table can never change again
    std::vector<uint64_t> link, nb;
    void init(uint32_t v)
    {
        V = v;
        words = (v + 63) / 64;
        nLinks = 0;
        link.assign((size_t)V * words, 0);
        nb.assign((size_t)V * words, 0);
    }
    // Every pair is linked: hasLink is true for all a != b, and addLink can only touch the neighbour sets, which are
    // read by nothing but the creation of new links (visibility_table.h:80-83, :113-114).
    bool complete() const { return nLinks == (uint64_t)V * (V - 1) / 2; }
    bool get(const std::vector<uint64_t> &m, uint32_t r, uint32_t c) const { return (m[(size_t)r * words + (c >> 6)] >> (c & 63)) & 1; }
    void set(std::vector<uint64_t> &m, uint32_t r, uint32_t c) { m[(size_t)r * words + (c >> 6)] |= 1ull << (c & 63); }
    bool hasLink(uint32_t a, uint32_t b) const
    {
        if (a == b) return false;
        return get(link, std::min(a, b), std::max(a, b));
    }
    // The reference walks a FIFO of neighbour ids (visibility_table.h:76-118).  What the walk leaves behind does not
    // depend on the order or on repeated visits: a vertex is expanded (its neighbour set queued) the first time it is
    // met without a link to `from`, its neighbour set only gains {from, to} during the walk (both are skipped when
    // met), and every later visit of the same vertex changes nothing.  So the reachable set is computed with bit
    // rows (pending |= nb[v] & ~visited) instead of queueing up to V ids per expansion.
    std::vector<uint64_t> pending, visited;
    bool addLink(uint32_t from_, uint32_t to_)
    {
        if (from_ == to_) return false;
        const uint32_t from = std::min(from_, to_), to = std::max(from_, to_);
        set(nb, from, to);
        set(nb, to, from);
        if (get(link, from, to)) return false;
        set(link, from, to);
        ++nLinks;
        pending.assign(words, 0);
        visited.assign(words, 0);
        const uint64_t *rf = &nb[(size_t)from * words], *rt = &nb[(size_t)to * words];
        for (uint32_t w = 0; w < words; w++) pending[w] = rf[w] | rt[w];
        for (;;) {
            uint32_t w = 0;
            while (w < words && pending[w] == 0) ++w;
            if (w == words) break;
            while (pending[w]) {
                const uint32_t v = w * 64 + (uint32_t)__builtin_ctzll(pending[w]);
                pending[w] &= pending[w] - 1;
                visited[v >> 6] |= 1ull << (v & 63);
                if (v == from || v == to) continue;
                const uint32_t first = std::min(v, from), second = std::max(v, from);
                if (!get(link, first, second)) {  // `!hasPair1 || !hasPair1` (:108)
                    set(link, first, second);
                    ++nLinks;
                    const uint64_t *rv = &nb[(size_t)v * words];
                    for (uint32_t x = 0; x < words; x++) pending[x] |= rv[x] & ~visited[x];
                }
                set(nb, v, from);
                set(nb, v, to);
            }
        }
        return true;
    }
};

struct AStarOut {
    bool valid = true;        // false: an entry below the cost floor reached the top of the queue (the caller repeats the search without a floor)
    double minPoppedF = 2.0;  // smallest combined cost among the popped nodes (the start node aside): the floor the search needed
    bool found = false;
    SE3 pose = se3Identity();
    uint32_t touched = 0;
    uint32_t pushes = 0;
    std::vector<uint32_t> expanded;  // vertices whose edge lists were read
    std::vector<double> expCost;     // (c0, c1) of the node at each of those expansions: what a child's cost is computed from
};

// Heap entries describe a child lazily: (parent node, entry of the parent's edge list).  The child's vertex and
// cost tuple are re-derived from the parent when (and only when) it is popped — the same IEEE operations on the
// same operands — so only the ~1 % of pushed nodes that are ever popped get an arena record.
struct HeapItem {
    double f;
    uint32_t parent;  // arena index of the expanded node that pushed this child (UINT32_MAX: the start node)
    uint32_t entry;   // index into the concatenated (committed ++ overlay) edge list the parent iterated
};
struct ArenaNode {
    uint32_t vertex, parent, depth;
    uint32_t listOwner;  // vertex whose edge list this node iterated when it was expanded
    double c0, c1;
};

struct AStarScratch {
    std::vector<HeapItem> heap;
    std::vector<ArenaNode> arena;
    std::vector<uint32_t> mark;  // per-vertex stamp of "expanded in this search"
    uint32_t epoch = 0;
    std::vector<uint32_t> path;
    uint64_t floorRetries = 0;    // searches repeated because the cost-floor guess was too high
    std::vector<double> childF;   // scratch of one expansion: combined cost / list entry of the admissible children
    std::vector<uint32_t> childE, childMove;
};

// Predicted edges of the open wave, layered over the committed graph.
struct OvAdj {
    Adj a;
    uint32_t pos;  // wave position that adds the edge
};
struct Overlay {
    std::vector<std::vector<OvAdj>> byVertex;        // appended in position order
    std::vector<Edge> edges;                         // index = Adj::edge - kOverlayBase
    std::vector<uint32_t> edgePos;
    std::unordered_map<uint64_t, uint32_t> lookup;   // (src,dst) -> overlay edge index
    std::vector<uint32_t> touchedVertices;
    void clear()
    {
        for (uint32_t v : touchedVertices) byVertex[v].clear();
        touchedVertices.clear();
        edges.clear();
        edgePos.clear();
        lookup.clear();
    }
    // drop every entry added by positions >= pos (entries are appended in position order everywhere)
    void truncate(uint32_t pos)
    {
        size_t keep = edges.size();
        while (keep > 0 && edgePos[keep - 1] >= pos) --keep;
        for (size_t ei = keep; ei < edges.size(); ei++) {
            const Edge &e = edges[ei];
            lookup.erase(edgeKey(e.src, e.dst));
            for (uint32_t v : {e.src, e.dst}) {
                std::vector<OvAdj> &l = byVertex[v];
                while (!l.empty() && l.back().pos >= pos) l.pop_back();
            }
        }
        edges.resize(keep);
        edgePos.resize(keep);
    }
    bool hasEither(uint32_t s, uint32_t d) const
    {
        return lookup.find(edgeKey(s, d)) != lookup.end() || lookup.find(edgeKey(d, s)) != lookup.end();
    }
    void add(const Edge &e, uint32_t pos)
    {
        const uint32_t ei = (uint32_t)edges.size();
        edges.push_back(e);
        edgePos.push_back(pos);
        lookup[edgeKey(e.src, e.dst)] = ei;
        if (byVertex[e.src].empty()) touchedVertices.push_back(e.src);
        byVertex[e.src].push_back(OvAdj{Adj{e.dst, ei, e.score}, pos});
        if (byVertex[e.dst].empty()) touchedVertices.push_back(e.dst);
        byVertex[e.dst].push_back(OvAdj{Adj{e.src, ei, e.score}, pos});
    }
};

struct GraphView {
    const Graph *g;
    const Overlay *ov;  // may be null
    uint32_t cutoff;    // overlay entries with pos < cutoff are visible
    const Edge *find(uint32_t s, uint32_t d) const
    {
        if (const Edge *e = g->find(s, d)) return e;
        if (ov) {
            auto it = ov->lookup.find(edgeKey(s, d));
            if (it != ov->lookup.end() && ov->edgePos[it->second] < cutoff) return &ov->edges[it->second];
        }
        return nullptr;
    }
};

// PoseGraphTraversal::recoverPath (graph_traversal.h:290-348): compose T_dst_src along the vertex path.
template <typename PathT>
bool recoverPath(const GraphView &gv, const PathT *path, size_t n, SE3 &pose)
{
    pose = se3Identity();  // :304
    for (size_t i = 1; i < n; ++i) {
        const uint32_t s = path[i - 1], d = path[i];
        if (const Edge *e = gv.find(s, d))
            pose = se3Mul(e->T, pose);  // :344
        else if (const Edge *e2 = gv.find(d, s))
            pose = se3Mul(se3Inverse(e2->T), pose);  // :342
        else
            return false;
    }
    return true;
}

// Pass 1 of an expansion over the committed entries, four at a time with AVX2 (runtime-dispatched; the scalar loop below
// is the definition).  Same IEEE operations per entry — compare + select for MIN/MAX (graph_traversal.h:843-848), two
// multiplications and one addition, never fused — so the costs are bit-identical to the scalar loop's.
#ifdef PGB_HAVE_AVX2_PATH
static const bool kUseAvx2 = __builtin_cpu_supports("avx2") && !(getenv("PGB_NO_AVX2") && atoi(getenv("PGB_NO_AVX2")) != 0);
__attribute__((target("avx2"))) size_t evalEntriesAvx2(const Adj *ra, uint32_t n, const uint32_t *mark, uint32_t epoch,
                                                       const double *simTo, double c0, double c1, double wgt, double omw,
                                                       double *cf, uint32_t *ce, size_t cnt, uint32_t &entryOut)
{
    const __m256d vc0 = _mm256_set1_pd(c0), vc1 = _mm256_set1_pd(c1), vw = _mm256_set1_pd(wgt), vo = _mm256_set1_pd(omw);
    const __m256d zero = _mm256_setzero_pd();
    const __m128i vep = _mm_set1_epi32((int)epoch);
    uint32_t e = 0;
    for (; e + 4 <= n; e += 4) {
        // Adj = {u32 next, u32 edge, f64 score}: two 32-byte loads hold entries (e, e+1) and (e+2, e+3)
        const __m256d a0 = _mm256_loadu_pd(reinterpret_cast<const double *>(ra + e));
        const __m256d a1 = _mm256_loadu_pd(reinterpret_cast<const double *>(ra + e + 2));
        const __m256d sc = _mm256_permute4x64_pd(_mm256_unpackhi_pd(a0, a1), 0xD8);  // scores of e, e+1, e+2, e+3
        const __m256i hd = _mm256_castpd_si256(_mm256_permute4x64_pd(_mm256_unpacklo_pd(a0, a1), 0xD8));  // (next, edge) x 4
        const __m128i nx = _mm256_castsi256_si128(_mm256_permutevar8x32_epi32(hd, _mm256_setr_epi32(0, 2, 4, 6, 0, 0, 0, 0)));
        const __m128i mk = _mm_i32gather_epi32(reinterpret_cast<const int *>(mark), nx, 4);
        const __m256d h = _mm256_i32gather_pd(simTo, nx, 8);
        const __m256d ec = _mm256_blendv_pd(vc0, sc, _mm256_cmp_pd(vc0, sc, _CMP_GT_OQ));  // c0 > score ? score : c0
        const __m256d nd = _mm256_blendv_pd(vc1, h, _mm256_cmp_pd(vc1, h, _CMP_LT_OQ));    // c1 < h ? h : c1
        const __m256d f = _mm256_add_pd(_mm256_mul_pd(vw, ec), _mm256_mul_pd(vo, nd));
        const int neg = _mm256_movemask_pd(_mm256_cmp_pd(sc, zero, _CMP_LT_OQ));           // score < 0
        const int seen = _mm_movemask_ps(_mm_castsi128_ps(_mm_cmpeq_epi32(mk, vep)));      // mark[next] == epoch
        const int ok = ~(neg | seen) & 15;
        alignas(32) double fo[4];
        _mm256_store_pd(fo, f);
#pragma GCC unroll 4
        for (int k = 0; k < 4; k++) {
            cf[cnt] = fo[k];
            ce[cnt] = e + (uint32_t)k;
            cnt += (ok >> k) & 1;
        }
    }
    entryOut = e;
    return cnt;
}
#endif

#ifdef PGB_HAVE_AVX2_PATH
// The same pass eight entries at a time where the CPU has AVX-512 (compress stores replace the scalar compaction).
static const bool kUseAvx512 = __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512vl") &&
                               !(getenv("PGB_NO_AVX512") && atoi(getenv("PGB_NO_AVX512")) != 0);
__attribute__((target("avx512f,avx512vl,avx2"))) size_t evalEntriesAvx512(const Adj *ra, uint32_t n, const uint32_t *mark, uint32_t epoch,
                                                                         const double *simTo, double c0, double c1, double wgt,
                                                                         double omw, double *cf, uint32_t *ce, size_t cnt,
                                                                         uint32_t &entryOut)
{
    const __m512d vc0 = _mm512_set1_pd(c0), vc1 = _mm512_set1_pd(c1), vw = _mm512_set1_pd(wgt), vo = _mm512_set1_pd(omw);
    const __m512d zero = _mm512_setzero_pd();
    const __m256i vep = _mm256_set1_epi32((int)epoch);
    const __m512i idxScore = _mm512_setr_epi64(1, 3, 5, 7, 9, 11, 13, 15), idxHead = _mm512_setr_epi64(0, 2, 4, 6, 8, 10, 12, 14);
    __m256i vent = _mm256_setr_epi32(0, 1, 2, 3, 4, 5, 6, 7);
    const __m256i eight = _mm256_set1_epi32(8);
    uint32_t e = 0;
    for (; e + 8 <= n; e += 8) {
        // Adj = {u32 next, u32 edge, f64 score}: two 64-byte loads hold entries e..e+3 and e+4..e+7
        const __m512d a0 = _mm512_loadu_pd(reinterpret_cast<const double *>(ra + e));
        const __m512d a1 = _mm512_loadu_pd(reinterpret_cast<const double *>(ra + e + 4));
        const __m512d sc = _mm512_permutex2var_pd(a0, idxScore, a1);
        const __m256i nx = _mm512_cvtepi64_epi32(_mm512_castpd_si512(_mm512_permutex2var_pd(a0, idxHead, a1)));  // low halves: next
        const __m256i mk = _mm256_i32gather_epi32(reinterpret_cast<const int *>(mark), nx, 4);
        const __m512d h = _mm512_i32gather_pd(nx, simTo, 8);
        const __m512d ec = _mm512_mask_blend_pd(_mm512_cmp_pd_mask(vc0, sc, _CMP_GT_OQ), vc0, sc);  // c0 > score ? score : c0
        const __m512d nd = _mm512_mask_blend_pd(_mm512_cmp_pd_mask(vc1, h, _CMP_LT_OQ), vc1, h);    // c1 < h ? h : c1
        const __m512d f = _mm512_add_pd(_mm512_mul_pd(vw, ec), _mm512_mul_pd(vo, nd));
        const __mmask8 ok = (__mmask8)(~_mm512_cmp_pd_mask(sc, zero, _CMP_LT_OQ)) & _mm256_cmpneq_epi32_mask(mk, vep);
        _mm512_mask_compressstoreu_pd(cf + cnt, ok, f);
        _mm256_mask_compressstoreu_epi32(ce + cnt, ok, vent);
        cnt += (size_t)__builtin_popcount(ok);
        vent = _mm256_add_epi32(vent, eight);
    }
    entryOut = e;
    return cnt;
}
#endif

// AStarTraversal<ImageSimilarityHeuristics>::getPath with the arguments of pose_graph_builder.h:834-841.
//
// The open list is std::priority_queue's binary heap, replayed slot by slot (std::push_heap / std::pop_heap of
// libstdc++: the pop order among equal costs depends on the heap layout, and children of one expansion mostly share
// their cost, SURVEY App. A.3) — but ORDERED only where it can matter.  `floorF` is a guess of the smallest cost the
// search will ever pop.  A child below it takes its slot in the array (slot numbers are what the layout is made of)
// WITHOUT the climb of std::push_heap.  As long as no such entry reaches the top, every entry >= floorF ("live") sits in
// exactly the slot the fully ordered queue would give it.  Induction over the queue operations, with the invariant
// that all ancestors of a live entry are live:
//   push   a live child climbs while its parent is smaller (std::__push_heap): past every non-live ancestor whatever
//          their mutual order — they move down the climbed path — and past smaller live ones, which move down one slot
//          of the path exactly as in the ordered queue; a non-live child cannot displace a live entry;
//   pop    std::__adjust_heap moves the larger child into the hole level by level (right child on ties): where at least
//          one child is live the choice is made among live entries by their values, and once both are non-live no live
//          entry lies underneath (invariant), so the rest of the descent only permutes non-live entries; the entry X of
//          the last slot is then pushed up from the leaf: a live X passes every non-live entry and every smaller live
//          entry of the hole's path (they return to the slots they came from) and stops below the first live entry
//          >= X; a non-live X stays underneath the live part of the path.
// Which slots hold live entries, and which live entry sits where, is therefore the same as in the ordered queue after
// every operation, and so is the sequence of popped entries.  In a dense view graph 60-90 % of the children are below
// anything that is ever popped, and their climbs — random walks through equally irrelevant entries, one mispredicted
// loop exit each — were ~70 % of the search time.  If an entry below the floor does reach the top, the guess was too
// high: out.valid = false and the caller repeats the search without a floor (the plain replay).
void aStar(const GraphView &gv, const double *sim /*transposed*/, uint32_t V, uint32_t from, uint32_t to, size_t maxDepth,
           double weight, AStarScratch &S, AStarOut &out, double floorF = -1.0)
{
    const Graph &g = *gv.g;
    out.found = false;
    out.valid = true;
    out.minPoppedF = 2.0;
    out.touched = 0;
    out.pushes = 0;
    out.expanded.clear();
    out.expCost.clear();
    if (S.mark.size() != V) { S.mark.assign(V, 0); S.epoch = 0; }
    if (++S.epoch == 0) { std::fill(S.mark.begin(), S.mark.end(), 0); S.epoch = 1; }
    S.arena.clear();
    auto cmp = [](const HeapItem &a, const HeapItem &b) { return a.f < b.f; };  // graph_traversal.h:669-673
    // the priority queue lives in a raw buffer (S.heap is only its storage; hs is the queue size)
    if (S.heap.size() < 1024) S.heap.resize(1024);
    HeapItem *H = S.heap.data();
    size_t hs = 0;
    H[hs++] = HeapItem{0.0, UINT32_MAX, 0};  // start node, cost (1,0,0)  :721
    const double oneMinusWeight = 1.0 - weight;
    // `edges` keeps its previous content when a vertex has no list (pose_graph.h:145-146).  Every vertex reached by
    // the search has at least the edge it was reached through, and the source has edges whenever hasLink holds, so
    // the stale case cannot occur; the owner is tracked only to keep the restatement literal.
    uint32_t listOwner = UINT32_MAX;
    const double *simTo = sim + (size_t)to * V;  // transposed table: simTo[next] = similarity(next, to)
    const uint32_t *mark = S.mark.data();
    const uint32_t epoch = S.epoch;
    // edge-list entry `idx` of vertex lv as seen by this search: committed entries first, then overlay entries
    auto entryAt = [&](uint32_t lv, uint32_t idx) -> const Adj & {
        const std::vector<Adj> &real = g.byVertex[lv];
        return idx < real.size() ? real[idx] : gv.ov->byVertex[lv][idx - real.size()].a;
    };
    while (hs > 0) {
        const HeapItem top = H[0];
        ++out.touched;  // :750
        std::pop_heap(H, H + hs, cmp);
        --hs;
        // materialise the popped node
        ArenaNode node;
        if (top.parent == UINT32_MAX) {
            node = ArenaNode{from, UINT32_MAX, 0, UINT32_MAX, 1.0, 0.0};
        } else {
            if (top.f < floorF) { out.valid = false; return; }  // the floor was a bad guess
            if (top.f < out.minPoppedF) out.minPoppedF = top.f;
            const ArenaNode &pn = S.arena[top.parent];
            const Adj &e = entryAt(pn.listOwner, top.entry);
            uint32_t next = e.next;
            if (pn.listOwner != pn.vertex) next = e.next == pn.vertex ? pn.listOwner : e.next;
            const double h = simTo[next];  // already clamped
            node.vertex = next;
            node.parent = top.parent;
            node.depth = pn.depth + 1;
            node.listOwner = UINT32_MAX;
            node.c0 = pn.c0 > e.score ? e.score : pn.c0;
            node.c1 = pn.c1 < h ? h : pn.c1;
        }
        if (node.depth > maxDepth) continue;  // :755
        const uint32_t v = node.vertex;
        if (v == to) {  // :766
            S.path.clear();
            S.path.push_back(v);
            for (uint32_t k = node.parent; k != UINT32_MAX; k = S.arena[k].parent) S.path.push_back(S.arena[k].vertex);
            std::reverse(S.path.begin(), S.path.end());
            SE3 pose;
            const bool ok = recoverPath(gv, S.path.data(), S.path.size(), pose);
            if (ok) {
                out.found = true;
                out.pose = pose;
                break;  // one path is tested, then the search ends (:792-800 with kMaximumPathNumber = 1)
            }
            continue;
        }
        S.mark[v] = epoch;  // nodeStates[v] = Open  :814
        // `expanded` = the vertices whose edge lists this search ITERATED (:820-866): what a later graph change must touch
        // to invalidate the result.  A node popped at the maximum depth is marked but pushes nothing.
        if (node.depth < maxDepth) {
            out.expanded.push_back(v);
            out.expCost.push_back(node.c0);
            out.expCost.push_back(node.c1);
        }
        const std::vector<Adj> &real = g.byVertex[v];
        const std::vector<OvAdj> *ovl = gv.ov ? &gv.ov->byVertex[v] : nullptr;
        const bool hasOv = ovl && !ovl->empty() && (*ovl)[0].pos < gv.cutoff;
        if (!real.empty() || hasOv) listOwner = v;  // :817
        node.listOwner = listOwner;
        const uint32_t ni = (uint32_t)S.arena.size();
        S.arena.push_back(node);
        if (node.depth < maxDepth && listOwner != UINT32_MAX) {  // :820
            const uint32_t lv = listOwner;
            const double c0 = node.c0, c1 = node.c1;
            // Children are pushed with std::push_heap semantics, spelled out (libstdc++ std::__push_heap: sift the hole
            // up while parent < value) on a raw buffer sized for the whole edge list up front.
            const std::vector<Adj> &rl = g.byVertex[lv];
            const std::vector<OvAdj> *ol = gv.ov ? &gv.ov->byVertex[lv] : nullptr;
            const size_t room = hs + rl.size() + (ol ? ol->size() : 0);
            if (S.heap.size() < room) {
                S.heap.resize(std::max(room, 2 * S.heap.size()));
                H = S.heap.data();
            }
            HeapItem *const first = H;
            const size_t hs0 = hs;
            const double wgt = weight;
            uint32_t entry = 0;
            // Two passes over the edge list.  Pass 1 evaluates every entry without a data-dependent branch (admissible
            // children are compacted into a scratch array by a predicated store); pass 2 replays std::push_heap for them
            // in list order, so the sift-up's unpredictable exit does not sit between two gathers.
            const size_t listLen = rl.size() + (ol ? ol->size() : 0);
            if (S.childF.size() < listLen + 8) { S.childF.resize(listLen + 8); S.childE.resize(listLen + 8); }  // (+8: a compress store may be issued at the very end)
            double *cf = S.childF.data();
            uint32_t *ce = S.childE.data();
            size_t cnt = 0;
            auto eval = [&](const Adj &e, uint32_t ent) __attribute__((always_inline)) {
                uint32_t next = e.next;     // (v == dst) ? src : dst  :838-840
                if (lv != v) next = e.next == v ? lv : e.next;  // stale list of another vertex (unreachable, see above)
                // kMinimumInlierRatio is `const bool` receiving 0.0 (:613, :839); nodeStates.find(next) != end  :855-856
                const bool ok = !(e.score < 0.0) && mark[next] != epoch;
                const double edgeCost = c0 > e.score ? e.score : c0;  // MIN :843
                const double h = simTo[next];  // std::clamp(getSimilarity(next, to), 0, 1)  :594 (pre-clamped table)
                const double nextToDest = c1 < h ? h : c1;  // MAX :847
                cf[cnt] = wgt * edgeCost + oneMinusWeight * nextToDest;  // :851-852
                ce[cnt] = ent;
                cnt += ok ? 1 : 0;
            };
            const Adj *ra = rl.data();
            const uint32_t nr = (uint32_t)rl.size();
#ifdef PGB_HAVE_AVX2_PATH
            if (kUseAvx512 && lv == v) cnt = evalEntriesAvx512(ra, nr, mark, epoch, simTo, c0, c1, wgt, oneMinusWeight, cf, ce, cnt, entry);
            else if (kUseAvx2 && lv == v) cnt = evalEntriesAvx2(ra, nr, mark, epoch, simTo, c0, c1, wgt, oneMinusWeight, cf, ce, cnt, entry);
#endif
            for (; entry < nr; ++entry) eval(ra[entry], entry);
            if (ol)
                for (const OvAdj &oe : *ol) {
                    if (oe.pos >= gv.cutoff) break;
                    eval(oe.a, entry++);
                }
            // Pass 2.  A sequential std::push_heap of child i touches only ancestors of its slot; ancestors that were in the
            // heap before this expansion can only grow while its children are pushed, so a child that is not larger than
            // its parent NOW stays where it is appended.  All children are appended first, the ones that move are then
            // replayed in list order (when the heap is smaller than the batch, parents may be new slots: replay them all).
            if (hs >= cnt) {
                size_t nMove = 0;
                uint32_t *mv = S.childMove.size() < cnt ? (S.childMove.resize(listLen), S.childMove.data()) : S.childMove.data();
                for (size_t i = 0; i < cnt; i++) {
                    const size_t slot = hs + i;
                    first[slot] = HeapItem{cf[i], ni, ce[i]};
                    mv[nMove] = (uint32_t)i;
                    nMove += (first[(slot - 1) / 2].f < cf[i]) & (cf[i] >= floorF) ? 1 : 0;  // slot >= 1 here (hs >= cnt >= 1)
                }
                for (size_t k = 0; k < nMove; k++) {
                    const size_t i = mv[k];
                    const double combined = cf[i];
                    size_t hole = hs + i;
                    while (hole > 0) {
                        const size_t parent = (hole - 1) / 2;
                        if (!(first[parent].f < combined)) break;
                        first[hole] = first[parent];
                        hole = parent;
                    }
                    first[hole] = HeapItem{combined, ni, ce[i]};
                }
                hs += cnt;
            } else
                for (size_t i = 0; i < cnt; i++) {
                    const double combined = cf[i];
                    size_t hole = hs++;
                    if (combined >= floorF)
                        while (hole > 0) {
                            const size_t parent = (hole - 1) / 2;
                            if (!(first[parent].f < combined)) break;
                            first[hole] = first[parent];
                            hole = parent;
                        }
                    first[hole] = HeapItem{combined, ni, ce[i]};
                }
            out.pushes += (uint32_t)(hs - hs0);
        }
    }
}

// What a position contributes to the graph: nothing, or an edge with a pose/score.
struct Outcome {
    bool known = false;     // verdict available
    bool accepted = false;
    uint8_t branch = 0;
    uint32_t inliers = 0;
    double q[4] = {0, 0, 0, 1}, t[3] = {0, 0, 0};
    bool sameEdge(const Outcome &o) const
    {
        if (known != o.known || accepted != o.accepted) return false;
        if (!accepted) return true;
        return inliers == o.inliers && !memcmp(q, o.q, sizeof q) && !memcmp(t, o.t, sizeof t);
    }
};

struct Item {
    uint32_t pairId = UINT32_MAX;  // UINT32_MAX: queued pair without registered correspondences
    uint32_t src = 0, dst = 0;
    uint32_t nCorr = 0;
    bool staticSkip = false;  // no correspondences / fewer than minimum_point_number (pose_graph_builder.h:550-551)
    bool dupSkip = false;     // the graph (committed, or predicted by an earlier wave position) already has this pair
                              // in either direction: the reference skips it before anything else (:438-443)
    bool searched = false;    // search result below is consistent with the current overlay
    bool visible = false;
    bool hasHyp = false;
    SE3 hyp = se3Identity();
    std::vector<uint32_t> expanded;
    std::vector<double> expCost;  // (c0, c1) per entry of `expanded` (empty: not recorded, e.g. a device search)
    double tauMin = 2.0;          // smallest cost the current search result popped (2: nothing but the start node)
    uint32_t touched = 0, pushes = 0;
    double floorSeen = -1.0;  // smallest cost the position's last search popped (< 0: none yet): the next search's floor guess
    bool needGpu = false;
    Outcome pred;             // what the overlay currently assumes for this position
    const pgi_verdict *finalV = nullptr, *pathV = nullptr;
    bool mine = true;         // this rank searches / verifies the position (pair owner); others learn it by exchange
    bool remoteKnown = false; // a record of the owner has been imported
    pgi_verdict remoteV;      // the owner's path verdict for the position (remote positions only)
};

struct Change {  // a wave position whose actual outcome differs from the prediction the overlay was built from
    uint32_t k, u, w;
    bool existence;      // the edge appears or disappears (otherwise only its score / pose changes)
    double sOld, sNew;   // inlier ratios of the predicted and of the actual edge
};

// The fine staleness rule for ONE expansion of a search: the expansion's node had the cost tuple (c0, c1), `h` is the
// heuristic of the changed edge's other endpoint, the edge's score goes sOld -> sNew, tauMin is the smallest combined cost
// the search popped.  The child pushed through the edge costs weight * min(c0, score) + (1 - weight) * max(c1, h)
// (graph_traversal.h:843-852, same operations); if that is below tauMin under both scores, the child is an entry that
// never leaves the queue and whose value decides nothing (aStar's cost-floor argument with floor = tauMin), so the search
// is bit for bit the same with either score.
inline bool scoreChangeIsInert(double c0, double c1, double h, double sOld, double sNew, double wgt, double omw, double tauMin)
{
    const double nd = c1 < h ? h : c1;
    const double fOld = wgt * (c0 > sOld ? sOld : c0) + omw * nd;
    const double fNew = wgt * (c0 > sNew ? sNew : c0) + omw * nd;
    return fOld < tauMin && fNew < tauMin;
}

struct HypKey {
    uint32_t pair;
    uint64_t bits[7];
    bool operator==(const HypKey &o) const { return pair == o.pair && !memcmp(bits, o.bits, sizeof bits); }
};
struct HypKeyHash {
    size_t operator()(const HypKey &k) const
    {
        uint64_t h = 1469598103934665603ull ^ k.pair;
        for (int i = 0; i < 7; i++) { h ^= k.bits[i]; h *= 1099511628211ull; }
        return (size_t)h;
    }
};
struct PathVerdict {
    bool ok;
    pgi_verdict v;
};

inline HypKey makeKey(uint32_t pair, const SE3 &h)
{
    HypKey k;
    k.pair = pair;
    memcpy(k.bits, h.q, 32);
    memcpy(k.bits + 4, h.t, 24);
    return k;
}

double nowSec() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// Minimal persistent worker pool (the reference spawns one OpenMP worker per core, pose_graph_builder.h:391-397).
struct Pool {
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cvWork, cvDone;
    std::function<void(int)> job;
    uint64_t generation = 0;
    int active = 0;
    bool quit = false;
    void start(int n)
    {
        for (int t = 1; t < n; t++)
            threads.emplace_back([this, t]() {
                uint64_t seen = 0;
                for (;;) {
                    std::function<void(int)> j;
                    {
                        std::unique_lock<std::mutex> lk(m);
                        cvWork.wait(lk, [&]() { return quit || generation != seen; });
                        if (quit) return;
                        seen = generation;
                        j = job;
                    }
                    j(t);
                    {
                        std::lock_guard<std::mutex> lk(m);
                        if (--active == 0) cvDone.notify_all();
                    }
                }
            });
    }
    void run(const std::function<void(int)> &j)
    {
        {
            std::lock_guard<std::mutex> lk(m);
            job = j;
            active = (int)threads.size();
            ++generation;
        }
        cvWork.notify_all();
        j(0);
        std::unique_lock<std::mutex> lk(m);
        cvDone.wait(lk, [&]() { return active == 0; });
    }
    ~Pool()
    {
        {
            std::lock_guard<std::mutex> lk(m);
            quit = true;
        }
        cvWork.notify_all();
        for (auto &t : threads) t.join();
    }
};

}  // namespace

struct pgb_builder {
    std::mutex driveMu;  // guards the host state between pgb_run_wave and pgb_set_fallback_verdicts_some (other thread)
    std::vector<pgb_item> driveItems;
    std::vector<uint32_t> driveIds, driveHoff;
    std::vector<double> driveHyp;
    std::vector<pgi_verdict> driveVerdicts;
    pgb_config cfg;
    Pool pool;
    uint32_t V = 0;
    std::vector<double> sim;  // transposed
    uint64_t P = 0;
    std::vector<uint32_t> pairViews;
    std::vector<uint64_t> mOffset;
    std::unordered_map<uint64_t, uint32_t> pairIndex;
    // similarity-ordered queue, materialised in pop order (the queue is static: imagesimilarity_graph.h:149-157)
    std::vector<std::pair<uint32_t, uint32_t>> order;
    size_t nextInOrder = 0;
    std::deque<Item> pending;  // re-queued items, in queue order, ahead of `order[nextInOrder..]`
    Graph graph;
    Visibility vis, visPred;
    std::vector<Visibility> visCkpt;  // simulated table before positions 32, 64, ... of the open wave (rebuildOverlay)
    Overlay overlay;
    std::vector<Item> wave;
    bool waveOpen = false;
    int rounds = 0;
    int rank = 0, world = 1;
    int phase = 0;                 // 0 search/resolve, 1 waiting for the record exchange, 2 compare
    int status = 0;                // PGB_WAVE_* of the open wave
    std::vector<uint32_t> minChangedPos;  // per vertex: smallest wave position whose outcome changed this round
    std::vector<Change> changes;          // the round's changed positions, in position order
    std::vector<std::vector<uint32_t>> changesOf;  // per vertex: indices into `changes` of the edges touching it
    std::vector<pgi_verdict> fbCache;
    std::vector<uint8_t> fbHave;
    std::unordered_map<HypKey, PathVerdict, HypKeyHash> pathCache;
    std::vector<pgb_log> log;
    pgb_counters ctr;
    std::vector<AStarScratch> scratch;
    // device search backend (pgb_set_search_backend): the engine's pgi_graph_apply / pgi_graph_search
    pgb_graph_apply_fn gpuApply = nullptr;
    pgb_graph_search_fn gpuSearch = nullptr;
    void *gpuEngine = nullptr;
    uint32_t gpuMinBatch = 0;
    int32_t searchError = 0;     // first engine status of a failed device search (surfaced by pgb_run_wave)
    bool gpuCheck = false;       // PGB_SEARCH_CHECK=1: every device search is repeated on the host and compared
    bool ovDirty = true;         // the overlay changed since it was last mirrored to the device
    double hybridShare = 0.3;    // share of a round's estimated search work the host pool takes beside the device
    uint32_t gpuBudget = 0;      // push budget of the round's device queries (0: unlimited)
    std::vector<double> srcFloor, dstFloor;  // per view: smallest popped cost of the last search from / to it (floor guesses)
    std::vector<uint32_t> srcCost;  // per source view: pushes of the last search that started there (cost estimate)
    double meanCost = 0.0;       // running mean of pushes per search
    std::vector<pgi_adj_entry> gpuEntries, commitEntries;
    std::vector<uint32_t> gpuCommitted, gpuTotal, gpuBits, gpuTodo;
    std::vector<pgi_query> gpuQueries;
    std::vector<pgi_search_result> gpuResults;
    // pgb_run_hashing: one entry per log record
    std::vector<uint8_t> matchSource;
    std::vector<uint32_t> guidedRows;
};

namespace {

Outcome outcomeOf(const pgi_verdict *v)
{
    Outcome o;
    o.known = v != nullptr;
    if (v && v->accepted) {
        o.accepted = true;
        o.branch = v->branch;
        o.inliers = v->inlier_count;
        memcpy(o.q, v->q, sizeof o.q);
        memcpy(o.t, v->t, sizeof o.t);
    }
    return o;
}

Edge edgeOf(const Item &it, const Outcome &o)
{
    Edge e;
    e.src = it.src; e.dst = it.dst;
    memcpy(e.T.q, o.q, 32);
    memcpy(e.T.t, o.t, 24);
    e.score = (double)o.inliers / (double)it.nCorr;  // pose_graph_builder.h:645-646
    e.inlierNumber = o.inliers; e.nCorr = it.nCorr; e.branch = o.branch;
    return e;
}

// Rebuild the overlay and the simulated visibility from the current predictions, starting at wave position `from`
// (the first position whose prediction changed: everything before it is unchanged, and so is the state those
// positions leave behind); positions whose hasLink answer changed lose their search result.  The simulated table is
// checkpointed every kCkptStride positions so that a late `from` only replays the tail of the wave.
constexpr uint32_t kCkptStride = 32;
// pose_graph_builder.h:438-443 as the sequential run would answer it at this position: the overlay holds exactly the
// edges predicted by the earlier positions while rebuildOverlay walks the wave in order.
inline bool isDuplicate(const pgb_builder *b, const Item &it)
{
    return b->graph.hasEdge(it.src, it.dst) || b->graph.hasEdge(it.dst, it.src) || b->overlay.hasEither(it.src, it.dst);
}
void rebuildOverlay(pgb_builder *b, uint32_t from = 0)
{
    PgiNvtxRange nvtxRange("pgb:rebuild overlay + simulated visibility");
    const double t0 = nowSec();
    b->ovDirty = true;
    bool allLinked = true;
    for (const Item &it : b->wave)
        if (!it.staticSkip && !b->vis.hasLink(it.src, it.dst)) { allLinked = false; break; }
    if (allLinked) {
        // Every pair the wave can commit is already linked in the committed table.  addLink on an existing link only
        // inserts into the two neighbour sets and returns (visibility_table.h:62-73), so no link can appear during this
        // wave and hasLink answers what the committed table answers: nothing needs to be simulated.  (The neighbour
        // sets are updated by the real commit, in order.)
        b->overlay.truncate(from);
        if (from == 0) b->overlay.clear();
        for (uint32_t k = from; k < b->wave.size(); k++) {
            Item &it = b->wave[k];
            const bool vis = b->vis.hasLink(it.src, it.dst);
            const bool dup = isDuplicate(b, it);
            if (it.searched && (vis != it.visible || dup != it.dupSkip)) it.searched = false;
            it.visible = vis;
            it.dupSkip = dup;
            if (!it.staticSkip && !dup && it.pred.known && it.pred.accepted) b->overlay.add(edgeOf(it, it.pred), k);
        }
        b->visCkpt.clear();
        b->ctr.sec_visibility += nowSec() - t0;
        return;
    }
    uint32_t start = (from / kCkptStride) * kCkptStride;
    if (start > 0 && start / kCkptStride - 1 >= b->visCkpt.size()) start = 0;  // no checkpoint that far (first build)
    if (start == 0) {
        b->overlay.clear();
        b->visPred = b->vis;
    } else {
        b->overlay.truncate(start);
        b->visPred = b->visCkpt[start / kCkptStride - 1];
    }
    for (uint32_t k = start; k < b->wave.size(); k++) {
        if (k > start && k % kCkptStride == 0) {
            const size_t ci = k / kCkptStride - 1;
            if (b->visCkpt.size() <= ci) b->visCkpt.resize(ci + 1);
            b->visCkpt[ci] = b->visPred;
        }
        Item &it = b->wave[k];
        const bool vis = b->visPred.hasLink(it.src, it.dst);  // pose_graph_builder.h:456-457 at position k
        const bool dup = isDuplicate(b, it);
        if (it.searched && (vis != it.visible || dup != it.dupSkip)) it.searched = false;
        it.visible = vis;
        it.dupSkip = dup;
        if (!it.staticSkip && !dup && it.pred.known && it.pred.accepted) {
            b->overlay.add(edgeOf(it, it.pred), k);
            b->visPred.addLink(it.src, it.dst);  // :692
        }
    }
    b->ctr.sec_visibility += nowSec() - t0;
}

// Margin under the remembered floors for the next guess.
static const double kFloorMargin = 0.01;

void searchPosition(pgb_builder *b, uint32_t k, AStarScratch &S)
{
    Item &it = b->wave[k];
    it.hasHyp = false;
    it.expanded.clear();
    it.expCost.clear();
    it.tauMin = 2.0;
    it.touched = it.pushes = 0;
    if (b->cfg.use_path_finding && it.visible && !it.staticSkip && !it.dupSkip) {  // :569-570
        AStarOut o;
        GraphView gv{&b->graph, &b->overlay, k};
        // Cost-floor guess (see aStar): what this position's previous search needed, else what the last searches from the
        // same source view and to the same destination view needed (neighbouring queue positions behave alike), minus a
        // margin.  The tables are hints shared by the pool threads without synchronisation — any value is a valid guess.
        double floorF = -1.0;
        double g = it.floorSeen;
        if (g < 0.0 && b->srcFloor[it.src] >= 0.0 && b->dstFloor[it.dst] >= 0.0) g = std::min(b->srcFloor[it.src], b->dstFloor[it.dst]);
        if (g >= 0.0) floorF = g - kFloorMargin;
        aStar(gv, b->sim.data(), b->V, it.src, it.dst, (size_t)b->cfg.maximum_search_depth,
              b->cfg.traversal_heuristics_weight, S, o, floorF);
        if (!o.valid && floorF - 0.05 > 0.0) {  // guessed too high: once more with a wide margin, then without a floor
            S.floorRetries++;
            aStar(gv, b->sim.data(), b->V, it.src, it.dst, (size_t)b->cfg.maximum_search_depth,
                  b->cfg.traversal_heuristics_weight, S, o, floorF - 0.05);
        }
        if (!o.valid) {
            S.floorRetries++;
            aStar(gv, b->sim.data(), b->V, it.src, it.dst, (size_t)b->cfg.maximum_search_depth,
                  b->cfg.traversal_heuristics_weight, S, o);
        }
        if (o.minPoppedF <= 1.0) it.floorSeen = b->srcFloor[it.src] = b->dstFloor[it.dst] = o.minPoppedF;
        it.hasHyp = o.found;
        it.hyp = o.pose;
        it.expanded.swap(o.expanded);
        it.expCost.swap(o.expCost);
        it.tauMin = o.minPoppedF;
        it.touched = o.touched;
        it.pushes = o.pushes;
    }
    it.searched = true;
}

void searchOnHost(pgb_builder *b, const std::vector<uint32_t> &todoIn)
{
    if (b->cfg.host_threads <= 1 || todoIn.size() < 4) {
        for (uint32_t k : todoIn) searchPosition(b, k, b->scratch[0]);
    } else {
        // search costs are heavy-tailed (the longest search of a round is ~10x the mean): hand the threads the
        // longest-looking searches first (a position's previous search is the estimate), so that no thread starts a
        // long one when the others are about to run dry
        std::vector<uint32_t> todo(todoIn);
        std::stable_sort(todo.begin(), todo.end(), [&](uint32_t x, uint32_t y) { return b->wave[x].pushes > b->wave[y].pushes; });
        std::atomic<size_t> next(0);
        b->pool.run([&](int tid) {
            for (;;) {
                const size_t i = next.fetch_add(1);
                if (i >= todo.size()) break;
                searchPosition(b, todo[i], b->scratch[tid]);
            }
        });
    }
}

// Mirror the open wave's overlay to the device graph: every predicted entry with its slot behind the committed
// entries of its vertex (tag = wave position + 1), plus the per-vertex counts.
int32_t uploadOverlay(pgb_builder *b)
{
    const uint32_t V = b->V;
    b->gpuEntries.clear();
    b->gpuCommitted.resize(V);
    b->gpuTotal.resize(V);
    for (uint32_t v = 0; v < V; v++) b->gpuCommitted[v] = b->gpuTotal[v] = (uint32_t)b->graph.byVertex[v].size();
    for (uint32_t v : b->overlay.touchedVertices) {
        const std::vector<OvAdj> &l = b->overlay.byVertex[v];
        const uint32_t base = b->gpuCommitted[v];
        for (uint32_t j = 0; j < l.size(); j++)
            b->gpuEntries.push_back(pgi_adj_entry{v, base + j, l[j].a.next, l[j].pos + 1u, l[j].a.score});
        b->gpuTotal[v] = base + (uint32_t)l.size();
    }
    const int32_t rc = b->gpuApply(b->gpuEngine, (uint32_t)b->gpuEntries.size(), b->gpuEntries.data(), b->gpuCommitted.data(),
                                   b->gpuTotal.data());
    if (rc == 0) b->ovDirty = false;
    return rc;
}

// Search the positions of `todo` with the device backend (K6, pgi_graph_search); positions the device could not
// finish (slab overflow) and trivially hypothesis-free positions are completed on the host.
int32_t searchOnDevice(pgb_builder *b, const std::vector<uint32_t> &todo, std::vector<uint32_t> &redo)
{
    const double t0 = nowSec();
    redo.clear();
    if (b->ovDirty) {
        const int32_t rc = uploadOverlay(b);
        if (rc != 0) return rc;
    }
    const uint32_t words = (b->V + 31) / 32;
    b->gpuQueries.clear();
    b->gpuTodo.clear();
    for (uint32_t k : todo) {
        Item &it = b->wave[k];
        if (b->cfg.use_path_finding && it.visible && !it.staticSkip && !it.dupSkip) {  // pose_graph_builder.h:569-570
            b->gpuQueries.push_back(pgi_query{it.src, it.dst, k, b->gpuBudget});
            b->gpuTodo.push_back(k);
        } else {
            it.hasHyp = false;
            it.expanded.clear();
            it.touched = it.pushes = 0;
            it.searched = true;
        }
    }
    const uint32_t n = (uint32_t)b->gpuQueries.size();
    if (n == 0) return 0;
    b->gpuResults.resize(n);
    b->gpuBits.resize((size_t)n * words);
    const int32_t rc = b->gpuSearch(b->gpuEngine, n, b->gpuQueries.data(), (uint32_t)b->cfg.maximum_search_depth,
                                    b->cfg.traversal_heuristics_weight, b->gpuResults.data(), b->gpuBits.data());
    if (rc != 0) return rc;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t k = b->gpuTodo[i];
        Item &it = b->wave[k];
        const pgi_search_result &r = b->gpuResults[i];
        if (r.status != 0) { redo.push_back(k); continue; }
        it.touched = r.touched;
        it.pushes = r.pushes;
        it.expanded.clear();
        it.expCost.clear();  // not recorded by the device search: the coarse staleness rule applies
        const uint32_t *bits = b->gpuBits.data() + (size_t)i * words;
        for (uint32_t w = 0; w < words; w++) {
            uint32_t x = bits[w];
            while (x) {
                it.expanded.push_back(w * 32 + (uint32_t)__builtin_ctz(x));
                x &= x - 1;
            }
        }
        it.hasHyp = false;
        if (r.found) {
            GraphView gv{&b->graph, &b->overlay, k};
            SE3 pose;
            if (recoverPath(gv, r.path, r.path_len, pose)) {
                it.hasHyp = true;
                it.hyp = pose;
            } else
                redo.push_back(k);  // (cannot happen: the path's edges are in the graph the search saw)
        }
        it.searched = true;
    }
    b->ctr.gpu_searches += n - redo.size();
    b->ctr.gpu_search_redo += redo.size();
    b->ctr.sec_search_gpu += nowSec() - t0;
    return 0;
}

// PGB_SEARCH_CHECK=1: repeat every device search of the round on the host and compare what the wave logic consumes.
void checkDeviceSearches(pgb_builder *b)
{
    for (uint32_t k : b->gpuTodo) {
        Item &it = b->wave[k];
        const bool hasHyp = it.hasHyp;
        const SE3 hyp = it.hyp;
        std::vector<uint32_t> exp = it.expanded;
        const uint32_t touched = it.touched, pushes = it.pushes;
        searchPosition(b, k, b->scratch[0]);
        std::vector<uint32_t> expHost = it.expanded;
        std::sort(exp.begin(), exp.end());
        exp.erase(std::unique(exp.begin(), exp.end()), exp.end());  // (a position redone on the host lists re-expansions)
        std::sort(expHost.begin(), expHost.end());
        expHost.erase(std::unique(expHost.begin(), expHost.end()), expHost.end());
        const bool same = hasHyp == it.hasHyp && (!hasHyp || !memcmp(&hyp, &it.hyp, sizeof(SE3))) && touched == it.touched &&
                          pushes == it.pushes && exp == expHost;
        if (!same) {
            if (b->ctr.search_mismatches < 10)
                fprintf(stderr, "[pgb] device/host search mismatch at wave position %u (%u -> %u): found %d/%d touched %u/%u pushes %u/%u expanded %zu/%zu\n",
                        k, it.src, it.dst, (int)hasHyp, (int)it.hasHyp, touched, it.touched, pushes, it.pushes, exp.size(), expHost.size());
            b->ctr.search_mismatches++;
        }
    }
}

// Search the stale positions below `limit` (pgb_config.reserved can restrict the re-search to a window behind the
// first stale position; unlimited by default).
void searchStale(pgb_builder *b, uint32_t limit)
{
    PgiNvtxRange nvtxRange("pgb:A* round (stale positions, thread pool)");
    const double t0 = nowSec();
    std::vector<uint32_t> todo;
    for (uint32_t k = 0; k < b->wave.size() && k < limit; k++)
        if (b->wave[k].mine && !b->wave[k].searched) todo.push_back(k);
    bool done = false;
    if (b->gpuSearch && todo.size() >= b->gpuMinBatch && b->V <= 65535u && b->cfg.maximum_search_depth <= 7) {
        // Device and host pool work on the round together.  The device's time for a round is the time of its longest
        // search (one warp per search), the pool's is the sum of its searches over the threads, so the pool takes the
        // searches expected to be the longest — a position's previous search is the estimate — up to a share of the
        // estimated work that is adapted round by round until both finish together.
        std::vector<uint32_t> hostPart, devPart;
        if (b->cfg.host_threads > 1) {
            std::vector<std::pair<uint64_t, uint32_t>> est;
            est.reserve(todo.size());
            uint64_t total = 0;
            if (b->srcCost.size() != b->V) b->srcCost.assign(b->V, 0);
            const uint64_t typical = (uint64_t)std::max(1.0, b->meanCost);
            for (uint32_t k : todo) {
                // a position's previous search, else the last search from the same source view, else the running mean
                const Item &it = b->wave[k];
                const uint64_t c = it.pushes ? it.pushes : (b->srcCost[it.src] ? b->srcCost[it.src] : typical);
                est.emplace_back(c, k);
                total += c;
            }
            std::sort(est.begin(), est.end(), [](const auto &x, const auto &y) { return x.first != y.first ? x.first > y.first : x.second < y.second; });
            const double budget = b->hybridShare * (double)total;
            uint64_t acc = 0;
            for (const auto &e : est) {
                if ((double)acc < budget) { hostPart.push_back(e.second); acc += e.first; }
                else devPart.push_back(e.second);
            }
            std::sort(devPart.begin(), devPart.end());
            // the device gives up on a search that turns out more than twice as long as the longest one it was meant to
            // get (and at least 4x the typical search): the pool repeats those few
            const uint64_t longest = hostPart.size() < est.size() ? est[hostPart.size()].first : 0;  // est is sorted, longest first
            b->gpuBudget = (uint32_t)std::min<uint64_t>(0x7fffffffu, std::max<uint64_t>(2 * longest, 4 * typical) + 4096);
        } else {
            devPart = todo;
            b->gpuBudget = 0;
        }
        std::vector<uint32_t> redo;
        int32_t rc = 0;
        double tDev = 0.0, tHost = 0.0;
        if (hostPart.empty()) {
            const double t1 = nowSec();
            rc = searchOnDevice(b, devPart, redo);
            tDev = nowSec() - t1;
        } else {
            std::thread dev([&]() {
                const double t1 = nowSec();
                rc = searchOnDevice(b, devPart, redo);
                tDev = nowSec() - t1;
            });
            const double t1 = nowSec();
            searchOnHost(b, hostPart);
            tHost = nowSec() - t1;
            dev.join();
            // move the share towards the point where both sides take the same time
            if (tDev > 0.0 && tHost > 0.0) {
                const double ratio = tDev / tHost;
                const double step = ratio > 1.0 ? std::min(ratio, 1.25) : std::max(ratio, 0.8);
                b->hybridShare = std::min(0.9, std::max(0.02, b->hybridShare * step));
            }
            b->ctr.sec_search_host_part += tHost;
        }
        if (rc == 0) {
            if (!redo.empty()) searchOnHost(b, redo);
            if (b->gpuCheck) checkDeviceSearches(b);
            done = true;
        } else {
            b->searchError = rc;
            fprintf(stderr, "[pgb] device search failed with status %d\n", (int)rc);
        }
    }
    if (!done) searchOnHost(b, todo);
    if (b->srcCost.size() == b->V)
        for (uint32_t k : todo) {
            const Item &it = b->wave[k];
            if (!it.pushes) continue;
            b->srcCost[it.src] = it.pushes;
            b->meanCost = b->meanCost > 0.0 ? 0.999 * b->meanCost + 0.001 * (double)it.pushes : (double)it.pushes;
        }
    for (uint32_t k : todo) { b->ctr.astar_pops += b->wave[k].touched; b->ctr.astar_pushes += b->wave[k].pushes; }
    b->ctr.astar_runs += todo.size();
    if (b->rounds > 0) b->ctr.astar_reruns += todo.size();
    b->ctr.sec_astar += nowSec() - t0;
}

// Resolve the verdict of every position from the caches.  Returns the number of positions that need the engine.
uint32_t resolveVerdicts(pgb_builder *b)
{
    uint32_t need = 0;
    for (Item &it : b->wave) {
        it.needGpu = false;
        if (!it.mine) continue;  // remote positions are resolved by their owner (import)
        it.finalV = it.pathV = nullptr;
        if (it.staticSkip || it.dupSkip || !it.searched) continue;  // unsearched positions wait for the window to reach them
        if (it.hasHyp) {
            auto pc = b->pathCache.find(makeKey(it.pairId, it.hyp));
            if (pc == b->pathCache.end()) { it.needGpu = true; ++need; continue; }
            it.pathV = &pc->second.v;
            if (pc->second.ok) it.finalV = it.pathV;
        }
        if (!it.finalV) {
            if (!b->fbHave[it.pairId]) { it.needGpu = true; ++need; continue; }
            it.finalV = &b->fbCache[it.pairId];
        }
    }
    return need;
}

void commitPosition(pgb_builder *b, Item &it)
{
    pgb_log lg;
    memset(&lg, 0, sizeof lg);
    lg.src = it.src; lg.dst = it.dst;
    lg.pair_index = it.pairId == UINT32_MAX ? -1 : (int64_t)it.pairId;
    lg.n_corr = it.nCorr;
    b->ctr.pairs_popped++;
    if (b->graph.hasEdge(it.src, it.dst) || b->graph.hasEdge(it.dst, it.src)) {  // pose_graph_builder.h:438-443
        b->ctr.skipped++;
        b->log.push_back(lg);
        return;
    }
    lg.visible = it.visible;
    if (it.staticSkip) {  // :550-551
        b->ctr.skipped++;
        b->log.push_back(lg);
        return;
    }
    const pgi_verdict *final = it.finalV;
    lg.had_path = it.hasHyp;
    lg.touched_nodes = it.touched;
    if (it.hasHyp) { memcpy(lg.hyp, it.hyp.q, 32); memcpy(lg.hyp + 4, it.hyp.t, 24); }
    if (it.pathV) { lg.test_passed = it.pathV->test_passed; lg.test_count = it.pathV->test_count; }
    lg.branch = final->accepted ? final->branch : 0;
    lg.inlier_number = final->inlier_count;
    memcpy(lg.E, final->E, sizeof lg.E);
    if (!final->accepted) {  // :641-642
        b->ctr.rejected++;
        b->log.push_back(lg);
        return;
    }
    const Edge e = edgeOf(it, outcomeOf(final));
    const uint32_t ei = (uint32_t)b->graph.edges.size();
    b->graph.edges.push_back(e);
    b->graph.lookup[edgeKey(e.src, e.dst)] = ei;
    b->graph.byVertex[e.src].push_back(Adj{e.dst, ei, e.score});  // pose_graph.h:219-220
    b->graph.byVertex[e.dst].push_back(Adj{e.src, ei, e.score});
    if (b->gpuApply) {
        b->commitEntries.push_back(pgi_adj_entry{e.src, (uint32_t)b->graph.byVertex[e.src].size() - 1, e.dst, 0u, e.score});
        b->commitEntries.push_back(pgi_adj_entry{e.dst, (uint32_t)b->graph.byVertex[e.dst].size() - 1, e.src, 0u, e.score});
    }
    const double tv = nowSec();
    b->vis.addLink(e.src, e.dst);  // :692
    b->ctr.sec_visibility += nowSec() - tv;
    lg.committed = 1;
    memcpy(lg.q, final->q, 32);
    memcpy(lg.t, final->t, 24);
    lg.score = e.score;
    b->log.push_back(lg);
    b->ctr.committed++;
    if (final->branch == 1) b->ctr.path_accepted++; else b->ctr.fallback_accepted++;
}

// Iterate the open wave towards its fixed point.  Returns the number of positions committed (0 while the wave still
// waits for engine verdicts or for the record exchange between ranks); b->status says what it waits for.
uint32_t advanceWave(pgb_builder *b)
{
    const uint32_t n = (uint32_t)b->wave.size();
    for (;;) {
        if (b->phase == 0) {
            uint32_t firstStale = n;
            for (uint32_t k = 0; k < n; k++)
                if (b->wave[k].mine && !b->wave[k].searched) { firstStale = k; break; }
            // optional re-search window behind the first stale position (0 = unlimited: measured best on cfg2, the
            // re-search cascade is intrinsic rather than wasted look-ahead)
            const uint32_t window = b->cfg.reserved > 0 ? (uint32_t)b->cfg.reserved : n;
            const uint32_t limit = firstStale + window < n ? firstStale + window : n;
            searchStale(b, limit);
            if (resolveVerdicts(b) > 0) { b->status = PGB_WAVE_NEED_GPU; return 0; }  // engine round trip; wave stays open
            if (b->world > 1) { b->phase = 1; b->status = PGB_WAVE_NEED_EXCHANGE; return 0; }
            b->phase = 2;
        }
        if (b->phase == 1) { b->status = PGB_WAVE_NEED_EXCHANGE; return 0; }  // waiting for pgb_import_records
        // ---- phase 2: actual outcomes vs. the predictions the overlay was built from (identical on every rank) ----
        std::fill(b->minChangedPos.begin(), b->minChangedPos.end(), UINT32_MAX);
        uint32_t firstChanged = UINT32_MAX;
        bool allKnown = true;
        b->changes.clear();
        for (uint32_t k = 0; k < n; k++) {
            Item &it = b->wave[k];
            if (it.staticSkip || it.dupSkip) continue;
            if (it.mine ? !it.searched : !it.remoteKnown) { allKnown = false; continue; }
            const Outcome act = outcomeOf(it.finalV);
            if (!act.sameEdge(it.pred)) {
                const bool hadEdge = it.pred.known && it.pred.accepted;
                b->changes.push_back(Change{k, it.src, it.dst, hadEdge != act.accepted,
                                            hadEdge ? (double)it.pred.inliers / (double)it.nCorr : 0.0,
                                            act.accepted ? (double)act.inliers / (double)it.nCorr : 0.0});
                it.pred = act;
                if (firstChanged == UINT32_MAX) firstChanged = k;
                b->minChangedPos[it.src] = std::min(b->minChangedPos[it.src], k);
                b->minChangedPos[it.dst] = std::min(b->minChangedPos[it.dst], k);
            }
        }
        b->phase = 0;
        if (firstChanged == UINT32_MAX) {
            if (allKnown) break;  // fixed point: every search saw exactly the sequential graph
            ++b->rounds;
            continue;             // nothing changed among the known positions: keep searching
        }
        ++b->rounds;
        // Which search results does the round invalidate?  A search reads the edge lists of the vertices it expanded
        // (graph_traversal.h:817) and nothing else, so position m can only be affected by a changed position k < m whose
        // edge touches one of them.  If the edge merely changed its score (or pose), the finer rule of the cost floor
        // applies (aStar): the child that expansion pushed through the edge has a combined cost computed from the node's
        // (c0, c1) and the score; if it is below the smallest cost the search ever popped (tauMin) under the predicted AND
        // under the actual score, it was and remains an entry that never leaves the queue and whose value decides
        // nothing — the search is bit for bit the same.  An edge that appears or disappears shifts the slots of the
        // children behind it and always invalidates.
        if (!b->changes.empty()) {
            for (std::vector<uint32_t> &l : b->changesOf) l.clear();
            if (b->changesOf.size() != b->V) b->changesOf.assign(b->V, {});
            for (uint32_t ci = 0; ci < b->changes.size(); ci++) {
                b->changesOf[b->changes[ci].u].push_back(ci);
                b->changesOf[b->changes[ci].w].push_back(ci);
            }
            const double wgt = b->cfg.traversal_heuristics_weight, omw = 1.0 - wgt;
            for (uint32_t m = firstChanged + 1; m < n; m++) {
                Item &it = b->wave[m];
                if (!it.mine || !it.searched) continue;
                const bool fine = it.expCost.size() == 2 * it.expanded.size();
                const double *simTo = b->sim.data() + (size_t)it.dst * b->V;
                for (size_t x = 0; x < it.expanded.size() && it.searched; x++) {
                    const uint32_t v = it.expanded[x];
                    if (b->minChangedPos[v] >= m) continue;
                    if (!fine) { it.searched = false; break; }
                    const double c0 = it.expCost[2 * x], c1 = it.expCost[2 * x + 1];
                    for (uint32_t ci : b->changesOf[v]) {
                        const Change &c = b->changes[ci];
                        if (c.k >= m) break;  // (lists are in position order)
                        if (c.existence) { it.searched = false; break; }
                        const uint32_t other = c.u == v ? c.w : c.u;
                        if (!scoreChangeIsInert(c0, c1, simTo[other], c.sOld, c.sNew, wgt, omw, it.tauMin)) { it.searched = false; break; }
                    }
                }
                if (it.searched) ++b->ctr.stale_spared;  // (counts positions that were examined and kept)
            }
        }
        rebuildOverlay(b, firstChanged);
    }
    const double t0 = nowSec();
    PgiNvtxRange nvtxCommit("pgb:commit wave in order");
    b->commitEntries.clear();
    for (Item &it : b->wave) commitPosition(b, it);
    b->wave.clear();
    b->waveOpen = false;
    b->status = PGB_WAVE_DONE;
    b->overlay.clear();
    if (b->gpuApply) {  // mirror the committed edges of the wave to the device graph
        b->gpuCommitted.resize(b->V);
        for (uint32_t v = 0; v < b->V; v++) b->gpuCommitted[v] = (uint32_t)b->graph.byVertex[v].size();
        const int32_t rc = b->gpuApply(b->gpuEngine, (uint32_t)b->commitEntries.size(), b->commitEntries.data(),
                                       b->gpuCommitted.data(), b->gpuCommitted.data());
        if (rc != 0 && b->searchError == 0) b->searchError = rc;
        b->ovDirty = false;  // device graph == committed graph, no overlay
    }
    b->ctr.sec_commit += nowSec() - t0;
    return n;
}

}  // namespace

extern "C" {

int32_t pgb_create(const pgb_config *cfg, uint64_t n_views, const double *sim, uint64_t n_pairs,
                   const uint32_t *pair_views, const uint64_t *m_offset, pgb_builder **out)
{
    if (!cfg || !sim || !out || (n_pairs && (!pair_views || !m_offset)) || n_views > 0x7fffffffULL) return -1;
    pgb_builder *b = new pgb_builder();
    b->cfg = *cfg;
    if (b->cfg.host_threads <= 0) b->cfg.host_threads = (int32_t)std::max(1u, std::thread::hardware_concurrency());
    b->V = (uint32_t)n_views;
    b->sim.resize(n_views * n_views);  // stored TRANSPOSED and already clamped to [0,1] (std::clamp at graph_traversal.h:594
                                       // is the only consumer): sim[to * V + next] = clamp(similarity(next, to), 0, 1)
    for (uint64_t r = 0; r < n_views; r++)
        for (uint64_t c = 0; c < n_views; c++) {
            const double v = sim[r * n_views + c];
            b->sim[c * n_views + r] = v < 0.0 ? 0.0 : (1.0 < v ? 1.0 : v);
        }
    b->P = n_pairs;
    b->pairViews.assign(pair_views, pair_views + 2 * n_pairs);
    b->mOffset.assign(m_offset, m_offset + n_pairs + 1);
    for (uint64_t p = 0; p < n_pairs; p++) b->pairIndex[edgeKey(pair_views[2 * p], pair_views[2 * p + 1])] = (uint32_t)p;
    // SimilarityTable::loadFromFile queue construction (imagesimilarity_graph.h:141-163): the table is pre-filled
    // with 1.0f (:58-65); (i,j) is queued while row i is filled iff i != j, thr <= s_ij and s_ji != s_ij at that time.
    {
        const size_t V = n_views;
        std::vector<double> table(V * V, (double)1.0f);
        std::priority_queue<std::tuple<double, size_t, size_t>> q;
        for (size_t i = 0; i < V; i++)
            for (size_t j = 0; j < V; j++) {
                table[i * V + j] = sim[i * V + j];
                if (i != j && cfg->similarity_threshold <= table[i * V + j] && table[j * V + i] != table[i * V + j])
                    q.emplace(std::make_tuple(table[i * V + j], i, j));
            }
        b->order.reserve(q.size());
        while (!q.empty()) {  // std::less on the tuple: larger similarity, then larger i, then larger j first (App. A.1)
            b->order.emplace_back((uint32_t)std::get<1>(q.top()), (uint32_t)std::get<2>(q.top()));
            q.pop();
        }
    }
    b->graph.byVertex.resize(n_views);
    b->overlay.byVertex.resize(n_views);
    b->vis.init((uint32_t)n_views);
    b->minChangedPos.assign(n_views, UINT32_MAX);
    b->srcFloor.assign(n_views, -1.0);
    b->dstFloor.assign(n_views, -1.0);
    b->fbCache.resize(n_pairs);
    b->fbHave.assign(n_pairs, 0);
    memset(&b->ctr, 0, sizeof b->ctr);
    b->scratch.resize(b->cfg.host_threads);
    b->pool.start(b->cfg.host_threads);
    *out = b;
    return 0;
}

void pgb_destroy(pgb_builder *b) { delete b; }

uint64_t pgb_remaining(pgb_builder *b) { return b ? b->pending.size() + (b->order.size() - b->nextInOrder) + b->wave.size() : 0; }

int32_t pgb_set_fallback_verdicts(pgb_builder *b, const pgi_verdict *verdicts, uint64_t n_pairs)
{
    if (!b || !verdicts || n_pairs != b->P) return -1;
    for (uint64_t p = 0; p < n_pairs; p++) {
        b->fbCache[p] = verdicts[p];
        b->fbHave[p] = 1;
    }
    return 0;
}

int32_t pgb_set_fallback_verdicts_some(pgb_builder *b, const uint32_t *pair_ids, const pgi_verdict *verdicts, uint64_t n)
{
    if (!b || !verdicts || !pair_ids) return -1;
    std::lock_guard<std::mutex> lk(b->driveMu);
    for (uint64_t i = 0; i < n; i++) {
        if (pair_ids[i] >= b->P) return -1;
        b->fbCache[pair_ids[i]] = verdicts[i];
        b->fbHave[pair_ids[i]] = 1;
    }
    return 0;
}

uint64_t pgb_queue_size(pgb_builder *b) { return b ? b->order.size() : 0; }
void pgb_queue_pairs(pgb_builder *b, uint32_t *out)
{
    for (size_t i = 0; i < b->order.size(); i++) {
        auto pi = b->pairIndex.find(edgeKey(b->order[i].first, b->order[i].second));
        out[i] = pi == b->pairIndex.end() ? UINT32_MAX : pi->second;
    }
}

static uint32_t emitItems(pgb_builder *b, pgb_item *items)
{
    const uint32_t n = (uint32_t)b->wave.size();
    for (uint32_t i = 0; i < n; i++) {
        const Item &it = b->wave[i];
        pgb_item &o = items[i];
        o.pair_id = it.pairId;
        o.src = it.src; o.dst = it.dst;
        o.has_hyp = it.hasHyp; o.need_gpu = it.needGpu; o.visible = it.visible; o.pad = 0;
        memcpy(o.hyp, it.hyp.q, 32);
        memcpy(o.hyp + 4, it.hyp.t, 24);
    }
    return n;
}

uint32_t pgb_next_wave(pgb_builder *b, uint32_t max_items, pgb_item *items)
{
    if (!b || !items) return 0;
    if (b->waveOpen) return emitItems(b, items);  // still waiting for verdicts of the open wave
    // 1. gather positions in queue order: re-queued ones first, then fresh pops
    while (b->wave.size() < max_items) {
        Item it;
        if (!b->pending.empty()) {
            it = std::move(b->pending.front());
            b->pending.pop_front();
        } else if (b->nextInOrder < b->order.size()) {
            it.src = b->order[b->nextInOrder].first;
            it.dst = b->order[b->nextInOrder].second;
            ++b->nextInOrder;
            auto pi = b->pairIndex.find(edgeKey(it.src, it.dst));
            if (pi != b->pairIndex.end()) {
                it.pairId = pi->second;
                it.nCorr = (uint32_t)(b->mOffset[it.pairId + 1] - b->mOffset[it.pairId]);
            }
            it.staticSkip = it.pairId == UINT32_MAX || it.nCorr < b->cfg.minimum_point_number;
        } else
            break;
        it.searched = false;
        it.remoteKnown = false;
        it.mine = true;
        if (b->world > 1 && !it.staticSkip) {
            it.mine = (int)(it.pairId % (uint32_t)b->world) == b->rank;  // interleaved ownership balances every wave
        }
        // prediction: the pair's hypothesis-independent fallback verdict, if already known
        const bool fbKnown = !it.staticSkip && b->fbHave[it.pairId];
        it.pred = fbKnown ? outcomeOf(&b->fbCache[it.pairId]) : Outcome();
        b->wave.push_back(std::move(it));
        if (!b->wave.back().staticSkip && !fbKnown) break;  // nothing can be predicted behind an unknown outcome
    }
    if (b->wave.empty()) return 0;
    b->waveOpen = true;
    b->rounds = 0;
    b->phase = 0;
    b->ctr.waves++;
    b->ctr.items_speculated += b->wave.size();
    rebuildOverlay(b);
    advanceWave(b);  // searches, resolves from the caches and stops at the first engine round trip / exchange / commit
    return emitItems(b, items);
}

uint32_t pgb_commit_wave(pgb_builder *b, const pgi_verdict *verdicts, uint32_t n_verdicts)
{
    if (!b || !b->waveOpen) return 0;
    // absorb the engine's verdicts into the caches (pure functions of (pair, hypothesis) / of the pair)
    uint32_t vi = 0;
    for (Item &it : b->wave) {
        if (!it.needGpu) continue;
        if (vi >= n_verdicts || !verdicts) break;
        const pgi_verdict &v = verdicts[vi++];
        if (it.hasHyp) {
            PathVerdict pv;
            pv.ok = v.branch == 1;
            pv.v = v;
            b->pathCache[makeKey(it.pairId, it.hyp)] = pv;
        }
        if (v.status & 1u) {  // the fallback ran: its verdict is a function of the pair alone
            b->fbCache[it.pairId] = v;
            b->fbHave[it.pairId] = 1;
        }
    }
    return advanceWave(b);
}

int32_t pgb_set_partition(pgb_builder *b, int32_t rank, int32_t world)
{
    if (!b || world < 1 || rank < 0 || rank >= world || b->waveOpen) return -1;
    if (world > 1 && b->cfg.lazy_fallback) return -1;  // records carry path verdicts only: fallback verdicts must be prefetched
    b->rank = rank;
    b->world = world;
    return 0;
}

int32_t pgb_wave_status(pgb_builder *b) { return (b && b->waveOpen) ? b->status : PGB_WAVE_DONE; }

int32_t pgb_set_search_backend(pgb_builder *b, pgb_graph_apply_fn apply, pgb_graph_search_fn search, void *engine,
                               uint32_t min_batch)
{
    if (!b || b->waveOpen || ((apply == nullptr) != (search == nullptr))) return -1;
    b->gpuApply = apply;
    b->gpuSearch = search;
    b->gpuEngine = engine;
    b->gpuMinBatch = min_batch;
    b->ovDirty = true;
    if (const char *e = getenv("PGB_SEARCH_CHECK")) b->gpuCheck = atoi(e) != 0;
    if (!apply) return 0;
    // bring the device graph up to the committed graph (normally empty at this point)
    std::vector<pgi_adj_entry> entries;
    b->gpuCommitted.resize(b->V);
    for (uint32_t v = 0; v < b->V; v++) {
        const std::vector<Adj> &l = b->graph.byVertex[v];
        b->gpuCommitted[v] = (uint32_t)l.size();
        for (uint32_t j = 0; j < l.size(); j++) entries.push_back(pgi_adj_entry{v, j, l[j].next, 0u, l[j].score});
    }
    return apply(engine, (uint32_t)entries.size(), entries.data(), b->gpuCommitted.data(), b->gpuCommitted.data());
}

void pgb_copy_sim_table(pgb_builder *b, double *out) { memcpy(out, b->sim.data(), b->sim.size() * sizeof(double)); }

int32_t pgb_run_wave(pgb_builder *b, uint32_t wave_size, pgb_submit_fn submit, pgb_wait_fn wait, void *engine, uint32_t flags,
                     pgb_drive_stats *stats)
{
    PgiNvtxRange nvtxRange("pgb:run_wave");
    if (!b || !submit || !wait || wave_size == 0) return -1;
    double t0 = nowSec();
    uint32_t n;
    int32_t status;
    {
        std::lock_guard<std::mutex> lk(b->driveMu);
        b->driveItems.resize(wave_size);
        n = pgb_next_wave(b, wave_size, b->driveItems.data());
        status = pgb_wave_status(b);
        if (b->searchError) return b->searchError;
    }
    double t1 = nowSec();
    if (stats) stats->host_s += t1 - t0;
    while (status == PGB_WAVE_NEED_GPU) {
        // the (pair, hypothesis) tuples of this round, in wave order
        b->driveIds.clear();
        b->driveHyp.clear();
        b->driveHoff.assign(1, 0u);
        for (uint32_t i = 0; i < n; i++) {
            const pgb_item &it = b->driveItems[i];
            if (!it.need_gpu) continue;
            b->driveIds.push_back(it.pair_id);
            if (it.has_hyp) b->driveHyp.insert(b->driveHyp.end(), it.hyp, it.hyp + 7);
            b->driveHoff.push_back((uint32_t)(b->driveHyp.size() / 7));
        }
        const uint32_t m = (uint32_t)b->driveIds.size();
        b->driveVerdicts.resize(std::max<uint32_t>(m, 1));
        int32_t rc = submit(engine, m, b->driveIds.data(), b->driveHoff.data(), b->driveHyp.empty() ? nullptr : b->driveHyp.data(), flags);
        if (rc < 0) return rc;
        rc = wait(engine, b->driveVerdicts.data(), nullptr);
        if (rc < 0) return rc;
        for (uint32_t i = 0; i < m; i++) b->driveVerdicts[i].pair_id = b->driveIds[i];
        t0 = nowSec();
        if (stats) { stats->engine_s += t0 - t1; stats->rounds += 1; stats->items += m; }
        {
            std::lock_guard<std::mutex> lk(b->driveMu);
            pgb_commit_wave(b, b->driveVerdicts.data(), m);
            if (b->searchError) return b->searchError;
            status = pgb_wave_status(b);
            if (status != PGB_WAVE_DONE) n = pgb_next_wave(b, wave_size, b->driveItems.data());
        }
        t1 = nowSec();
        if (stats) stats->host_s += t1 - t0;
    }
    return status;
}
uint32_t pgb_wave_size(pgb_builder *b) { return b ? (uint32_t)b->wave.size() : 0; }

int32_t pgb_run_hashing(pgb_builder *b, const uint32_t *matches, const pgb_hashing_config *hc, pgb_submit_fn submit,
                        pgb_wait_fn wait, pgb_register_extra_fn register_extra, pgb_guided_fn guided, void *engine,
                        pgb_hashing_stats *stats)
{
    PgiNvtxRange nvtxRange("pgb:run_hashing");
    if (!b || !hc || !submit || !wait || !register_extra || !guided || (b->mOffset.back() && !matches)) return -1;
    if (b->waveOpen || !b->pending.empty() || b->log.size() != b->matchSource.size()) return -1;
    pgb_hashing_stats local;
    memset(&local, 0, sizeof local);
    pgb_hashing_stats &st = stats ? *stats : local;
    std::unique_ptr<pgb_tracklets, void (*)(pgb_tracklets *)> tracklets(pgb_tracklets_create(b->V), pgb_tracklets_destroy);
    const uint64_t maxTracks = hc->maximum_tracklet_number, maxGuided = hc->maximum_point_number;
    std::vector<uint64_t> qS(maxTracks + 1), qD(maxTracks + 1), addS, addD;
    std::vector<uint32_t> quick, gm((size_t)2 * maxGuided);
    std::vector<double> gv(maxGuided);
    std::vector<uint8_t> mask, ones;
    AStarScratch &S = b->scratch[0];
    const uint32_t flagsBase = PGI_WAVE_PATH | PGI_WAVE_FALLBACK | PGI_WAVE_MASKS;
    while (b->nextInOrder < b->order.size()) {
        Item it;
        it.src = b->order[b->nextInOrder].first;
        it.dst = b->order[b->nextInOrder].second;
        ++b->nextInOrder;
        ++st.positions;
        uint8_t source = PGB_MATCH_SKIPPED;
        uint32_t guidedAdded = 0;
        const auto finish = [&]() {
            commitPosition(b, it);
            b->matchSource.push_back(source);
            b->guidedRows.push_back(guidedAdded);
        };
        if (b->graph.hasEdge(it.src, it.dst) || b->graph.hasEdge(it.dst, it.src)) {  // pose_graph_builder.h:438-443
            finish();
            continue;
        }
        it.visible = b->vis.hasLink(it.src, it.dst);  // :456-457
        auto pi = b->pairIndex.find(edgeKey(it.src, it.dst));
        if (pi != b->pairIndex.end()) it.pairId = pi->second;
        // quick matching from the tracks the two views share (:492-520)
        double t0 = nowSec();
        const int64_t nq = pgb_tracklets_get_correspondences(tracklets.get(), it.src, it.dst, maxTracks, qS.data(), qD.data(), qS.size());
        st.sec_tracklets += nowSec() - t0;
        if (nq < 0) return -1;
        const bool isQuick = (uint64_t)nq >= b->cfg.minimum_point_number;
        if (isQuick)
            it.nCorr = (uint32_t)nq;
        else  // matchFeatures' list (:522-547)
            it.nCorr = it.pairId == UINT32_MAX ? 0u : (uint32_t)(b->mOffset[it.pairId + 1] - b->mOffset[it.pairId]);
        if (it.nCorr < b->cfg.minimum_point_number) {  // :550-551
            it.staticSkip = true;
            finish();
            continue;
        }
        source = isQuick ? PGB_MATCH_QUICK : PGB_MATCH_FULL;
        ++(isQuick ? st.quick_matched : st.full_matched);
        uint32_t flags = flagsBase, pid = it.pairId;
        t0 = nowSec();
        if (isQuick) {
            quick.resize((size_t)2 * nq);
            for (int64_t i = 0; i < nq; i++) { quick[2 * i] = (uint32_t)qS[i]; quick[2 * i + 1] = (uint32_t)qD[i]; }
            const uint32_t pv[2] = {it.src, it.dst};
            const uint64_t off[2] = {0, (uint64_t)nq};
            const int32_t rc = register_extra(engine, 1, pv, off, quick.data());
            if (rc < 0) return rc;
            flags |= PGI_WAVE_EXTRA;
            pid = 0;
        }
        st.sec_engine += nowSec() - t0;
        // A* on the committed graph (:569-603)
        if (b->cfg.use_path_finding && it.visible) {
            t0 = nowSec();
            AStarOut o;
            GraphView gv0{&b->graph, nullptr, 0};
            aStar(gv0, b->sim.data(), b->V, it.src, it.dst, (size_t)b->cfg.maximum_search_depth, b->cfg.traversal_heuristics_weight, S, o);
            it.hasHyp = o.found;
            it.hyp = o.pose;
            it.touched = o.touched;
            const double dt = nowSec() - t0;
            st.sec_astar += dt;
            b->ctr.sec_astar += dt;
            b->ctr.astar_runs++;
            b->ctr.astar_pops += o.touched;
            b->ctr.astar_pushes += o.pushes;
        }
        // estimatePose on the chosen matches: a wave of one, with its inlier mask
        t0 = nowSec();
        double hyp[7];
        memcpy(hyp, it.hyp.q, 32);
        memcpy(hyp + 4, it.hyp.t, 24);
        const uint32_t hoff[2] = {0, it.hasHyp ? 1u : 0u};
        pgi_verdict v;
        mask.assign(it.nCorr, 0);
        int32_t rc = submit(engine, 1, &pid, hoff, it.hasHyp ? hyp : nullptr, flags);
        if (rc < 0) return rc;
        rc = wait(engine, &v, mask.data());
        if (rc < 0) return rc;
        st.sec_engine += nowSec() - t0;
        b->ctr.waves++;
        b->ctr.items_speculated++;
        v.pair_id = it.pairId;
        it.finalV = &v;
        it.pathV = it.hasHyp ? &v : nullptr;
        commitPosition(b, it);
        if (v.accepted) {
            uint64_t n = 0;
            const uint8_t *m = nullptr;
            if (isQuick) {  // guidedMatching with the committed pose (:663-676, :717-783)
                t0 = nowSec();
                double pose[7];
                memcpy(pose, v.q, 32);
                memcpy(pose + 4, v.t, 24);
                uint32_t gn = 0;
                rc = guided(engine, it.src, it.dst, pose, hc->bin_number, (uint32_t)maxGuided, gm.data(), gv.data(), &gn);
                if (rc < 0) return rc;
                st.sec_guided += nowSec() - t0;
                st.guided_calls++;
                st.guided_rows += gn;
                guidedAdded = gn;
                n = std::min<uint64_t>(gn, maxGuided);
                addS.resize(n);
                addD.resize(n);
                for (uint64_t i = 0; i < n; i++) { addS[i] = gm[2 * i]; addD[i] = gm[2 * i + 1]; }
                ones.assign(n, 1);
                m = ones.data();
            } else {  // the matchFeatures list under estimatePose's inlier mask (:697-703)
                n = it.nCorr;
                const uint32_t *pm = matches + 2 * b->mOffset[it.pairId];
                addS.resize(n);
                addD.resize(n);
                for (uint64_t i = 0; i < n; i++) { addS[i] = pm[2 * i]; addD[i] = pm[2 * i + 1]; }
                m = mask.data();
            }
            t0 = nowSec();
            if (pgb_tracklets_add(tracklets.get(), it.src, it.dst, n, addS.data(), addD.data(), m) != 0) return -1;
            st.sec_tracklets += nowSec() - t0;
            st.tracklet_adds++;
        }
        b->matchSource.push_back(source);
        b->guidedRows.push_back(guidedAdded);
    }
    return 0;
}

uint64_t pgb_copy_match_sources(pgb_builder *b, uint8_t *source_out, uint32_t *guided_rows_out)
{
    if (!b) return 0;
    const size_t n = b->matchSource.size();
    if (source_out && n) memcpy(source_out, b->matchSource.data(), n);
    if (guided_rows_out && n) memcpy(guided_rows_out, b->guidedRows.data(), n * 4);
    return n;
}

// One record per wave position; a rank fills the positions it owns and leaves the others zero, so a byte-wise SUM
// all-reduce merges the ranks' buffers.
void pgb_export_records(pgb_builder *b, pgb_record *out)
{
    const uint32_t n = (uint32_t)b->wave.size();
    memset(out, 0, (size_t)n * sizeof(pgb_record));
    for (uint32_t k = 0; k < n; k++) {
        const Item &it = b->wave[k];
        if (!it.mine || it.staticSkip || it.dupSkip) continue;
        pgb_record &r = out[k];
        r.valid = (it.searched && it.finalV) ? 1 : 0;
        r.has_hyp = it.hasHyp;
        r.has_path_verdict = it.pathV ? 1 : 0;
        r.final_is_path = (it.pathV && it.finalV == it.pathV) ? 1 : 0;
        r.touched = it.touched;
        if (it.pathV) r.v = *it.pathV;
        if (it.hasHyp) { memcpy(r.hyp, it.hyp.q, 32); memcpy(r.hyp + 4, it.hyp.t, 24); }
    }
}

uint32_t pgb_import_records(pgb_builder *b, const pgb_record *in)
{
    if (!b || !b->waveOpen || b->phase != 1) return 0;
    const uint32_t n = (uint32_t)b->wave.size();
    for (uint32_t k = 0; k < n; k++) {
        Item &it = b->wave[k];
        if (it.mine || it.staticSkip || it.dupSkip) continue;
        const pgb_record &r = in[k];
        it.remoteKnown = r.valid != 0;
        it.hasHyp = r.has_hyp != 0;
        memcpy(it.hyp.q, r.hyp, 32);
        memcpy(it.hyp.t, r.hyp + 4, 24);
        it.touched = r.touched;
        it.pathV = it.finalV = nullptr;
        if (r.has_path_verdict) { it.remoteV = r.v; it.pathV = &it.remoteV; }
        if (r.final_is_path)
            it.finalV = &it.remoteV;
        else if (b->fbHave[it.pairId])
            it.finalV = &b->fbCache[it.pairId];
        else
            it.remoteKnown = false;  // (cannot happen: with several ranks the fallback verdicts are prefetched)
    }
    b->phase = 2;
    return advanceWave(b);
}

uint64_t pgb_edge_count(pgb_builder *b) { return b ? b->graph.edges.size() : 0; }
void pgb_copy_edges(pgb_builder *b, pgb_edge *out)
{
    for (size_t i = 0; i < b->graph.edges.size(); i++) {
        const Edge &e = b->graph.edges[i];
        pgb_edge &o = out[i];
        memset(&o, 0, sizeof o);
        o.src = e.src; o.dst = e.dst;
        memcpy(o.q, e.T.q, 32);
        memcpy(o.t, e.T.t, 24);
        o.score = e.score; o.inlier_number = e.inlierNumber; o.n_corr = e.nCorr; o.branch = e.branch;
    }
}
uint64_t pgb_log_count(pgb_builder *b) { return b ? b->log.size() : 0; }
void pgb_copy_log(pgb_builder *b, pgb_log *out) { memcpy(out, b->log.data(), b->log.size() * sizeof(pgb_log)); }
void pgb_get_counters(pgb_builder *b, pgb_counters *out)
{
    *out = b->ctr;
    out->floor_retries = 0;
    for (const AStarScratch &s : b->scratch) out->floor_retries += s.floorRetries;
}

int32_t pgb_astar(pgb_builder *b, uint32_t src, uint32_t dst, double *hyp_q_t, uint32_t *touched_nodes)
{
    if (!b || src >= b->V || dst >= b->V) return -1;
    AStarOut o;
    GraphView gv{&b->graph, nullptr, 0};
    aStar(gv, b->sim.data(), b->V, src, dst, (size_t)b->cfg.maximum_search_depth, b->cfg.traversal_heuristics_weight,
          b->scratch[0], o);
    if (hyp_q_t) { memcpy(hyp_q_t, o.pose.q, 32); memcpy(hyp_q_t + 4, o.pose.t, 24); }
    if (touched_nodes) *touched_nodes = o.touched;
    return o.found ? 1 : 0;
}

}  // extern "C"
