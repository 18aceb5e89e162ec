// pgi_api.cu — C-ABI (include/pgi.h) over the sm_100a kernels of pgi_kernels.cuh.
// Host-side plumbing only: device memory, one stream per context, pinned staging, CUDA-event timing.
// No CPU compute path exists here: without a usable device every entry point returns PGI_ERR_CUDA.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/pgi.h"
#include "pgi_kernels.cuh"
#include "pgi_astar.cuh"
#include "pgi_matcher.cuh"
#include "pgi_guided_batch.cuh"
#include "pgi_match_scene.cuh"
#include "pgi_nvtx.h"

using namespace pgi;

namespace {

// A device (or pinned host) allocation of `capacity()` elements of T, freed with its owner. Move-only.
template <typename T, bool Pinned>
class CudaBuf {
public:
    CudaBuf() = default;
    CudaBuf(CudaBuf &&o) noexcept : p_(std::exchange(o.p_, nullptr)), cap_(std::exchange(o.cap_, 0)) {}
    CudaBuf &operator=(CudaBuf o) noexcept  // the old allocation leaves with `o`
    {
        std::swap(p_, o.p_);
        std::swap(cap_, o.cap_);
        return *this;
    }
    ~CudaBuf() { release(); }

    T *data() const { return p_; }
    size_t capacity() const { return cap_; }

    // Room for n elements (at least one). The old allocation is freed before the new one is made, so peak memory does
    // not rise, and its contents are lost. A failed grow leaves the buffer empty.
    cudaError_t grow(size_t n)
    {
        if (p_ && n <= cap_) return cudaSuccess;
        cudaError_t e = release();
        if (e == cudaSuccess) {
            const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
            e = Pinned ? cudaMallocHost((void **)&p_, bytes) : cudaMalloc((void **)&p_, bytes);
        }
        if (e != cudaSuccess) {
            p_ = nullptr;
            cudaGetLastError();  // a failed allocation must not be reported again by a later launch check
            return e;
        }
        cap_ = n;
        return cudaSuccess;
    }

private:
    cudaError_t release()
    {
        cudaError_t e = cudaSuccess;
        if (p_) e = Pinned ? cudaFreeHost(p_) : cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
        return e;
    }

    T *p_ = nullptr;
    size_t cap_ = 0;
};

template <typename T>
using DevBuf = CudaBuf<T, false>;
template <typename T>
using PinnedBuf = CudaBuf<T, true>;

// A stream or event, destroyed with its owner; converts to the runtime handle.
template <typename H, cudaError_t (*Destroy)(H)>
struct Owned {
    H h = nullptr;
    Owned() = default;
    Owned(const Owned &) = delete;
    Owned &operator=(const Owned &) = delete;
    ~Owned() { if (h) Destroy(h); }
    operator H() const { return h; }
};
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

// The pairs a context verifies: normalised correspondences (4 doubles per row), offsets, thresholds, sampler tables.
struct Registration {
    DevBuf<double> corr;
    DevBuf<uint64_t> offset;
    DevBuf<double> thr;
    DevBuf<uint32_t> pairTable, sampler;
    DevBuf<uint16_t> itersTab;
    DevBuf<uint64_t> itersOff;
    uint64_t nPairs = 0, nRows = 0;
    uint32_t maxN = 0;
    std::vector<uint64_t> h_offset;
};

// Device arrays with one entry per wave slot, re-created together when the slot count or the bit stride grows.
struct DevSlots {
    uint32_t cap = 0;  // slots; 0 until every array is allocated
    DevBuf<uint32_t> pairId, hypOffset, bits;
    DevBuf<SlotState> state;
    DevBuf<uint64_t> maskOffset;
    DevBuf<pgi_verdict> verdicts;
    DevBuf<uint32_t> k3Scratch;  // K3 vote totals + arrival ticket (zero between launches)
};

// Pinned staging of the per-slot wave inputs and verdicts.
struct HostSlots {
    uint32_t cap = 0;
    PinnedBuf<uint32_t> pairId, hypOffset;
    PinnedBuf<uint64_t> maskOffset;
    PinnedBuf<pgi_verdict> verdicts;
};

// Scratch of the fallback kernels (K4, K5), sized for DevSlots::cap; created by the first fallback wave.
struct FallbackScratch {
    DevBuf<double> sols;
    DevBuf<uint8_t> counts;
    DevBuf<float4> solsF;
    DevBuf<uint32_t> dkList, dkCtl;  // work list of K4b (K4a -> K4b -> K4c)
};

// What K9 (matchPairs) reads and writes: descriptors, keypoint offsets and pair views of the views it matches, its
// per-chunk scratch, and the match list with the ratios beside it.
struct MatchStaging {
    DevBuf<uint64_t> kpOff;
    DevBuf<uint2> pv, m;
    DevBuf<float> desc, ratio;
    DevBuf<unsigned char> k9Scratch;

    // The match list is the one allocation that grows while it is filled: to max(need, 2 x capacity, 1024) rows,
    // with its first `keep` rows copied over.
    cudaError_t growMatches(uint64_t need, uint64_t keep, cudaStream_t s)
    {
        if (need <= m.capacity() && need <= ratio.capacity() && m.data() && ratio.data()) return cudaSuccess;
        const size_t cap = std::max<size_t>({need, 2 * std::min(m.capacity(), ratio.capacity()), 1024});
        DevBuf<uint2> m2;
        DevBuf<float> ratio2;
        cudaError_t e;
        if ((e = m2.grow(cap)) != cudaSuccess || (e = ratio2.grow(cap)) != cudaSuccess) return e;
        if (keep && ((e = cudaMemcpyAsync(m2.data(), m.data(), keep * sizeof(uint2), cudaMemcpyDeviceToDevice, s)) != cudaSuccess ||
                     (e = cudaMemcpyAsync(ratio2.data(), ratio.data(), keep * sizeof(float), cudaMemcpyDeviceToDevice, s)) != cudaSuccess ||
                     (e = cudaStreamSynchronize(s)) != cudaSuccess))
            return e;
        m = std::move(m2);
        ratio = std::move(ratio2);
        return cudaSuccess;
    }
};

// The compact inputs of the last scene registration. Kept between registrations: cudaMalloc / cudaFree of GB-sized
// buffers costs up to hundreds of milliseconds and synchronises the device.  The descriptors stay resident for K9 and K10.
struct SceneStaging : MatchStaging {
    DevBuf<double> focal, size;
    DevBuf<float2> kp;
    uint64_t rows = 0;
    bool matches = false;  // m / ratio hold the matches of the last descriptor registration
    // what pgi_register_extra_pairs and pgi_guided_match_views read on the host: the last registration's views
    bool staged = false;   // a scene registration completed its upload
    bool hasDesc = false;  // desc holds dim floats per keypoint of this scene
    uint32_t dim = 0;
    double thrPx = 0.0;
    std::vector<uint64_t> hKpOff;
    std::vector<double> hFocal, hSize;
};

// K6: device mirror of the pose graph and the per-search slabs (pgi_graph_*). V is 0 until pgi_graph_init built it.
struct Graph {
    uint32_t V = 0, cap = 0, words = 0, heapCap = 0, arenaCap = 0, slots = 0;
    DevBuf<AdjDev> adj;
    DevBuf<uint32_t> counts;  // [0, V): committed entries per vertex, [V, 2V): committed + predicted
    PinnedBuf<uint32_t> hCounts;
    DevBuf<double> simT;
    DevBuf<HeapItemDev> heaps;
    DevBuf<ArenaNodeDev> arenas;
    DevBuf<uint32_t> nextQuery;
    struct {
        uint32_t cap = 0;
        DevBuf<ApplyEntry> dev;
        PinnedBuf<ApplyEntry> host;
    } apply;
    struct {
        uint32_t cap = 0;
        DevBuf<pgi_query> queries;
        DevBuf<pgi_search_result> results;
        DevBuf<uint32_t> expBits;
        PinnedBuf<pgi_query> hQueries;
        PinnedBuf<pgi_search_result> hResults;
        PinnedBuf<uint32_t> hExpBits;
    } search;
};

constexpr int kMaxChunks = 64;
constexpr uint32_t kK5MaxSmemPts = 11264;  // 176 KB of float4 + 22 KB of queues; also keeps point slots per thread <= 64 (mask bits)
constexpr uint32_t kK4bCtasPerSm = 2;       // fewer lanes = more polynomials per lane = better refill balance
constexpr uint32_t kAstarSlotsPerSm = 16;   // K6 searches resident per SM (heap + arena slabs each)
static_assert(kAstarSlotsPerSm % kAstarWarps == 0, "K6 slots come in whole CTAs");

}  // namespace

// Members are destroyed in reverse order: the buffers first, then the events and the stream.
struct pgi_ctx {
    pgi_config cfg;
    Stream stream;
    Event evBegin, evStart, evK1, evK2, evK3, evFbEnd;
    Event evChunk[kMaxChunks][2];
    Event evS0, evS1;
    std::string err;
    Registration own, tmp;
    Registration extra;            // pgi_register_extra_pairs: rows built from caller-supplied matches (PGI_WAVE_EXTRA)
    DevBuf<uint2> extraPv, extraM; // their pair views and matches, as K0 reads them
    DevBuf<unsigned char> guidedBatch;  // K10 scratch of one chunk
    std::vector<GuidedPairIn> guidedIn;
    std::vector<uint64_t> guidedOff;
    MatchStaging pairMatch;             // pgi_match_features: its two views, apart from the registered scene
    DevBuf<uint64_t> pairMatchOff;
    const Registration *reg = &own;  // own, or the owner's after pgi_share_pairs
    // wave buffers
    DevSlots slots;
    HostSlots hostSlots;
    FallbackScratch fb;
    uint32_t bitsStride = 0;  // only grows
    DevBuf<double> hyp;       // 7 per hypothesis
    PinnedBuf<double> hHyp;
    DevBuf<uint8_t> masks;
    DevBuf<unsigned long long> counters;
    PinnedBuf<unsigned long long> hCounters;
    SceneStaging scene;
    uint32_t numSms = 148;
    // in flight
    bool inFlight = false;
    uint32_t waveN = 0, waveFlags = 0;
    uint64_t waveMaskRows = 0;
    int nChunks = 0;
    bool fbLaunched = false;
    pgi_stats stats;
    Graph graph;
    pgi_search_stats sstats;
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char buf__[256];                                                                       \
            snprintf(buf__, sizeof buf__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                     __FILE__, __LINE__);                                                          \
            ctx->err = buf__;                                                                      \
            return e__ == cudaErrorMemoryAllocation ? PGI_ERR_NOMEM : PGI_ERR_CUDA;                \
        }                                                                                          \
    } while (0)

// cv::RNG (multiply-with-carry) on the host, for the sampler tables.
struct HostRng {
    uint64_t state;
    explicit HostRng(uint64_t s) : state(s ? s : 0xffffffffULL) {}
    uint32_t next()
    {
        state = (uint64_t)(uint32_t)state * 4164903690U + (uint32_t)(state >> 32);
        return (uint32_t)state;
    }
    int uniform(int a, int b) { return a == b ? a : (int)(next() % (uint32_t)(b - a) + a); }
};

// Per distinct N: the uniform sampler's (iteration -> 5 indices) table (persistent-pool partial
// Fisher-Yates driven by cv::RNG(0), SURVEY App. B.5) and the termination table
// iterations(inlier count) = ceil(log(1-0.99)/log(1-(k/N)^5)) clamped to [1, maxIters].
pgi_status buildTables(pgi_ctx *ctx, Registration &r)
{
    const uint32_t maxIters = ctx->cfg.fallback_max_iters;
    std::map<uint32_t, uint32_t> tableOfN;
    std::vector<uint32_t> pairTable(r.nPairs);
    for (uint64_t p = 0; p < r.nPairs; p++) {
        const uint32_t N = (uint32_t)(r.h_offset[p + 1] - r.h_offset[p]);
        auto it = tableOfN.find(N);
        if (it == tableOfN.end()) it = tableOfN.emplace(N, (uint32_t)tableOfN.size()).first;
        pairTable[p] = it->second;
    }
    const size_t T = tableOfN.size();
    std::vector<uint32_t> sampler(T * maxIters * 5, 0);
    std::vector<uint64_t> itersOff(T, 0);
    std::vector<uint16_t> itersTab;
    std::vector<std::pair<uint32_t, uint32_t>> order(tableOfN.begin(), tableOfN.end());
    std::sort(order.begin(), order.end(), [](auto &a, auto &b) { return a.second < b.second; });
    std::vector<int> pool;
    for (auto &kv : order) {
        const int N = (int)kv.first;
        const uint32_t t = kv.second;
        itersOff[t] = itersTab.size();
        for (int k = 0; k <= N; k++) {
            int it;
            const double w = N > 0 ? (double)k / (double)N : 0.0;
            const double p5 = w * w * w * w * w;
            if (p5 <= 0.0)
                it = (int)maxIters;
            else if (p5 >= 1.0)
                it = 1;
            else {
                const double v = std::log(1.0 - 0.99) / std::log(1.0 - p5);
                it = v >= (double)maxIters ? (int)maxIters : (int)std::ceil(v);
                if (it < 1) it = 1;
            }
            itersTab.push_back((uint16_t)it);
        }
        if (N >= 5) {
            pool.resize(N);
            for (int i = 0; i < N; i++) pool[i] = i;
            HostRng rng(0);
            uint32_t *out = sampler.data() + (size_t)t * maxIters * 5;
            for (uint32_t itn = 0; itn < maxIters; itn++) {
                int size = N;
                for (int i = 0; i < 5; i++) {
                    const int j = rng.uniform(0, size);
                    out[(size_t)itn * 5 + i] = (uint32_t)pool[j];
                    std::swap(pool[j], pool[--size]);
                }
            }
        }
    }
    CK(r.pairTable.grow(r.nPairs));
    CK(r.sampler.grow(sampler.size()));
    CK(r.itersTab.grow(itersTab.size()));
    CK(r.itersOff.grow(T));
    CK(cudaMemcpyAsync(r.pairTable.data(), pairTable.data(), pairTable.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(r.sampler.data(), sampler.data(), sampler.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(r.itersTab.data(), itersTab.data(), itersTab.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(r.itersOff.data(), itersOff.data(), itersOff.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->stats.h2d_bytes += pairTable.size() * 4 + sampler.size() * 4 + itersTab.size() * 2 + itersOff.size() * 8;
    return PGI_OK;
}

pgi_status registerDense(pgi_ctx *ctx, Registration &r, uint64_t nPairs, const uint64_t *offset, const double *corr,
                         const double *thr)
{
    if (!offset || (!corr && offset[nPairs] > 0) || !thr) { ctx->err = "null argument"; return PGI_ERR_INVALID; }
    for (uint64_t p = 0; p < nPairs; p++)
        if (offset[p + 1] < offset[p] || offset[p + 1] - offset[p] > 0x7fffffffULL) { ctx->err = "bad corr_offset"; return PGI_ERR_INVALID; }
    r.nPairs = nPairs;
    r.nRows = offset[nPairs];
    r.h_offset.assign(offset, offset + nPairs + 1);
    r.maxN = 0;
    for (uint64_t p = 0; p < nPairs; p++) r.maxN = std::max<uint32_t>(r.maxN, (uint32_t)(offset[p + 1] - offset[p]));
    CK(r.corr.grow(r.nRows * 4));
    CK(r.offset.grow(nPairs + 1));
    CK(r.thr.grow(nPairs));
    if (r.nRows) CK(cudaMemcpyAsync(r.corr.data(), corr, r.nRows * 32, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(r.offset.data(), offset, (nPairs + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (nPairs) CK(cudaMemcpyAsync(r.thr.data(), thr, nPairs * 8, cudaMemcpyHostToDevice, ctx->stream));
    ctx->stats.h2d_bytes += r.nRows * 32 + (nPairs + 1) * 8 + nPairs * 8;
    return buildTables(ctx, r);
}

pgi_status ensureWave(pgi_ctx *ctx, const Registration &r, uint32_t n, uint32_t nHyp, uint32_t flags, uint64_t maskRows)
{
    const uint32_t stride = (r.maxN + 31) / 32 + 1;
    if (n > ctx->slots.cap || stride > ctx->bitsStride) {
        const uint32_t cap = std::max<uint32_t>(std::max(n, ctx->slots.cap), 64);
        // the fallback scratch is sized for the old slot count: released here, re-created by the next fallback wave
        ctx->fb = FallbackScratch();
        ctx->slots = DevSlots();
        ctx->bitsStride = std::max(stride, ctx->bitsStride);
        CK(ctx->slots.pairId.grow(cap));
        CK(ctx->slots.hypOffset.grow((size_t)cap + 1));
        CK(ctx->slots.state.grow(cap));
        CK(ctx->slots.bits.grow((size_t)cap * 2 * ctx->bitsStride));
        CK(ctx->slots.maskOffset.grow((size_t)cap + 1));
        CK(ctx->slots.verdicts.grow(cap));
        CK(ctx->slots.k3Scratch.grow((size_t)cap * 8));
        CK(cudaMemsetAsync(ctx->slots.k3Scratch.data(), 0, (size_t)cap * 8 * 4, ctx->stream));
        ctx->slots.cap = cap;
    }
    if (flags & PGI_WAVE_FALLBACK) {
        const size_t slots = (size_t)ctx->slots.cap * kFbChunk;
        CK(ctx->fb.sols.grow(slots * 90));
        CK(ctx->fb.counts.grow(slots));
        CK(ctx->fb.solsF.grow(slots * 30));
        CK(ctx->fb.dkList.grow(slots));
        CK(ctx->fb.dkCtl.grow(2));
    }
    if ((size_t)nHyp * 7 > ctx->hyp.capacity())
        CK(ctx->hyp.grow((size_t)std::max<uint32_t>(nHyp, std::max<uint32_t>(ctx->slots.cap, 64)) * 7));
    if ((flags & PGI_WAVE_MASKS) && maskRows > ctx->masks.capacity()) CK(ctx->masks.grow(maskRows));
    if (n > ctx->hostSlots.cap) {
        const uint32_t cap = std::max<uint32_t>(std::max(n, ctx->hostSlots.cap), 64);
        ctx->hostSlots = HostSlots();
        CK(ctx->hostSlots.pairId.grow(cap));
        CK(ctx->hostSlots.hypOffset.grow((size_t)cap + 1));
        CK(ctx->hostSlots.maskOffset.grow((size_t)cap + 1));
        CK(ctx->hostSlots.verdicts.grow(cap));
        ctx->hostSlots.cap = cap;
    }
    if ((size_t)nHyp * 7 > ctx->hHyp.capacity())
        CK(ctx->hHyp.grow((size_t)std::max<uint32_t>(nHyp, std::max<uint32_t>(ctx->hostSlots.cap, 64)) * 7));
    return PGI_OK;
}

pgi_status submitWave(pgi_ctx *ctx, const Registration &r, uint32_t n, const uint32_t *pairId, const uint32_t *hypOffset,
                      const double *hyp, uint32_t flags, const double *thrOverride, uint32_t testMinOverride, bool scoreOnly)
{
    if (ctx->inFlight) { ctx->err = "a wave is already in flight"; return PGI_ERR_STATE; }
    if (n == 0) { ctx->waveN = 0; ctx->inFlight = true; ctx->fbLaunched = false; ctx->nChunks = 0; ctx->waveFlags = flags; return PGI_OK; }
    if (!pairId || !hypOffset) { ctx->err = "null argument"; return PGI_ERR_INVALID; }
    if (!r.offset.data()) { ctx->err = "no pairs registered"; return PGI_ERR_STATE; }
    const uint32_t nHyp = hypOffset[n];
    if (nHyp && !hyp) { ctx->err = "hypotheses missing"; return PGI_ERR_INVALID; }
    uint64_t maskRows = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (pairId[i] >= r.nPairs) { ctx->err = "pair_id out of range"; return PGI_ERR_INVALID; }
        if (hypOffset[i + 1] < hypOffset[i]) { ctx->err = "hyp_offset not monotone"; return PGI_ERR_INVALID; }
    }
    pgi_status st = ensureWave(ctx, r, n, nHyp, flags, 0);
    if (st != PGI_OK) return st;
    const DevSlots &d = ctx->slots;
    const HostSlots &h = ctx->hostSlots;
    for (uint32_t i = 0; i < n; i++) {
        h.maskOffset.data()[i] = maskRows;
        maskRows += r.h_offset[pairId[i] + 1] - r.h_offset[pairId[i]];
    }
    h.maskOffset.data()[n] = maskRows;
    if ((st = ensureWave(ctx, r, n, nHyp, flags, maskRows)) != PGI_OK) return st;
    memcpy(h.pairId.data(), pairId, (size_t)n * 4);
    memcpy(h.hypOffset.data(), hypOffset, ((size_t)n + 1) * 4);
    if (nHyp) memcpy(ctx->hHyp.data(), hyp, (size_t)nHyp * 56);
    cudaStream_t s = ctx->stream;
    CK(cudaEventRecord(ctx->evBegin, s));
    CK(cudaMemcpyAsync(d.pairId.data(), h.pairId.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d.hypOffset.data(), h.hypOffset.data(), ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d.maskOffset.data(), h.maskOffset.data(), ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, s));
    if (nHyp) CK(cudaMemcpyAsync(ctx->hyp.data(), ctx->hHyp.data(), (size_t)nHyp * 56, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(ctx->counters.data(), 0, 3 * sizeof(unsigned long long), s));
    ctx->stats.h2d_bytes += (size_t)n * 4 + ((size_t)n + 1) * 12 + (size_t)nHyp * 56;

    WaveArgs a;
    a.corr = r.corr.data(); a.offset = r.offset.data(); a.thr = r.thr.data(); a.pairTable = r.pairTable.data();
    a.samplerTab = r.sampler.data(); a.itersTab = r.itersTab.data(); a.itersTabOff = r.itersOff.data();
    a.n = n; a.pairId = d.pairId.data(); a.hypOffset = d.hypOffset.data(); a.hyp = ctx->hyp.data(); a.state = d.state.data();
    a.bits = d.bits.data(); a.bitsStride = ctx->bitsStride; a.masks = ctx->masks.data(); a.maskOffset = d.maskOffset.data();
    a.verdicts = d.verdicts.data(); a.flags = flags; a.minInliers = ctx->cfg.min_inliers;
    a.testMinInliers = testMinOverride ? testMinOverride : ctx->cfg.test_min_inliers;
    a.fbMaxIters = ctx->cfg.fallback_max_iters; a.thrMultiplier = ctx->cfg.threshold_multiplier;
    a.thrOverride = thrOverride ? *thrOverride : 0.0;
    a.hasThrOverride = thrOverride ? 1u : 0u;
    a.fbSols = ctx->fb.sols.data(); a.fbSolsF = ctx->fb.solsF.data(); a.fbCounts = ctx->fb.counts.data(); a.counters = ctx->counters.data();
    a.k3Scratch = d.k3Scratch.data(); a.dkList = ctx->fb.dkList.data(); a.dkCtl = ctx->fb.dkCtl.data();

    CK(cudaEventRecord(ctx->evStart, s));  // kernel-only timing: the wave's small H2D copies are before this event
    // full waves stream the correspondences through shared memory with bulk async copies (persistent CTAs, one per SM);
    // small waves and waves that want byte masks take the one-CTA-per-pair kernel
    if (n >= 2u * ctx->numSms && !(flags & PGI_WAVE_MASKS)) {
        const int k1Smem = kK1Stages * kK1TileRows * 32 + (int)sizeof(K1Meta);
        CK(cudaFuncSetAttribute(k1_score_hypotheses_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, k1Smem));
        k1_score_hypotheses_tma<<<std::min<uint32_t>(n, ctx->numSms), kK1TmaThreads, k1Smem, s>>>(a);
    } else
        k1_score_hypotheses<<<n, kCtaThreads, 0, s>>>(a);
    CK(cudaEventRecord(ctx->evK1, s));
    ctx->stats.launches += 1;
    ctx->fbLaunched = false;
    ctx->nChunks = 0;
    if (!scoreOnly) {
        // the solve is one long serial chain per pair: on small waves give every pair a warp of its own (no divergence
        // serialisation between pairs, all SMs used); large waves pack 64 pairs per CTA for throughput
        if (n <= 4096u)
            k2_fivept_first_solution<<<n, 32, 0, s>>>(a, 1);
        else
            k2_fivept_first_solution<<<(n + 63) / 64, 64, 0, s>>>(a, 0);
        CK(cudaEventRecord(ctx->evK2, s));
        ctx->stats.launches += 1;
        if (flags & PGI_WAVE_FALLBACK) {
            const int chunks = (int)((ctx->cfg.fallback_max_iters + kFbChunk - 1) / kFbChunk);
            // FP32 staging area of K5: the largest pair if it fits, else 0 (those pairs take the FP64-only path)
            uint32_t smemPts = r.maxN <= kK5MaxSmemPts ? std::max<uint32_t>(r.maxN, 1) : kK5MaxSmemPts;
            // + per-warp compaction queues: 8 warps x min(smemPts, 2048) uint16
            const size_t k5Smem = (size_t)smemPts * 16 + (size_t)8 * (smemPts < kK5QueuePts ? ((smemPts + 31u) & ~31u) : kK5QueuePts) * 2 +
                                  (size_t)((smemPts + 31) / 32) * 4;  // + inlier bit mask of the LO refit
            if (k5Smem > 40 * 1024)  // static shared memory (~4 KB) counts towards the 48 KB default limit
                CK(cudaFuncSetAttribute(k5_fallback_score, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k5Smem));
            ctx->nChunks = std::min(chunks, kMaxChunks);
            for (int c = 0; c < ctx->nChunks; c++) {
                const uint32_t threads = n * kFbChunk;
                CK(cudaMemsetAsync(ctx->fb.dkCtl.data(), 0, 8, s));
                k4a_polynomial<<<(threads + 127) / 128, 128, 0, s>>>(a, c);
                k4b_roots<<<std::min<uint32_t>((threads + 127) / 128, ctx->numSms * kK4bCtasPerSm), 128, 0, s>>>(a);
                k4c_solutions<<<(threads + 127) / 128, 128, 0, s>>>(a, c);
                CK(cudaEventRecord(ctx->evChunk[c][0], s));
                k5_fallback_score<<<n, kCtaThreads, k5Smem, s>>>(a, c, c == ctx->nChunks - 1 ? 1 : 0, smemPts);
                CK(cudaEventRecord(ctx->evChunk[c][1], s));
                ctx->stats.launches += 4;
            }
            ctx->fbLaunched = true;
        }
        CK(cudaEventRecord(ctx->evFbEnd, s));
        // small waves are latency bound: cover each pair by several point-range CTAs until the grid fills the GPU
        const uint32_t split = n >= 592u ? 1u : std::min(8u, (592u + n - 1) / n);
        k3_decompose_vote<<<n * split, kK3Threads, 0, s>>>(a, split);
        ctx->stats.launches += 1;
    } else {
        CK(cudaEventRecord(ctx->evK2, s));
        CK(cudaEventRecord(ctx->evFbEnd, s));
    }
    CK(cudaEventRecord(ctx->evK3, s));
    CK(cudaGetLastError());
    ctx->inFlight = true;
    ctx->waveN = n;
    ctx->waveFlags = flags;
    ctx->waveMaskRows = maskRows;
    ctx->stats.pairs += n;
    return PGI_OK;
}

// A failed CUDA call inside a wait must not leave the context "in flight" for ever (every later submit would answer
// PGI_ERR_STATE): whatever the exit path, the wave is over once the wait returns.
struct WaveEndGuard {
    pgi_ctx *ctx;
    ~WaveEndGuard()
    {
        if (ctx->inFlight) {
            cudaStreamSynchronize(ctx->stream);  // best effort: nothing of the failed wave may still be running
            ctx->inFlight = false;
        }
    }
};

pgi_status finishWave(pgi_ctx *ctx)
{
    // caller has synchronised the stream
    if (ctx->waveN == 0) { ctx->inFlight = false; return PGI_OK; }
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evK1)); ctx->stats.ms_score += ms;
    CK(cudaEventElapsedTime(&ms, ctx->evK1, ctx->evK2)); ctx->stats.ms_fivept += ms;
    if (ctx->fbLaunched) {
        for (int c = 0; c < ctx->nChunks; c++) {
            CK(cudaEventElapsedTime(&ms, c == 0 ? ctx->evK2 : ctx->evChunk[c - 1][1], ctx->evChunk[c][0]));
            ctx->stats.ms_fallback_solve += ms;
            CK(cudaEventElapsedTime(&ms, ctx->evChunk[c][0], ctx->evChunk[c][1]));
            ctx->stats.ms_fallback_score += ms;
        }
    }
    CK(cudaEventElapsedTime(&ms, ctx->evFbEnd, ctx->evK3)); ctx->stats.ms_decompose += ms;
    CK(cudaEventElapsedTime(&ms, ctx->evBegin, ctx->evK3)); ctx->stats.ms_total += ms;
    ctx->stats.corr_evals += ctx->hCounters.data()[0];
    ctx->stats.fallback_pairs += ctx->hCounters.data()[1];
    ctx->stats.fallback_models += ctx->hCounters.data()[2];
    ctx->inFlight = false;
    return PGI_OK;
}

// K0 (createCorrespondenceMatrix) over the staged scene's views and keypoints (ctx->scene) for the pair views pv and
// matches m (device arrays: the scene's own, or the extra pairs') into r,
// whose offset, h_offset, nPairs, nRows and maxN are set and whose corr / thr hold nRows / nPairs entries; then the
// sampler tables.
pgi_status buildCorrespondences(pgi_ctx *ctx, Registration &r, double thr_px, const uint2 *pv, const uint2 *m)
{
    cudaStream_t s = ctx->stream;
    const SceneStaging &sc = ctx->scene;
    const uint64_t n_pairs = r.nPairs;
    if (n_pairs) {
        CK(cudaEventRecord(ctx->evStart, s));
        const uint32_t gx = std::max<uint32_t>(1, std::min<uint32_t>((r.maxN + 255) / 256, 64));
        const uint32_t gy = (uint32_t)std::min<uint64_t>(n_pairs, 65535), gz = (uint32_t)((n_pairs + gy - 1) / gy);
        k0_build_correspondences<<<dim3(gx, gy, gz), 256, 0, s>>>(sc.focal.data(), sc.size.data(), sc.kpOff.data(), sc.kp.data(),
                                                                   n_pairs, pv, r.offset.data(), m, thr_px,
                                                                   reinterpret_cast<double4 *>(r.corr.data()), r.thr.data());
        CK(cudaEventRecord(ctx->evK1, s));
        CK(cudaGetLastError());
        ctx->stats.launches += 1;
    }
    CK(cudaStreamSynchronize(s));
    if (n_pairs) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evK1));
        ctx->stats.ms_correspondences += ms;
    }
    return buildTables(ctx, r);
}

// PGI_ERR_INVALID if one of the n device values is not finite (a NaN distance never enters a 2-NN, so it would silently
// drop neighbours).  Synchronises the stream.
pgi_status checkFinite(pgi_ctx *ctx, const float *x, uint64_t n)
{
    cudaStream_t s = ctx->stream;
    uint32_t *d_flag = reinterpret_cast<uint32_t *>(ctx->counters.data());
    uint32_t flag = 0;
    CK(cudaMemsetAsync(d_flag, 0, 4, s));
    if (n) {
        k9_check_finite<<<(uint32_t)std::min<uint64_t>((n + 1023) / 1024, 4 * ctx->numSms), 1024, 0, s>>>(x, n, d_flag);
        CK(cudaGetLastError());
        ctx->stats.launches += 1;
    }
    CK(cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += 4;
    if (flag) { ctx->err = "non-finite descriptor value"; return PGI_ERR_INVALID; }
    return PGI_OK;
}

// Uploads the scene's descriptors (nKp x dim, row-aligned with the staged keypoints); they stay resident for K9 and K10.
pgi_status uploadDescriptors(pgi_ctx *ctx, const float *desc, uint64_t nKp, uint32_t dim)
{
    SceneStaging &sc = ctx->scene;
    sc.hasDesc = false;
    CK(sc.desc.grow(nKp * dim));
    if (nKp) CK(cudaMemcpyAsync(sc.desc.data(), desc, nKp * dim * 4, cudaMemcpyHostToDevice, ctx->stream));
    ctx->stats.h2d_bytes += nKp * dim * 4;
    if (pgi_status st = checkFinite(ctx, sc.desc.data(), nKp * dim); st != PGI_OK) return st;
    sc.hasDesc = true;
    sc.dim = dim;
    return PGI_OK;
}

// Grows the staging both scene registrations share and queues its upload: focal lengths, image sizes, keypoint
// offsets, keypoints and pair views.
pgi_status stageScene(pgi_ctx *ctx, uint64_t n_views, const double *focal, const double *size_wh, const uint64_t *kp_offset,
                      const float *kp_xy, uint64_t n_pairs, const uint32_t *pair_views)
{
    SceneStaging &sc = ctx->scene;
    const uint64_t nKp = kp_offset[n_views];
    sc.staged = sc.hasDesc = false;
    sc.hKpOff.assign(kp_offset, kp_offset + n_views + 1);
    sc.hFocal.assign(focal, focal + n_views);
    sc.hSize.assign(size_wh, size_wh + 2 * n_views);
    CK(sc.focal.grow(n_views));
    CK(sc.size.grow(n_views * 2));
    CK(sc.kpOff.grow(n_views + 1));
    CK(sc.kp.grow(nKp));
    CK(sc.pv.grow(n_pairs));
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(sc.focal.data(), focal, n_views * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(sc.size.data(), size_wh, n_views * 16, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(sc.kpOff.data(), kp_offset, (n_views + 1) * 8, cudaMemcpyHostToDevice, s));
    if (nKp) CK(cudaMemcpyAsync(sc.kp.data(), kp_xy, nKp * 8, cudaMemcpyHostToDevice, s));
    if (n_pairs) CK(cudaMemcpyAsync(sc.pv.data(), pair_views, n_pairs * 8, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += n_views * 24 + (n_views + 1) * 8 + nKp * 8 + n_pairs * 8;
    return PGI_OK;
}

// E = [t]x R of the pose (pose.h:46-55), as the matcher reads it from Pose::getEssentialMatrix (matcher.h:218)
void essentialOfPose(const double *q, double *E)
{
    double R[9];
    const double tx = 2.0 * q[0], ty = 2.0 * q[1], tz = 2.0 * q[2];
    const double twx = tx * q[3], twy = ty * q[3], twz = tz * q[3], txx = tx * q[0], txy = ty * q[0], txz = tz * q[0];
    const double tyy = ty * q[1], tyz = tz * q[1], tzz = tz * q[2];
    R[0] = 1.0 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
    R[3] = txy + twz; R[4] = 1.0 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1.0 - (txx + tyy);
    const double Cx[9] = {0.0, -q[6], q[5], q[6], 0.0, -q[4], -q[5], q[4], 0.0};
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) E[i * 3 + j] = Cx[i * 3 + 0] * R[j] + (Cx[i * 3 + 1] * R[3 + j] + Cx[i * 3 + 2] * R[6 + j]);
}

// What a K9 or K10 run took: device time of its chunks (CUDA events), descriptor distances, rows, chunks.
struct MatchRun {
    float ms = 0;
    uint64_t dist = 0, rows = 0, chunks = 0;
};

// K9 for the n_pairs pairs staged in st (desc, kpOff, pv; kp_offset and pair_views are the host copies of the last two,
// maxK the largest view): pair p's rows, sorted by (ratio bits, query), go to st.m / st.ratio at offset[p] .. offset[p + 1]
// - 1.  The caller sets offset[0] = 0.  Scratch (forward states, backward partials, staged sorted rows) is sized for a
// chunk of pairs only.
pgi_status matchPairs(pgi_ctx *ctx, MatchStaging &st, uint32_t dim, uint32_t maxK, uint64_t n_pairs, const uint64_t *kp_offset,
                      const uint32_t *pair_views, uint64_t *offset, MatchRun &run)
{
    cudaStream_t s = ctx->stream;
    const uint32_t stride = std::max<uint32_t>(maxK, 1), maxSB = (stride + kK9Rows - 1) / kK9Rows;
    uint32_t keyCap = 1;
    while (keyCap < stride) keyCap <<= 1;
    const size_t perPair = (size_t)maxSB * stride * sizeof(Nn2) + (size_t)stride * (sizeof(Nn2) + 8 + 4) + 4;
    const size_t kScratchBudget = (size_t)512 << 20;
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>({kScratchBudget / perPair, 65535, std::max<uint64_t>(n_pairs, 1)}));
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t oF = 0, oB = oF + al(chunk * stride * sizeof(Nn2)), oM = oB + al(chunk * maxSB * stride * sizeof(Nn2)),
                 oR = oM + al(chunk * stride * 8), oC = oR + al(chunk * stride * 4), total = oC + al(chunk * 4);
    CK(st.k9Scratch.grow(total));
    Nn2 *d_fwd = reinterpret_cast<Nn2 *>(st.k9Scratch.data() + oF), *d_bpart = reinterpret_cast<Nn2 *>(st.k9Scratch.data() + oB);
    uint2 *d_sm = reinterpret_cast<uint2 *>(st.k9Scratch.data() + oM);
    float *d_sr = reinterpret_cast<float *>(st.k9Scratch.data() + oR);
    uint32_t *d_cnt = reinterpret_cast<uint32_t *>(st.k9Scratch.data() + oC);
    const size_t finishSmem = (size_t)keyCap * 8 + (size_t)stride * 4;
    CK(cudaFuncSetAttribute(k9_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)finishSmem));
    for (uint64_t c0 = 0; c0 < n_pairs; c0 += chunk) {
        const uint32_t cp = (uint32_t)std::min<uint64_t>(chunk, n_pairs - c0);
        uint32_t sbUsed = 0;
        for (uint64_t p = c0; p < c0 + cp; p++) {
            const uint64_t nS = kp_offset[pair_views[2 * p] + 1] - kp_offset[pair_views[2 * p]];
            const uint64_t nD = kp_offset[pair_views[2 * p + 1] + 1] - kp_offset[pair_views[2 * p + 1]];
            sbUsed = std::max<uint32_t>(sbUsed, (uint32_t)((nS + kK9Rows - 1) / kK9Rows));
            run.dist += nS * nD;
        }
        CK(cudaEventRecord(ctx->evStart, s));
        {
            PgiNvtxRange chunkRange("pgi:k9 chunk");
            if (sbUsed) {
                if (dim == 128)
                    k9_knn2_tile<128><<<dim3(sbUsed, cp), kK9Threads, 0, s>>>(st.desc.data(), st.kpOff.data(), st.pv.data(), c0, stride, maxSB, d_fwd, d_bpart);
                else
                    k9_knn2_tile<64><<<dim3(sbUsed, cp), kK9Threads, 0, s>>>(st.desc.data(), st.kpOff.data(), st.pv.data(), c0, stride, maxSB, d_fwd, d_bpart);
                ctx->stats.launches += 1;
            }
            k9_finish<<<cp, kK9FinishThreads, finishSmem, s>>>(st.kpOff.data(), st.pv.data(), c0, stride, keyCap, maxSB, d_fwd, d_bpart, d_cnt, d_sm, d_sr);
            k9_offsets<<<1, 1024, 0, s>>>(d_cnt, cp, offset, c0);
            CK(cudaGetLastError());
            ctx->stats.launches += 2;
        }
        uint64_t end = 0;
        CK(cudaMemcpyAsync(&end, offset + c0 + cp, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        ctx->stats.d2h_bytes += 8;
        CK(st.growMatches(end, run.rows, s));
        k9_scatter<<<cp, 256, 0, s>>>(offset, c0, stride, d_cnt, d_sm, d_sr, st.m.data(), st.ratio.data());
        CK(cudaEventRecord(ctx->evK1, s));
        CK(cudaGetLastError());
        ctx->stats.launches += 1;
        CK(cudaEventSynchronize(ctx->evK1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evK1));
        run.ms += ms;
        run.rows = end;
        run.chunks++;
    }
    return PGI_OK;
}

// One guided-matching case of the registered scene: views src -> dst at pose q (T_dst_src), K = [f 0 w/2; 0 f h/2; 0 0 1]
// of each view (pose_graph_builder.h:284-286).
GuidedPairIn scenePairIn(const SceneStaging &sc, uint32_t src, uint32_t dst, const double *q, int32_t bin_number)
{
    GuidedPairIn in;
    memset(&in, 0, sizeof in);
    essentialOfPose(q, in.E);
    const double fS = sc.hFocal[src], wS = sc.hSize[2 * src], hS = sc.hSize[2 * src + 1];
    const double fD = sc.hFocal[dst], wD = sc.hSize[2 * dst], hD = sc.hSize[2 * dst + 1];
    const double Ks[9] = {fS, 0.0, wS / 2.0, 0.0, fS, hS / 2.0, 0.0, 0.0, 1.0};
    const double Kd[9] = {fD, 0.0, wD / 2.0, 0.0, fD, hD / 2.0, 0.0, 0.0, 1.0};
    memcpy(in.Ks, Ks, sizeof Ks);
    memcpy(in.Kd, Kd, sizeof Kd);
    in.wS = (int)wS; in.hS = (int)hS; in.wD = (int)wD; in.hD = (int)hD; in.binNumber = bin_number;
    in.kS0 = sc.hKpOff[src]; in.kD0 = sc.hKpOff[dst];
    in.nS = (uint32_t)(sc.hKpOff[src + 1] - in.kS0); in.nD = (uint32_t)(sc.hKpOff[dst + 1] - in.kD0);
    return in;
}

// K10 for the n_pairs cases `in` (host array) on the keypoints kp and the descriptors desc (dim 64 or 128) they index:
// pair k's rows go to offsets_out[k] .. offsets_out[k + 1] - 1 of matches_out / values_out.  max_points > 0: guidedMatching's
// selection (pose_graph_builder.h:760-782); 0: match()'s rows and adapted ratios in source order.  Every argument error
// comes before any device work.  Scratch is sized for the batch's largest views and bounded per chunk of pairs (512 MB).
// prep_or_null receives the first pair's preparation.
pgi_status runGuided(pgi_ctx *ctx, const float2 *kp, const float *desc, uint32_t dim, const GuidedPairIn *in, uint64_t n_pairs,
                     uint32_t max_points, uint64_t *offsets_out, uint32_t *matches_out, double *values_out, uint64_t capacity_rows,
                     GuidedPrep *prep_or_null, MatchRun &run)
{
    uint64_t need = 0;
    uint32_t maxS = 0, maxD = 0;
    for (uint64_t p = 0; p < n_pairs; p++) {
        // the selection sorts 16-bit source indices; without it any view size works
        if (max_points && (in[p].nS > kK10MaxKp || in[p].nD > kK10MaxKp)) {
            ctx->err = "batched guided matching supports at most 16384 keypoints per view";
            return PGI_ERR_INVALID;
        }
        need += max_points ? std::min<uint64_t>(in[p].nS, max_points) : in[p].nS;
        maxS = std::max(maxS, in[p].nS);
        maxD = std::max(maxD, in[p].nD);
    }
    if (need > capacity_rows) { ctx->err = "capacity_rows is below the rows the batch can produce"; return PGI_ERR_INVALID; }
    if (need && (!matches_out || !values_out)) { ctx->err = "null argument"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    offsets_out[0] = 0;
    if (n_pairs == 0) return PGI_OK;
    cudaStream_t s = ctx->stream;

    const uint32_t strideS = std::max<uint32_t>(maxS, 1), strideD = std::max<uint32_t>(maxD, 1);
    const uint32_t dstBlocks = (strideD + kK10DstBlock - 1) / kK10DstBlock;
    const uint32_t rowCap = max_points ? std::min(strideS, max_points) : strideS;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t perPair = sizeof(GuidedPairIn) + sizeof(GuidedPairDev) + (size_t)strideD * 5 + (size_t)dstBlocks * kMatchMaxBins * 4 +
                           (size_t)strideS * (4 + 8 + 8 + 8) + 4 + 8 + (size_t)rowCap * 16;
    const size_t kScratchBudget = (size_t)512 << 20;
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>({kScratchBudget / perPair, 65535, n_pairs}));
    const size_t oIn = 0, oDev = oIn + al(chunk * sizeof(GuidedPairIn)), oBin = oDev + al(chunk * sizeof(GuidedPairDev)),
                 oList = oBin + al(chunk * strideD), oBlk = oList + al(chunk * strideD * 4),
                 oCand = oBlk + al(chunk * dstBlocks * kMatchMaxBins * 4), oRatio = oCand + al(chunk * strideS * 4),
                 oSM = oRatio + al(chunk * strideS * 8), oSV = oSM + al(chunk * strideS * 8), oCnt = oSV + al(chunk * strideS * 8),
                 oOff = oCnt + al(chunk * 4), oRM = oOff + al((chunk + 1) * 8), oRV = oRM + al(chunk * rowCap * 8),
                 oEv = oRV + al(chunk * rowCap * 8), total = oEv + 256;
    CK(ctx->guidedBatch.grow(total));
    unsigned char *d = ctx->guidedBatch.data();
    GuidedScratch g;
    g.in = reinterpret_cast<const GuidedPairIn *>(d + oIn);
    g.dev = reinterpret_cast<GuidedPairDev *>(d + oDev);
    g.binOfD = d + oBin;
    g.binList = reinterpret_cast<uint32_t *>(d + oList);
    g.blockOff = reinterpret_cast<uint32_t *>(d + oBlk);
    g.cand = reinterpret_cast<uint32_t *>(d + oCand);
    g.candRatio = reinterpret_cast<double *>(d + oRatio);
    g.stageM = reinterpret_cast<uint2 *>(d + oSM);
    g.stageV = reinterpret_cast<double *>(d + oSV);
    g.counts = reinterpret_cast<uint32_t *>(d + oCnt);
    g.strideS = strideS; g.strideD = strideD; g.dstBlocks = dstBlocks;
    uint64_t *d_off = reinterpret_cast<uint64_t *>(d + oOff);
    uint2 *d_rowsM = reinterpret_cast<uint2 *>(d + oRM);
    double *d_rowsV = reinterpret_cast<double *>(d + oRV);
    unsigned long long *d_evals = reinterpret_cast<unsigned long long *>(d + oEv);
    uint32_t sortCap = 0;
    if (max_points) {
        sortCap = 1;
        while (sortCap < strideS) sortCap <<= 1;
    }
    const size_t selectSmem = (size_t)sortCap * (8 + 2);
    CK(cudaFuncSetAttribute(k10_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)selectSmem));
    CK(cudaMemsetAsync(d_evals, 0, 8, s));
    CK(cudaMemsetAsync(d_off, 0, 8, s));
    std::vector<uint64_t> &hoff = ctx->guidedOff;
    uint64_t base = 0;
    unsigned long long evals = 0;  // every chunk adds to d_evals: the copy after the last chunk is the total
    for (uint64_t c0 = 0; c0 < n_pairs; c0 += chunk) {
        const uint32_t cp = (uint32_t)std::min<uint64_t>(chunk, n_pairs - c0);
        uint32_t sBlocks = 0, dBlocks = 0;
        for (uint32_t k = 0; k < cp; k++) {
            sBlocks = std::max<uint32_t>(sBlocks, (in[c0 + k].nS + kK10SrcPerCta - 1) / kK10SrcPerCta);
            dBlocks = std::max<uint32_t>(dBlocks, (in[c0 + k].nD + kK10DstBlock - 1) / kK10DstBlock);
        }
        CK(cudaMemcpyAsync(d + oIn, in + c0, (size_t)cp * sizeof(GuidedPairIn), cudaMemcpyHostToDevice, s));
        ctx->stats.h2d_bytes += (size_t)cp * sizeof(GuidedPairIn);
        CK(cudaEventRecord(ctx->evStart, s));
        {
            PgiNvtxRange chunkRange("pgi:k10 chunk");
            k10_prepare<<<(cp + 63) / 64, 64, 0, s>>>(g, cp);
            if (dBlocks) {
                k10_bin_count<<<dim3(dBlocks, cp), kK10DstBlock, 0, s>>>(g, kp);
                k10_bin_offsets<<<cp, kMatchMaxBins, 0, s>>>(g);
                k10_bin_scatter<<<dim3(dBlocks, cp), kK10DstBlock, 0, s>>>(g);
                ctx->stats.launches += 3;
            }
            if (sBlocks) {
                if (dim == 128)
                    k10_match<128><<<dim3(sBlocks, cp), kK10Threads, 0, s>>>(g, kp, desc, d_evals);
                else
                    k10_match<64><<<dim3(sBlocks, cp), kK10Threads, 0, s>>>(g, kp, desc, d_evals);
                ctx->stats.launches += 1;
            }
            k10_select<<<cp, kK10SelectThreads, selectSmem, s>>>(g, max_points, sortCap);
            k9_offsets<<<1, 1024, 0, s>>>(g.counts, cp, d_off, 0);
            k10_scatter<<<cp, 256, 0, s>>>(g, d_off, d_rowsM, d_rowsV);
            ctx->stats.launches += 4;
        }
        CK(cudaEventRecord(ctx->evK1, s));
        CK(cudaGetLastError());
        hoff.resize(cp + 1);
        CK(cudaMemcpyAsync(hoff.data(), d_off, (size_t)(cp + 1) * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(&evals, d_evals, 8, cudaMemcpyDeviceToHost, s));
        if (prep_or_null && c0 == 0) {
            CK(cudaMemcpyAsync(prep_or_null, &g.dev[0].p, sizeof(GuidedPrep), cudaMemcpyDeviceToHost, s));
            ctx->stats.d2h_bytes += sizeof(GuidedPrep);
        }
        CK(cudaStreamSynchronize(s));
        const uint64_t rows = hoff[cp];
        if (rows > capacity_rows - base) { ctx->err = "K10 produced more rows than its bound"; return PGI_ERR_CUDA; }
        for (uint32_t k = 0; k < cp; k++) offsets_out[c0 + k + 1] = base + hoff[k + 1];
        if (rows) {
            CK(cudaMemcpyAsync(matches_out + 2 * base, d_rowsM, rows * 8, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(values_out + base, d_rowsV, rows * 8, cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
        }
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evK1));
        run.ms += ms;
        ctx->stats.d2h_bytes += (size_t)(cp + 2) * 8 + rows * 16;
        base += rows;
        run.chunks++;
    }
    run.dist += evals;
    run.rows = base;
    return PGI_OK;
}

}  // namespace

extern "C" {

const char *pgi_version(void) { return "pgi 0.1 (sm_100a)"; }

int32_t pgi_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; d++) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, d) == cudaSuccess && p.major == 10) ok++;
    }
    return ok;
}

pgi_status pgi_create(const pgi_config *cfg, pgi_ctx **out)
{
    if (!cfg || !out) return PGI_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= cfg->device || cfg->device < 0) { cudaGetLastError(); return PGI_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return PGI_ERR_CUDA;
    if (prop.major != 10) return PGI_ERR_CUDA;  // kernels are sm_100a-only; there is no other path
    // until it is handed out, a failure destroys the half-built context
    std::unique_ptr<pgi_ctx, decltype(&pgi_destroy)> ctx(new pgi_ctx(), pgi_destroy);
    ctx->cfg = *cfg;
    ctx->numSms = (uint32_t)std::max(1, prop.multiProcessorCount);
    if (ctx->cfg.min_inliers == 0) ctx->cfg.min_inliers = 20;
    if (ctx->cfg.test_min_inliers == 0) ctx->cfg.test_min_inliers = 5;
    if (ctx->cfg.fallback_max_iters == 0) ctx->cfg.fallback_max_iters = 1000;
    if (ctx->cfg.fallback_max_iters > (uint32_t)kMaxChunks * kFbChunk) ctx->cfg.fallback_max_iters = kMaxChunks * kFbChunk;
    if (ctx->cfg.threshold_multiplier == 0.0) ctx->cfg.threshold_multiplier = 3.0 / 2.0;
    memset(&ctx->stats, 0, sizeof ctx->stats);
    memset(&ctx->sstats, 0, sizeof ctx->sstats);
    if (cudaSetDevice(cfg->device) != cudaSuccess) return PGI_ERR_CUDA;
    {
        // flags bit 0: background context (lowest stream priority) — used for the hypothesis-independent fallback
        // prefetch so that the latency-critical wave kernels of the foreground context get SM slots first
        int prioLow = 0, prioHigh = 0;
        cudaDeviceGetStreamPriorityRange(&prioLow, &prioHigh);
        const int prio = (ctx->cfg.flags & 1u) ? prioLow : prioHigh;
        if (cudaStreamCreateWithPriority(&ctx->stream.h, cudaStreamNonBlocking, prio) != cudaSuccess) return PGI_ERR_CUDA;
    }
    Event *evs[] = {&ctx->evBegin, &ctx->evStart, &ctx->evK1, &ctx->evK2, &ctx->evK3, &ctx->evFbEnd};
    for (Event *e : evs)
        if (cudaEventCreate(&e->h) != cudaSuccess) return PGI_ERR_CUDA;
    for (auto &chunk : ctx->evChunk)
        for (Event &e : chunk)
            if (cudaEventCreate(&e.h) != cudaSuccess) return PGI_ERR_CUDA;
    if (ctx->counters.grow(3) != cudaSuccess) return PGI_ERR_NOMEM;
    if (ctx->hCounters.grow(3) != cudaSuccess) return PGI_ERR_NOMEM;
    memset(ctx->hCounters.data(), 0, 3 * sizeof(unsigned long long));
    *out = ctx.release();
    return PGI_OK;
}

pgi_status pgi_destroy(pgi_ctx *ctx)
{
    if (!ctx) return PGI_OK;
    cudaSetDevice(ctx->cfg.device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);  // nothing still running may use a buffer freed below
    delete ctx;
    cudaGetLastError();
    return PGI_OK;
}

const char *pgi_last_error(pgi_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

pgi_status pgi_register_pairs(pgi_ctx *ctx, uint64_t n_pairs, const uint64_t *corr_offset, const double *corr_xy4,
                              const double *thr_norm)
{
    PgiNvtxRange nvtxRange("pgi:register_pairs");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->reg = &ctx->own;
    return registerDense(ctx, ctx->own, n_pairs, corr_offset, corr_xy4, thr_norm);
}

pgi_status pgi_register_scene(pgi_ctx *ctx, uint64_t n_views, const double *focal, const double *size_wh,
                              const uint64_t *kp_offset, const float *kp_xy, uint64_t n_pairs,
                              const uint32_t *pair_views, const uint64_t *m_offset, const uint32_t *matches,
                              double thr_px)
{
    PgiNvtxRange nvtxRange("pgi:register_scene (H2D + K0)");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    if (!focal || !size_wh || !kp_offset || !kp_xy || !pair_views || !m_offset || (!matches && m_offset[n_pairs])) {
        ctx->err = "null argument";
        return PGI_ERR_INVALID;
    }
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->reg = &ctx->own;
    Registration &r = ctx->own;
    const uint64_t nRows = m_offset[n_pairs];
    for (uint64_t p = 0; p < n_pairs; p++) {
        if (pair_views[2 * p] >= n_views || pair_views[2 * p + 1] >= n_views) { ctx->err = "view id out of range"; return PGI_ERR_INVALID; }
        if (m_offset[p + 1] < m_offset[p] || m_offset[p + 1] - m_offset[p] > 0x7fffffffULL) { ctx->err = "bad m_offset"; return PGI_ERR_INVALID; }
    }
    r.nPairs = n_pairs;
    r.nRows = nRows;
    r.h_offset.assign(m_offset, m_offset + n_pairs + 1);
    r.maxN = 0;
    for (uint64_t p = 0; p < n_pairs; p++) r.maxN = std::max<uint32_t>(r.maxN, (uint32_t)(m_offset[p + 1] - m_offset[p]));
    CK(r.corr.grow(nRows * 4));
    CK(r.offset.grow(n_pairs + 1));
    CK(r.thr.grow(n_pairs));
    CK(ctx->scene.m.grow(nRows));
    if (pgi_status st = stageScene(ctx, n_views, focal, size_wh, kp_offset, kp_xy, n_pairs, pair_views); st != PGI_OK) return st;
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(ctx->scene.m.data(), matches, nRows * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(r.offset.data(), m_offset, (n_pairs + 1) * 8, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += nRows * 8 + (n_pairs + 1) * 8;
    ctx->scene.matches = false;  // m now holds the caller's matches
    ctx->scene.staged = true;
    ctx->scene.thrPx = thr_px;
    return buildCorrespondences(ctx, r, thr_px, ctx->scene.pv.data(), ctx->scene.m.data());
}

pgi_status pgi_register_scene_descriptors(pgi_ctx *ctx, uint64_t n_views, const double *focal, const double *size_wh,
                                          const uint64_t *kp_offset, const float *kp_xy, const float *desc, uint32_t dim,
                                          uint64_t n_pairs, const uint32_t *pair_views, double thr_px, uint64_t *m_offset_out)
{
    PgiNvtxRange nvtxRange("pgi:register_scene_descriptors (H2D + K9 match + K0)");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    if (!focal || !size_wh || !kp_offset || (!kp_xy && kp_offset[n_views]) || (!desc && kp_offset[n_views]) || !pair_views ||
        !m_offset_out) {
        ctx->err = "null argument";
        return PGI_ERR_INVALID;
    }
    if (dim != 128 && dim != 64) { ctx->err = "descriptors must have 64 or 128 dimensions"; return PGI_ERR_INVALID; }
    uint32_t maxK = 0;
    if (kp_offset[0] != 0) { ctx->err = "kp_offset[0] must be 0"; return PGI_ERR_INVALID; }
    for (uint64_t v = 0; v < n_views; v++) {
        if (kp_offset[v + 1] < kp_offset[v]) { ctx->err = "kp_offset is not monotone"; return PGI_ERR_INVALID; }
        const uint64_t k = kp_offset[v + 1] - kp_offset[v];
        if (k > kK9MaxKp) {
            char buf[160];
            snprintf(buf, sizeof buf, "view %llu has %llu keypoints; batched matching supports at most %u per view",
                     (unsigned long long)v, (unsigned long long)k, kK9MaxKp);
            ctx->err = buf;
            return PGI_ERR_INVALID;
        }
        maxK = std::max<uint32_t>(maxK, (uint32_t)k);
    }
    for (uint64_t p = 0; p < n_pairs; p++)
        if (pair_views[2 * p] >= n_views || pair_views[2 * p + 1] >= n_views) { ctx->err = "view id out of range"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->reg = &ctx->own;
    Registration &r = ctx->own;
    SceneStaging &sc = ctx->scene;
    cudaStream_t s = ctx->stream;
    const uint64_t nKp = kp_offset[n_views];
    sc.matches = false;
    CK(r.offset.grow(n_pairs + 1));
    CK(r.thr.grow(n_pairs));
    if (pgi_status st = stageScene(ctx, n_views, focal, size_wh, kp_offset, kp_xy, n_pairs, pair_views); st != PGI_OK) return st;
    CK(cudaMemsetAsync(r.offset.data(), 0, 8, s));
    if (pgi_status st = uploadDescriptors(ctx, desc, nKp, dim); st != PGI_OK) return st;
    MatchRun run;
    if (pgi_status st = matchPairs(ctx, sc, dim, maxK, n_pairs, kp_offset, pair_views, r.offset.data(), run); st != PGI_OK) return st;
    const uint64_t rows = run.rows;
    ctx->stats.ms_match += run.ms;
    ctx->stats.dist_evals += run.dist;
    ctx->stats.match_pairs += n_pairs;
    ctx->stats.match_rows += rows;
    // the offsets are the caller's m_offset and the registration's host copy; the matches stay on the device for K0
    r.nPairs = n_pairs;
    r.nRows = rows;
    r.h_offset.resize(n_pairs + 1);
    CK(cudaMemcpyAsync(r.h_offset.data(), r.offset.data(), (n_pairs + 1) * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += (n_pairs + 1) * 8;
    memcpy(m_offset_out, r.h_offset.data(), (n_pairs + 1) * 8);
    r.maxN = 0;
    for (uint64_t p = 0; p < n_pairs; p++) r.maxN = std::max<uint32_t>(r.maxN, (uint32_t)(r.h_offset[p + 1] - r.h_offset[p]));
    CK(r.corr.grow(rows * 4));
    sc.rows = rows;
    sc.matches = true;
    sc.staged = true;
    sc.thrPx = thr_px;
    return buildCorrespondences(ctx, r, thr_px, ctx->scene.pv.data(), ctx->scene.m.data());
}

pgi_status pgi_read_scene_matches(pgi_ctx *ctx, uint32_t *matches_out, double *ratios_or_null, uint64_t capacity_rows)
{
    if (!ctx) return PGI_ERR_INVALID;
    if (!ctx->scene.matches) { ctx->err = "no descriptor registration to read matches from"; return PGI_ERR_STATE; }
    const uint64_t n = ctx->scene.rows;
    if (capacity_rows < n || (!matches_out && n)) { ctx->err = "capacity too small"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    if (!n) return PGI_OK;
    std::vector<float> r(ratios_or_null ? n : 0);
    CK(cudaMemcpyAsync(matches_out, ctx->scene.m.data(), n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (ratios_or_null) CK(cudaMemcpyAsync(r.data(), ctx->scene.ratio.data(), n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (uint64_t i = 0; i < r.size(); i++) ratios_or_null[i] = (double)r[i];  // feature_utils.h:182: float widened
    ctx->stats.d2h_bytes += n * 8 + r.size() * 4;
    return PGI_OK;
}

pgi_status pgi_share_pairs(pgi_ctx *ctx, pgi_ctx *owner)
{
    if (!ctx || !owner || ctx == owner) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    if (ctx->cfg.device != owner->cfg.device) { ctx->err = "contexts are on different devices"; return PGI_ERR_INVALID; }
    if (ctx->cfg.fallback_max_iters != owner->cfg.fallback_max_iters) { ctx->err = "fallback_max_iters differ"; return PGI_ERR_INVALID; }
    ctx->own = Registration();  // not used while shared; a later pgi_register_* starts it afresh
    ctx->reg = owner->reg;
    return PGI_OK;
}

namespace {
pgi_status readPair(pgi_ctx *ctx, const Registration &r, uint32_t pair_id, double *corr_xy4, uint64_t capacity_rows,
                    uint64_t *n_rows, double *thr_norm)
{
    if (pair_id >= r.nPairs) { ctx->err = "pair_id out of range"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    const uint64_t n = r.h_offset[pair_id + 1] - r.h_offset[pair_id];
    if (n_rows) *n_rows = n;
    if (corr_xy4) {
        if (capacity_rows < n) { ctx->err = "capacity too small"; return PGI_ERR_INVALID; }
        CK(cudaMemcpyAsync(corr_xy4, r.corr.data() + 4 * r.h_offset[pair_id], n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (thr_norm) CK(cudaMemcpyAsync(thr_norm, r.thr.data() + pair_id, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PGI_OK;
}
}  // namespace

pgi_status pgi_read_pair(pgi_ctx *ctx, uint32_t pair_id, double *corr_xy4, uint64_t capacity_rows, uint64_t *n_rows,
                         double *thr_norm)
{
    if (!ctx) return PGI_ERR_INVALID;
    return readPair(ctx, *ctx->reg, pair_id, corr_xy4, capacity_rows, n_rows, thr_norm);
}

pgi_status pgi_read_extra_pair(pgi_ctx *ctx, uint32_t pair_id, double *corr_xy4, uint64_t capacity_rows, uint64_t *n_rows,
                               double *thr_norm)
{
    if (!ctx) return PGI_ERR_INVALID;
    return readPair(ctx, ctx->extra, pair_id, corr_xy4, capacity_rows, n_rows, thr_norm);
}

pgi_status pgi_register_extra_pairs(pgi_ctx *ctx, uint64_t n_pairs, const uint32_t *pair_views, const uint64_t *m_offset,
                                    const uint32_t *matches)
{
    PgiNvtxRange nvtxRange("pgi:register_extra_pairs (H2D + K0)");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    const SceneStaging &sc = ctx->scene;
    if (!sc.staged) { ctx->err = "pgi_register_extra_pairs needs a scene registration first"; return PGI_ERR_STATE; }
    if ((n_pairs && !pair_views) || !m_offset || (!matches && m_offset[n_pairs])) { ctx->err = "null argument"; return PGI_ERR_INVALID; }
    if (m_offset[0] != 0) { ctx->err = "m_offset[0] must be 0"; return PGI_ERR_INVALID; }
    const uint64_t V = sc.hFocal.size();
    for (uint64_t p = 0; p < n_pairs; p++) {
        const uint32_t s = pair_views[2 * p], d = pair_views[2 * p + 1];
        if (s >= V || d >= V) { ctx->err = "view id out of range"; return PGI_ERR_INVALID; }
        if (m_offset[p + 1] < m_offset[p] || m_offset[p + 1] - m_offset[p] > 0x7fffffffULL) { ctx->err = "bad m_offset"; return PGI_ERR_INVALID; }
        // K0 reads the keypoints the indices name: an index past the view's keypoints is rejected here
        const uint64_t nS = sc.hKpOff[s + 1] - sc.hKpOff[s], nD = sc.hKpOff[d + 1] - sc.hKpOff[d];
        for (uint64_t i = m_offset[p]; i < m_offset[p + 1]; i++)
            if (matches[2 * i] >= nS || matches[2 * i + 1] >= nD) { ctx->err = "keypoint index out of range"; return PGI_ERR_INVALID; }
    }
    CK(cudaSetDevice(ctx->cfg.device));
    Registration &r = ctx->extra;
    const uint64_t nRows = m_offset[n_pairs];
    r.nPairs = n_pairs;
    r.nRows = nRows;
    r.h_offset.assign(m_offset, m_offset + n_pairs + 1);
    r.maxN = 0;
    for (uint64_t p = 0; p < n_pairs; p++) r.maxN = std::max<uint32_t>(r.maxN, (uint32_t)(m_offset[p + 1] - m_offset[p]));
    CK(r.corr.grow(nRows * 4));
    CK(r.offset.grow(n_pairs + 1));
    CK(r.thr.grow(n_pairs));
    CK(ctx->extraPv.grow(n_pairs));
    CK(ctx->extraM.grow(nRows));
    cudaStream_t s = ctx->stream;
    if (n_pairs) CK(cudaMemcpyAsync(ctx->extraPv.data(), pair_views, n_pairs * 8, cudaMemcpyHostToDevice, s));
    if (nRows) CK(cudaMemcpyAsync(ctx->extraM.data(), matches, nRows * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(r.offset.data(), m_offset, (n_pairs + 1) * 8, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += n_pairs * 8 + nRows * 8 + (n_pairs + 1) * 8;
    return buildCorrespondences(ctx, r, sc.thrPx, ctx->extraPv.data(), ctx->extraM.data());
}

pgi_status pgi_set_scene_descriptors(pgi_ctx *ctx, const float *desc, uint32_t dim)
{
    PgiNvtxRange nvtxRange("pgi:set_scene_descriptors (H2D)");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    SceneStaging &sc = ctx->scene;
    if (!sc.staged) { ctx->err = "pgi_set_scene_descriptors needs a scene registration first"; return PGI_ERR_STATE; }
    if (dim != 128 && dim != 64) { ctx->err = "descriptors must have 64 or 128 dimensions"; return PGI_ERR_INVALID; }
    const uint64_t nKp = sc.hKpOff.back();
    if (!desc && nKp) { ctx->err = "null argument"; return PGI_ERR_INVALID; }
    for (size_t v = 0; v + 1 < sc.hKpOff.size(); v++)
        if (sc.hKpOff[v + 1] - sc.hKpOff[v] > kK10MaxKp) {
            char buf[160];
            snprintf(buf, sizeof buf, "view %zu has %llu keypoints; guided matching supports at most %u per view", v,
                     (unsigned long long)(sc.hKpOff[v + 1] - sc.hKpOff[v]), kK10MaxKp);
            ctx->err = buf;
            return PGI_ERR_INVALID;
        }
    CK(cudaSetDevice(ctx->cfg.device));
    return uploadDescriptors(ctx, desc, nKp, dim);
}

pgi_status pgi_submit_wave(pgi_ctx *ctx, uint32_t n, const uint32_t *pair_id, const uint32_t *hyp_offset,
                           const double *hyp_q_t, uint32_t flags)
{
    PgiNvtxRange nvtxRange("pgi:submit_wave (H2D hypotheses + K1/K2/K4/K5/K3 launches)");
    if (!ctx) return PGI_ERR_INVALID;
    CK(cudaSetDevice(ctx->cfg.device));
    // PGI_WAVE_EXTRA selects the registration of pgi_register_extra_pairs; the kernels never see the bit
    const Registration &r = (flags & PGI_WAVE_EXTRA) ? ctx->extra : *ctx->reg;
    return submitWave(ctx, r, n, pair_id, hyp_offset, hyp_q_t, flags & ~(uint32_t)PGI_WAVE_EXTRA, nullptr, 0, false);
}

pgi_status pgi_wait_wave(pgi_ctx *ctx, pgi_verdict *out, uint8_t *masks_or_null)
{
    PgiNvtxRange nvtxRange("pgi:wait_wave (sync + D2H verdicts)");
    if (!ctx) return PGI_ERR_INVALID;
    if (!ctx->inFlight) { ctx->err = "no wave in flight"; return PGI_ERR_STATE; }
    WaveEndGuard guard{ctx};
    CK(cudaSetDevice(ctx->cfg.device));
    const uint32_t n = ctx->waveN;
    if (n) {
        if (!out) { ctx->err = "null output"; return PGI_ERR_INVALID; }
        CK(cudaMemcpyAsync(ctx->hostSlots.verdicts.data(), ctx->slots.verdicts.data(), (size_t)n * sizeof(pgi_verdict), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->hCounters.data(), ctx->counters.data(), 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        if (masks_or_null && (ctx->waveFlags & PGI_WAVE_MASKS) && ctx->waveMaskRows)
            CK(cudaMemcpyAsync(masks_or_null, ctx->masks.data(), ctx->waveMaskRows, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        memcpy(out, ctx->hostSlots.verdicts.data(), (size_t)n * sizeof(pgi_verdict));
        ctx->stats.d2h_bytes += (size_t)n * sizeof(pgi_verdict) + 24 + ((masks_or_null && (ctx->waveFlags & PGI_WAVE_MASKS)) ? ctx->waveMaskRows : 0);
    }
    return finishWave(ctx);
}

pgi_status pgi_wait_wave_device(pgi_ctx *ctx, void *verdicts_device)
{
    PgiNvtxRange nvtxRange("pgi:wait_wave_device");
    if (!ctx) return PGI_ERR_INVALID;
    if (!ctx->inFlight) { ctx->err = "no wave in flight"; return PGI_ERR_STATE; }
    WaveEndGuard guard{ctx};
    CK(cudaSetDevice(ctx->cfg.device));
    const uint32_t n = ctx->waveN;
    if (n) {
        if (!verdicts_device) { ctx->err = "null output"; return PGI_ERR_INVALID; }
        CK(cudaMemcpyAsync(verdicts_device, ctx->slots.verdicts.data(), (size_t)n * sizeof(pgi_verdict), cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->hCounters.data(), ctx->counters.data(), 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->stats.d2h_bytes += 24;
    }
    return finishWave(ctx);
}

int32_t pgi_estimate_pose(pgi_ctx *ctx, const double *corr_xy4, uint64_t n, double thr_norm, const double *guesses_q_t,
                          uint32_t n_guesses, double *pose_q_t_out, uint8_t *mask_out, uint64_t *inlier_number_out,
                          pgi_verdict *verdict_or_null)
{
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    if (n > 0x7fffffffULL) { ctx->err = "too many correspondences"; return PGI_ERR_INVALID; }
    if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return PGI_ERR_CUDA;
    const uint64_t off[2] = {0, n};
    pgi_status st = registerDense(ctx, ctx->tmp, 1, off, corr_xy4, &thr_norm);
    if (st != PGI_OK) return st;
    const uint32_t pid = 0, hoff[2] = {0, n_guesses};
    const uint32_t flags = PGI_WAVE_PATH | PGI_WAVE_FALLBACK | PGI_WAVE_NO_TEST | (mask_out ? PGI_WAVE_MASKS : 0u);
    st = submitWave(ctx, ctx->tmp, 1, &pid, hoff, guesses_q_t, flags, nullptr, 0, false);
    if (st != PGI_OK) return st;
    pgi_verdict v;
    st = pgi_wait_wave(ctx, &v, mask_out);
    if (st != PGI_OK) return st;
    if (pose_q_t_out) {
        for (int k = 0; k < 4; k++) pose_q_t_out[k] = v.q[k];
        for (int k = 0; k < 3; k++) pose_q_t_out[4 + k] = v.t[k];
    }
    if (inlier_number_out) *inlier_number_out = v.inlier_count;
    if (verdict_or_null) *verdict_or_null = v;
    return v.accepted ? 1 : 0;
}

int32_t pgi_test_pose(pgi_ctx *ctx, const double *corr_xy4, uint64_t n, double thr, uint64_t min_inliers,
                      const double *pose_q_t, uint64_t *inlier_number_out)
{
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    if (!pose_q_t || n > 0x7fffffffULL || min_inliers == 0 || min_inliers > 0xffffffffULL) { ctx->err = "bad argument"; return PGI_ERR_INVALID; }
    if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return PGI_ERR_CUDA;
    const uint64_t off[2] = {0, n};
    const double thrReg = thr;
    pgi_status st = registerDense(ctx, ctx->tmp, 1, off, corr_xy4, &thrReg);
    if (st != PGI_OK) return st;
    const uint32_t pid = 0, hoff[2] = {0, 1};
    st = submitWave(ctx, ctx->tmp, 1, &pid, hoff, pose_q_t, PGI_WAVE_PATH, &thr, (uint32_t)min_inliers, true);
    if (st != PGI_OK) return st;
    // score-only wave: read the slot state instead of a verdict
    SlotState s;
    CK(cudaMemcpyAsync(&s, ctx->slots.state.data(), sizeof s, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->hCounters.data(), ctx->counters.data(), 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    st = finishWave(ctx);
    if (st != PGI_OK) return st;
    if (inlier_number_out) *inlier_number_out = s.testCount;
    return (s.flags & ST_TEST_PASSED) ? 1 : 0;
}

// ---- K6: device pose graph + batched A* -------------------------------------------------------------------
pgi_status pgi_graph_init(pgi_ctx *ctx, uint32_t n_views, const double *sim_to_next)
{
    if (!ctx) return PGI_ERR_INVALID;
    if (!sim_to_next || n_views == 0 || n_views > 65535u) { ctx->err = "bad graph size (1..65535 views)"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->stream));
    const uint32_t V = n_views;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->cfg.device));
    uint32_t heapCap = 0;
    if (const char *e = getenv("PGI_ASTAR_HEAP")) heapCap = (uint32_t)std::max(1024, atoi(e));
    if (!heapCap) {
        const uint64_t want = (uint64_t)V * V / 2;
        heapCap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(want, 65536), 1u << 20);
    }
    const uint32_t slots = (uint32_t)prop.multiProcessorCount * kAstarSlotsPerSm;
    const uint32_t arenaCap = 16384;
    if (ctx->graph.V != V || ctx->graph.heapCap != heapCap || ctx->graph.slots != slots) {
        // the old graph is released first; the new one only replaces it once every allocation succeeded
        ctx->graph = Graph();
        Graph g;
        CK(g.adj.grow((size_t)V * V));
        CK(g.counts.grow((size_t)2 * V));
        CK(g.simT.grow((size_t)V * V));
        CK(g.heaps.grow((size_t)slots * heapCap));
        CK(g.arenas.grow((size_t)slots * arenaCap));
        CK(g.nextQuery.grow(1));
        CK(g.hCounts.grow((size_t)2 * V));
        g.V = V; g.cap = V; g.words = (V + 31) / 32;
        g.heapCap = heapCap; g.arenaCap = arenaCap; g.slots = slots;
        ctx->graph = std::move(g);
    }
    CK(cudaMemsetAsync(ctx->graph.counts.data(), 0, (size_t)2 * V * 4, ctx->stream));
    CK(cudaMemcpyAsync(ctx->graph.simT.data(), sim_to_next, (size_t)V * V * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->sstats.h2d_bytes += (uint64_t)V * V * 8;
    if (!ctx->evS0) CK(cudaEventCreate(&ctx->evS0.h));
    if (!ctx->evS1) CK(cudaEventCreate(&ctx->evS1.h));
    return PGI_OK;
}

pgi_status pgi_graph_apply(pgi_ctx *ctx, uint32_t n_entries, const pgi_adj_entry *entries, const uint32_t *committed_count,
                           const uint32_t *total_count)
{
    if (!ctx) return PGI_ERR_INVALID;
    Graph &g = ctx->graph;
    if (!g.V) { ctx->err = "pgi_graph_init has not been called"; return PGI_ERR_STATE; }
    if ((n_entries && !entries) || !committed_count || !total_count) { ctx->err = "null argument"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    const uint32_t V = g.V;
    for (uint32_t v = 0; v < V; v++)
        if (total_count[v] < committed_count[v] || total_count[v] > g.cap) { ctx->err = "bad edge-list count"; return PGI_ERR_INVALID; }
    for (uint32_t i = 0; i < n_entries; i++)
        if (entries[i].vertex >= V || entries[i].next >= V || entries[i].index >= g.cap) { ctx->err = "edge-list entry out of range"; return PGI_ERR_INVALID; }
    if (n_entries > g.apply.cap) {
        const uint32_t cap = std::max<uint32_t>(n_entries * 2, 4096);
        g.apply = {};
        CK(g.apply.host.grow(cap));
        CK(g.apply.dev.grow(cap));
        g.apply.cap = cap;
    }
    static_assert(sizeof(ApplyEntry) == sizeof(pgi_adj_entry), "apply entry layout");
    cudaStream_t s = ctx->stream;
    memcpy(g.hCounts.data(), committed_count, (size_t)V * 4);
    memcpy(g.hCounts.data() + V, total_count, (size_t)V * 4);
    CK(cudaMemcpyAsync(g.counts.data(), g.hCounts.data(), (size_t)2 * V * 4, cudaMemcpyHostToDevice, s));
    if (n_entries) {
        memcpy(g.apply.host.data(), entries, (size_t)n_entries * sizeof(ApplyEntry));
        CK(cudaMemcpyAsync(g.apply.dev.data(), g.apply.host.data(), (size_t)n_entries * sizeof(ApplyEntry), cudaMemcpyHostToDevice, s));
        k6_graph_apply<<<(n_entries + 255) / 256, 256, 0, s>>>(g.adj.data(), g.cap, g.apply.dev.data(), n_entries);
        CK(cudaGetLastError());
        ctx->sstats.launches += 1;
    }
    CK(cudaStreamSynchronize(s));  // the pinned staging buffers are reused by the next call
    ctx->sstats.h2d_bytes += (uint64_t)2 * V * 4 + (uint64_t)n_entries * sizeof(ApplyEntry);
    return PGI_OK;
}

pgi_status pgi_graph_search(pgi_ctx *ctx, uint32_t n, const pgi_query *queries, uint32_t max_depth, double weight,
                            pgi_search_result *results, uint32_t *expanded_bits)
{
    PgiNvtxRange nvtxRange("pgi:graph_search (K6)");
    if (!ctx) return PGI_ERR_INVALID;
    Graph &g = ctx->graph;
    if (!g.V) { ctx->err = "pgi_graph_init has not been called"; return PGI_ERR_STATE; }
    if (n == 0) return PGI_OK;
    if (!queries || !results || !expanded_bits || max_depth > 7) { ctx->err = "bad argument"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    const uint32_t V = g.V, words = g.words;
    for (uint32_t i = 0; i < n; i++)
        if (queries[i].src >= V || queries[i].dst >= V) { ctx->err = "query vertex out of range"; return PGI_ERR_INVALID; }
    auto &q = g.search;
    if (n > q.cap) {
        const uint32_t cap = std::max<uint32_t>(n, 4096);
        q = {};
        CK(q.queries.grow(cap));
        CK(q.results.grow(cap));
        CK(q.expBits.grow((size_t)cap * words));
        CK(q.hQueries.grow(cap));
        CK(q.hResults.grow(cap));
        CK(q.hExpBits.grow((size_t)cap * words));
        q.cap = cap;
    }
    cudaStream_t s = ctx->stream;
    memcpy(q.hQueries.data(), queries, (size_t)n * sizeof(pgi_query));
    CK(cudaMemcpyAsync(q.queries.data(), q.hQueries.data(), (size_t)n * sizeof(pgi_query), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(g.nextQuery.data(), 0, 4, s));
    SearchArgs a;
    a.adj = g.adj.data(); a.cap = g.cap; a.ccnt = g.counts.data(); a.cnt = g.counts.data() + V; a.simT = g.simT.data();
    a.V = V; a.words = words; a.n = n; a.queries = q.queries.data(); a.maxDepth = max_depth;
    a.weight = weight; a.oneMinusWeight = 1.0 - weight;
    a.heaps = g.heaps.data(); a.heapCap = g.heapCap; a.arenas = g.arenas.data(); a.arenaCap = g.arenaCap;
    a.results = q.results.data(); a.expandedBits = q.expBits.data(); a.nextQuery = g.nextQuery.data();
    const uint32_t ctas = std::min<uint32_t>((n + kAstarWarps - 1) / kAstarWarps, g.slots / kAstarWarps);
    const size_t smem = (size_t)kAstarWarps * ((size_t)kStageItems * sizeof(HeapItemDev) + (size_t)kChunk * 2 + (size_t)2 * words * 4);
    CK(cudaFuncSetAttribute(k6_astar_search, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
    CK(cudaEventRecord(ctx->evS0, s));
    k6_astar_search<<<ctas, kAstarWarps * 32, smem, s>>>(a);
    CK(cudaEventRecord(ctx->evS1, s));
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(q.hResults.data(), q.results.data(), (size_t)n * sizeof(pgi_search_result), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(q.hExpBits.data(), q.expBits.data(), (size_t)n * words * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memcpy(results, q.hResults.data(), (size_t)n * sizeof(pgi_search_result));
    memcpy(expanded_bits, q.hExpBits.data(), (size_t)n * words * 4);
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->evS0, ctx->evS1));
    pgi_search_stats &st = ctx->sstats;
    st.ms_search += ms;
    st.launches += 1;
    st.queries += n;
    uint32_t longest = 0;
    for (uint32_t i = 0; i < n; i++) {
        st.pops += results[i].touched;
        st.pushes += results[i].pushes;
        st.overflows += results[i].status != 0;
        st.kcycles_sum += results[i].kcycles;
        longest = std::max(longest, results[i].kcycles);
    }
    st.kcycles_longest += longest;
    st.h2d_bytes += (uint64_t)n * sizeof(pgi_query);
    st.d2h_bytes += (uint64_t)n * (sizeof(pgi_search_result) + (uint64_t)words * 4);
    return PGI_OK;
}

pgi_status pgi_graph_stats(pgi_ctx *ctx, pgi_search_stats *out, int32_t reset)
{
    if (!ctx) return PGI_ERR_INVALID;
    if (out) *out = ctx->sstats;
    if (reset) memset(&ctx->sstats, 0, sizeof ctx->sstats);
    return PGI_OK;
}

pgi_status pgi_guided_match(pgi_ctx *ctx, uint32_t n_src, const float *kp_src, const float *desc_src, uint32_t n_dst,
                            const float *kp_dst, const float *desc_dst, uint32_t dim, const double *pose_q_t,
                            const double *K_src, const double *K_dst, const int32_t *size_src, const int32_t *size_dst,
                            int32_t bin_number, uint32_t *matches_out, double *ratios_out, uint32_t *n_out,
                            double *prepared_or_null)
{
    PgiNvtxRange nvtxRange("pgi:guided_match (K10 on one pair)");
    if (!ctx) return PGI_ERR_INVALID;
    if (!pose_q_t || !K_src || !K_dst || !size_src || !size_dst || !n_out || (n_src && (!kp_src || !desc_src || !matches_out || !ratios_out)) ||
        (n_dst && (!kp_dst || !desc_dst)) || bin_number > kMatchMaxBins) {
        ctx->err = "bad argument";
        return PGI_ERR_INVALID;
    }
    if (dim != 128 && dim != 64) { ctx->err = "descriptors must have 64 or 128 dimensions"; return PGI_ERR_INVALID; }
    CK(cudaSetDevice(ctx->cfg.device));
    *n_out = 0;
    if (n_src == 0 || n_dst == 0) return PGI_OK;
    // the pair as a scene of two views: [desc_src; desc_dst], then [kp_src; kp_dst] (256-byte aligned: dim * 4 is)
    cudaStream_t s = ctx->stream;
    const size_t nKp = (size_t)n_src + n_dst, oKp = nKp * dim * 4;
    DevBuf<unsigned char> staged;
    CK(staged.grow(oKp + nKp * 8));
    unsigned char *d = staged.data();
    CK(cudaMemcpyAsync(d, desc_src, (size_t)n_src * dim * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d + (size_t)n_src * dim * 4, desc_dst, (size_t)n_dst * dim * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d + oKp, kp_src, (size_t)n_src * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d + oKp + (size_t)n_src * 8, kp_dst, (size_t)n_dst * 8, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += nKp * (8 + dim * 4);
    GuidedPairIn in;
    memset(&in, 0, sizeof in);
    essentialOfPose(pose_q_t, in.E);
    memcpy(in.Ks, K_src, sizeof in.Ks);
    memcpy(in.Kd, K_dst, sizeof in.Kd);
    in.wS = size_src[0]; in.hS = size_src[1]; in.wD = size_dst[0]; in.hD = size_dst[1]; in.binNumber = bin_number;
    in.kS0 = 0; in.kD0 = n_src;
    in.nS = n_src; in.nD = n_dst;
    uint64_t off[2];
    GuidedPrep prep;
    MatchRun run;
    if (pgi_status st = runGuided(ctx, reinterpret_cast<const float2 *>(d + oKp), reinterpret_cast<const float *>(d), dim, &in, 1, 0,
                                  off, matches_out, ratios_out, n_src, &prep, run);
        st != PGI_OK)
        return st;
    ctx->stats.ms_guided += run.ms;
    ctx->stats.guided_calls += 1;
    *n_out = (uint32_t)off[1];
    if (prepared_or_null) {
        for (int k = 0; k < 9; k++) prepared_or_null[k] = prep.F[k];
        prepared_or_null[9] = prep.ex; prepared_or_null[10] = prep.ey; prepared_or_null[11] = prep.minAngle;
        prepared_or_null[12] = prep.range; prepared_or_null[13] = prep.binsRaw;
    }
    return PGI_OK;
}

pgi_status pgi_guided_match_views(pgi_ctx *ctx, uint32_t src, uint32_t dst, const double *pose_q_t, int32_t bin_number,
                                  uint32_t max_points, uint32_t *matches_out, double *values_out, uint32_t *n_out)
{
    PgiNvtxRange nvtxRange("pgi:guided_match_views (K10 on one pair of the resident scene)");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    const SceneStaging &sc = ctx->scene;
    if (!sc.staged) { ctx->err = "pgi_guided_match_views needs a scene registration first"; return PGI_ERR_STATE; }
    if (!sc.hasDesc) {
        ctx->err = "the registered scene has no descriptors (pgi_register_scene_descriptors or pgi_set_scene_descriptors)";
        return PGI_ERR_STATE;
    }
    const uint64_t V = sc.hFocal.size();
    if (src >= V || dst >= V) { ctx->err = "view id out of range"; return PGI_ERR_INVALID; }
    if (!pose_q_t || !n_out || (max_points && (!matches_out || !values_out)) || bin_number > kMatchMaxBins) {
        ctx->err = "bad argument";
        return PGI_ERR_INVALID;
    }
    CK(cudaSetDevice(ctx->cfg.device));
    *n_out = 0;
    const GuidedPairIn in = scenePairIn(sc, src, dst, pose_q_t, bin_number);
    if (in.nS == 0 || in.nD == 0 || max_points == 0) return PGI_OK;
    uint64_t off[2];
    MatchRun run;
    if (pgi_status st = runGuided(ctx, sc.kp.data(), sc.desc.data(), sc.dim, &in, 1, max_points, off, matches_out, values_out,
                                  std::min(in.nS, max_points), nullptr, run);
        st != PGI_OK)
        return st;
    ctx->stats.ms_guided += run.ms;
    ctx->stats.guided_calls += 1;
    *n_out = (uint32_t)off[1];
    return PGI_OK;
}

pgi_status pgi_guided_match_pairs(pgi_ctx *ctx, uint64_t n_pairs, const uint32_t *pair_views, const double *poses_q_t,
                                  int32_t bin_number, uint32_t max_points, uint64_t *offsets_out,
                                  uint32_t *matches_out, double *values_out, uint64_t capacity_rows)
{
    PgiNvtxRange nvtxRange("pgi:guided_match_pairs (K10 on the resident scene)");
    if (!ctx) return PGI_ERR_INVALID;
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    const SceneStaging &sc = ctx->scene;
    if (!sc.staged) { ctx->err = "pgi_guided_match_pairs needs a scene registration first"; return PGI_ERR_STATE; }
    if (!sc.hasDesc) {
        ctx->err = "the registered scene has no descriptors (pgi_register_scene_descriptors or pgi_set_scene_descriptors)";
        return PGI_ERR_STATE;
    }
    if (!offsets_out || (n_pairs && (!pair_views || !poses_q_t)) || bin_number > kMatchMaxBins) {
        ctx->err = "bad argument";
        return PGI_ERR_INVALID;
    }
    const uint64_t V = sc.hFocal.size();
    std::vector<GuidedPairIn> &in = ctx->guidedIn;
    in.resize(n_pairs);
    for (uint64_t p = 0; p < n_pairs; p++) {
        const uint32_t src = pair_views[2 * p], dst = pair_views[2 * p + 1];
        if (src >= V || dst >= V) { ctx->err = "view id out of range"; return PGI_ERR_INVALID; }
        in[p] = scenePairIn(sc, src, dst, poses_q_t + 7 * p, bin_number);
    }
    MatchRun run;
    if (pgi_status st = runGuided(ctx, sc.kp.data(), sc.desc.data(), sc.dim, in.data(), n_pairs, max_points, offsets_out, matches_out,
                                  values_out, capacity_rows, nullptr, run);
        st != PGI_OK)
        return st;
    ctx->stats.ms_guided_pairs += run.ms;
    ctx->stats.guided_pairs += n_pairs;
    ctx->stats.guided_dist_evals += run.dist;
    ctx->stats.guided_chunks += run.chunks;
    return PGI_OK;
}

pgi_status pgi_match_features(pgi_ctx *ctx, uint32_t n_src, const float *desc_src, uint32_t n_dst, const float *desc_dst,
                              uint32_t dim, uint32_t *matches_out, double *ratios_out, uint32_t *n_out)
{
    PgiNvtxRange nvtxRange("pgi:match_features (K9 on one pair)");
    if (!ctx) return PGI_ERR_INVALID;
    // the finite check's flag word and K9's timing events are the ones a wave in flight reads back
    if (ctx->inFlight) { ctx->err = "a wave is in flight"; return PGI_ERR_STATE; }
    if (!n_out || (n_src && (!desc_src || !matches_out || !ratios_out)) || (n_dst && !desc_dst) || (dim != 128 && dim != 64)) {
        ctx->err = "bad argument (descriptors must have 64 or 128 dimensions)";
        return PGI_ERR_INVALID;
    }
    if (n_src > kK9MaxKp || n_dst > kK9MaxKp) {
        ctx->err = "descriptor matching supports at most 16384 descriptors per side";
        return PGI_ERR_INVALID;
    }
    CK(cudaSetDevice(ctx->cfg.device));
    *n_out = 0;
    if (n_src == 0 || n_dst == 0) return PGI_OK;
    // the pair as a scene of two views, staged apart from the registered scene: [desc_src; desc_dst], pair (0, 1)
    MatchStaging &st = ctx->pairMatch;
    cudaStream_t s = ctx->stream;
    const uint64_t kpOff[3] = {0, n_src, (uint64_t)n_src + n_dst};
    const uint32_t pv[2] = {0, 1};
    CK(st.desc.grow(kpOff[2] * dim));
    CK(cudaMemcpyAsync(st.desc.data(), desc_src, (size_t)n_src * dim * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(st.desc.data() + (size_t)n_src * dim, desc_dst, (size_t)n_dst * dim * 4, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += kpOff[2] * dim * 4;
    if (pgi_status e = checkFinite(ctx, st.desc.data(), kpOff[2] * dim); e != PGI_OK) return e;
    CK(st.kpOff.grow(3));
    CK(st.pv.grow(1));
    CK(ctx->pairMatchOff.grow(2));
    CK(cudaMemcpyAsync(st.kpOff.data(), kpOff, sizeof kpOff, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(st.pv.data(), pv, sizeof pv, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(ctx->pairMatchOff.data(), 0, 8, s));
    ctx->stats.h2d_bytes += sizeof kpOff + sizeof pv;
    MatchRun run;
    if (pgi_status e = matchPairs(ctx, st, dim, std::max(n_src, n_dst), 1, kpOff, pv, ctx->pairMatchOff.data(), run); e != PGI_OK)
        return e;
    const uint32_t n = (uint32_t)run.rows;
    std::vector<float> r(n);
    if (n) {
        CK(cudaMemcpyAsync(matches_out, st.m.data(), (size_t)n * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(r.data(), st.ratio.data(), (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    for (uint32_t i = 0; i < n; i++) ratios_out[i] = (double)r[i];  // feature_utils.h:182: float widened
    *n_out = n;
    ctx->stats.d2h_bytes += (size_t)n * 12;
    return PGI_OK;
}

pgi_status pgi_get_stats(pgi_ctx *ctx, pgi_stats *out)
{
    if (!ctx || !out) return PGI_ERR_INVALID;
    *out = ctx->stats;
    return PGI_OK;
}

pgi_status pgi_reset_stats(pgi_ctx *ctx)
{
    if (!ctx) return PGI_ERR_INVALID;
    memset(&ctx->stats, 0, sizeof ctx->stats);
    return PGI_OK;
}

// ---- unit-level device entry points for the parity tests -----------------------------------------
namespace {
__global__ void kdbg_sampson(const double4 *rows, uint64_t n, const double *E9, double *out)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double E[9];
    for (int k = 0; k < 9; k++) E[k] = E9[k];
    const double4 c = rows[i];
    out[i] = sampsonSq(c.x, c.y, c.z, c.w, E);
}
__global__ void kdbg_five_point(const double *x1, const double *x2, uint32_t n, int dkMaxIters, double dkTolSq, double *Eout,
                                int *count)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double a[10], b[10];
    for (int k = 0; k < 10; k++) { a[k] = x1[10 * (size_t)i + k]; b[k] = x2[10 * (size_t)i + k]; }
    // 1000 sweeps (with or without a tolerance) = K2's configuration: the exact cycle jump; fewer sweeps = K4's plain loop
    count[i] = dkMaxIters >= 1000 ? fivePoint<true>(a, b, Eout + 90 * (size_t)i, 10, dkMaxIters, dkTolSq)
                                  : fivePoint<false>(a, b, Eout + 90 * (size_t)i, 10, dkMaxIters, dkTolSq);
}
}  // namespace

pgi_status pgi_dbg_sampson(pgi_ctx *ctx, const double *corr_xy4, uint64_t n, const double *E, double *out)
{
    if (!ctx || !corr_xy4 || !E || !out) return PGI_ERR_INVALID;
    CK(cudaSetDevice(ctx->cfg.device));
    DevBuf<double4> d_c;
    DevBuf<double> d_E, d_o;
    CK(d_c.grow(n));
    CK(d_E.grow(9));
    CK(d_o.grow(n));
    CK(cudaMemcpy(d_c.data(), corr_xy4, n * 32, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_E.data(), E, 72, cudaMemcpyHostToDevice));
    if (n) kdbg_sampson<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_c.data(), n, d_E.data(), d_o.data());
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(out, d_o.data(), n * 8, cudaMemcpyDeviceToHost));
    ctx->stats.launches += 1;
    return PGI_OK;
}

pgi_status pgi_dbg_five_point(pgi_ctx *ctx, const double *x1, const double *x2, uint32_t n_problems, int32_t dk_max_iters,
                              double dk_tol_sq, double *E_out, int32_t *count_out)
{
    if (!ctx || !x1 || !x2 || !E_out || !count_out) return PGI_ERR_INVALID;
    CK(cudaSetDevice(ctx->cfg.device));
    DevBuf<double> d_a, d_b, d_E;
    DevBuf<int> d_c;
    const size_t n = std::max<uint32_t>(n_problems, 1);
    CK(d_a.grow(n * 10));
    CK(d_b.grow(n * 10));
    CK(d_E.grow(n * 90));
    CK(d_c.grow(n));
    CK(cudaMemset(d_E.data(), 0, n * 720));
    CK(cudaMemcpy(d_a.data(), x1, (size_t)n_problems * 80, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_b.data(), x2, (size_t)n_problems * 80, cudaMemcpyHostToDevice));
    if (n_problems) kdbg_five_point<<<(n_problems + 63) / 64, 64, 0, ctx->stream>>>(d_a.data(), d_b.data(), n_problems, dk_max_iters, dk_tol_sq, d_E.data(), d_c.data());
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    CK(cudaMemcpy(E_out, d_E.data(), (size_t)n_problems * 720, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(count_out, d_c.data(), (size_t)n_problems * 4, cudaMemcpyDeviceToHost));
    ctx->stats.launches += 1;
    return PGI_OK;
}

pgi_status pgi_dbg_pose_from_essential(pgi_ctx *ctx, const double *E, const double *corr_xy4, uint64_t n, double *R,
                                       double *t, uint64_t *votes)
{
    if (!ctx || !E || !corr_xy4 || !R || !t || !votes || n > 0x7fffffffULL) return PGI_ERR_INVALID;
    CK(cudaSetDevice(ctx->cfg.device));
    DevBuf<double4> d_c;
    DevBuf<double> d_E, d_R, d_t;
    DevBuf<unsigned long long> d_v;
    CK(d_c.grow(n));
    CK(d_E.grow(9));
    CK(d_R.grow(9));
    CK(d_t.grow(3));
    CK(d_v.grow(4));
    CK(cudaMemcpy(d_c.data(), corr_xy4, n * 32, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_E.data(), E, 72, cudaMemcpyHostToDevice));
    kdbg_pose_from_essential<<<1, kCtaThreads, 0, ctx->stream>>>(d_E.data(), d_c.data(), (uint32_t)n, d_R.data(), d_t.data(), d_v.data());
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    unsigned long long hv[4];
    CK(cudaMemcpy(R, d_R.data(), 72, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(t, d_t.data(), 24, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hv, d_v.data(), 32, cudaMemcpyDeviceToHost));
    for (int k = 0; k < 4; k++) votes[k] = hv[k];
    ctx->stats.launches += 1;
    return PGI_OK;
}

pgi_status pgi_dbg_fp64_peak(pgi_ctx *ctx, int32_t fused, double *tflops_out)
{
    if (!ctx || !tflops_out) return PGI_ERR_INVALID;
    CK(cudaSetDevice(ctx->cfg.device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->cfg.device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 14;
    DevBuf<double> d;
    CK(d.grow((size_t)blocks * threads));
    k_fp64_peak<<<blocks, threads, 0, ctx->stream>>>(d.data(), 64, fused);  // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CK(cudaEventRecord(ctx->evStart, ctx->stream));
        k_fp64_peak<<<blocks, threads, 0, ctx->stream>>>(d.data(), iters, fused);
        CK(cudaEventRecord(ctx->evK1, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evK1));
        const double flops = (double)blocks * threads * iters * 8.0 * 2.0;  // 8 chains x (mul + add)
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    ctx->stats.launches += 6;
    *tflops_out = best;
    return PGI_OK;
}

}  // extern "C"
