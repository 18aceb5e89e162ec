// ORACLE — TEST INFRASTRUCTURE ONLY (see pgo_geom.hpp header).
// extern "C" surface of pgo_hashing.hpp, loaded through ctypes by oracle/pgo_hashing.py.  Never linked into the product.
#include <cstdint>
#include <cstring>

#include "pgo_hashing.hpp"

using namespace pgo;

extern "C" {

// The hashing run over the compact scene (the container of SURVEY App. D plus desc[sum K x dim]).  Returns a handle.
void *pgo_run_scene_hashing(uint64_t V, const double *focal, const double *size, const double *sim, const uint64_t *kpOffset,
                            const float *kp, const float *desc, int dim, uint64_t P, const uint32_t *pairViews,
                            const uint64_t *mOffset, const uint32_t *matches, double simThreshold, double thrPx,
                            uint64_t minInliers, uint64_t minPoints, uint64_t maxDepth, double weight, int usePathFinding,
                            uint64_t maxTracklets, uint64_t maxPointsHashing, int binNumber)
{
    host::Scene sc;
    sc.V = V; sc.focal = focal; sc.size = size; sc.sim = sim; sc.kpOffset = kpOffset; sc.kp = kp;
    sc.P = P; sc.pairViews = pairViews; sc.mOffset = mOffset; sc.matches = matches;
    host::Config cfg;
    cfg.similarityThreshold = simThreshold; cfg.inlierOutlierThreshold = thrPx; cfg.minimumInlierNumber = minInliers;
    cfg.minimumPointNumber = minPoints; cfg.maximumSearchDepth = maxDepth; cfg.traversalHeuristicsWeight = weight;
    cfg.usePathFinding = usePathFinding != 0;
    host::HashingConfig hc;
    hc.maximumTrackletNumber = maxTracklets; hc.maximumPointNumberForEpipolarHashing = maxPointsHashing; hc.binNumber = binNumber;
    return new host::HashingResult(host::runHashing(sc, desc, dim, cfg, hc));
}
uint64_t pgo_hashing_pairlog_size() { return sizeof(host::PairLog); }
uint64_t pgo_hashing_log_count(void *h) { return ((host::HashingResult *)h)->run.log.size(); }
uint64_t pgo_hashing_edge_count(void *h) { return ((host::HashingResult *)h)->run.edges.size(); }
// log[n], source[n], guided[n]; edges: src[e], dst[e], out[e x 8] = {qx, qy, qz, qw, tx, ty, tz, score}
void pgo_hashing_copy(void *h, void *log, uint8_t *source, uint32_t *guided, uint32_t *src, uint32_t *dst, double *out)
{
    const host::HashingResult &r = *(host::HashingResult *)h;
    std::memcpy(log, r.run.log.data(), r.run.log.size() * sizeof(host::PairLog));
    std::memcpy(source, r.matchSource.data(), r.matchSource.size());
    std::memcpy(guided, r.guidedRows.data(), r.guidedRows.size() * sizeof(uint32_t));
    for (size_t i = 0; i < r.run.edges.size(); i++) {
        const host::Edge &e = r.run.edges[i];
        src[i] = (uint32_t)e.src; dst[i] = (uint32_t)e.dst;
        const SE3 &T = e.T;
        out[8 * i] = T.q.x; out[8 * i + 1] = T.q.y; out[8 * i + 2] = T.q.z; out[8 * i + 3] = T.q.w;
        out[8 * i + 4] = T.t.x; out[8 * i + 5] = T.t.y; out[8 * i + 6] = T.t.z; out[8 * i + 7] = e.score;
    }
}
void pgo_hashing_free(void *h) { delete (host::HashingResult *)h; }

}  // extern "C"
