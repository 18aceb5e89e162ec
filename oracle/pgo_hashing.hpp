// ORACLE — TEST INFRASTRUCTURE ONLY (see pgo_geom.hpp header).
//
// pgo_hashing.hpp — processImages (pose_graph_builder.h:352-715) with the epipolar-hashing branch, sequential
// (core_number = 1): pgo_host.hpp's run() plus quick matching from the tracklets (:492-520), the matchFeatures list as the
// alternative (:522-547) and the tracklet updates after an accepted pair (:657-707).  Built from pgo_host.hpp's PoseGraph,
// VisibilityTable, aStar and queue, pgo_matcher.hpp's guided matcher and pgo_tracklets.hpp; with no tracklet ever
// returning kMinimumPointNumber_ rows it commits what run() commits.  Parity unpinned (DESIGN.md §7a gives the reading).
#pragma once
#include <algorithm>
#include <cstdint>
#include <map>
#include <tuple>
#include <utility>
#include <vector>

#include "pgo_host.hpp"
#include "pgo_matcher.hpp"
#include "pgo_tracklets.hpp"

namespace pgo {
namespace host {

struct HashingConfig {
    size_t maximumTrackletNumber = 5000;                // maximum_tracklet_number
    size_t maximumPointNumberForEpipolarHashing = 100;  // maximum_point_number_for_epipolar_hashing
    int binNumber = 45;                                 // HashingBasedMatcherWithPose<false, 45>
};

struct HashingResult {
    RunResult run;
    // per log record: 0 skipped, 1 quick-matched from the tracklets, 2 matchFeatures' list; rows guidedMatching added
    std::vector<uint8_t> matchSource;
    std::vector<uint32_t> guidedRows;
};

// desc: sum K x dim descriptors, row-aligned with sc.kp.
inline HashingResult runHashing(const Scene &sc, const float *desc, int dim, const Config &cfg, const HashingConfig &hc)
{
    HashingResult res;
    RunResult &out = res.run;
    PoseGraph graph;
    VisibilityTable vis;
    Tracklets tracklets;
    auto queue = buildPairQueue(sc, cfg.similarityThreshold);
    std::map<std::pair<uint32_t, uint32_t>, size_t> pairIndex;
    for (size_t p = 0; p < sc.P; p++) pairIndex[{sc.pairViews[2 * p], sc.pairViews[2 * p + 1]}] = p;
    std::vector<double> corr;
    std::vector<uint8_t> mask;
    std::vector<uint32_t> quick;
    while (!queue.empty()) {
        const auto vp = queue.top();
        queue.pop();
        const ViewId src = std::get<1>(vp), dst = std::get<2>(vp);
        PairLog lg{};
        lg.src = (uint32_t)src; lg.dst = (uint32_t)dst; lg.pairIndex = -1;
        uint8_t source = 0;
        uint32_t guided = 0;
        auto logPair = [&]() {
            out.log.push_back(lg);
            res.matchSource.push_back(source);
            res.guidedRows.push_back(guided);
        };
        if (graph.hasEdge(src, dst) || graph.hasEdge(dst, src)) {  // :438-443
            out.skipped++;
            logPair();
            continue;
        }
        const bool visible = vis.hasLink(src, dst);  // :456-457
        lg.visible = visible;
        size_t n = 0;
        const uint32_t *rows = nullptr;  // the chosen matches: the quick matches or matchFeatures' list
        const auto q = tracklets.getCorrespondences(src, dst, hc.maximumTrackletNumber);  // :492-520
        const bool quickMatched = q.size() >= cfg.minimumPointNumber;
        if (quickMatched) {
            quick.resize(2 * q.size());
            for (size_t i = 0; i < q.size(); i++) {
                quick[2 * i] = (uint32_t)std::get<0>(q[i]);
                quick[2 * i + 1] = (uint32_t)std::get<1>(q[i]);
            }
            n = q.size();
            rows = quick.data();
        }
        auto pit = pairIndex.find({(uint32_t)src, (uint32_t)dst});
        if (pit != pairIndex.end()) {
            const size_t p = pit->second;
            lg.pairIndex = (int64_t)p;
            if (!quickMatched) {  // matchFeatures (:522-547)
                n = (size_t)(sc.mOffset[p + 1] - sc.mOffset[p]);
                rows = sc.matches + 2 * sc.mOffset[p];
            }
        }
        lg.nCorr = (uint32_t)n;
        if (n < cfg.minimumPointNumber) {  // :550-551
            out.skipped++;
            logPair();
            continue;
        }
        source = quickMatched ? 1 : 2;
        corr.resize(n * 4);
        double thrNorm = 0.0;
        const double f = sc.focal[src], cx = sc.size[2 * src] / 2.0, cy = sc.size[2 * src + 1] / 2.0;  // :284-286
        createCorrespondenceMatrix(sc.kp + 2 * sc.kpOffset[src], sc.kp + 2 * sc.kpOffset[dst], rows, n, f, f, cx, cy,
                                   cfg.inlierOutlierThreshold, corr.data(), thrNorm);
        std::vector<SE3> poses;
        if (cfg.usePathFinding && visible) {  // :569-603
            AStarResult ar = aStar(graph, sc, src, dst, cfg.maximumSearchDepth, cfg.traversalHeuristicsWeight);
            lg.touchedNodes = (uint32_t)ar.touchedNodes;
            lg.hadPath = ar.pathFound;
            if (ar.pathFound) {
                size_t cnt = 0;
                const bool ok = inTraversalTest(corr.data(), n, ar.pose, 1.5 * thrNorm, 5, cnt);  // :798-811, GT:790
                lg.testPassed = ok;
                lg.testCount = (uint32_t)cnt;
                if (ok) poses.push_back(ar.pose);
            }
        }
        mask.clear();
        EstimateResult er = estimatePose(corr.data(), n, thrNorm, cfg.minimumInlierNumber, poses.data(), poses.size(), mask);
        lg.branch = (uint8_t)er.branch;
        lg.inlierNumber = (uint32_t)er.inlierNumber;
        for (int k = 0; k < 9; k++) lg.E[k] = er.E[k];
        if (!er.success) {  // :641-642
            out.rejected++;
            logPair();
            continue;
        }
        const double ratio = (double)er.inlierNumber / (double)n;  // :645-646
        Edge e{src, dst, er.pose, ratio};
        graph.addEdge(src, dst, e);  // :649-654
        vis.addLink(src, dst);       // :692
        out.edges.push_back(e);
        lg.committed = 1;
        lg.q[0] = er.pose.q.x; lg.q[1] = er.pose.q.y; lg.q[2] = er.pose.q.z; lg.q[3] = er.pose.q.w;
        lg.t[0] = er.pose.t.x; lg.t[1] = er.pose.t.y; lg.t[2] = er.pose.t.z;
        lg.score = ratio;
        if (er.branch == 1) out.pathAccepted++; else out.fallbackAccepted++;
        std::vector<std::pair<size_t, size_t>> add;
        std::vector<uint8_t> addMask;
        if (quickMatched) {  // guidedMatching with the committed pose, every selected row an inlier (:663-676, :717-783)
            const double fd = sc.focal[dst];
            const double Ks[9] = {f, 0.0, sc.size[2 * src] / 2.0, 0.0, f, sc.size[2 * src + 1] / 2.0, 0.0, 0.0, 1.0};
            const double Kd[9] = {fd, 0.0, sc.size[2 * dst] / 2.0, 0.0, fd, sc.size[2 * dst + 1] / 2.0, 0.0, 0.0, 1.0};
            double E[9];
            essentialFromPose(er.pose, E);
            const matcher::Prepared P = matcher::prepare(E, Ks, Kd, (int)sc.size[2 * src], (int)sc.size[2 * src + 1],
                                                         (int)sc.size[2 * dst], (int)sc.size[2 * dst + 1], hc.binNumber);
            std::vector<std::pair<uint32_t, uint32_t>> gm;
            std::vector<double> gr;
            matcher::match(sc.kp + 2 * sc.kpOffset[src], (size_t)(sc.kpOffset[src + 1] - sc.kpOffset[src]),
                           desc + (size_t)dim * sc.kpOffset[src], sc.kp + 2 * sc.kpOffset[dst],
                           (size_t)(sc.kpOffset[dst + 1] - sc.kpOffset[dst]), desc + (size_t)dim * sc.kpOffset[dst], dim, P, gm, gr);
            std::vector<std::tuple<uint32_t, uint32_t, double>> sel;
            matcher::selectMatches(gm, gr, hc.maximumPointNumberForEpipolarHashing, sel);
            for (const auto &m : sel) add.emplace_back(std::get<0>(m), std::get<1>(m));
            addMask.assign(add.size(), 1);
            guided = (uint32_t)add.size();
        } else {  // the matchFeatures list under estimatePose's inlier mask (:697-703)
            for (size_t i = 0; i < n; i++) add.emplace_back(rows[2 * i], rows[2 * i + 1]);
            addMask.assign(n, 0);
            std::copy(mask.begin(), mask.begin() + std::min(mask.size(), n), addMask.begin());
        }
        tracklets.add(src, dst, add, addMask);
        logPair();
    }
    return res;
}

}  // namespace host
}  // namespace pgo
