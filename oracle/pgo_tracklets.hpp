// ORACLE — TEST INFRASTRUCTURE ONLY (see pgo_geom.hpp header).
//
// pgo_tracklets.hpp — reconstruction::Tracklets (point_track.h:541-712) for the C++ oracle host: a port of
// oracle/pgo_tracklets.py statement by statement, with the Python containers mapped back onto the reference's kinds
// (dict with setdefault -> std::map / std::unordered_map with operator[], list -> std::vector).  It shares no code with the
// product's pgb_tracklets.cpp.  Parity unpinned, as the Python restatement: the reference has no tests or fixtures for
// Tracklets (SURVEY §4).
#pragma once
#include <cstddef>
#include <cstdint>
#include <map>
#include <set>
#include <tuple>
#include <unordered_map>
#include <utility>
#include <vector>

namespace pgo {

class Tracklets {
public:
    typedef std::pair<size_t, size_t> ViewPoint;  // (view, point)

    // :575-636; the third tuple member is never written (value-initialised)
    std::vector<std::tuple<size_t, size_t, double>> getCorrespondences(size_t viewIdSource_, size_t viewIdDestination_,
                                                                       size_t maximumCorrespondenceNumber_) const
    {
        std::vector<std::tuple<size_t, size_t, double>> matches_;
        const auto its = tmpViewToTracks.find(viewIdSource_);
        if (its == tmpViewToTracks.end()) return matches_;  // :583-588
        const auto itd = tmpViewToTracks.find(viewIdDestination_);
        if (itd == tmpViewToTracks.end()) return matches_;  // :590-596
        const std::vector<size_t> &tracksSrc = its->second, &tracksDst = itd->second;
        const std::set<size_t> trackMap(tracksSrc.begin(), tracksSrc.end());  // :602-606
        for (const size_t trackIdx : tracksDst) {                             // :608
            if (trackMap.find(trackIdx) == trackMap.end()) continue;
            std::tuple<size_t, size_t, double> pair{0, 0, 0.0};
            int cnt = 0;
            for (const ViewPoint &p : tmpTracks[trackIdx]) {  // :614-627
                if (p.first == viewIdSource_) {
                    std::get<0>(pair) = p.second;
                    cnt += 1;
                } else if (p.first == viewIdDestination_) {
                    std::get<1>(pair) = p.second;
                    cnt += 1;
                }
                if (cnt == 2) break;
            }
            matches_.push_back(pair);                                     // :629
            if (matches_.size() > maximumCorrespondenceNumber_) break;    // :631-632
        }
        return matches_;
    }

    // :638-712.  matches_: (source point, destination point) per row.
    void add(size_t imageIdxSource_, size_t imageIdxDestination_, const std::vector<std::pair<size_t, size_t>> &matches_,
             const std::vector<uint8_t> &inlierMask_)
    {
        for (size_t pointIdx = 0; pointIdx < matches_.size(); pointIdx++) {
            if (!inlierMask_[pointIdx]) continue;  // :650-651
            const ViewPoint pairSource(imageIdxSource_, matches_[pointIdx].first);
            const ViewPoint pairDestination(imageIdxDestination_, matches_[pointIdx].second);
            size_t it = pointPairs[pairSource];  // :655-657
            if (it == 0) {
                it = pointPairs[pairSource] = pointPairNumber;
                pointPairNumber += 1;
            }
            size_t jt = pointPairs[pairDestination];  // :659-661
            if (jt == 0) {
                jt = pointPairs[pairDestination] = pointPairNumber;
                pointPairNumber += 1;
            }
            std::vector<size_t> &tracksSource = tmpPairToTracks[it];       // :663
            std::vector<size_t> &tracksDestination = tmpPairToTracks[jt];  // :664
            const size_t trackNumDestination = tracksDestination.size();    // :665
            bool added = false;
            // :668-679 — the Python restatement iterates a copy when both names are one list
            const std::vector<size_t> sourceCopy = &tracksSource == &tracksDestination ? tracksSource : std::vector<size_t>();
            const std::vector<size_t> &loop = &tracksSource == &tracksDestination ? sourceCopy : tracksSource;
            for (size_t k = 0; k < loop.size(); k++) {
                const size_t trackIdx = loop[k];
                std::vector<ViewPoint> &track = tmpTracks[trackIdx];
                if (contains(track, pairDestination)) continue;
                tmpViewToTracks[imageIdxDestination_].push_back(trackIdx);
                track.push_back(pairDestination);
                tracksDestination.push_back(trackIdx);
                added = true;
            }
            for (size_t trackIdxIdx = 0; trackIdxIdx < trackNumDestination; trackIdxIdx++) {  // :681-693
                const size_t trackIdx = tracksDestination[trackIdxIdx];
                std::vector<ViewPoint> &track = tmpTracks[trackIdx];
                if (contains(track, pairSource)) continue;
                tmpViewToTracks[imageIdxSource_].push_back(trackIdx);
                track.push_back(pairSource);
                tracksSource.push_back(trackIdx);
                added = true;
            }
            if (!added) {  // :695-703
                const size_t idx = tmpTracks.size();
                tmpTracks.push_back({pairSource, pairDestination});
                tmpViewToTracks[imageIdxSource_].push_back(idx);
                tmpViewToTracks[imageIdxDestination_].push_back(idx);
                tracksSource.push_back(idx);
                tracksDestination.push_back(idx);
            }
        }
    }

    size_t trackCount() const { return tmpTracks.size(); }

private:
    static bool contains(const std::vector<ViewPoint> &track, const ViewPoint &p)
    {
        for (const ViewPoint &q : track)
            if (q == p) return true;
        return false;
    }
    size_t pointPairNumber = 0;                                         // :552, :565
    std::map<ViewPoint, size_t> pointPairs;                             // operator[] default-constructs 0
    std::vector<std::vector<ViewPoint>> tmpTracks;                      // :556
    std::unordered_map<size_t, std::vector<size_t>> tmpViewToTracks;    // :557
    std::unordered_map<size_t, std::vector<size_t>> tmpPairToTracks;    // :558
};

}  // namespace pgo
