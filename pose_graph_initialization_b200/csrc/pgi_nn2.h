// pgi_nn2.h — the 2-NN state of matchFeatures' knnMatch(k = 2) scan (feature_utils.h:151-163) as a mergeable value.
//
// The reference (and oracle.match_features) scans train indices in ascending order with strict `<`, starting from
// d1 = d2 = FLT_MAX:
//   if (v < d1) { d2 = d1; d1 = v; i1 = idx; } else if (v < d2) d2 = v;
// Its result is a function of the multiset of distances, not of the scan:
//   d1 = the minimum of the distances below FLT_MAX (FLT_MAX if there is none; NaN and values >= FLT_MAX never enter),
//   i1 = the lowest index reaching d1 (kNn2None if d1 == FLT_MAX),
//   d2 = the second order statistic of the same multiset padded with FLT_MAX (d2 == d1 on a tie).
// So the results of disjoint index subsets merge exactly, in any order and grouping (nn2Merge is commutative and
// associative): K9 scans the columns a thread owns, then merges across lanes, warps and CTAs.
// tests/test_nn2_merge_property.py compiles this header with g++ and checks random partitions against the sequential scan.
//
// Compiles as plain C++ (g++) and as CUDA device code.
#pragma once
#include <cfloat>
#include <cstdint>
#include <cstring>
#ifdef __CUDACC__
#define PGI_NN2_FN __host__ __device__ inline
#else
#define PGI_NN2_FN inline
#endif

namespace pgi {

constexpr uint32_t kNn2None = 0xffffffffu;

struct Nn2 {
    float d1, d2;
    uint32_t i1;
};

PGI_NN2_FN Nn2 nn2Empty() { return Nn2{FLT_MAX, FLT_MAX, kNn2None}; }

// one step of the sequential scan; within one state, indices must be pushed in ascending order
PGI_NN2_FN void nn2Push(Nn2 &s, float v, uint32_t idx)
{
    if (v < s.d1) { s.d2 = s.d1; s.d1 = v; s.i1 = idx; }
    else if (v < s.d2) s.d2 = v;
}

PGI_NN2_FN float nn2Min(float a, float b) { return b < a ? b : a; }
PGI_NN2_FN float nn2Max(float a, float b) { return a < b ? b : a; }

// the state of the union of two disjoint index sets (neither state ever holds a NaN)
PGI_NN2_FN Nn2 nn2Merge(const Nn2 &a, const Nn2 &b)
{
    Nn2 r;
    r.d1 = nn2Min(a.d1, b.d1);
    r.i1 = a.d1 < b.d1 ? a.i1 : (b.d1 < a.d1 ? b.i1 : (a.i1 < b.i1 ? a.i1 : b.i1));
    r.d2 = nn2Min(nn2Max(a.d1, b.d1), nn2Min(a.d2, b.d2));
    return r;
}

// sort key of a surviving match: the ratio d1 / d2 is a non-negative float below 0.90 (never NaN), so its bit pattern
// orders like its value, and the query index below it breaks ties as std::sort on (ratio, &matches[i]) does
// (feature_utils.h:188).  One unique 64-bit key per survivor.
PGI_NN2_FN uint64_t matchKey(float ratio, uint32_t query)
{
    uint32_t bits;
#ifdef __CUDA_ARCH__
    bits = __float_as_uint(ratio);
#else
    memcpy(&bits, &ratio, 4);
#endif
    return ((uint64_t)bits << 32) | query;
}

}  // namespace pgi
