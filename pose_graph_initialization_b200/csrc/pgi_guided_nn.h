// pgi_guided_nn.h — the best / second-best state of the guided matcher's candidate scan (matcher.h:366-384) as a value that
// merges over consecutive runs of a bin.
//
// The reference (matcher.h:362-384) walks a source keypoint's bin in list order.  Every bin entry whose gate
// `d2 >= 0.75 * 0.75` is false is a candidate (a NaN d2 is one); for each candidate it computes the descriptor distance
// acc and steps
//   if (acc < best) { second = best; best = acc; bestIndex = nb; }        (best = second = DBL_MAX, bestIndex = -1 at first)
// Restated over the candidate sequence:
//   best, bestIndex = the FIRST strict minimum of acc among candidates with acc < DBL_MAX (DBL_MAX, -1 if there is none);
//   second          = min(DBL_MAX, acc of the candidates before bestIndex's position) — the best-so-far at the moment the
//                     final best was found, which is not in general the second-smallest acc.
// Since best is also min(DBL_MAX, every acc of the run), the state of a run followed by a later run is
//   later.best < earlier.best ? (later.best, min(earlier.best, later.second), later.index) : earlier
// so the states of consecutive runs merge exactly in any grouping that keeps their order (guidedMerge is associative, not
// commutative): K10 evaluates 32 consecutive candidates at a time, one per lane, and merges the lanes in order.
// tests/test_guided_nn_property.py compiles this header with g++ and checks random ordered partitions against the loop.
//
// Compiles as plain C++ (g++) and as CUDA device code.
#pragma once
#include <cfloat>
#include <cstdint>
#ifdef __CUDACC__
#define PGI_GNN_FN __host__ __device__ inline
#else
#define PGI_GNN_FN inline
#endif

namespace pgi {

struct GuidedNn {
    double best, second;
    int32_t bestIndex;  // destination keypoint, -1: none
    int32_t count;      // candidates seen: countSnn
};

PGI_GNN_FN GuidedNn guidedEmpty() { return GuidedNn{DBL_MAX, DBL_MAX, -1, 0}; }

// one step of the reference's sequential loop: candidate nb with descriptor distance acc, after every candidate before it
PGI_GNN_FN void guidedPush(GuidedNn &s, double acc, int32_t nb)
{
    s.count += 1;
    if (acc < s.best) { s.second = s.best; s.best = acc; s.bestIndex = nb; }
}

// the state of run a followed by run b
PGI_GNN_FN GuidedNn guidedMerge(const GuidedNn &a, const GuidedNn &b)
{
    GuidedNn r = a;
    r.count = a.count + b.count;
    if (b.best < a.best) {
        r.second = b.second < a.best ? b.second : a.best;
        r.best = b.best;
        r.bestIndex = b.bestIndex;
    }
    return r;
}

}  // namespace pgi
