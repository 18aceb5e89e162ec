// pgi_matcher.cuh — the device functions of guided matching (SURVEY §8f-3), which K10 (pgi_guided_batch.cuh) runs:
//
//   HashingBasedMatcherWithPose<false, 45>::match     matcher.h:199-405
//   (called from PoseGraphBuilder::guidedMatching       pose_graph_builder.h:717-783)
//
//   guidedPrepare: F = Kd^-T E Ks^-1, epipole from the 3x3 Jacobi SVD of F, angular range from the destination image's
//           corners (matcher.h:218-277) — the same operations in the same order as oracle/pgo_matcher.hpp;
//   guidedDestinationBin / guidedSourceBin: the bin of a destination keypoint's epipolar line's normal angle
//           (matcher.h:285-299), of a source keypoint's ray from the epipole (:333-345);
//   guidedEpipolarSq, guidedIsCandidate: squared symmetric epipolar distance (FP64, matcher.h:351-360) against 0.75^2;
//   guidedDescriptorSq: the squared descriptor distance (float differences accumulated in double, matcher.h:371-375);
//   guidedAdaptedRatio, guidedAccepted: the count-corrected Lowe ratio and the acceptance (matcher.h:386-406) of a
//           source keypoint's best / second-best state (pgi_guided_nn.h).
// atan2 is evaluated in double-double arithmetic and rounded once (pgi_atan2.h): the correctly rounded value, which is
// what glibc returns for all but ~2.5e-4 of arguments (CUDA's own atan2 is a 2-ulp function and differed from the host
// in the angular range of one of five test scenes).
#pragma once
#include <climits>
#include <cstdint>
#include <cuda_runtime.h>

#include "pgi_atan2.h"
#include "pgi_guided_nn.h"
#include "pgi_math.cuh"

namespace pgi {

constexpr int kMatchMaxBins = 192;

PGI_DEV void inverse3(const double *m, double *inv)  // Eigen compute_inverse_size3 (see oracle/pgo_matcher.hpp)
{
    auto cof = [&](int i, int j) {
        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
        return m[i1 * 3 + j1] * m[i2 * 3 + j2] - m[i1 * 3 + j2] * m[i2 * 3 + j1];
    };
    const double c00 = cof(0, 0), c10 = cof(1, 0), c20 = cof(2, 0);
    const double det = c00 * m[0] + (c10 * m[3] + c20 * m[6]);
    const double invdet = 1.0 / det;
    inv[0] = c00 * invdet; inv[1] = c10 * invdet; inv[2] = c20 * invdet;
    inv[3] = cof(0, 1) * invdet; inv[4] = cof(1, 1) * invdet; inv[5] = cof(2, 1) * invdet;
    inv[6] = cof(0, 2) * invdet; inv[7] = cof(1, 2) * invdet; inv[8] = cof(2, 2) * invdet;
}
PGI_DEV void mul3(const double *A, const double *B, double *C)
{
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) C[i * 3 + j] = sum3(A[i * 3 + 0] * B[0 * 3 + j], A[i * 3 + 1] * B[1 * 3 + j], A[i * 3 + 2] * B[2 * 3 + j]);
}
PGI_DEV double lineAngle(double ny, double nx)
{
    const double kRadianToDegree = 180.0 / 3.14159265358979323846;
    double angle = kRadianToDegree * pgi_atan::atan2cr(ny, nx) + 180.0;
    if (angle > 180) angle -= 180;
    return angle;
}
PGI_DEV int binOfAngle(double angle, double minAngle, double angularRange, int binNumber)
{
    angle = (binNumber - 1) * (angle - minAngle) / angularRange;
    const double r = round(angle);
    // the host's conversion (x86 cvttsd2si): NaN and out-of-range values become INT_MIN, i.e. bin 0 (cvt.rzi saturates)
    const int b = (r >= -2147483648.0 && r < 2147483648.0) ? (int)r : INT_MIN;
    const int lo = b < 0 ? 0 : b;  // MAX(0, .)
    return lo < binNumber - 1 ? lo : binNumber - 1;
}

// The per-pair preparation (matcher.h:218-277): F = Kd^-T E Ks^-1, the epipole from the 3x3 Jacobi SVD of F, the angular
// range from the destination image's corners, the bin count.  K10 runs it on one thread per pair.
struct GuidedPrep {
    double F[9];
    double ex, ey, minAngle, range;
    int binsRaw;  // binNumber, or the angular range's integer part for binNumber <= 0
    int bins;     // binsRaw clamped to [0, kMatchMaxBins]: the bins the kernels use (0: no match)
};

PGI_DEV void guidedPrepare(const double *E, const double *Ks, const double *Kd, int wS, int hS, int wD, int hD, int binNumber,
                           GuidedPrep &p)
{
    double KdInv[9], KsInv[9], KdInvT[9], T[9];
    inverse3(Kd, KdInv);
    inverse3(Ks, KsInv);
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) KdInvT[i * 3 + j] = KdInv[j * 3 + i];
    mul3(KdInvT, E, T);
    mul3(T, KsInv, p.F);
    double U[1], V[9], S[3];
    eigenJacobiSvd<3, false, true>(p.F, U, V, S);
    const double *F = p.F;
    const double ez = V[8];
    const double ex = V[2] / ez, ey = V[5] / ez;
    const bool inImage = ex >= 0 && ex < wS && ey >= 0 && ey < hS;
    double minAngle = 180, maxAngle = 0;
    if (!inImage) {
        const double corners[8] = {0, 0, (double)wD, 0, (double)wD, (double)hD, 0, (double)hD};
        for (int c = 0; c < 8; c += 2) {
            const double x = corners[c], y = corners[c + 1];
            const double nx = F[0] * x + F[3] * y + F[6];
            const double ny = F[1] * x + F[4] * y + F[7];
            const double angle = lineAngle(ny, nx);
            minAngle = minAngle < angle ? minAngle : angle;
            maxAngle = maxAngle > angle ? maxAngle : angle;
        }
    }
    p.ex = ex; p.ey = ey;
    p.minAngle = minAngle;
    p.range = maxAngle - minAngle;
    p.binsRaw = binNumber <= 0 ? (int)p.range : binNumber;
    p.bins = p.binsRaw < 0 ? 0 : (p.binsRaw > kMatchMaxBins ? kMatchMaxBins : p.binsRaw);
}

// bin of destination keypoint (x, y): the angle of its epipolar line's normal (matcher.h:285-299)
PGI_DEV int guidedDestinationBin(const double *F, double x, double y, double minAngle, double range, int bins)
{
    const double nx = F[0] * x + F[3] * y + F[6];
    const double ny = F[1] * x + F[4] * y + F[7];
    return binOfAngle(lineAngle(ny, nx), minAngle, range, bins);
}

// bin of source keypoint (x1, y1): the angle of its ray from the epipole (matcher.h:333-345)
PGI_DEV int guidedSourceBin(double x1, double y1, double ex, double ey, double minAngle, double range, int bins)
{
    const double vx = x1 - ex, vy = y1 - ey;
    return binOfAngle(lineAngle(vx, -vy), minAngle, range, bins);
}

// squared symmetric epipolar distance (FP64, matcher.h:351-360)
PGI_DEV double guidedEpipolarSq(const double *F, double x1, double y1, double x2, double y2)
{
    const double rxc = F[0] * x2 + F[3] * y2 + F[6];
    const double ryc = F[1] * x2 + F[4] * y2 + F[7];
    const double rwc = F[2] * x2 + F[5] * y2 + F[8];
    const double r = (x1 * rxc + y1 * ryc + rwc);
    const double rx = F[0] * x1 + F[1] * y1 + F[2];
    const double ry = F[3] * x1 + F[4] * y1 + F[5];
    const double a1 = rxc * rxc + ryc * ryc;
    const double b1 = rx * rx + ry * ry;
    return r * r * (a1 + b1) / (a1 * b1);
}

// the gate of matcher.h:362, literally: a NaN distance passes it
PGI_DEV bool guidedIsCandidate(double d2) { return !(d2 >= 0.75 * 0.75); }

// squared descriptor distance: float differences widened to double, accumulated in dimension order (matcher.h:371-375)
PGI_DEV double guidedDescriptorSq(const float *ds, const float *dd, uint32_t dim)
{
    double acc = 0;
    for (uint32_t m = 0; m < dim; m++) {
        const double dist = (double)(ds[m] - dd[m]);  // float subtraction, widened (matcher.h:373)
        acc += dist * dist;
    }
    return acc;
}

// count-corrected Lowe ratio (matcher.h:386-399) of a source keypoint's final scan state
PGI_DEV double guidedAdaptedRatio(const GuidedNn &s)
{
    double corr = 1.0;
    if (s.count < 20) corr = 0.65 * 0.65;
    if (s.count < 10) corr = 0.6 * 0.6;
    if (s.count < 5) corr = 0.5 * 0.5;
    if (s.count < 3) corr = 0.25 * 0.25;
    return (s.best / s.second) / corr;
}

// acceptance (matcher.h:400-406)
PGI_DEV bool guidedAccepted(const GuidedNn &s, double adapted)
{
    bool ok = false;
    if (!(adapted < 0.00001)) ok = s.bestIndex > -1 && ((adapted < 0.8 * 0.8) || (s.count == 1));
    return ok;
}

}  // namespace pgi
