// pgi_atan2.h — atan2 evaluated in double-double arithmetic and rounded once.
//
// matcher.h:285-299 and :330-340 bin keypoints by `atan2` of an epipolar line's normal; the reference calls the host
// libm, whose last bit depends on the libm version (glibc 2.39: correctly rounded in 99.97 % of random arguments, off by
// one ulp in the rest — measured against this file and mpmath).  CUDA's atan2 is a 2-ulp function, and an angle that
// differs in its last bit shows up in the matcher's angular range and, rarely, in a bin index.  The guided matcher therefore evaluates
// the one canonical answer, the correctly rounded atan2, itself: y/x as a double-double quotient, reduced against a
// 65-entry table of atan(k/64) (double-double), odd series on the remainder (|z| <= 1/128), quadrant fix-ups with
// double-double pi — about 100 bits before the final rounding, so the result is the correctly rounded one except for
// arguments within ~2^-45 ulp of a rounding boundary.  tests/test_atan2_cr.py compiles this header with g++ and
// requires the result to be the correctly rounded one (mpmath) wherever it differs from the host libm.
//
// Compiles as plain C++ (g++) and as CUDA device code; fma() is the exact fused multiply-add in both (it is spelled out,
// so -fmad=false / -ffp-contract=off do not affect it).
#pragma once
#include <cmath>
#ifdef __CUDACC__
#define PGI_ATAN_FN __device__ inline
#define PGI_ATAN_TAB __device__
#else
#define PGI_ATAN_FN inline
#define PGI_ATAN_TAB
#endif

namespace pgi_atan {

struct dd {
    double h, l;
};
PGI_ATAN_FN dd fastTwoSum(double a, double b)  // |a| >= |b|
{
    const double s = a + b;
    return dd{s, b - (s - a)};
}
PGI_ATAN_FN dd twoSum(double a, double b)
{
    const double s = a + b, bb = s - a;
    return dd{s, (a - (s - bb)) + (b - bb)};
}
PGI_ATAN_FN dd twoProd(double a, double b)
{
    const double p = a * b;
    return dd{p, fma(a, b, -p)};
}
PGI_ATAN_FN dd ddAdd(dd a, dd b)
{
    dd s = twoSum(a.h, b.h);
    const dd t = twoSum(a.l, b.l);
    s.l += t.h;
    s = fastTwoSum(s.h, s.l);
    s.l += t.l;
    return fastTwoSum(s.h, s.l);
}
PGI_ATAN_FN dd ddMul(dd a, dd b)
{
    dd p = twoProd(a.h, b.h);
    p.l += a.h * b.l + a.l * b.h;
    return fastTwoSum(p.h, p.l);
}
PGI_ATAN_FN dd ddDiv(dd n, dd d)
{
    const double q1 = n.h / d.h;
    // n - q1 * d, exactly in the leading parts
    const dd p = twoProd(q1, d.h);
    double r = (n.h - p.h) - p.l;  // n.h - p.h is exact (q1 * d.h ~ n.h)
    r += n.l - q1 * d.l;
    const double q2 = r / d.h;
    return fastTwoSum(q1, q2);
}

PGI_ATAN_TAB static const double kTab[65][2] = {
    {0x0.0p+0, 0x0.0p+0},
    {0x1.fff555bbb729bp-7, -0x1.220c39d4dff50p-61},
    {0x1.ffd55bba97625p-6, -0x1.5ec431444912cp-60},
    {0x1.7fb818430da2ap-5, -0x1.86ef8f794f105p-63},
    {0x1.ff55bb72cfdeap-5, -0x1.c934d86d23f1dp-60},
    {0x1.3f59f0e7c559dp-4, 0x1.ac4ce285df847p-58},
    {0x1.7ee182602f10fp-4, -0x1.cfb654c0c3d98p-58},
    {0x1.be39ebe6f07c3p-4, 0x1.f7b8f29a05987p-58},
    {0x1.fd5ba9aac2f6ep-4, -0x1.cd37686760c17p-59},
    {0x1.1e1fafb043727p-3, -0x1.b485914dacf8cp-59},
    {0x1.3d6eee8c6626cp-3, 0x1.61a3b0ce9281bp-57},
    {0x1.5c9811e3ec26ap-3, -0x1.054ab2c010f3dp-58},
    {0x1.7b97b4bce5b02p-3, 0x1.347b0b4f881cap-58},
    {0x1.9a6a8e96c8626p-3, 0x1.cf601e7b4348ep-59},
    {0x1.b90d7529260a2p-3, 0x1.17b10d2e0e5abp-61},
    {0x1.d77d5df205736p-3, 0x1.c648d1534597ep-57},
    {0x1.f5b75f92c80ddp-3, 0x1.8ab6e3cf7afbdp-57},
    {0x1.09dc597d86362p-2, 0x1.62e47390cb865p-56},
    {0x1.18bf5a30bf178p-2, 0x1.30ca4748b1bf9p-57},
    {0x1.278372057ef46p-2, -0x1.077cdd36dfc81p-56},
    {0x1.362773707ebccp-2, -0x1.963a544b672d8p-57},
    {0x1.44aa436c2af0ap-2, -0x1.5d5e43c55b3bap-56},
    {0x1.530ad9951cd4ap-2, -0x1.2566480884082p-57},
    {0x1.614840309cfe2p-2, -0x1.a725715711f00p-56},
    {0x1.6f61941e4def1p-2, -0x1.c63aae6f6e918p-56},
    {0x1.7d5604b63b3f7p-2, 0x1.69c885c2b249ap-56},
    {0x1.8b24d394a1b25p-2, 0x1.b6d0ba3748fa8p-56},
    {0x1.98cd5454d6b18p-2, 0x1.9e6c988fd0a77p-56},
    {0x1.a64eec3cc23fdp-2, -0x1.24dec1b50b7ffp-56},
    {0x1.b3a911da65c6cp-2, 0x1.ae187b1ca5040p-56},
    {0x1.c0db4c94ec9f0p-2, -0x1.cc1ce70934c34p-56},
    {0x1.cde53432c1351p-2, -0x1.a2cfa4418f1adp-56},
    {0x1.dac670561bb4fp-2, 0x1.a2b7f222f65e2p-56},
    {0x1.e77eb7f175a34p-2, 0x1.0e53dc1bf3435p-56},
    {0x1.f40dd0b541418p-2, -0x1.a3992dc382a23p-57},
    {0x1.0039c73c1a40cp-1, -0x1.b32c949c9d593p-55},
    {0x1.0657e94db30d0p-1, -0x1.d5b495f6349e6p-56},
    {0x1.0c6145b5b43dap-1, 0x1.974fa13b5404fp-58},
    {0x1.1255d9bfbd2a9p-1, -0x1.2bdaee1c0ee35p-58},
    {0x1.1835a88be7c13p-1, 0x1.c621cec00c301p-55},
    {0x1.1e00babdefeb4p-1, -0x1.928df287a668fp-58},
    {0x1.23b71e2cc9e6ap-1, 0x1.c421c9f38224ep-57},
    {0x1.2958e59308e31p-1, -0x1.09e73b0c6c087p-56},
    {0x1.2ee628406cbcap-1, 0x1.c5d5e9ff0cf8dp-55},
    {0x1.345f01cce37bbp-1, 0x1.1021137c71102p-55},
    {0x1.39c391cd4171ap-1, -0x1.2304331d8bf46p-55},
    {0x1.3f13fb89e96f4p-1, 0x1.ecf8b492644f0p-56},
    {0x1.445065b795b56p-1, -0x1.f76d0163f79c8p-56},
    {0x1.4978fa3269ee1p-1, 0x1.2419a87f2a458p-56},
    {0x1.4e8de5bb6ec04p-1, 0x1.4a33dbeb3796cp-55},
    {0x1.538f57b89061fp-1, -0x1.1bb74abda520cp-55},
    {0x1.587d81f732fbbp-1, -0x1.5e5c9d8c5a950p-56},
    {0x1.5d58987169b18p-1, 0x1.0028e4bc5e7cap-57},
    {0x1.6220d115d7b8ep-1, -0x1.2b785350ee8c1p-57},
    {0x1.66d663923e087p-1, -0x1.6ea6febe8bbbap-56},
    {0x1.6b798920b3d99p-1, -0x1.a80386188c50ep-55},
    {0x1.700a7c5784634p-1, -0x1.8c34d25aadef6p-56},
    {0x1.748978fba8e0fp-1, 0x1.7b2a6165884a1p-59},
    {0x1.78f6bbd5d315ep-1, 0x1.406a089803740p-55},
    {0x1.7d528289fa093p-1, 0x1.560821e2f3aa9p-55},
    {0x1.819d0b7158a4dp-1, -0x1.bf76229d3b917p-56},
    {0x1.85d69576cc2c5p-1, 0x1.6b66e7fc8b8c3p-57},
    {0x1.89ff5ff57f1f8p-1, -0x1.55b9a5e177a1bp-55},
    {0x1.8e17aa99cc05ep-1, -0x1.ec182ab042f61p-56},
    {0x1.921fb54442d18p-1, 0x1.1a62633145c07p-55},
};

// atan of t in [0, 1] (double-double in, double-double out)
PGI_ATAN_FN dd atanUnit(dd t)
{
    const int k = (int)rint(t.h * 64.0);
    dd z = t;
    if (k > 0) {
        const double c = (double)k * (1.0 / 64.0);
        const dd num = twoSum(t.h - c, t.l);  // t.h - c is exact (Sterbenz)
        dd pc = twoProd(t.h, c);
        pc.l += t.l * c;
        dd den = twoSum(1.0, pc.h);
        den.l += pc.l;
        den = fastTwoSum(den.h, den.l);
        z = ddDiv(num, den);
    }
    // atan(z) = z + z^3 * (-1/3 + w/5 - w^2/7 + w^3/9 - w^4/11 + w^5/13), w = z^2 <= 2^-14
    const dd w = ddMul(z, z);
    const double wh = w.h;
    const double q = wh * (1.0 / 5.0 - wh * (1.0 / 7.0 - wh * (1.0 / 9.0 - wh * (1.0 / 11.0 - wh * (1.0 / 13.0 - wh * (1.0 / 15.0))))));
    const dd s = ddAdd(dd{-0x1.5555555555555p-2, -0x1.5555555555555p-56}, dd{q, 0.0});
    const dd corr = ddMul(ddMul(z, w), s);
    const dd a = ddAdd(z, corr);
    return ddAdd(dd{kTab[k][0], kTab[k][1]}, a);
}

// atan2(y, x) for finite arguments, correctly rounded (see the header comment)
PGI_ATAN_FN double atan2cr(double y, double x)
{
    const double ax = fabs(x), ay = fabs(y);
    if (!(ax <= 1.79769313486231570815e+308) || !(ay <= 1.79769313486231570815e+308)) return atan2(y, x);  // inf / nan: library semantics
    const dd piHalf{0x1.921fb54442d18p+0, 0x1.1a62633145c07p-54}, pi{0x1.921fb54442d18p+1, 0x1.1a62633145c07p-53};
    if (ay == 0.0) return (copysign(1.0, x) < 0.0) ? copysign(pi.h, y) : copysign(0.0, y);
    if (ax == 0.0) return copysign(piHalf.h, y);
    const bool swap = ay > ax;
    const double lo = swap ? ax : ay, hi = swap ? ay : ax;
    const double th = lo / hi;
    if (th < 0x1p-900) return atan2(y, x);  // quotient underflows towards subnormals: not a keypoint geometry, library semantics
    const double tl = fma(-th, hi, lo) / hi;
    dd a = atanUnit(fastTwoSum(th, tl));
    if (swap) a = ddAdd(piHalf, dd{-a.h, -a.l});
    if ((copysign(1.0, x) < 0.0)) a = ddAdd(pi, dd{-a.h, -a.l});
    return copysign(a.h, y);
}

}  // namespace pgi_atan
