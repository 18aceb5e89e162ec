"""pgi_atan2.h (the atan2 guided matching evaluates on the device) compiled for the host: it must return the correctly rounded
atan2.  Wherever it differs from the host libm (glibc is off by one ulp for ~2.5e-4 of arguments) mpmath decides, and
it must never be the one that is wrong."""
import math
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = r"""
#include "%s"
#include <cstdio>
#include <cstring>
#include <random>
int main() {
    std::mt19937_64 g(7);
    std::uniform_real_distribution<double> U(-2000, 2000), S(-1, 1);
    long n = 0, bad = 0;
    for (long i = 0; i < 3000000; i++) {
        double y, x;
        switch (i %% 4) {
        case 0: y = U(g); x = U(g); break;                       // pixel-sized line normals
        case 1: y = S(g) * 1e-3; x = U(g); break;                // nearly horizontal
        case 2: y = U(g); x = S(g) * 1e-5; break;                // nearly vertical
        default: y = std::ldexp(S(g), (int)(g() %% 80) - 40); x = std::ldexp(S(g), (int)(g() %% 80) - 40);
        }
        const double a = std::atan2(y, x), b = pgi_atan::atan2cr(y, x);
        n++;
        if (memcmp(&a, &b, 8)) { printf("%%a %%a %%a %%a\n", y, x, a, b); bad++; }
    }
    const double sp[][2] = {{0, 1}, {0, -1}, {-0.0, -1}, {1, 0}, {-1, 0}, {1, 1}, {-1, -1}, {3, -0.0}, {-3, 0.0}, {1e-300, 1e300}, {5, 5e-320}};
    for (auto &p : sp) {
        const double a = std::atan2(p[0], p[1]), b = pgi_atan::atan2cr(p[0], p[1]);
        if (memcmp(&a, &b, 8)) { printf("special %%a %%a %%a %%a\n", p[0], p[1], a, b); }
    }
    fprintf(stderr, "%%ld %%ld\n", n, bad);
    return 0;
}
"""


def test_device_atan2_is_the_correctly_rounded_one(tmp_path):
    mp = pytest.importorskip("mpmath")
    src = tmp_path / "h.cpp"
    src.write_text(HARNESS % os.path.join(ROOT, "pose_graph_initialization_b200", "csrc", "pgi_atan2.h"))
    exe = tmp_path / "h"
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-o", str(exe), str(src)], check=True)
    r = subprocess.run([str(exe)], check=True, capture_output=True, text=True)
    n, bad = (int(x) for x in r.stderr.split())
    assert n == 3000000 and bad < n * 1e-3  # the host libm itself is almost always correctly rounded
    mp.mp.prec = 300
    for line in r.stdout.splitlines():
        assert not line.startswith("special"), line
        y, x, libm, mine = (float.fromhex(t) for t in line.split())
        exact = mp.atan2(mp.mpf(y), mp.mpf(x))
        err_mine = abs(mp.mpf(mine) - exact) / math.ulp(mine)
        err_libm = abs(mp.mpf(libm) - exact) / math.ulp(libm)
        assert err_mine <= 0.5 < err_libm, line
