// geodesy.cuh -- latLonToECEF (processor.go:125-148) for the kernels of solve.cu and window_fix.cu.
// Both translation units are compiled with -fmad=false, so the two copies round alike.
#pragma once
#include "common.cuh"

namespace tdoa {

constexpr double kA = 6378137.0;
constexpr double kF = 1.0 / 298.257223563;
constexpr double kPi = 3.14159265358979323846;

__device__ inline void llh_to_ecef(double lat, double lon, double elev, double *xyz)
{
    const double e2 = 2 * kF - kF * kF;
    const double lr = lat * kPi / 180, lo = lon * kPi / 180;
    const double sl = sin(lr), cl = cos(lr), so = sin(lo), co = cos(lo);
    const double N = kA / sqrt(1 - e2 * sl * sl);
    xyz[0] = (N + elev) * cl * co;
    xyz[1] = (N + elev) * cl * so;
    xyz[2] = (N * (1 - e2) + elev) * sl;
}

}  // namespace tdoa
