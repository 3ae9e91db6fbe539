// ls_core.cuh -- the least-squares fix of one set (k_solve_ls in solve.cu, and every candidate of the station check
// k_window_exclude in exclude.cu).  Both translation units are compiled with -fmad=false, so one statement gives
// one result in either kernel: a candidate's solve is, bit for bit, tdoa_solve_ls on the stations without it.
//
// SURVEY.md 8f rank 4 (no reference equivalent; oracle: orc_solve_ls, same statement):
// all P = S(S-1)/2 range differences, Levenberg-Marquardt in the local east/north/up
// frame of the current estimate (dims = 2: the elevation of the start point is kept,
// which is what three stations can support; dims = 3: elevation is solved too).
//   f_p(x) = (|x - s_j| - |x - s_i|) - rd_p,  row_p = g_j - g_i,  g_k = ENU components of
//   the unit vector from station k to x;  (J'J + lambda diag(J'J)) d = -J'f;  a step is
//   taken only if it lowers sum f^2 (lambda / 3), else lambda * 4, at most 8 tries;
//   stop after 60 iterations, when no try succeeds, or when |d| < 1e-6 m.
// used (may be nullptr): per set and pair, 0 leaves the pair out of the cost, the normal equations
// and the rms; fewer than `dims` used pairs, or used pairs touching fewer than dims + 1 stations,
// give status 2 with the start point and no iteration (tdoa_process_windows).  skip: a station bit mask on top of
// used (needs used): every pair that touches a station of skip is left out as an unused one is.
#pragma once
#include <cstdint>

#include "geodesy.cuh"
#include "graph_ls.cuh"

namespace tdoa {

constexpr int kLsMaxStations = 64;

struct LsPoint {
    double lat, lon, h;  // degrees, degrees, metres
};

struct LsFix {
    LsPoint p;
    double rms;
    int status, iters;
};

__device__ __forceinline__ bool ls_pair_out(const uint8_t *used, unsigned long long skip, int q, int i, int j)
{
    return used && (!used[q] || ((skip >> i | skip >> j) & 1ull));
}

__device__ inline double ls_cost(const double *s_st, int n_st, const double *rd, const uint8_t *used, unsigned long long skip,
                                 const LsPoint &p, double *r_out)
{
    double x[3];
    llh_to_ecef(p.lat, p.lon, p.h, x);
    for (int k = 0; k < n_st; k++) {
        const double dx = x[0] - s_st[3 * k], dy = x[1] - s_st[3 * k + 1], dz = x[2] - s_st[3 * k + 2];
        r_out[k] = sqrt(dx * dx + dy * dy + dz * dz);
    }
    double c = 0.0;
    int q = 0;
    for (int i = 0; i < n_st; i++)
        for (int j = i + 1; j < n_st; j++, q++) {
            if (ls_pair_out(used, skip, q, i, j)) continue;
            const double f = (r_out[j] - r_out[i]) - rd[q];
            c += f * f;
        }
    return c;
}

// d = -(A + lambda diag A)^-1 b for the leading n x n part (n = 2 or 3); false: singular
__device__ inline bool ls_step(const double (&A)[3][3], const double (&b)[3], double lambda, int n, double (&d)[3])
{
    double M[3][3];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) M[i][j] = A[i][j];
    for (int i = 0; i < 3; i++) M[i][i] = A[i][i] + lambda * A[i][i];
    d[0] = d[1] = d[2] = 0.0;
    if (n == 2) {
        const double det = M[0][0] * M[1][1] - M[0][1] * M[1][0];
        if (!(fabs(det) > 1e-300)) return false;
        d[0] = -(b[0] * M[1][1] - b[1] * M[0][1]) / det;
        d[1] = -(M[0][0] * b[1] - M[1][0] * b[0]) / det;
        return true;
    }
    const double c00 = M[1][1] * M[2][2] - M[1][2] * M[2][1];
    const double c01 = M[1][2] * M[2][0] - M[1][0] * M[2][2];
    const double c02 = M[1][0] * M[2][1] - M[1][1] * M[2][0];
    const double det = M[0][0] * c00 + M[0][1] * c01 + M[0][2] * c02;
    if (!(fabs(det) > 1e-300)) return false;
    const double c10 = M[0][2] * M[2][1] - M[0][1] * M[2][2];
    const double c11 = M[0][0] * M[2][2] - M[0][2] * M[2][0];
    const double c12 = M[0][1] * M[2][0] - M[0][0] * M[2][1];
    const double c20 = M[0][1] * M[1][2] - M[0][2] * M[1][1];
    const double c21 = M[0][2] * M[1][0] - M[0][0] * M[1][2];
    const double c22 = M[0][0] * M[1][1] - M[0][1] * M[1][0];
    d[0] = -(c00 * b[0] + c10 * b[1] + c20 * b[2]) / det;
    d[1] = -(c01 * b[0] + c11 * b[1] + c21 * b[2]) / det;
    d[2] = -(c02 * b[0] + c12 * b[1] + c22 * b[2]) / det;
    return true;
}

// the start of set `set`: init_llh[set], or (init == nullptr) the mean of the station coordinates
__device__ inline LsPoint ls_start(const double *llh, int n_st, const double *init_llh, int set)
{
    LsPoint p;
    if (init_llh) {
        p.lat = init_llh[3 * set]; p.lon = init_llh[3 * set + 1]; p.h = init_llh[3 * set + 2];
    } else {
        p.lat = p.lon = p.h = 0.0;
        for (int k = 0; k < n_st; k++) { p.lat += llh[3 * k]; p.lon += llh[3 * k + 1]; p.h += llh[3 * k + 2]; }
        p.lat /= n_st; p.lon /= n_st; p.h /= n_st;
    }
    return p;
}

// the fix of one set from p; s_st: the station ECEF
__device__ inline LsFix ls_fix(const double *s_st, int n_st, const double *rd, const uint8_t *used, unsigned long long skip,
                               int dims, LsPoint p)
{
    int P = n_st * (n_st - 1) / 2;
    const double e2 = 2 * kF - kF * kF;
    if (used) {   // too few measurements: no iteration
        const int n_used = ls_used_pairs(used, n_st, dims, skip);
        if (n_used < 0) return LsFix{p, 0.0, 2, 0};
        P = n_used;
    }
    double r[kLsMaxStations], g[kLsMaxStations][3];
    double lambda = 1e-3;
    double cost = ls_cost(s_st, n_st, rd, used, skip, p, r);
    int it = 0, st = 0;
    for (; it < 60; it++) {
        const double lr = p.lat * kPi / 180, lo = p.lon * kPi / 180;
        const double sl = sin(lr), cl = cos(lr), so = sin(lo), co = cos(lo);
        const double w = sqrt(1 - e2 * sl * sl);
        const double Nr = kA / w, Mr = kA * (1 - e2) / (w * w * w);
        double x[3];
        llh_to_ecef(p.lat, p.lon, p.h, x);
        for (int k = 0; k < n_st; k++) {
            const double ux = (x[0] - s_st[3 * k]) / r[k], uy = (x[1] - s_st[3 * k + 1]) / r[k], uz = (x[2] - s_st[3 * k + 2]) / r[k];
            g[k][0] = -so * ux + co * uy;
            g[k][1] = -sl * co * ux - sl * so * uy + cl * uz;
            g[k][2] = cl * co * ux + cl * so * uy + sl * uz;
        }
        double A[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, b[3] = {0, 0, 0};
        int q = 0;
        for (int i = 0; i < n_st; i++)
            for (int j = i + 1; j < n_st; j++, q++) {
                if (ls_pair_out(used, skip, q, i, j)) continue;
                const double f = (r[j] - r[i]) - rd[q];
                const double row[3] = {g[j][0] - g[i][0], g[j][1] - g[i][1], g[j][2] - g[i][2]};
                for (int a = 0; a < 3; a++) {
                    b[a] += row[a] * f;
                    for (int c = 0; c < 3; c++) A[a][c] += row[a] * row[c];
                }
            }
        bool moved = false;
        double d[3] = {0, 0, 0};
        for (int tr = 0; tr < 8 && !moved; tr++) {
            if (!ls_step(A, b, lambda, dims, d)) { lambda *= 10.0; continue; }
            LsPoint c = p;
            c.lat = p.lat + d[1] / (Mr + p.h) * 180.0 / kPi;
            c.lon = p.lon + d[0] / ((Nr + p.h) * cl) * 180.0 / kPi;
            if (dims == 3) c.h = p.h + d[2];
            double rc[kLsMaxStations];
            const double cc = ls_cost(s_st, n_st, rd, used, skip, c, rc);
            if (cc < cost) {
                p = c; cost = cc; moved = true;
                for (int k = 0; k < n_st; k++) r[k] = rc[k];
                lambda = fmax(lambda / 3.0, 1e-12);
            } else {
                lambda *= 4.0;
            }
        }
        if (!moved) break;
        if (sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]) < 1e-6) { it++; break; }
    }
    if (!(cost == cost)) st = 1;  // NaN: degenerate geometry
    return LsFix{p, P > 0 ? sqrt(cost / P) : 0.0, st, it};
}

}  // namespace tdoa
