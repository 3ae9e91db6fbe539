// solve.cu -- geodesy, the reference's 2x2 damped Newton fix, and the dense lat-lon
// grid multilateration.
//
// Replaces latLonToECEF (processor.go:125-148), distance3D / calculateBaseline
// (:151-163), solveTDOA (:932-1020) and ecefToLatLon (:1023-1045).  All f64, written
// in the reference's operation order.  The grid solve has no reference equivalent
// (oracle: orc_grid_solve).
#include <algorithm>
#include <type_traits>

#include "geodesy.cuh"
#include "graph_ls.cuh"
#include "kernels.h"
#include "ls_core.cuh"

namespace tdoa {

namespace {

__device__ void ecef_to_llh(double x, double y, double z, double *llh)
{
    const double e2 = 2 * kF - kF * kF;
    const double p = sqrt(x * x + y * y);
    const double lon = atan2(y, x);
    double lat = atan2(z, p * (1 - e2));
    for (int i = 0; i < 5; i++) {
        const double N = kA / sqrt(1 - e2 * sin(lat) * sin(lat));
        const double elev = p / cos(lat) - N;
        lat = atan2(z, p * (1 - e2 * N / (N + elev)));
    }
    const double N = kA / sqrt(1 - e2 * sin(lat) * sin(lat));
    const double elev = p / cos(lat) - N;
    llh[0] = lat * 180.0 / kPi;
    llh[1] = lon * 180.0 / kPi;
    llh[2] = elev;
}

__global__ void k_baselines(const double *llh, int n_st, double *out)
{
    // pair p = (i, j), i < j lexicographic (processor.go:803-809)
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int P = n_st * (n_st - 1) / 2;
    if (p >= P) return;
    int i = 0, rem = p;
    while (rem >= n_st - 1 - i) { rem -= n_st - 1 - i; i++; }
    const int j = i + 1 + rem;
    double a[3], b[3];
    llh_to_ecef(llh[3 * i], llh[3 * i + 1], llh[3 * i + 2], a);
    llh_to_ecef(llh[3 * j], llh[3 * j + 1], llh[3 * j + 2], b);
    const double dx = b[0] - a[0], dy = b[1] - a[1], dz = b[2] - a[2];
    out[p] = sqrt(dx * dx + dy * dy + dz * dz);
}

// processor.go:932-1020: stations 0..2 only, rd[0] and rd[1] only, start at the ECEF of
// the mean lat/lon/elev, <= 10 iterations, residual test before the update, Jacobian in
// X,Y, Cramer, |det| < 1e-10 -> singular, step 0.5, Z frozen.  One thread per set.
__global__ void k_solve(const double *llh, const double *rd_all, int n_sets, int rd_stride, double *out_llh,
                        int *status, int *iters)
{
    const int set = blockIdx.x * blockDim.x + threadIdx.x;
    if (set >= n_sets) return;
    const double *rd = rd_all + (size_t)set * rd_stride;
    double s[3][3];
    for (int k = 0; k < 3; k++) llh_to_ecef(llh[3 * k], llh[3 * k + 1], llh[3 * k + 2], s[k]);
    const double clat = (llh[0] + llh[3] + llh[6]) / 3.0;
    const double clon = (llh[1] + llh[4] + llh[7]) / 3.0;
    const double cel = (llh[2] + llh[5] + llh[8]) / 3.0;
    double x[3];
    llh_to_ecef(clat, clon, cel, x);
    int it, st = 0;
    for (it = 0; it < 10; it++) {
        double r[3];
        for (int k = 0; k < 3; k++)
            r[k] = sqrt((x[0] - s[k][0]) * (x[0] - s[k][0]) + (x[1] - s[k][1]) * (x[1] - s[k][1]) +
                        (x[2] - s[k][2]) * (x[2] - s[k][2]));
        const double res1 = (r[1] - r[0]) - rd[0];
        const double res2 = (r[2] - r[0]) - rd[1];
        if (fabs(res1) < 1.0 && fabs(res2) < 1.0) break;
        const double dx1 = (x[0] - s[0][0]) / r[0], dy1 = (x[1] - s[0][1]) / r[0];
        const double dx2 = (x[0] - s[1][0]) / r[1], dy2 = (x[1] - s[1][1]) / r[1];
        const double dx3 = (x[0] - s[2][0]) / r[2], dy3 = (x[1] - s[2][1]) / r[2];
        const double J11 = dx2 - dx1, J12 = dy2 - dy1, J21 = dx3 - dx1, J22 = dy3 - dy1;
        const double det = J11 * J22 - J12 * J21;
        if (fabs(det) < 1e-10) { st = 1; break; }
        const double dx = (-res1 * J22 + res2 * J12) / det;
        const double dy = (res1 * J21 - res2 * J11) / det;
        x[0] += 0.5 * dx;
        x[1] += 0.5 * dy;
    }
    if (iters) iters[set] = it;
    status[set] = st;
    double o[3] = {0.0, 0.0, 0.0};
    if (!st) ecef_to_llh(x[0], x[1], x[2], o);
    out_llh[3 * set] = o[0];
    out_llh[3 * set + 1] = o[1];
    out_llh[3 * set + 2] = o[2];
}

// solveTDOA of the SHIPPED BINARY (ELF 0x4a0360; oracle: orc_solve_binary, same statement, pinned
// by the iteration traces the binary prints): measurements with |rd| > 20400 m are dropped and
// the rest compacted; fewer than two -> status 1; any count but two -> status 2 (the binary solves
// with exactly two); res1 = (r2 - r1) - valid[0], res2 = (r3 - r1) - valid[1]; both < 1 m ->
// converged; |det| < 1e-12 -> 0.1 of a single-equation step in X (status 3 if neither equation
// can be used); else the Newton step times 0.7, a step longer than 1000 m first scaled to 1000 m;
// at most 10 iterations; Z is never updated.
// info[4] = {status, n_valid, n_iter, converged}; trace[10][5] = {det, res1, res2, step, code}
// (code 0 plain step, 1 limited step, 2 / 3 single equation 1 / 2).
__global__ void k_solve_binary(const double *llh, const double *rd, int n_rd, double *out_llh, int *info, double *trace)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    double valid[2] = {0.0, 0.0};
    int nv = 0;
    for (int k = 0; k < n_rd; k++)
        if (fabs(rd[k]) <= 20400.0) {
            if (nv < 2) valid[nv] = rd[k];
            nv++;
        }
    int status = 0, n_iter = 0, converged = 0;
    double o[3] = {0.0, 0.0, 0.0};
    if (nv < 2) {
        status = 1;
    } else {
        double s[3][3];
        for (int k = 0; k < 3; k++) llh_to_ecef(llh[3 * k], llh[3 * k + 1], llh[3 * k + 2], s[k]);
        double x[3];
        llh_to_ecef((llh[0] + llh[3] + llh[6]) / 3.0, (llh[1] + llh[4] + llh[7]) / 3.0, (llh[2] + llh[5] + llh[8]) / 3.0, x);
        for (int it = 0; it < 10 && status == 0; it++) {
            double r[3];
            for (int k = 0; k < 3; k++)
                r[k] = sqrt((x[0] - s[k][0]) * (x[0] - s[k][0]) + (x[1] - s[k][1]) * (x[1] - s[k][1]) +
                            (x[2] - s[k][2]) * (x[2] - s[k][2]));
            const double dx1 = (x[0] - s[0][0]) / r[0], dy1 = (x[1] - s[0][1]) / r[0];
            const double dx2 = (x[0] - s[1][0]) / r[1], dy2 = (x[1] - s[1][1]) / r[1];
            const double dx3 = (x[0] - s[2][0]) / r[2], dy3 = (x[1] - s[2][1]) / r[2];
            if (nv != 2) { status = 2; break; }
            const double res1 = (r[1] - r[0]) - valid[0];
            const double res2 = (r[2] - r[0]) - valid[1];
            const double J11 = dx2 - dx1, J12 = dy2 - dy1, J21 = dx3 - dx1, J22 = dy3 - dy1;
            if (fabs(res1) < 1.0 && fabs(res2) < 1.0) { converged = 1; break; }
            const double det = J22 * J11 - J21 * J12;
            n_iter = it + 1;
            double t_step = 0.0, t_code = 0.0;
            // trace may be NULL (tdoa_b200.h): one guarded store per iteration
            auto record = [&]() {
                if (trace) {
                    double *tr = trace + 5 * it;
                    tr[0] = det; tr[1] = res1; tr[2] = res2; tr[3] = t_step; tr[4] = t_code;
                }
            };
            if (fabs(det) < 1e-12) {
                double d = 0.0;
                if (fabs(J11) > fabs(J21) && fabs(J12) > 1e-10) { d = -res1 / J11; t_code = 2.0; }
                else if (fabs(J21) > 1e-10) { d = -res2 / J21; t_code = 3.0; }
                else { status = 3; record(); break; }
                x[0] += d * 0.1;
            } else {
                const double dx = (-res1 * J22 + J12 * res2) / det;
                const double dy = (res1 * J21 - J11 * res2) / det;
                const double step = sqrt(dx * dx + dy * dy);
                double scale = 0.7;
                if (step > 1000.0) { scale = 1000.0 / step * 0.7; t_code = 1.0; }
                t_step = step;
                x[0] += dx * scale;
                x[1] += dy * scale;
            }
            record();
        }
        if (status == 0) ecef_to_llh(x[0], x[1], x[2], o);
    }
    out_llh[0] = o[0]; out_llh[1] = o[1]; out_llh[2] = o[2];
    info[0] = status; info[1] = nv; info[2] = n_iter; info[3] = converged;
}

// ---------------------------------------------------------------- least-squares fix
// The statement and its body are in ls_core.cuh (the station check of exclude.cu runs the same function).
__global__ void k_solve_ls(const double *llh, int n_st, const double *rd_all, int n_sets, int rd_stride,
                           const double *init_llh, int dims, double *out_llh, double *out_rms, int *status, int *iters,
                           const uint8_t *used_all)
{
    extern __shared__ double s_st[];  // station ECEF
    for (int k = threadIdx.x; k < n_st; k += blockDim.x) llh_to_ecef(llh[3 * k], llh[3 * k + 1], llh[3 * k + 2], s_st + 3 * k);
    __syncthreads();
    const int set = blockIdx.x * blockDim.x + threadIdx.x;
    if (set >= n_sets) return;
    const double *rd = rd_all + (size_t)set * rd_stride;
    const uint8_t *used = used_all ? used_all + (size_t)set * rd_stride : nullptr;
    const LsFix F = ls_fix(s_st, n_st, rd, used, 0ull, dims, ls_start(llh, n_st, init_llh, set));
    out_llh[3 * set] = F.p.lat;
    out_llh[3 * set + 1] = F.p.lon;
    out_llh[3 * set + 2] = F.p.h;
    if (out_rms) out_rms[set] = F.rms;
    status[set] = F.status;
    if (iters) iters[set] = F.iters;
}

// ---------------------------------------------------------------- grid multilateration
// cost(cell, set) = sum over pairs i<j (lexicographic) of ((r_j - r_i) - rd_ij)^2, f64,
// terms added in pair order (as orc_grid_solve); arg-min, lowest linear index wins ties.
// The S ranges of a cell do not depend on the set, so one thread computes them once
// and sweeps every set; per-CTA minima go to scratch and a second kernel reduces them.
// Masked statement (tdoa_grid_masked, the windowed seed): the sum runs over the pairs with used[p] != 0 only, in the
// same order; an unused slot is never read (NaN there is fine); a set that is not searched -- no used pair, or the
// windowed fix's status-2 rule -- has no arg-min: index -1, cost NaN, out_llh left as it was.  used == NULL is the
// unmasked statement, and the kernels' kMasked = false instantiations are the unmasked kernels unchanged.
constexpr int kGridThreads = 128;
constexpr int kMaxStations = 16;
constexpr int kMaxPairs = kMaxStations * (kMaxStations - 1) / 2;
// a set's row of the ranked table: c[16], sum rd^2, 2 sum |rd|, unused pairs m, searched (1 / 0); a masked row then
// holds the m unused pairs as one byte each, i * 16 + j, in pair order
constexpr int kRankTab = 20;
constexpr int kRankTabMasked = kRankTab + (kMaxPairs + 7) / 8 + 1;   // 36 doubles: 16-byte aligned rows

struct GridDesc {
    double lat0, lon0, dlat, dlon;
    int nlat, nlon;
    double elev;
};

__device__ __forceinline__ GridDesc read_desc(const double *g)
{
    GridDesc d;
    d.lat0 = g[0]; d.lon0 = g[1]; d.dlat = g[2]; d.dlon = g[3];
    d.nlat = (int)g[4]; d.nlon = (int)g[5]; d.elev = g[6];
    return d;
}

template <bool kMasked>
__global__ void __launch_bounds__(kGridThreads) k_grid_cost(const double *llh, int n_st, const double *gdesc,
                                                           const double *rd_all, int n_sets, int rd_stride,
                                                           double *cta_cost, i64 *cta_idx, const uint8_t *used_all,
                                                           const double *tab)
{
    extern __shared__ double sm[];  // [n_st*3] station ECEF, then [kGridThreads] cost + idx scratch
    double *s_st = sm;
    double *s_cost = sm + 3 * kMaxStations;
    i64 *s_idx = reinterpret_cast<i64 *>(s_cost + kGridThreads);
    const GridDesc G = read_desc(gdesc);
    if (threadIdx.x < n_st) llh_to_ecef(llh[3 * threadIdx.x], llh[3 * threadIdx.x + 1], llh[3 * threadIdx.x + 2],
                                        s_st + 3 * threadIdx.x);
    __syncthreads();
    const i64 n_cells = (i64)G.nlat * G.nlon;
    const i64 cell = (i64)blockIdx.x * kGridThreads + threadIdx.x;
    double r[kMaxStations];
    const bool live = cell < n_cells;
    if (live) {
        const int a = (int)(cell / G.nlon), b = (int)(cell % G.nlon);
        double x[3];
        llh_to_ecef(G.lat0 + a * G.dlat, G.lon0 + b * G.dlon, G.elev, x);
#pragma unroll
        for (int k = 0; k < kMaxStations; k++) {
            if (k < n_st) {
                const double dx = x[0] - s_st[3 * k], dy = x[1] - s_st[3 * k + 1], dz = x[2] - s_st[3 * k + 2];
                r[k] = sqrt(dx * dx + dy * dy + dz * dz);
            } else {
                r[k] = 0.0;
            }
        }
    }
    for (int set = 0; set < n_sets; set++) {
        const double *rd = rd_all + (size_t)set * rd_stride;
        const uint8_t *used = kMasked ? used_all + (size_t)set * rd_stride : nullptr;
        const bool searched = !kMasked || tab[(size_t)set * kRankTabMasked + 19] != 0.0;
        double cost = 0.0;
        if (live && searched) {
            int p = 0;
#pragma unroll
            for (int i = 0; i < kMaxStations; i++) {
#pragma unroll
                for (int j = i + 1; j < kMaxStations; j++) {
                    if (j < n_st) {
                        if (!kMasked || used[p]) {
                            const double e = (r[j] - r[i]) - rd[p];
                            cost = __dadd_rn(cost, __dmul_rn(e, e));
                        }
                        p++;
                    }
                }
            }
        }
        // block arg-min (lowest index wins ties)
        s_cost[threadIdx.x] = cost;
        s_idx[threadIdx.x] = live && searched ? cell : (i64)-1;
        __syncthreads();
        for (int o = kGridThreads / 2; o > 0; o >>= 1) {
            if (threadIdx.x < o) {
                const i64 ia = s_idx[threadIdx.x], ib = s_idx[threadIdx.x + o];
                const double ca = s_cost[threadIdx.x], cb = s_cost[threadIdx.x + o];
                const bool take_b = ib >= 0 && (ia < 0 || cb < ca || (cb == ca && ib < ia));
                if (take_b) { s_cost[threadIdx.x] = cb; s_idx[threadIdx.x] = ib; }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            cta_cost[(size_t)set * gridDim.x + blockIdx.x] = s_cost[0];
            cta_idx[(size_t)set * gridDim.x + blockIdx.x] = s_idx[0];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) k_grid_reduce(const double *gdesc, const double *cta_cost, const i64 *cta_idx,
                                                    int n_cta, double *best_cost, i64 *best_idx, double *out_llh)
{
    __shared__ double s_cost[256];
    __shared__ i64 s_idx[256];
    const int set = blockIdx.x;
    double c = 0.0;
    i64 ix = -1;
    for (int i = threadIdx.x; i < n_cta; i += 256) {
        const double cc = cta_cost[(size_t)set * n_cta + i];
        const i64 ii = cta_idx[(size_t)set * n_cta + i];
        if (ii >= 0 && (ix < 0 || cc < c || (cc == c && ii < ix))) { c = cc; ix = ii; }
    }
    s_cost[threadIdx.x] = c;
    s_idx[threadIdx.x] = ix;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            const i64 ia = s_idx[threadIdx.x], ib = s_idx[threadIdx.x + o];
            const double ca = s_cost[threadIdx.x], cb = s_cost[threadIdx.x + o];
            if (ib >= 0 && (ia < 0 || cb < ca || (cb == ca && ib < ia))) { s_cost[threadIdx.x] = cb; s_idx[threadIdx.x] = ib; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const GridDesc G = read_desc(gdesc);
        const i64 bi = s_idx[0];
        best_cost[set] = bi >= 0 ? s_cost[0] : __longlong_as_double(0x7ff8000000000000ll);   // no arg-min: NaN
        best_idx[set] = bi;
        if (bi >= 0) {
            out_llh[3 * set] = G.lat0 + (double)(bi / G.nlon) * G.dlat;
            out_llh[3 * set + 1] = G.lon0 + (double)(bi % G.nlon) * G.dlon;
            out_llh[3 * set + 2] = G.elev;
        }
    }
}

}  // namespace

void launch_baselines(const double *d_llh, int n_st, double *d_out, cudaStream_t st)
{
    const int P = n_st * (n_st - 1) / 2;
    if (P <= 0) return;
    k_baselines<<<(P + 63) / 64, 64, 0, st>>>(d_llh, n_st, d_out);
}

void launch_solve(const double *d_llh, const double *d_rd, int n_sets, int rd_stride, double *d_out_llh,
                  int *d_status, int *d_iters, cudaStream_t st)
{
    if (n_sets <= 0) return;
    k_solve<<<(n_sets + 63) / 64, 64, 0, st>>>(d_llh, d_rd, n_sets, rd_stride, d_out_llh, d_status, d_iters);
}

void launch_solve_binary(const double *d_llh, const double *d_rd, int n_rd, double *d_out_llh, int *d_info, double *d_trace,
                         cudaStream_t st)
{
    k_solve_binary<<<1, 32, 0, st>>>(d_llh, d_rd, n_rd, d_out_llh, d_info, d_trace);
}

// ProcessTDOA between the pair loops and the solver (processor.go:821, :853, :899-903; shipped
// binary: "REFERENCE SIGNAL SYNCHRONIZATION"): dt = delay / fs per pair; SOURCE keeps the
// target differences, the binary's modes subtract the reference differences pair by pair;
// range difference = dt * c.  EXTENDED adds the sub-sample offset to the delay.
__global__ void k_range_diffs(const PeakRec *ref, const PeakRec *tgt, int n_pairs, double fs, int mode, double *td_out,
                              double *rd_out)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    double lt = (double)tgt[p].lag, lr = (double)ref[p].lag;
    if (mode == TDOA_MODE_EXTENDED) { lt += (double)tgt[p].frac; lr += (double)ref[p].frac; }
    const double tt = lt / fs, tr = lr / fs;
    const double td = mode == TDOA_MODE_SOURCE ? tt : tt - tr;
    td_out[p] = td;
    rd_out[p] = td * 299792458.0;
}

void launch_range_diffs(const PeakRec *d_ref, const PeakRec *d_tgt, int n_pairs, double fs, int mode, double *d_td,
                        double *d_rd, cudaStream_t st)
{
    if (n_pairs > 0) k_range_diffs<<<(n_pairs + 63) / 64, 64, 0, st>>>(d_ref, d_tgt, n_pairs, fs, mode, d_td, d_rd);
}

int solve_ls_max_stations() { return kLsMaxStations; }

void launch_solve_ls(const double *d_llh, int n_st, const double *d_rd, int n_sets, int rd_stride, const double *d_init,
                     int dims, double *d_out_llh, double *d_rms, int *d_status, int *d_iters, cudaStream_t st,
                     const uint8_t *d_used)
{
    if (n_sets <= 0) return;
    k_solve_ls<<<(n_sets + 31) / 32, 32, 3 * n_st * sizeof(double), st>>>(d_llh, n_st, d_rd, n_sets, rd_stride, d_init, dims,
                                                                       d_out_llh, d_rms, d_status, d_iters, d_used);
}

// ---------------------------------------------------------------- grid multilateration, ranked
// The cost above spends 4 f64 operations per (cell, set, pair): 480 per cell and set at 16 stations.  Expanded
// around q_k = r_k - r_0 (the cost only sees differences of ranges) it separates into a part of the cell, a
// part of the set and ONE dot product that couples them:
//     cost = [S sum q_k^2 - (sum q_k)^2]  -  2 sum_k q_k c_k  +  sum_p rd_p^2 ,
//     c_k  = sum_{i<k} rd_ik - sum_{j>k} rd_kj      (S = stations; c_k and sum rd^2 come from the host, per set)
// i.e. 16 fused multiply-adds per cell and set.  That form only RANKS cells (it cancels ~1e11 m^2 down to the
// cost): its rounding error is bounded by tol = kGridKappa * (2 S sum q^2 + 4 max|q| sum|rd| + sum rd^2), so the
// statement's arg-min x* satisfies f(x*) - tol(x*) <= min_x (f(x) + tol(x)) =: U.  k_grid_rank leaves per CTA and
// set the minima of f - tol and f + tol; k_grid_bound takes U; k_grid_refine revisits only the CTAs that can
// hold a cell under U and lists those cells (normally one per set); k_grid_exact evaluates the listed cells by the
// statement itself -- pair by pair in its order -- and k_grid_pick runs the statement's selection (strict <,
// lowest index on ties) on them.  The
// index and the cost are the statement's, bit for bit; config 5 (10^6 cells x 64 sets) 7.5 ms -> see DESIGN.md.
constexpr int kRankThreads = 128;
constexpr int kRankCells = 2;                    // cells per thread
constexpr int kRankSpan = kRankThreads * kRankCells;
constexpr double kGridKappa = 4e-13;             // ~3600 ulp of the largest partial result: far above the ~200 roundings
constexpr int kRankMaxSets = 512;                // per launch (shared memory: 64 B per set)

struct RankCell {
    double q[kMaxStations];
    double a;      // S sum q^2 - (sum q)^2
    double t0;     // 2 S sum q^2
    double qmax;
    bool live;
};

__device__ __forceinline__ void rank_cell(const GridDesc &G, const double *s_st, int n_st, i64 cell, i64 n_cells,
                                          RankCell &c, double *r_out)
{
    c.live = cell < n_cells;
    double r[kMaxStations];
    if (c.live) {
        const int a = (int)(cell / G.nlon), b = (int)(cell % G.nlon);
        double x[3];
        llh_to_ecef(G.lat0 + a * G.dlat, G.lon0 + b * G.dlon, G.elev, x);
#pragma unroll
        for (int k = 0; k < kMaxStations; k++) {
            if (k < n_st) {
                const double dx = x[0] - s_st[3 * k], dy = x[1] - s_st[3 * k + 1], dz = x[2] - s_st[3 * k + 2];
                r[k] = sqrt(dx * dx + dy * dy + dz * dz);
            } else {
                r[k] = 0.0;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < kMaxStations; k++) r[k] = 0.0;
    }
    double sq = 0.0, sl = 0.0, qm = 0.0;
#pragma unroll
    for (int k = 0; k < kMaxStations; k++) {
        const double q = k < n_st ? r[k] - r[0] : 0.0;
        c.q[k] = q;
        sq = __fma_rn(q, q, sq);
        sl += q;
        qm = fmax(qm, fabs(q));
    }
    c.a = (double)n_st * sq - sl * sl;
    c.t0 = 2.0 * (double)n_st * sq;
    c.qmax = qm;
    if (r_out) {
#pragma unroll
        for (int k = 0; k < kMaxStations; k++) r_out[k] = r[k];
    }
}

// f and tol of one cell for one set; tab = the set's row (c[16], B, C1; masked: m, searched, the unused pairs).
// Masked, the bracket loses the unused pairs' terms: a - sum_unused (q_j - q_i)^2 (m FMA more per cell and set);
// a set that is not searched gives NaN, which no bound comparison lets through.
template <bool kMasked>
__device__ __forceinline__ void rank_eval(const RankCell &c, const double2 *__restrict__ tab, double &lo, double &hi)
{
    double mid = 0.0;
#pragma unroll
    for (int m = 0; m < kMaxStations / 2; m++) {
        const double2 cc = __ldg(tab + m);
        mid = __fma_rn(c.q[2 * m], cc.x, mid);
        mid = __fma_rn(c.q[2 * m + 1], cc.y, mid);
    }
    const double2 bc = __ldg(tab + kMaxStations / 2);   // (sum rd^2, 2 sum |rd|)
    double a = c.a;
    if (kMasked) {
        const double2 ms = __ldg(tab + kMaxStations / 2 + 1);   // (unused pairs, searched)
        if (ms.y == 0.0) {
            lo = hi = __longlong_as_double(0x7ff8000000000000ll);
            return;
        }
        const uint8_t *code = reinterpret_cast<const uint8_t *>(tab + kRankTab / 2);
        double su = 0.0;
        for (int m = 0; m < (int)ms.x; m++) {
            const int k = __ldg(code + m);
            const double d = c.q[k & 15] - c.q[k >> 4];
            su = __fma_rn(d, d, su);
        }
        a = a - su;
    }
    const double f = __fma_rn(-2.0, mid, a + bc.x);
    const double tol = kGridKappa * (c.t0 + __fma_rn(2.0 * c.qmax, bc.y, bc.x));
    lo = f - tol;
    hi = f + tol;
}

__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

template <bool kMasked>
__global__ void __launch_bounds__(kRankThreads) k_grid_rank(const double *llh, int n_st, const double *gdesc,
                                                            const double *tab, int n_sets, double *cta_lo, double *cta_hi)
{
    constexpr int kTab = kMasked ? kRankTabMasked : kRankTab;
    extern __shared__ double sm[];   // [3 * 16] station ECEF, then [n_sets][4 warps] lo, [n_sets][4 warps] hi
    double *s_st = sm;
    double *s_lo = sm + 3 * kMaxStations;
    double *s_hi = s_lo + (size_t)n_sets * (kRankThreads / 32);
    const GridDesc G = read_desc(gdesc);
    if (threadIdx.x < n_st) llh_to_ecef(llh[3 * threadIdx.x], llh[3 * threadIdx.x + 1], llh[3 * threadIdx.x + 2],
                                        s_st + 3 * threadIdx.x);
    __syncthreads();
    const i64 n_cells = (i64)G.nlat * G.nlon;
    const i64 base = (i64)blockIdx.x * kRankSpan + threadIdx.x;
    RankCell c0, c1;
    rank_cell(G, s_st, n_st, base, n_cells, c0, nullptr);
    rank_cell(G, s_st, n_st, base + kRankThreads, n_cells, c1, nullptr);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    for (int set = 0; set < n_sets; set++) {
        const double2 *row = reinterpret_cast<const double2 *>(tab + (size_t)set * kTab);
        double lo0, hi0, lo1, hi1;
        rank_eval<kMasked>(c0, row, lo0, hi0);
        rank_eval<kMasked>(c1, row, lo1, hi1);
        double lo = fmin(c0.live ? lo0 : inf, c1.live ? lo1 : inf);
        double hi = fmin(c0.live ? hi0 : inf, c1.live ? hi1 : inf);
        lo = warp_min(lo);
        hi = warp_min(hi);
        if (lane == 0) { s_lo[set * (kRankThreads / 32) + wid] = lo; s_hi[set * (kRankThreads / 32) + wid] = hi; }
    }
    __syncthreads();
    for (int set = threadIdx.x; set < n_sets; set += kRankThreads) {
        double lo = inf, hi = inf;
#pragma unroll
        for (int w = 0; w < kRankThreads / 32; w++) {
            lo = fmin(lo, s_lo[set * (kRankThreads / 32) + w]);
            hi = fmin(hi, s_hi[set * (kRankThreads / 32) + w]);
        }
        cta_lo[(size_t)set * gridDim.x + blockIdx.x] = lo;
        cta_hi[(size_t)set * gridDim.x + blockIdx.x] = hi;
    }
}

__global__ void __launch_bounds__(256) k_grid_bound(const double *cta_hi, int n_cta, double *bound)
{
    __shared__ double s_m[8];
    const int set = blockIdx.x;
    double m = __longlong_as_double(0x7ff0000000000000ll);
    for (int i = threadIdx.x; i < n_cta; i += 256) m = fmin(m, cta_hi[(size_t)set * n_cta + i]);
    m = warp_min(m);
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 1; w < 8; w++) m = fmin(m, s_m[w]);
        bound[set] = m;
    }
}

struct GridCand { i64 cell; double cost; int set; int pad; };

template <bool kMasked>
__global__ void __launch_bounds__(kRankThreads) k_grid_refine(const double *llh, int n_st, const double *gdesc,
                                                              const double *tab, const double *rd_all, int n_sets,
                                                              int rd_stride, const double *cta_lo, const double *bound,
                                                              GridCand *cands, int cap, int *n_cand)
{
    constexpr int kTab = kMasked ? kRankTabMasked : kRankTab;
    __shared__ double s_st[3 * kMaxStations];
    __shared__ int s_sets[kRankMaxSets];
    __shared__ int s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    for (int set = threadIdx.x; set < n_sets; set += kRankThreads)
        if (cta_lo[(size_t)set * gridDim.x + blockIdx.x] <= bound[set] && (!kMasked || tab[(size_t)set * kTab + 19] != 0.0))
            s_sets[atomicAdd(&s_n, 1)] = set;
    __syncthreads();
    const int ns = s_n;
    if (ns == 0) return;   // nearly every CTA
    const GridDesc G = read_desc(gdesc);
    if (threadIdx.x < n_st) llh_to_ecef(llh[3 * threadIdx.x], llh[3 * threadIdx.x + 1], llh[3 * threadIdx.x + 2],
                                        s_st + 3 * threadIdx.x);
    __syncthreads();
    const i64 n_cells = (i64)G.nlat * G.nlon;
    for (int h = 0; h < kRankCells; h++) {
        const i64 cell = (i64)blockIdx.x * kRankSpan + h * kRankThreads + threadIdx.x;
        RankCell c;
        rank_cell(G, s_st, n_st, cell, n_cells, c, nullptr);
        if (!c.live) continue;
        for (int u = 0; u < ns; u++) {
            const int set = s_sets[u];
            double lo, hi;
            rank_eval<kMasked>(c, reinterpret_cast<const double2 *>(tab + (size_t)set * kTab), lo, hi);
            if (!(lo <= bound[set])) continue;
            const int slot = atomicAdd(n_cand, 1);
            if (slot < cap) cands[slot] = GridCand{cell, 0.0, set, 0};
        }
    }
}

// The statement itself (k_grid_cost / orc_grid_solve) on the surviving (cell, set) pairs, one thread each: pair by
// pair, in order, no contraction.  (Inside k_grid_refine the survivors of all sets sit in two or three
// neighbouring cells, i.e. in one warp, and their 120-term chains ran one after the other: 0.41 ms of 0.75.)
template <bool kMasked>
__global__ void __launch_bounds__(kRankThreads) k_grid_exact(const double *llh, int n_st, const double *gdesc,
                                                             const double *rd_all, int rd_stride, GridCand *cands, int cap,
                                                             const int *n_cand, const uint8_t *used_all)
{
    __shared__ double s_st[3 * kMaxStations];
    const int n = min(*n_cand, cap);
    if ((int)(blockIdx.x * kRankThreads) >= n) return;
    const GridDesc G = read_desc(gdesc);
    if (threadIdx.x < n_st) llh_to_ecef(llh[3 * threadIdx.x], llh[3 * threadIdx.x + 1], llh[3 * threadIdx.x + 2],
                                        s_st + 3 * threadIdx.x);
    __syncthreads();
    const int i = blockIdx.x * kRankThreads + threadIdx.x;
    if (i >= n) return;
    const GridCand g = cands[i];
    RankCell c;
    double r[kMaxStations];
    rank_cell(G, s_st, n_st, g.cell, (i64)G.nlat * G.nlon, c, r);
    const double *rd = rd_all + (size_t)g.set * rd_stride;
    const uint8_t *used = kMasked ? used_all + (size_t)g.set * rd_stride : nullptr;
    double cost = 0.0;
    int p = 0;
#pragma unroll
    for (int a = 0; a < kMaxStations; a++) {
#pragma unroll
        for (int b = a + 1; b < kMaxStations; b++) {
            if (b < n_st) {
                if (!kMasked || used[p]) {
                    const double e = (r[b] - r[a]) - rd[p];
                    cost = __dadd_rn(cost, __dmul_rn(e, e));
                }
                p++;
            }
        }
    }
    cands[i].cost = cost;
}

__global__ void __launch_bounds__(128) k_grid_pick(const double *gdesc, const GridCand *cands, int cap, const int *n_cand,
                                                  double *best_cost, i64 *best_idx, double *out_llh)
{
    __shared__ double s_cost[128];
    __shared__ i64 s_idx[128];
    const int set = blockIdx.x;
    const int n = min(*n_cand, cap);
    double c = 0.0;
    i64 ix = -1;
    for (int i = threadIdx.x; i < n; i += 128) {
        const GridCand g = cands[i];
        if (g.set == set && (ix < 0 || g.cost < c || (g.cost == c && g.cell < ix))) { c = g.cost; ix = g.cell; }
    }
    s_cost[threadIdx.x] = c;
    s_idx[threadIdx.x] = ix;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            const i64 ia = s_idx[threadIdx.x], ib = s_idx[threadIdx.x + o];
            const double ca = s_cost[threadIdx.x], cb = s_cost[threadIdx.x + o];
            if (ib >= 0 && (ia < 0 || cb < ca || (cb == ca && ib < ia))) { s_cost[threadIdx.x] = cb; s_idx[threadIdx.x] = ib; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const GridDesc G = read_desc(gdesc);
        const i64 bi = s_idx[0];
        best_cost[set] = bi >= 0 ? s_cost[0] : __longlong_as_double(0x7ff8000000000000ll);   // no arg-min: NaN
        best_idx[set] = bi;
        if (bi >= 0) {
            out_llh[3 * set] = G.lat0 + (double)(bi / G.nlon) * G.dlat;
            out_llh[3 * set + 1] = G.lon0 + (double)(bi % G.nlon) * G.dlon;
            out_llh[3 * set + 2] = G.elev;
        }
    }
}

// One set's row of the ranked table from its range differences (c_k, sum rd^2 and 2 sum |rd| over the used pairs,
// the unused pairs), on the host for tdoa_grid / tdoa_grid_masked and in k_grid_rows for the windowed seed.  Products
// and sums are separate roundings on both sides (solve.cu is compiled without contraction).
__host__ __device__ inline void grid_row_fill(const double *rd, const uint8_t *used, int n_st, bool searched, double *row)
{
    double c[kMaxStations];
    for (int k = 0; k < kMaxStations; k++) c[k] = 0.0;
    double b = 0.0;
    int p = 0, m = 0;
    uint8_t *code = reinterpret_cast<uint8_t *>(row + kRankTab);
    for (int i = 0; i < n_st; i++)
        for (int j = i + 1; j < n_st; j++, p++) {
            if (used && !used[p]) {
                code[m++] = (uint8_t)(i * 16 + j);
                continue;
            }
            c[j] += rd[p];
            c[i] -= rd[p];
            b += rd[p] * rd[p];
        }
    // the bound takes sum |rd| over the terms of every c_k (not sum |c_k|: a c_k that cancels keeps its rounding)
    double c1 = 0.0;
    p = 0;
    for (int i = 0; i < n_st; i++)
        for (int j = i + 1; j < n_st; j++, p++)
            if (!used || used[p]) c1 += 2.0 * (rd[p] < 0 ? -rd[p] : rd[p]);
    for (int k = 0; k < kMaxStations; k++) row[k] = c[k];
    row[16] = b;
    row[17] = c1;
    row[18] = (double)m;
    row[19] = searched ? 1.0 : 0.0;
}

// the windowed seed's rows, one thread per set: searched unless the least-squares step would refuse the set (status 2)
__global__ void k_grid_rows(const double *rd_all, const uint8_t *used_all, int n_sets, int rd_stride, int n_st, int dims,
                            double *tab)
{
    const int set = blockIdx.x * blockDim.x + threadIdx.x;
    if (set >= n_sets) return;
    const uint8_t *used = used_all + (size_t)set * rd_stride;
    grid_row_fill(rd_all + (size_t)set * rd_stride, used, n_st, ls_used_pairs(used, n_st, dims) >= 0,
                  tab + (size_t)set * kRankTabMasked);
}

int grid_rank_tab_doubles(bool masked) { return masked ? kRankTabMasked : kRankTab; }
int grid_rank_chunks(int n_sets) { return (n_sets + kRankMaxSets - 1) / kRankMaxSets; }

// the candidate table of a chunk of n_sets sets
static int rank_cand_cap(int n_sets) { return 64 * n_sets + 1024; }

bool grid_rank_overflowed(const int *h_count, int n_sets)
{
    for (int c = 0; c < grid_rank_chunks(n_sets); c++)
        if (h_count[c] > rank_cand_cap(std::min(kRankMaxSets, n_sets - c * kRankMaxSets))) return true;
    return false;
}

static int rank_n_cta(int nlat, int nlon)
{
    const i64 cells = (i64)nlat * nlon;
    return (int)((cells + kRankSpan - 1) / kRankSpan);
}

// one chunk's scratch, which every chunk reuses: [n_sets][n_cta] lo, [n_sets][n_cta] hi, [n_sets] bound, candidates, counter
size_t grid_rank_scratch_bytes(int nlat, int nlon, int n_sets)
{
    n_sets = std::min(n_sets, kRankMaxSets);
    const size_t n_cta = (size_t)rank_n_cta(nlat, nlon);
    return (2 * n_cta * (size_t)n_sets + (size_t)n_sets) * sizeof(double) +
           (size_t)rank_cand_cap(n_sets) * sizeof(GridCand) + 64;
}

// Host rows (tdoa_grid, tdoa_grid_masked): the range differences are on the host already, and building the rows there
// keeps the ranked arg-min at five launches per 512 sets.  used == nullptr: the unmasked row; masked, a set without a
// used pair is not searched.  Returns whether the set is searched.
bool grid_rank_row(const double *rd, const uint8_t *used, int n_st, double *row)
{
    const bool searched = !used || ls_used_pairs(used, n_st, 0) >= 0;
    grid_row_fill(rd, used, n_st, searched, row);
    return searched;
}

void launch_grid_rows(const double *d_rd, const uint8_t *d_used, int n_sets, int rd_stride, int n_st, int dims, double *d_tab,
                      cudaStream_t st)
{
    if (n_sets > 0) k_grid_rows<<<(n_sets + 63) / 64, 64, 0, st>>>(d_rd, d_used, n_sets, rd_stride, n_st, dims, d_tab);
}

// five launches per chunk of kRankMaxSets sets.  d_count: grid_rank_chunks(n_sets) ints, read back by the caller after
// the stream has drained -- grid_rank_overflowed means the table is incomplete (launch_grid_cells then).
void launch_grid_ranked(const double *d_llh, int n_st, const double *d_grid_desc, int nlat, int nlon, const double *d_tab,
                        const double *d_rd, int n_sets, int rd_stride, double *d_best_cost, i64 *d_best_idx,
                        double *d_out_llh, void *d_scratch, int *d_count, cudaStream_t st, const uint8_t *d_used)
{
    const int n_cta = rank_n_cta(nlat, nlon);
    if (n_cta <= 0 || n_sets <= 0) return;
    cudaMemsetAsync(d_count, 0, (size_t)grid_rank_chunks(n_sets) * sizeof(int), st);
    auto chunks = [&](auto masked) {
        constexpr bool kMasked = decltype(masked)::value;
        constexpr int kTab = kMasked ? kRankTabMasked : kRankTab;
        for (int c = 0, s0 = 0; s0 < n_sets; c++, s0 += kRankMaxSets) {
            const int ns = std::min(kRankMaxSets, n_sets - s0), cap = rank_cand_cap(ns);
            const double *tab = d_tab + (size_t)s0 * kTab, *rd = d_rd + (size_t)s0 * rd_stride;
            double *cta_lo = reinterpret_cast<double *>(d_scratch);
            double *cta_hi = cta_lo + (size_t)n_cta * ns;
            double *bound = cta_hi + (size_t)n_cta * ns;
            GridCand *cands = reinterpret_cast<GridCand *>(bound + ns);
            const size_t smem = (3 * kMaxStations + 2 * (size_t)ns * (kRankThreads / 32)) * sizeof(double);
            const int n_exact = (cap + kRankThreads - 1) / kRankThreads;
            k_grid_rank<kMasked><<<n_cta, kRankThreads, smem, st>>>(d_llh, n_st, d_grid_desc, tab, ns, cta_lo, cta_hi);
            k_grid_bound<<<ns, 256, 0, st>>>(cta_hi, n_cta, bound);
            k_grid_refine<kMasked><<<n_cta, kRankThreads, 0, st>>>(d_llh, n_st, d_grid_desc, tab, rd, ns, rd_stride, cta_lo,
                                                                   bound, cands, cap, d_count + c);
            k_grid_exact<kMasked><<<n_exact, kRankThreads, 0, st>>>(d_llh, n_st, d_grid_desc, rd, rd_stride, cands, cap,
                                                                    d_count + c,
                                                                    kMasked ? d_used + (size_t)s0 * rd_stride : nullptr);
            k_grid_pick<<<ns, 128, 0, st>>>(d_grid_desc, cands, cap, d_count + c, d_best_cost + s0, d_best_idx + s0,
                                            d_out_llh + 3 * s0);
        }
    };
    if (d_used) chunks(std::true_type{}); else chunks(std::false_type{});
}

static int grid_n_cta(int nlat, int nlon)
{
    const i64 cells = (i64)nlat * nlon;
    return (int)((cells + kGridThreads - 1) / kGridThreads);
}

size_t grid_scratch_bytes(int nlat, int nlon, int n_sets)
{
    return (size_t)grid_n_cta(nlat, nlon) * (size_t)n_sets * (sizeof(double) + sizeof(i64));
}

void launch_grid_cells(const double *d_llh, int n_st, const double *d_grid_desc, int nlat, int nlon,
                       const double *d_rd, int n_sets, int rd_stride, double *d_best_cost, i64 *d_best_idx,
                       double *d_out_llh, void *d_scratch, cudaStream_t st, const uint8_t *d_used, const double *d_tab)
{
    const int n_cta = grid_n_cta(nlat, nlon);
    if (n_cta <= 0 || n_sets <= 0) return;
    double *cta_cost = reinterpret_cast<double *>(d_scratch);
    i64 *cta_idx = reinterpret_cast<i64 *>(cta_cost + (size_t)n_cta * n_sets);
    const size_t smem = (3 * kMaxStations + kGridThreads) * sizeof(double) + kGridThreads * sizeof(i64);
    auto cells = [&](auto masked) {
        k_grid_cost<decltype(masked)::value><<<n_cta, kGridThreads, smem, st>>>(d_llh, n_st, d_grid_desc, d_rd, n_sets, rd_stride,
                                                                                cta_cost, cta_idx, d_used, d_tab);
    };
    if (d_used) cells(std::true_type{}); else cells(std::false_type{});
    k_grid_reduce<<<n_sets, 256, 0, st>>>(d_grid_desc, cta_cost, cta_idx, n_cta, d_best_cost, d_best_idx, d_out_llh);
}

}  // namespace tdoa
