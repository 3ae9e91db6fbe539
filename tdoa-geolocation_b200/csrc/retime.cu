// retime.cu -- re-timed target correlation (tdoa_process_windows_retimed; no reference equivalent; restated in
// tests/retime_oracle.py).
//
// Clock error belongs to a station, not to a pair: the REF fit's pair slopes satisfy beta_ij = c_j - c_i.  Once
// every station's TGT plane is re-timed by its own rate, every pair of planes is drift-free and a TGT window can be
// as long as the block.
//   k_station_rates  one CTA: the station rates c[S] from the per-pair REF fits (k_window_ref_fit), a small dense
//                    least-squares solve in f64 (statement in include/tdoa_b200.h, tdoa_process_windows_retimed)
//   k_retime         the gather x~[n] = x[n + delta(n)] of one preprocessed plane, 8 B per sample.  delta is a step
//                    function that changes at most once per 1/|c| samples, so a tile evaluates the f64 formula at
//                    its two ends and at its few change points only (a binary search each), stages the source run
//                    it needs in shared memory with 16-byte loads and writes 16-byte stores.
// Both follow the statement operation for operation (__dmul_rn / __dadd_rn / __dsub_rn / __ddiv_rn / __dsqrt_rn:
// no contraction), so the restatement reproduces the bits.
#include <cuda_runtime.h>

#include <cstdint>

#include "kernels.h"

namespace tdoa {

namespace {

constexpr int kRatesMaxStations = 64;
constexpr int kRetimeTile = 4096;      // output samples per CTA
constexpr int kRetimeThreads = 256;
constexpr int kRetimeMaxSteps = 32;    // change points a tile takes on the staged path
constexpr int kRetimeLoads = (kRetimeTile + kRetimeMaxSteps + 8) / 4 / kRetimeThreads + 1;   // 16-byte loads per thread

__global__ void __launch_bounds__(kRatesMaxStations) k_station_rates(const double *__restrict__ fit, int n_st,
                                                                     double *__restrict__ rate, double *__restrict__ clock)
{
    __shared__ double A[kRatesMaxStations][kRatesMaxStations + 1];
    __shared__ double b[kRatesMaxStations];
    __shared__ int comp[kRatesMaxStations], fitted[kRatesMaxStations];
    const int t = threadIdx.x, S = n_st;
    if (t == 0) {
        // components of the fitted-pair graph: every station ends labelled with the smallest index of its component
        for (int k = 0; k < S; k++) { comp[k] = k; fitted[k] = 0; }
        for (bool changed = true; changed;) {
            changed = false;
            for (int i = 0, p = 0; i < S; i++)
                for (int j = i + 1; j < S; j++, p++) {
                    if (!(fit[(size_t)kWindowFitDoubles * p + 3] >= 2.0)) continue;
                    const int m = min(comp[i], comp[j]);
                    if (comp[i] != m || comp[j] != m) { comp[i] = comp[j] = m; changed = true; }
                }
        }
        // normal equations of the fitted pairs, plus one all-ones block per component (the zero-sum gauge)
        for (int i = 0; i < S; i++) {
            b[i] = 0.0;
            for (int j = 0; j < S; j++) A[i][j] = comp[i] == comp[j] ? 1.0 : 0.0;
        }
        for (int i = 0, p = 0; i < S; i++)
            for (int j = i + 1; j < S; j++, p++) {
                const double *f = fit + (size_t)kWindowFitDoubles * p;
                if (!(f[3] >= 2.0)) continue;
                A[i][i] += 1.0; A[j][j] += 1.0; A[i][j] -= 1.0; A[j][i] -= 1.0;
                b[i] = __dsub_rn(b[i], f[1]);
                b[j] = __dadd_rn(b[j], f[1]);
                fitted[i] = fitted[j] = 1;
            }
    }
    __syncthreads();
    // Cholesky, right-looking, row t on thread t: A[i][j] -= L[i][k] L[j][k] in k order
    for (int k = 0; k < S; k++) {
        if (t == k) A[k][k] = __dsqrt_rn(A[k][k]);
        __syncthreads();
        if (t > k && t < S) A[t][k] = __ddiv_rn(A[t][k], A[k][k]);
        __syncthreads();
        if (t > k && t < S)
            for (int j = k + 1; j <= t; j++) A[t][j] = __dsub_rn(A[t][j], __dmul_rn(A[t][k], A[j][k]));
        __syncthreads();
    }
    // L y = b, then L^T c = y, both column by column (b holds y, then c)
    for (int k = 0; k < S; k++) {
        if (t == k) b[k] = __ddiv_rn(b[k], A[k][k]);
        __syncthreads();
        if (t > k && t < S) b[t] = __dsub_rn(b[t], __dmul_rn(A[t][k], b[k]));
        __syncthreads();
    }
    for (int k = S - 1; k >= 0; k--) {
        if (t == k) b[k] = __ddiv_rn(b[k], A[k][k]);
        __syncthreads();
        if (t < k) b[t] = __dsub_rn(b[t], __dmul_rn(A[k][t], b[k]));
        __syncthreads();
    }
    if (t < S) {
        rate[t] = b[t];   // exactly 0 for a station without a fitted pair
        clock[t] = fitted[t] ? b[t] : __longlong_as_double(0x7ff8000000000000ll);
    }
}

// delta(n) = floor(c (n - n_c) + 0.5); n - n_c is exact (n < 2^52, n_c a multiple of 1/2)
__device__ __forceinline__ double retime_shift(double c, i64 n, double nc)
{
    return floor(__dadd_rn(__dmul_rn(c, __dsub_rn((double)n, nc)), 0.5));
}

__global__ void __launch_bounds__(kRetimeThreads) k_retime(const RetimeJob *__restrict__ jobs, const double *__restrict__ rates)
{
    const RetimeJob J = jobs[blockIdx.y];
    const i64 t0 = (i64)blockIdx.x * kRetimeTile;
    if (t0 >= J.n) return;
    const i64 t1 = min(t0 + (i64)kRetimeTile, J.n);
    const double c = rates[J.station];
    const double nc = __dmul_rn((double)(J.n - 1), 0.5);
    // delta is monotone in n (c fixed; every step rounds monotonically): its values on the tile lie between the ends
    const double d0 = retime_shift(c, t0, nc), d1 = retime_shift(c, t1 - 1, nc);
    if (!(fabs(d1 - d0) <= kRetimeMaxSteps && fabs(d0) < 0x1p40 && fabs(d1) < 0x1p40)) {
        // a rate far beyond any clock's (|c| > 1/128): the formula per sample; an index off the plane reads 0
        for (i64 n = t0 + threadIdx.x; n < t1; n += kRetimeThreads) {
            const double s = (double)n + retime_shift(c, n, nc);
            J.y[n] = s >= 0.0 && s < (double)J.n ? J.x[(i64)s] : 0.f;
        }
        return;
    }
    __shared__ __align__(16) float sh[kRetimeLoads * kRetimeThreads * 4];
    __shared__ i64 cp[kRetimeMaxSteps];
    const i64 s0 = (i64)d0;
    const int m = (int)fabs(d1 - d0), sgn = d1 < d0 ? -1 : 1;
    // change point k: the first n of the tile at which sgn (delta(n) - delta(t0)) >= k + 1 (delta(t1 - 1) is there)
    if (threadIdx.x < m) {
        const int k = threadIdx.x;
        i64 lo = t0 + 1, hi = t1 - 1;
        while (lo < hi) {
            const i64 mid = lo + (hi - lo) / 2;
            if (sgn * (retime_shift(c, mid, nc) - d0) >= (double)(k + 1)) hi = mid;
            else lo = mid + 1;
        }
        cp[k] = lo;
    }
    // the source samples of the tile that exist, [a, z), staged from the 16-byte boundary a4 at or below a
    const i64 lo_d = sgn > 0 ? s0 : s0 - m, hi_d = sgn > 0 ? s0 + m : s0;
    const i64 a = max(t0 + lo_d, (i64)0), z = min(t1 + hi_d, J.n);
    const i64 a4 = a & ~(i64)3;
    const bool aligned = (reinterpret_cast<uintptr_t>(J.x) & 15) == 0;
    float4 v[kRetimeLoads];
#pragma unroll
    for (int r = 0; r < kRetimeLoads; r++) {
        const i64 q = a4 + 4 * (i64)(threadIdx.x + r * kRetimeThreads);
        if (q >= z) continue;
        if (aligned && q + 4 <= J.n) {
            v[r] = __ldcs(reinterpret_cast<const float4 *>(J.x + q));
        } else {
            v[r].x = J.x[q];
            v[r].y = q + 1 < J.n ? J.x[q + 1] : 0.f;
            v[r].z = q + 2 < J.n ? J.x[q + 2] : 0.f;
            v[r].w = q + 3 < J.n ? J.x[q + 3] : 0.f;
        }
    }
#pragma unroll
    for (int r = 0; r < kRetimeLoads; r++) {
        const int u = threadIdx.x + r * kRetimeThreads;
        if (a4 + 4 * (i64)u < z) reinterpret_cast<float4 *>(sh)[u] = v[r];
    }
    __syncthreads();
    for (i64 q = t0 + 4 * (i64)threadIdx.x; q < t1; q += 4 * kRetimeThreads) {
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const i64 n = q + j;
            int level = 0;
            for (int k = 0; k < m; k++) level += cp[k] <= n;
            const i64 s = n + s0 + sgn * level;
            o[j] = n < t1 && s >= a && s < z ? sh[s - a4] : 0.f;
        }
        if (q + 4 <= t1) {
            __stcg(reinterpret_cast<float4 *>(J.y + q), make_float4(o[0], o[1], o[2], o[3]));
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (q + j < t1) J.y[q + j] = o[j];
        }
    }
}

}  // namespace

void launch_station_rates(const double *d_fit, int n_st, double *d_rate, double *d_clock, cudaStream_t st)
{
    k_station_rates<<<1, kRatesMaxStations, 0, st>>>(d_fit, n_st, d_rate, d_clock);
}

void launch_retime(const RetimeJob *d_jobs, int n_jobs, i64 max_n, const double *d_rates, cudaStream_t st)
{
    if (n_jobs <= 0 || max_n <= 0) return;
    const dim3 grid((unsigned)((max_n + kRetimeTile - 1) / kRetimeTile), (unsigned)n_jobs);
    k_retime<<<grid, kRetimeThreads, 0, st>>>(d_jobs, d_rates);
}

}  // namespace tdoa
