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
//   k_window_closure one CTA per TGT window (the _closure windowed calls, tdoa_closure): the same solve with the
//                    window's range differences in place of the slopes, and the drop of the pairs the rest of the
//                    window contradicts (statement in include/tdoa_b200.h, tdoa_closure; tests/closure_oracle.py)
// All three follow the statement operation for operation (__dmul_rn / __dadd_rn / __dsub_rn / __ddiv_rn / __dsqrt_rn:
// no contraction), so the restatement reproduces the bits.
#include <cuda_runtime.h>

#include <cstdint>

#include "graph_ls.cuh"
#include "kernels.h"

namespace tdoa {

namespace {

constexpr int kRatesMaxStations = kGraphLsMaxStations;
constexpr int kClosureThreads = 64;
constexpr int kClosureMaxPairs = kGraphLsMaxStations * (kGraphLsMaxStations - 1) / 2;
constexpr int kRetimeTile = 4096;      // output samples per CTA
constexpr int kRetimeThreads = 256;
constexpr int kRetimeMaxSteps = 32;    // change points a tile takes on the staged path
constexpr int kRetimeLoads = (kRetimeTile + kRetimeMaxSteps + 8) / 4 / kRetimeThreads + 1;   // 16-byte loads per thread

__global__ void __launch_bounds__(kRatesMaxStations) k_station_rates(const double *__restrict__ fit, int n_st,
                                                                     double *__restrict__ rate, double *__restrict__ clock)
{
    __shared__ GraphLsMatrix A[kRatesMaxStations];
    __shared__ double b[kRatesMaxStations];
    __shared__ int comp[kRatesMaxStations], deg[kRatesMaxStations];
    const int t = threadIdx.x, S = n_st;
    auto fitted = [&](int p) { return fit[(size_t)kWindowFitDoubles * p + 3] >= 2.0; };
    auto slope = [&](int p) { return fit[(size_t)kWindowFitDoubles * p + 1]; };
    graph_components(S, t, comp, fitted);
    graph_normal(S, t, comp, A, b, deg, fitted, slope);
    graph_ls_solve(S, t, A, b);
    if (t < S) {
        rate[t] = b[t];   // exactly 0 for a station without a fitted pair
        clock[t] = deg[t] ? b[t] : __longlong_as_double(0x7ff8000000000000ll);
    }
}

// One TGT window per CTA (include/tdoa_b200.h, tdoa_closure): station ranges tau from the window's used range
// differences, the residual of every usable pair, and the drop of the pair with the largest |residual| (with the
// pairs the degree rule takes after it) while that residual exceeds max_resid.  Each drop solves again from scratch,
// so every solve is the stated one.  used[P] in: the usable mask u (0 / 1); out: 0, 1 used, 2 dropped.  mask[P]
// (may be nullptr): the final 0 / 1 mask the fix reads.  resid[P] (may be nullptr): NaN where u = 0.
__global__ void __launch_bounds__(kClosureThreads) k_window_closure(const double *__restrict__ rd_all, uint8_t *used_all,
                                                                    uint8_t *mask_all, int n_st, int stride, int dims,
                                                                    double max_resid, int max_drop, double *resid_all,
                                                                    int *dropped)
{
    __shared__ GraphLsMatrix A[kGraphLsMaxStations];
    __shared__ double b[kGraphLsMaxStations];
    __shared__ int comp[kGraphLsMaxStations], deg[kGraphLsMaxStations];
    __shared__ uint8_t u[kClosureMaxPairs], m[kClosureMaxPairs], cut[kClosureMaxPairs];
    __shared__ uint8_t pi[kClosureMaxPairs], pj[kClosureMaxPairs];
    __shared__ double best_v[kClosureThreads / 32];
    __shared__ int best_p[kClosureThreads / 32];
    __shared__ int s_drops, s_go, s_keep;
    const int t = threadIdx.x, S = n_st, P = S * (S - 1) / 2;
    const double *rd = rd_all + (size_t)blockIdx.x * stride;
    uint8_t *used = used_all + (size_t)blockIdx.x * stride;
    double *resid = resid_all ? resid_all + (size_t)blockIdx.x * stride : nullptr;
    for (int i = 0, p = 0; i < S; i++)
        for (int j = i + 1; j < S; j++, p++)
            if (p % kClosureThreads == t) { pi[p] = (uint8_t)i; pj[p] = (uint8_t)j; }
    for (int p = t; p < P; p += kClosureThreads) { u[p] = m[p] = used[p] != 0; cut[p] = 0; }
    if (t == 0) s_drops = 0;
    __syncthreads();
    auto in_m = [&](int p) { return m[p] != 0; };
    auto rd_of = [&](int p) { return rd[p]; };
    for (;;) {
        graph_components(S, t, comp, in_m);
        graph_normal(S, t, comp, A, b, deg, in_m, rd_of);
        graph_ls_solve(S, t, A, b);
        // residuals of the usable pairs; the m-pair with the largest |e| (ties: the lowest p)
        double bv = -1.0;
        int bp = -1;
        for (int p = t; p < P; p += kClosureThreads) {
            double e = __longlong_as_double(0x7ff8000000000000ll);
            if (u[p]) {
                e = __dsub_rn(rd[p], __dsub_rn(b[pj[p]], b[pi[p]]));
                if (m[p] && fabs(e) > bv) { bv = fabs(e); bp = p; }
            }
            if (resid) resid[p] = e;
        }
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_down_sync(0xffffffffu, bv, off);
            const int op = __shfl_down_sync(0xffffffffu, bp, off);
            if (op >= 0 && (ov > bv || (ov == bv && op < bp))) { bv = ov; bp = op; }
        }
        if ((t & 31) == 0) { best_v[t >> 5] = bv; best_p[t >> 5] = bp; }
        __syncthreads();
        if (t == 0) {
            for (int w = 1; w < kClosureThreads / 32; w++)
                if (best_p[w] >= 0 && (best_v[w] > bv || (best_v[w] == bv && best_p[w] < bp))) { bv = best_v[w]; bp = best_p[w]; }
            // redundancy = used pairs - stations they touch + components among those stations
            int n2 = 0, touched = 0, comps = 0;
            for (int s = 0; s < S; s++) {
                n2 += deg[s];
                touched += deg[s] > 0;
                comps += deg[s] > 0 && comp[s] == s;
            }
            bool go = n2 / 2 - touched + comps >= 2 && !(max_drop > 0 && s_drops >= max_drop) && bp >= 0 && bv > max_resid;
            s_keep = 1;
            if (go) {
                // the tentative drop: q, then every station that lost a pair here and has one pair left loses it too
                unsigned long long lost = 0ull;
                int n_cut = 0;
                for (int q = bp; q >= 0;) {
                    const int i = pi[q], j = pj[q];
                    m[q] = 0; cut[q] = 1; n_cut++;
                    deg[i]--; deg[j]--;
                    lost |= (1ull << i) | (1ull << j);
                    q = -1;
                    for (int s = 0; s < S && q < 0; s++) {
                        if (!((lost >> s) & 1ull) || deg[s] != 1) continue;
                        for (int k = 0; k < S && q < 0; k++)
                            if (k != s && m[graph_pair(min(s, k), max(s, k), S)]) q = graph_pair(min(s, k), max(s, k), S);
                    }
                }
                if (ls_used_pairs(m, S, dims) < 0) { go = false; s_keep = 0; }
                else s_drops += n_cut;
            }
            s_go = go;
        }
        __syncthreads();
        const bool go = s_go, keep = s_keep;
        for (int p = t; p < P; p += kClosureThreads) {
            if (cut[p] && !keep) m[p] = 1;
            cut[p] = 0;
        }
        __syncthreads();
        if (!go) break;
    }
    for (int p = t; p < P; p += kClosureThreads) {
        if (mask_all) mask_all[(size_t)blockIdx.x * stride + p] = m[p];
        used[p] = u[p] ? (m[p] ? 1 : 2) : 0;
    }
    if (t == 0 && dropped) dropped[blockIdx.x] = s_drops;
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

void launch_window_closure(const double *d_rd, uint8_t *d_used, uint8_t *d_mask, int n_sets, int stride, int n_st, int dims,
                           double max_resid, int max_drop, double *d_resid, int *d_dropped, cudaStream_t st)
{
    if (n_sets > 0)
        k_window_closure<<<n_sets, kClosureThreads, 0, st>>>(d_rd, d_used, d_mask, n_st, stride, dims, max_resid, max_drop,
                                                           d_resid, d_dropped);
}

void launch_retime(const RetimeJob *d_jobs, int n_jobs, i64 max_n, const double *d_rates, cudaStream_t st)
{
    if (n_jobs <= 0 || max_n <= 0) return;
    const dim3 grid((unsigned)((max_n + kRetimeTile - 1) / kRetimeTile), (unsigned)n_jobs);
    k_retime<<<grid, kRetimeThreads, 0, st>>>(d_jobs, d_rates);
}

}  // namespace tdoa
