// graph_ls.cuh -- per-station values from per-pair differences, and the status-2 rule of a masked fix.
//
// The dense graph least-squares solve of k_station_rates (station clock rates from pair slopes) and
// k_window_closure (station ranges from a TGT window's range differences), both in retime.cu: find v[S] that
// minimises sum over the used pairs p = (i, j) of (v_j - v_i - d_p)^2 and sums to zero in each connected
// component of those pairs.  One CTA of at least S threads, station t on thread t.  Every f64 operation is an
// explicit __d*_rn intrinsic, so the bits do not depend on -fmad; the order is the one stated in
// include/tdoa_b200.h (tdoa_process_windows_retimed) and restated in tests/retime_oracle.py.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace tdoa {

constexpr int kGraphLsMaxStations = 64;
typedef double GraphLsMatrix[kGraphLsMaxStations + 1];   // a row of A (padded against bank conflicts)

// pair p = (i, j), i < j, in lexicographic order
__host__ __device__ __forceinline__ int graph_pair(int i, int j, int S) { return i * (2 * S - i - 1) / 2 + (j - i - 1); }

// The status-2 rule of a masked fix (k_solve_ls), of the grid seed (k_grid_rows), of a closure drop
// (k_window_closure) and of a station exclusion (k_window_exclude): the number of used pairs, or -1 when there are
// fewer than `dims` of them or they touch fewer than dims + 1 stations (dims = 0: no used pair).  skip: stations
// whose pairs count as unused.
__host__ __device__ __forceinline__ int ls_used_pairs(const uint8_t *used, int n_st, int dims, unsigned long long skip = 0ull)
{
    int n_used = 0, q = 0;
    unsigned long long touched = 0ull;
    for (int i = 0; i < n_st; i++)
        for (int j = i + 1; j < n_st; j++, q++)
            if (used[q] && !((skip >> i | skip >> j) & 1ull)) { n_used++; touched |= (1ull << i) | (1ull << j); }
#ifdef __CUDA_ARCH__
    const int n_touched = __popcll(touched);
#else
    const int n_touched = __builtin_popcountll(touched);
#endif
    return (n_used < dims || n_touched < dims + 1) ? -1 : n_used;
}

// Components of the used-pair graph: every station ends labelled with the smallest index of its component (a
// label is the minimum over its neighbours' labels, repeated until no label changes).  Called by every thread.
template <class Use>
__device__ void graph_components(int S, int t, int *comp, Use use)
{
    if (t < S) comp[t] = t;
    __syncthreads();
    for (;;) {
        int c = t < S ? comp[t] : 0;
        if (t < S) {
            for (int k = 0; k < t; k++)
                if (use(graph_pair(k, t, S))) c = min(c, comp[k]);
            for (int j = t + 1; j < S; j++)
                if (use(graph_pair(t, j, S))) c = min(c, comp[j]);
        }
        __syncthreads();
        const bool changed = t < S && c != comp[t];
        if (changed) comp[t] = c;
        if (!__syncthreads_or(changed)) break;
    }
}

// The normal equations of the used pairs plus one all-ones block per component (the zero-sum gauge): A and b as
// a pass over the pairs in pair order gives them, b[i] -= d_p, b[j] += d_p.  Row t on thread t: station t's pairs
// in pair order are (k, t) for k < t, then (t, j) for j > t, so b[t] takes its terms in that same order.  deg[t]:
// the used pairs of station t.  Called by every thread after graph_components.
template <class Use, class Val>
__device__ void graph_normal(int S, int t, const int *comp, GraphLsMatrix *A, double *b, int *deg, Use use, Val val)
{
    if (t < S) {
        double bt = 0.0;
        int d = 0;
        for (int j = 0; j < S; j++) A[t][j] = comp[t] == comp[j] ? 1.0 : 0.0;
        for (int k = 0; k < t; k++) {
            const int p = graph_pair(k, t, S);
            if (!use(p)) continue;
            A[t][t] += 1.0; A[t][k] -= 1.0;
            bt = __dadd_rn(bt, val(p));
            d++;
        }
        for (int j = t + 1; j < S; j++) {
            const int p = graph_pair(t, j, S);
            if (!use(p)) continue;
            A[t][t] += 1.0; A[t][j] -= 1.0;
            bt = __dsub_rn(bt, val(p));
            d++;
        }
        b[t] = bt;
        deg[t] = d;
    }
    __syncthreads();
}

// A = L L^T (right-looking Cholesky, row t on thread t: A[i][j] -= L[i][k] L[j][k] in k order), then L y = b and
// L^T v = y column by column; b ends holding v.  Called by every thread.
__device__ __forceinline__ void graph_ls_solve(int S, int t, GraphLsMatrix *A, double *b)
{
    for (int k = 0; k < S; k++) {
        if (t == k) A[k][k] = __dsqrt_rn(A[k][k]);
        __syncthreads();
        if (t > k && t < S) A[t][k] = __ddiv_rn(A[t][k], A[k][k]);
        __syncthreads();
        if (t > k && t < S)
            for (int j = k + 1; j <= t; j++) A[t][j] = __dsub_rn(A[t][j], __dmul_rn(A[t][k], A[j][k]));
        __syncthreads();
    }
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
}

}  // namespace tdoa
