// exclude.cu -- the station check of the windowed fixes (tdoa_exclude_stations, the _exclude windowed calls; no
// reference equivalent; statement in include/tdoa_b200.h, tdoa_exclusion_opts; restated in tests/exclusion_oracle.py).
//
// An error common to all of one station's pairs (a collector tuned to another programme, an antenna that is down) is
// a station value: the closure check cannot see it, but the range differences then disagree with one position.
//   k_window_exclude  one CTA per set, thread k = station k: every candidate solves the set without its station's
//                     pairs (ls_core.cuh's ls_fix, the 64-bit skip mask on top of the fix mask: no candidate mask is
//                     materialised), a block arg-min (least rms, lowest k on ties) picks the station to exclude, and
//                     the rounds repeat inside the CTA.  F, the set's fix without the check, is what k_solve_ls left
//                     in the output arrays; the kernel overwrites them only for a set where it excludes a station.
#include <cuda_runtime.h>

#include <cstdint>

#include "graph_ls.cuh"
#include "kernels.h"
#include "ls_core.cuh"

namespace tdoa {

namespace {

constexpr int kExcludeThreads = kLsMaxStations;

// the number of components of the graph of adj among the stations of `nodes` (adj restricted to nodes)
__device__ __forceinline__ int bit_components(const unsigned long long *adj, unsigned long long nodes)
{
    int comps = 0;
    for (unsigned long long rest = nodes; rest;) {
        unsigned long long seen = rest & (~rest + 1ull), front = seen;
        while (front) {
            unsigned long long next = 0ull;
            for (unsigned long long f = front; f; f &= f - 1ull) next |= adj[__ffsll((long long)f) - 1];
            next &= nodes;
            front = next & ~seen;
            seen |= next;
        }
        rest &= ~seen;
        comps++;
    }
    return comps;
}

// mask[P] (read): the fix mask m.  used[P] (may be nullptr; may be mask itself): an m-pair of an excluded station
// becomes 3.  final_mask[P] (may be nullptr): the final m as 0 / 1.  round[S], srms[S] per set; n_excl per set.
__global__ void __launch_bounds__(kExcludeThreads) k_window_exclude(const double *llh, int n_st, const double *rd_all,
                                                                    const uint8_t *mask_all, uint8_t *used_all,
                                                                    uint8_t *final_all, int stride, const double *init_llh,
                                                                    int dims, double max_rms, int max_exclude,
                                                                    double *out_llh, double *out_rms, int *status,
                                                                    int *iters, uint8_t *round_all, double *srms_all,
                                                                    int *n_excl)
{
    __shared__ double s_st[3 * kLsMaxStations];
    __shared__ unsigned long long adj[kLsMaxStations];
    __shared__ double s_srms[kLsMaxStations];
    __shared__ uint8_t s_round[kLsMaxStations];
    __shared__ double w_rms[kExcludeThreads / 32];
    __shared__ int w_k[kExcludeThreads / 32];
    __shared__ LsFix s_F;
    __shared__ unsigned long long s_E;
    __shared__ int s_nE, s_win;
    const int t = threadIdx.x, S = n_st, set = blockIdx.x;
    const double *rd = rd_all + (size_t)set * stride;
    const uint8_t *mask = mask_all + (size_t)set * stride;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (t < S) {
        llh_to_ecef(llh[3 * t], llh[3 * t + 1], llh[3 * t + 2], s_st + 3 * t);
        unsigned long long a = 0ull;
        for (int k = 0; k < S; k++)
            if (k != t && mask[graph_pair(min(t, k), max(t, k), S)]) a |= 1ull << k;
        adj[t] = a;
        s_srms[t] = nan;
        s_round[t] = 0;
    }
    if (t == 0) {
        s_F.p.lat = out_llh[3 * set]; s_F.p.lon = out_llh[3 * set + 1]; s_F.p.h = out_llh[3 * set + 2];
        s_F.rms = out_rms[set]; s_F.status = status[set]; s_F.iters = iters ? iters[set] : 0;
        s_E = 0ull;
        s_nE = 0;
    }
    __syncthreads();
    const LsPoint x0 = ls_start(llh, S, init_llh, set);
    const unsigned long long all = S == 64 ? ~0ull : (1ull << S) - 1ull;
    for (int round = 1;; round++) {
        const unsigned long long E = s_E;
        if (s_F.status != 0 || s_F.rms <= max_rms || (max_exclude > 0 && s_nE == max_exclude)) break;
        // station t is a candidate: it has an m-pair, and m without its pairs passes the status-2 rule with
        // redundancy (touched stations - components - dims) >= 1
        bool cand = false;
        const unsigned long long skip = E | (1ull << t);
        if (t < S && !((E >> t) & 1ull) && (adj[t] & ~E)) {
            unsigned long long touched = 0ull;
            int n2 = 0;
            for (unsigned long long rest = all & ~skip; rest; rest &= rest - 1ull) {
                const int s = __ffsll((long long)rest) - 1;
                const unsigned long long a = adj[s] & ~skip;
                if (a) { touched |= 1ull << s; n2 += __popcll(a); }
            }
            const int n_touched = __popcll(touched);
            if (n2 / 2 >= dims && n_touched >= dims + 1) cand = n_touched - bit_components(adj, touched) - dims >= 1;
        }
        LsFix F{};
        double key = 0.0;
        int k = -1;
        if (cand) {
            F = ls_fix(s_st, S, rd, mask, skip, dims, x0);
            if (round == 1) s_srms[t] = F.rms;
            if (F.status == 0) { key = F.rms; k = t; }
        }
        // the eligible candidate with the least rms, the lowest station on ties
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_down_sync(0xffffffffu, key, off);
            const int ok = __shfl_down_sync(0xffffffffu, k, off);
            if (ok >= 0 && (k < 0 || ov < key || (ov == key && ok < k))) { key = ov; k = ok; }
        }
        if ((t & 31) == 0) { w_rms[t >> 5] = key; w_k[t >> 5] = k; }
        __syncthreads();
        if (t == 0) {
            for (int w = 1; w < kExcludeThreads / 32; w++)
                if (w_k[w] >= 0 && (k < 0 || w_rms[w] < key || (w_rms[w] == key && w_k[w] < k))) { key = w_rms[w]; k = w_k[w]; }
            s_win = k >= 0 && key < s_F.rms ? k : -1;
        }
        __syncthreads();
        const int win = s_win;
        if (win < 0) break;
        if (t == win) {
            s_F = F;
            s_E = E | (1ull << t);
            s_nE++;
            s_round[t] = (uint8_t)round;
        }
        __syncthreads();
    }
    const unsigned long long E = s_E;
    if (t < S) {
        for (int j = t + 1; j < S; j++) {
            const size_t p = (size_t)set * stride + graph_pair(t, j, S);
            const bool m = mask_all[p] != 0, out = ((E >> t) | (E >> j)) & 1ull;
            if (final_all) final_all[p] = m && !out;
            if (used_all && m && out) used_all[p] = 3;
        }
        if (round_all) round_all[(size_t)set * S + t] = s_round[t];
        if (srms_all) srms_all[(size_t)set * S + t] = s_srms[t];
    }
    if (t == 0) {
        if (n_excl) n_excl[set] = s_nE;
        if (s_nE > 0) {
            out_llh[3 * set] = s_F.p.lat; out_llh[3 * set + 1] = s_F.p.lon; out_llh[3 * set + 2] = s_F.p.h;
            out_rms[set] = s_F.rms;
            status[set] = s_F.status;
            if (iters) iters[set] = s_F.iters;
        }
    }
}

}  // namespace

void launch_window_exclude(const double *d_llh, int n_st, const double *d_rd, const uint8_t *d_mask, uint8_t *d_used,
                           uint8_t *d_final, int n_sets, int stride, const double *d_init, int dims, double max_rms,
                           int max_exclude, double *d_out_llh, double *d_rms, int *d_status, int *d_iters, uint8_t *d_round,
                           double *d_srms, int *d_n_excl, cudaStream_t st)
{
    if (n_sets > 0)
        k_window_exclude<<<n_sets, kExcludeThreads, 0, st>>>(d_llh, n_st, d_rd, d_mask, d_used, d_final, stride, d_init, dims,
                                                             max_rms, max_exclude, d_out_llh, d_rms, d_status, d_iters,
                                                             d_round, d_srms, d_n_excl);
}

}  // namespace tdoa
