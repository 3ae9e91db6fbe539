// window_fix.cu -- from window tables to range differences, one fix per TGT window
// (tdoa_process_windows, tdoa_window_fixes; no reference equivalent; restated in tests/window_oracle.py;
// the grid seed of the _grid calls in tests/window_grid_oracle.py).
//
// An RTL-SDR's sample clock is off by ppm, so the lag between two collectors drifts linearly over
// the capture (1 ppm of relative rate = 2 samples per second at 2 Msps).  The reference correlates
// the REF blocks 1 and 3 as one signal, which evaluates the REF lag at block 2's centre: right for a
// TGT correlation over the whole of block 2, but a 1 s TGT window 16 s from that centre keeps
// 33 samples (5 km) of error per ppm.  Here the REF lag's linear track is fitted per pair across the
// REF windows and evaluated at each TGT window's time:
//   k_window_ref_fit  one thread per pair: least-squares line y = a + beta (t - t_mean) through the
//                     usable REF windows (sums in f64, window order), one optional refit without the
//                     windows whose residual exceeds max_resid, the REF transmitter's geometric term
//   k_window_rd       one thread per (TGT window, pair): rd = (y_tgt / fs - y_ref(t_w) / fs) * c
//                     (+ the geometric term) and the used mask that k_solve_ls reads.
// The _grid calls then seed each window's fix from the masked grid arg-min of its own used pairs (solve.cu):
//   k_grid_rows       the window's row of the ranked table (not searched: the least-squares step's status 2)
//   k_grid_rank ... k_grid_pick   (engine.cu's grid search, as in tdoa_grid) write the arg-min cell into the window's
//                     start point, which holds the start the window has without a grid; k_solve_ls starts there.
// The ranked pass is optimistic: when the grid search finds it incomplete after the call's one synchronisation, the
// call reruns the grid on every cell (k_grid_cost) and the fixes before it returns.
// The _closure calls check each window's range differences against each other first (retime.cu):
//   k_window_closure  one CTA per TGT window: drops the pairs the window's other pairs contradict, into a separate
//                     0 / 1 mask that k_grid_rows and k_solve_ls read in place of the used mask.
// The _exclude calls check each window's fix for one wrong station after it (exclude.cu):
//   k_window_exclude  one CTA per TGT window: solves again without each station in turn and excludes the station
//                     whose solve fits best, while the fix's rms exceeds max_rms; with a grid, k_grid_rows and the
//                     grid search run again on the final mask and k_solve_ls fixes every window from that seed.
// tdoa_process_windows_retimed runs the REF pair loop, k_window_ref_fit and k_station_rates (retime.cu) before the TGT
// pair loop, which re-times every plane by its station's rate; the fix stage is the same.
// Window times and the usable test are stated in include/tdoa_b200.h (tdoa_process_windows).
#include <cuda_runtime.h>

#include <cmath>
#include <vector>

#include "engine_internal.h"
#include "geodesy.cuh"
#include "graph_ls.cuh"

using namespace tdoa;

namespace tdoa {

namespace {

constexpr double kC = 299792458.0;

__device__ __forceinline__ bool record_usable(const PeakRec &r, float min_margin)
{
    if (r.flags & (TDOA_PEAK_EMPTY | TDOA_PEAK_EDGE)) return false;
    return !(min_margin > 0.f && r.margin < min_margin);
}

__device__ __forceinline__ double record_lag(const PeakRec &r) { return (double)r.lag + (double)r.frac; }

// pair p = (i, j), i < j lexicographic
__device__ __forceinline__ void pair_stations(int p, int n_st, int &i, int &j)
{
    int rem = p;
    i = 0;
    while (rem >= n_st - 1 - i) { rem -= n_st - 1 - i; i++; }
    j = i + 1 + rem;
}

// least-squares line through the REF windows of pair p that pass the usable test, the time test (a window
// with samples in blocks 1 and 3 has no time: NaN) and -- refit -- |y - line0(t)| <= max_resid
struct Line { double a, beta, t_mean; int n; };

__device__ Line fit_line(const PeakRec *ref, int n_ref, int P, int p, const double *t_ref, int n_st, int i, float min_margin,
                         const Line *line0, double max_resid)
{
    auto take = [&](int w, double &t, double &y) -> bool {
        const PeakRec r = ref[(size_t)w * P + p];
        t = t_ref[(size_t)w * n_st + i];
        if (!record_usable(r, min_margin) || isnan(t)) return false;
        y = record_lag(r);
        return !line0 || !(fabs(y - (line0->a + line0->beta * (t - line0->t_mean))) > max_resid);
    };
    int n = 0;
    double st = 0.0, sy = 0.0;
    for (int w = 0; w < n_ref; w++) {
        double t, y;
        if (take(w, t, y)) { n++; st += t; sy += y; }
    }
    Line L{0.0, 0.0, 0.0, n};
    if (n == 0) return L;
    L.t_mean = st / n;
    L.a = sy / n;
    double stt = 0.0, sty = 0.0;
    for (int w = 0; w < n_ref; w++) {
        double t, y;
        if (take(w, t, y)) {
            const double dt = t - L.t_mean;
            stt += dt * dt;
            sty += dt * (y - L.a);
        }
    }
    if (n > 1 && stt > 0.0) L.beta = sty / stt;
    return L;
}

__global__ void k_window_ref_fit(const PeakRec *ref, int n_ref, int n_st, const double *t_ref, const double *t_mid,
                                 const double *llh, const double *ref_tx, float min_margin, double max_resid, double *fit,
                                 double *ref_fit)
{
    const int P = n_st * (n_st - 1) / 2;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    int i, j;
    pair_stations(p, n_st, i, j);
    Line L = fit_line(ref, n_ref, P, p, t_ref, n_st, i, min_margin, nullptr, 0.0);
    if (max_resid > 0.0 && L.n > 0) {
        const Line L0 = L;
        L = fit_line(ref, n_ref, P, p, t_ref, n_st, i, min_margin, &L0, max_resid);
    }
    double geo = 0.0;
    if (ref_tx) {
        double x[3], a[3], b[3];
        llh_to_ecef(ref_tx[0], ref_tx[1], ref_tx[2], x);
        llh_to_ecef(llh[3 * i], llh[3 * i + 1], llh[3 * i + 2], a);
        llh_to_ecef(llh[3 * j], llh[3 * j + 1], llh[3 * j + 2], b);
        const double ri = sqrt((x[0] - a[0]) * (x[0] - a[0]) + (x[1] - a[1]) * (x[1] - a[1]) + (x[2] - a[2]) * (x[2] - a[2]));
        const double rj = sqrt((x[0] - b[0]) * (x[0] - b[0]) + (x[1] - b[1]) * (x[1] - b[1]) + (x[2] - b[2]) * (x[2] - b[2]));
        geo = rj - ri;
    }
    double *f = fit + (size_t)kWindowFitDoubles * p;
    f[0] = L.a; f[1] = L.beta; f[2] = L.t_mean; f[3] = (double)L.n; f[4] = geo;
    if (ref_fit) {
        ref_fit[3 * p] = L.n > 0 ? L.a + L.beta * (t_mid[i] - L.t_mean) : 0.0;
        ref_fit[3 * p + 1] = L.beta;
        ref_fit[3 * p + 2] = (double)L.n;
    }
}

__global__ void k_window_rd(const PeakRec *tgt, int n_tgt, int n_st, const double *t_tgt, const double *fit, float min_margin,
                            double fs, double *rd, uint8_t *used)
{
    const int P = n_st * (n_st - 1) / 2;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_tgt * P) return;
    const int w = k / P, p = k - w * P;
    int i, j;
    pair_stations(p, n_st, i, j);
    const double *f = fit + (size_t)kWindowFitDoubles * p;
    const PeakRec r = tgt[k];
    const bool ok = f[3] > 0.0 && record_usable(r, min_margin);
    double v = __longlong_as_double(0x7ff8000000000000ll);   // NaN: pair not used in this window
    if (ok) {
        const double y_ref = f[0] + f[1] * (t_tgt[(size_t)w * n_st + i] - f[2]);
        // k_range_diffs' order: dt = y_tgt / fs - y_ref / fs, rd = dt * c
        v = (record_lag(r) / fs - y_ref / fs) * kC + f[4];
    }
    rd[k] = v;
    used[k] = ok ? 1 : 0;
}

}  // namespace

void launch_window_ref_fit(const PeakRec *d_ref, int n_ref, int n_st, const double *d_t_ref, const double *d_t_mid,
                           const double *d_llh, const double *d_ref_tx, float min_margin, double max_resid, double *d_fit,
                           double *d_ref_fit, cudaStream_t st)
{
    const int P = n_st * (n_st - 1) / 2;
    if (P > 0)
        k_window_ref_fit<<<(P + 63) / 64, 64, 0, st>>>(d_ref, n_ref, n_st, d_t_ref, d_t_mid, d_llh, d_ref_tx, min_margin,
                                                       max_resid, d_fit, d_ref_fit);
}

void launch_window_rd(const PeakRec *d_tgt, int n_tgt, int n_st, const double *d_t_tgt, const double *d_fit, float min_margin,
                      double fs, double *d_rd, uint8_t *d_used, cudaStream_t st)
{
    const int n = n_tgt * (n_st * (n_st - 1) / 2);
    if (n > 0) k_window_rd<<<(n + 127) / 128, 128, 0, st>>>(d_tgt, n_tgt, n_st, d_t_tgt, d_fit, min_margin, fs, d_rd, d_used);
}

// ---------------------------------------------------------------- host side

namespace {

// the windows of one signal kind, as tdoa_xcorr takes them
struct WinGeom {
    int64_t start, len;
    int32_t n;
    int64_t hop;
};

// what the fix stage needs besides the tables: window times per (window, station), block-2 centres
struct WinTimes {
    int n_ref = 0, n_tgt = 0;
    std::vector<double> t_ref, t_tgt, t_mid;
    std::vector<ShardPart> parts;   // per kind: window lengths as the pair loops take them
};

// make_view's mapping is the one place that knows where a window lies in the capture
double window_time(const Station &s, int kind, i64 start, i64 len, i64 guard)
{
    const SigSrc v = make_view(s, kind, start, len, guard);
    if (s.nsamp / 3 > 0 && v.run0_len < len) return NAN;   // REF window across blocks 1 and 3
    return (double)v.run0_start + 0.5 * (double)(len - 1);
}

// the grid seed of the _grid calls: descriptor and optional outputs
struct GridSeed {
    const double *desc = nullptr;   // nullptr: no grid
    double *llh = nullptr, *cost = nullptr;
    int64_t *index = nullptr;
};

// the closure check of the _closure calls: options and optional outputs
struct Closure {
    const tdoa_closure_opts *opts = nullptr;   // nullptr: no check
    double *resid = nullptr;
    int32_t *dropped = nullptr;
};

// the station check of the _exclude calls: options and optional outputs
struct Exclusion {
    const tdoa_exclusion_opts *opts = nullptr;   // nullptr: no check
    uint8_t *round = nullptr;
    double *rms = nullptr;
    int32_t *excluded = nullptr;
};

int exclusion_opts_check(tdoa_engine *e, const char *fn, const tdoa_exclusion_opts *x)
{
    if (!x) return fail(e, TDOA_E_INVALID, "%s: exclusion options are NULL", fn);
    if (!(x->max_rms > 0.0)) return fail(e, TDOA_E_INVALID, "%s: max_rms must be > 0, got %g", fn, x->max_rms);
    if (x->max_exclude < 0) return fail(e, TDOA_E_INVALID, "%s: max_exclude must be >= 0, got %d", fn, x->max_exclude);
    return TDOA_OK;
}

int closure_opts_check(tdoa_engine *e, const char *fn, const tdoa_closure_opts *c)
{
    if (!c) return fail(e, TDOA_E_INVALID, "%s: closure options are NULL", fn);
    if (!(c->max_residual > 0.0)) return fail(e, TDOA_E_INVALID, "%s: max_residual must be > 0, got %g", fn, c->max_residual);
    if (c->max_drop < 0) return fail(e, TDOA_E_INVALID, "%s: max_drop must be >= 0, got %d", fn, c->max_drop);
    return TDOA_OK;
}

// grid: the seed of the _grid calls, nullptr without
int window_check(tdoa_engine *e, const char *fn, const double *stations_llh, const tdoa_window_opts *o, const WinGeom &ref,
                 const WinGeom &tgt, const double *fix_llh, const int32_t *fix_status, const GridSeed *grid, WinTimes &T,
                 const Closure &closure, const Exclusion &exclusion)
{
    const int32_t n_ref = ref.n, n_tgt = tgt.n;
    const int S = e->cfg.n_stations;
    if (!stations_llh || !o || !fix_llh || !fix_status) return fail(e, TDOA_E_INVALID, "%s: NULL argument", fn);
    if (e->cfg.mode == TDOA_MODE_SOURCE)
        return fail(e, TDOA_E_INVALID, "%s: SOURCE mode has no REF correction (processor.go:853)", fn);
    if (S < 3 || S > solve_ls_max_stations())
        return fail(e, TDOA_E_INVALID, "%s: 3..%d stations, got %d", fn, solve_ls_max_stations(), S);
    if (o->dims != 2 && o->dims != 3) return fail(e, TDOA_E_INVALID, "%s: dims must be 2 or 3, got %d", fn, o->dims);
    if (o->dims == 3 && S < 4) return fail(e, TDOA_E_INVALID, "%s: dims 3 needs at least 4 stations", fn);
    if (n_ref < 1 || n_tgt < 1)
        return fail(e, TDOA_E_INVALID, "%s: need >= 1 REF and >= 1 TGT window, got %d and %d", fn, n_ref, n_tgt);
    int rc;
    if (closure.opts && (rc = closure_opts_check(e, fn, closure.opts))) return rc;
    if (exclusion.opts && (rc = exclusion_opts_check(e, fn, exclusion.opts))) return rc;
    T.n_ref = n_ref; T.n_tgt = n_tgt;
    T.parts.assign(2, ShardPart{});
    for (int kind = 0; kind < 2; kind++) {
        const WinGeom &G = kind == TDOA_KIND_REF ? ref : tgt;
        ShardPart &Q = T.parts[kind];
        Q.kind = kind; Q.win_start = G.start; Q.hop = G.hop; Q.n_windows = G.n;
        if ((rc = window_lengths(e, kind, G.start, G.len, G.n, G.hop, Q.len))) return rc;
        std::vector<double> &t = kind == TDOA_KIND_REF ? T.t_ref : T.t_tgt;
        t.resize((size_t)Q.n_windows * S);
        for (int w = 0; w < Q.n_windows; w++)
            for (int st = 0; st < S; st++)
                t[(size_t)w * S + st] = window_time(e->stations[st], kind, G.start + (i64)w * G.hop, Q.len[st], e->cfg.guard_samples);
    }
    T.t_mid.resize(S);
    for (int st = 0; st < S; st++) {
        const i64 b = e->stations[st].nsamp / 3;
        T.t_mid[st] = (double)b + 0.5 * (double)(b - 1);
    }
    if (!grid) return TDOA_OK;
    if (!grid->desc) return fail(e, TDOA_E_INVALID, "%s: grid_desc is NULL", fn);
    if (S > 16) return fail(e, TDOA_E_INVALID, "%s: the grid takes 2..16 stations, got %d", fn, S);
    return grid_check(e, fn, S, grid->desc);
}

// the fix stage on device tables, queued on the engine's stream inside the caller's begin_call / end_call;
// the station table, times and options ride in the descriptor frame.  *synced: the stream was drained (the grid
// seed's check) and holds nothing more
int fix_stage(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o, const WinTimes &T, const PeakRec *d_ref,
              const PeakRec *d_tgt, double *ref_fit, double *range_diffs, uint8_t *pair_used, double *fix_llh, double *fix_rms,
              int32_t *fix_status, int32_t *fix_iters, const GridSeed *grid, const Closure &closure,
              const Exclusion &exclusion, bool *synced)
{
    const tdoa_exclusion_opts *X = exclusion.opts;
    *synced = false;
    const GridSeed G = grid ? *grid : GridSeed{};
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2, nt = T.n_tgt;
    int rc;
    const double *d_llh = nullptr, *d_t_ref = nullptr, *d_t_tgt = nullptr, *d_t_mid = nullptr, *d_ref_tx = nullptr,
                 *d_init = nullptr;
    if ((rc = upload(e, std::vector<double>(stations_llh, stations_llh + (size_t)3 * S), &d_llh)) ||
        (rc = upload(e, T.t_ref, &d_t_ref)) || (rc = upload(e, T.t_tgt, &d_t_tgt)) || (rc = upload(e, T.t_mid, &d_t_mid)))
        return rc;
    if (o->has_ref_tx && (rc = upload(e, std::vector<double>(o->ref_tx_llh, o->ref_tx_llh + 3), &d_ref_tx))) return rc;
    if (o->has_init || G.desc) {
        // the start of every window: init_llh, or (grid seed) the mean of the stations as k_solve_ls takes it
        double p0[3] = {0.0, 0.0, 0.0};
        if (o->has_init) {
            for (int k = 0; k < 3; k++) p0[k] = o->init_llh[k];
        } else {
            for (int s = 0; s < S; s++)
                for (int k = 0; k < 3; k++) p0[k] += stations_llh[3 * s + k];
            for (int k = 0; k < 3; k++) p0[k] /= S;
        }
        std::vector<double> init((size_t)3 * nt);
        for (int w = 0; w < nt; w++)
            for (int k = 0; k < 3; k++) init[(size_t)3 * w + k] = p0[k];
        if ((rc = upload(e, init, &d_init))) return rc;
    }
    double *d_fit = nullptr, *d_ref_fit = nullptr, *d_rd = nullptr, *d_fix = nullptr, *d_rms = nullptr;
    uint8_t *d_used = nullptr;
    int *d_status = nullptr, *d_iters = nullptr;
    if ((rc = alloc_t(e, &d_fit, (size_t)kWindowFitDoubles * P)) || (rc = alloc_t(e, &d_ref_fit, (size_t)3 * P)) ||
        (rc = alloc_t(e, &d_rd, (size_t)nt * P)) || (rc = alloc_t(e, &d_used, (size_t)nt * P)) ||
        (rc = alloc_t(e, &d_fix, (size_t)3 * nt)) || (rc = alloc_t(e, &d_rms, (size_t)nt)) ||
        (rc = alloc_t(e, &d_status, (size_t)nt)) || (rc = alloc_t(e, &d_iters, (size_t)nt)))
        return rc;
    // the closure check: the mask the grid rows and the fixes read (the used mask without a check)
    uint8_t *d_fix_used = d_used;
    double *d_cresid = nullptr;
    int *d_dropped = nullptr;
    if (closure.opts &&
        ((rc = alloc_t(e, &d_fix_used, (size_t)nt * P)) || (rc = alloc_t(e, &d_cresid, (size_t)nt * P)) ||
         (rc = alloc_t(e, &d_dropped, (size_t)nt))))
        return rc;
    // the station check: rounds and rms per (window, station), stations excluded per window
    uint8_t *d_round = nullptr;
    double *d_srms = nullptr;
    int *d_n_excl = nullptr;
    if (X && ((rc = alloc_t(e, &d_round, (size_t)nt * S)) || (rc = alloc_t(e, &d_srms, (size_t)nt * S)) ||
              (rc = alloc_t(e, &d_n_excl, (size_t)nt))))
        return rc;
    // the grid seed: the windows' start points (written by the grid where it finds a cell), the masked rows; with the
    // station check, a second search (g2) on the check's final mask, into the same start points
    GridSearch g, g2;
    double *d_start = nullptr, *d_tab = nullptr, *d_tab2 = nullptr;
    uint8_t *d_final = nullptr;
    if (G.desc) {
        const double *d_desc = nullptr;
        if ((rc = upload(e, std::vector<double>(G.desc, G.desc + 7), &d_desc)) || (rc = alloc_t(e, &d_start, (size_t)3 * nt)) ||
            (rc = alloc_t(e, &d_tab, (size_t)nt * grid_rank_tab_doubles(true))) || (rc = alloc_t(e, &g.d_cost, (size_t)nt)) ||
            (rc = alloc_t(e, &g.d_idx, (size_t)nt)))
            return rc;
        g.d_llh = d_llh; g.d_desc = d_desc; g.d_tab = d_tab; g.d_rd = d_rd; g.d_used = d_fix_used; g.d_out = d_start;
        g.n_sets = nt; g.rd_stride = P; g.n_st = S; g.nlat = (int)G.desc[4]; g.nlon = (int)G.desc[5];
        if (X) {
            g2 = g;
            if ((rc = alloc_t(e, &d_final, (size_t)nt * P)) ||
                (rc = alloc_t(e, &d_tab2, (size_t)nt * grid_rank_tab_doubles(true))) || (rc = alloc_t(e, &g2.d_cost, (size_t)nt)) ||
                (rc = alloc_t(e, &g2.d_idx, (size_t)nt)))
                return rc;
            g2.d_tab = d_tab2; g2.d_used = d_final;
        }
    }
    const GridSearch &g_seed = G.desc && X ? g2 : g;   // the search whose arg-min the seed outputs report
    // the grid (ranked, or every cell) between the range differences and the fixes
    auto seed_and_fix = [&](bool every_cell) -> int {
        if (G.desc) {
            CU(cudaMemcpyAsync(d_start, d_init, (size_t)3 * nt * sizeof(double), cudaMemcpyDeviceToDevice, e->stream));
            if (const int rc2 = grid_search_queue(e, g, every_cell)) return rc2;
        }
        launch_solve_ls(d_llh, S, d_rd, nt, P, G.desc ? d_start : d_init, o->dims, d_fix, d_rms, d_status, d_iters, e->stream,
                        d_fix_used);
        count_launch(e);
        if (X) {
            // d_used gets 3 on the excluded stations' pairs; without the closure check it is the fix mask itself,
            // which a rerun then reads as before (3 is in the mask as 1 is)
            launch_window_exclude(d_llh, S, d_rd, d_fix_used, d_used, d_final, nt, P, G.desc ? d_start : d_init, o->dims,
                                  X->max_rms, X->max_exclude, d_fix, d_rms, d_status, d_iters, d_round, d_srms, d_n_excl,
                                  e->stream);
            count_launch(e);
            if (G.desc) {   // seeded again from the grid arg-min over the final mask (the same seed where none is excluded)
                CU(cudaMemcpyAsync(d_start, d_init, (size_t)3 * nt * sizeof(double), cudaMemcpyDeviceToDevice, e->stream));
                launch_grid_rows(d_rd, d_final, nt, P, S, o->dims, d_tab2, e->stream);
                count_launch(e);
                if (const int rc2 = grid_search_queue(e, g2, every_cell)) return rc2;
                launch_solve_ls(d_llh, S, d_rd, nt, P, d_start, o->dims, d_fix, d_rms, d_status, d_iters, e->stream, d_final);
                count_launch(e);
            }
        }
        CU(cudaEventRecord(e->ev[2], e->stream));
        CU(cudaGetLastError());
        return TDOA_OK;
    };
    auto back = [&](void *dst, const void *src, size_t bytes) -> int {
        if (dst) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, e->stream));
        return TDOA_OK;
    };
    auto results = [&]() -> int {
        int rc2;
        if ((rc2 = back(fix_llh, d_fix, (size_t)3 * nt * sizeof(double))) || (rc2 = back(fix_rms, d_rms, (size_t)nt * sizeof(double))) ||
            (rc2 = back(fix_status, d_status, (size_t)nt * sizeof(int32_t))) ||
            (rc2 = back(fix_iters, d_iters, (size_t)nt * sizeof(int32_t))))
            return rc2;
        if (G.desc &&
            ((rc2 = back(G.llh, d_start, (size_t)3 * nt * sizeof(double))) ||
             (rc2 = back(G.cost, g_seed.d_cost, (size_t)nt * sizeof(double))) ||
             (rc2 = back(G.index, g_seed.d_idx, (size_t)nt * sizeof(int64_t)))))
            return rc2;
        if (X && ((rc2 = back(pair_used, d_used, (size_t)nt * P)) ||
                  (rc2 = back(exclusion.round, d_round, (size_t)nt * S)) ||
                  (rc2 = back(exclusion.rms, d_srms, (size_t)nt * S * sizeof(double))) ||
                  (rc2 = back(exclusion.excluded, d_n_excl, (size_t)nt * sizeof(int32_t)))))
            return rc2;
        return TDOA_OK;
    };
    CU(cudaEventRecord(e->ev[1], e->stream));
    launch_window_ref_fit(d_ref, T.n_ref, S, d_t_ref, d_t_mid, d_llh, d_ref_tx, o->min_margin, o->ref_max_residual, d_fit,
                          d_ref_fit, e->stream);
    launch_window_rd(d_tgt, nt, S, d_t_tgt, d_fit, o->min_margin, e->cfg.sample_rate, d_rd, d_used, e->stream);
    count_launch(e, 2);
    if (closure.opts) {
        launch_window_closure(d_rd, d_used, d_fix_used, nt, P, S, o->dims, closure.opts->max_residual, closure.opts->max_drop,
                              d_cresid, d_dropped, e->stream);
        count_launch(e);
    }
    if (G.desc) {
        launch_grid_rows(d_rd, d_fix_used, nt, P, S, o->dims, d_tab, e->stream);
        count_launch(e);
    }
    if ((rc = seed_and_fix(false))) return rc;
    if ((rc = back(ref_fit, d_ref_fit, (size_t)3 * P * sizeof(double))) ||
        (rc = back(range_diffs, d_rd, (size_t)nt * P * sizeof(double))) || (!X && (rc = back(pair_used, d_used, (size_t)nt * P))) ||
        (closure.opts && ((rc = back(closure.resid, d_cresid, (size_t)nt * P * sizeof(double))) ||
                          (rc = back(closure.dropped, d_dropped, (size_t)nt * sizeof(int32_t))))) ||
        (rc = results()))
        return rc;
    if (G.desc) {
        // the grid's check after the call's one synchronisation; its pageable read-back returns only when done, so
        // it is queued behind the fixes
        std::vector<int> h_status((size_t)nt);
        if ((rc = grid_search_fetch(e, g)) || (X && (rc = grid_search_fetch(e, g2)))) return rc;
        CU(cudaMemcpyAsync(h_status.data(), d_status, (size_t)nt * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        *synced = true;
        // an exclusion keeps the status-2 rule, so both searches searched the same windows
        std::vector<char> searched((size_t)nt);
        for (int w = 0; w < nt; w++) searched[w] = h_status[w] != 2;
        if (!grid_search_complete(g, searched) || (X && !grid_search_complete(g2, searched))) {
            if ((rc = seed_and_fix(true)) || (rc = results())) return rc;
            *synced = false;
        }
    }
    return TDOA_OK;
}

// synced: fix_stage drained the stream and queued nothing after (the frees and the frame's event need no wait)
int finish_fix_stage(tdoa_engine *e, bool synced)
{
    const int rc = end_call(e, !synced);
    if (rc) return rc;
    float t = 0.f;
    cudaEventElapsedTime(&t, e->ev[1], e->ev[2]);
    e->st.ms_fix = t;
    return TDOA_OK;
}

// the two device tables of tdoa_process_windows, and the station rates of the retimed call (re-timing rates, then
// the returned clock_rate): they outlive the pair loops' calls
struct Tables {
    cudaStream_t st;
    PeakRec *ref = nullptr, *tgt = nullptr;
    double *rates = nullptr;
    ~Tables()
    {
        if (ref) cudaFreeAsync(ref, st);
        if (tgt) cudaFreeAsync(tgt, st);
        if (rates) cudaFreeAsync(rates, st);
    }
};

// the station rates from the REF table, as one call of their own: k_window_ref_fit (the slopes only), k_station_rates
int station_rates(tdoa_engine *e, const tdoa_window_opts *o, const WinTimes &T, const PeakRec *d_ref, double *d_rates)
{
    int rc = begin_call(e);
    if (rc) return rc;
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    const double *d_t_ref = nullptr;
    double *d_fit = nullptr;
    if ((rc = upload(e, T.t_ref, &d_t_ref)) || (rc = alloc_t(e, &d_fit, (size_t)kWindowFitDoubles * P))) return rc;
    launch_window_ref_fit(d_ref, T.n_ref, S, d_t_ref, nullptr, nullptr, nullptr, o->min_margin, o->ref_max_residual, d_fit,
                          nullptr, e->stream);
    launch_station_rates(d_fit, S, d_rates, d_rates + S, e->stream);
    count_launch(e, 2);
    CU(cudaGetLastError());
    return end_call(e, false);
}

int window_fixes_impl(tdoa_engine *e, const char *fn, const double *stations_llh, const tdoa_window_opts *o, int64_t win_start,
                      int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop, const tdoa_peak *ref_in,
                      const tdoa_peak *tgt_in, double *ref_fit, double *range_diffs, uint8_t *pair_used, double *fix_llh,
                      double *fix_rms, int32_t *fix_status, int32_t *fix_iters, const GridSeed *grid,
                      const Closure &closure = Closure{}, const Exclusion &exclusion = Exclusion{})
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    WinTimes T;
    if ((rc = window_check(e, fn, stations_llh, o, WinGeom{win_start, win_len, n_ref_windows, hop},
                          WinGeom{win_start, win_len, n_tgt_windows, hop}, fix_llh, fix_status, grid, T, closure, exclusion)))
        return rc;
    if (!ref_in || !tgt_in) return fail(e, TDOA_E_INVALID, "%s: a table is NULL", fn);
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    PeakRec *d_ref = nullptr, *d_tgt = nullptr;
    if ((rc = alloc_t(e, &d_ref, (size_t)n_ref_windows * P)) || (rc = alloc_t(e, &d_tgt, (size_t)n_tgt_windows * P))) return rc;
    CU(cudaMemcpyAsync(d_ref, ref_in, (size_t)n_ref_windows * P * sizeof(PeakRec), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_tgt, tgt_in, (size_t)n_tgt_windows * P * sizeof(PeakRec), cudaMemcpyHostToDevice, e->stream));
    bool synced = false;
    if ((rc = fix_stage(e, stations_llh, o, T, d_ref, d_tgt, ref_fit, range_diffs, pair_used, fix_llh, fix_rms, fix_status,
                        fix_iters, grid, closure, exclusion, &synced)))
        return rc;
    return finish_fix_stage(e, synced);
}

// retimed: tdoa_process_windows_retimed -- the TGT planes re-timed by the station rates fitted from the REF table;
// clock_rate (may be NULL) receives those rates
int process_windows_impl(tdoa_engine *e, const char *fn, const double *stations_llh, const tdoa_window_opts *o,
                         const WinGeom &ref, const WinGeom &tgt, tdoa_peak *ref_out, tdoa_peak *tgt_out, double *ref_fit,
                         double *range_diffs, uint8_t *pair_used, double *fix_llh, double *fix_rms, int32_t *fix_status,
                         int32_t *fix_iters, const GridSeed *grid, bool retimed, double *clock_rate,
                         const Closure &closure = Closure{}, const Exclusion &exclusion = Exclusion{})
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    WinTimes T;
    if ((rc = window_check(e, fn, stations_llh, o, ref, tgt, fix_llh, fix_status, grid, T, closure, exclusion))) return rc;
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    Tables tab{e->stream};
    CU(cudaMallocAsync(reinterpret_cast<void **>(&tab.ref), (size_t)ref.n * P * sizeof(PeakRec), e->stream));
    CU(cudaMallocAsync(reinterpret_cast<void **>(&tab.tgt), (size_t)tgt.n * P * sizeof(PeakRec), e->stream));
    // the pair loop of one kind into its device table: dealt and gathered as tdoa_xcorr deals them, or on this GPU
    bool sharded[2] = {false, false};
    auto pass = [&](int kind, const double *d_rates) -> int {
        const WinGeom &G = kind == TDOA_KIND_REF ? ref : tgt;
        PeakRec *table = kind == TDOA_KIND_REF ? tab.ref : tab.tgt;
        if ((sharded[kind] = multi_wants(e, G.n))) {
            if (const int rc2 = begin_call(e)) return rc2;
            ShardPart Q = T.parts[kind];
            Q.out = reinterpret_cast<tdoa_peak *>(table); Q.out_is_device = true; Q.rates = d_rates;
            return xcorr_sharded(e, std::vector<ShardPart>{Q});
        }
        return xcorr_impl(e, kind, G.start, G.len, G.n, G.hop, kind == TDOA_KIND_REF ? ref_out : tgt_out, false, table, d_rates);
    };
    if (retimed) {
        // the TGT pass needs the rates, the rates need the gathered REF table: two meetings of the ranks
        CU(cudaMallocAsync(reinterpret_cast<void **>(&tab.rates), (size_t)2 * S * sizeof(double), e->stream));
        if ((rc = pass(TDOA_KIND_REF, nullptr)) || (rc = station_rates(e, o, T, tab.ref, tab.rates)) ||
            (rc = pass(TDOA_KIND_TGT, tab.rates)))
            return rc;
    } else if (multi_wants(e, ref.n + tgt.n)) {   // the tables tdoa_xcorr_windows gathers, left on this rank's device
        T.parts[TDOA_KIND_REF].out = reinterpret_cast<tdoa_peak *>(tab.ref);
        T.parts[TDOA_KIND_TGT].out = reinterpret_cast<tdoa_peak *>(tab.tgt);
        for (ShardPart &Q : T.parts) Q.out_is_device = true;
        if ((rc = xcorr_sharded(e, T.parts))) return rc;
        sharded[0] = sharded[1] = true;
    } else {         // tdoa_xcorr_windows on one GPU: the REF pair loop, then the TGT pair loop
        if ((rc = pass(TDOA_KIND_REF, nullptr)) || (rc = pass(TDOA_KIND_TGT, nullptr))) return rc;
    }
    if ((rc = begin_call(e))) return rc;
    if (sharded[TDOA_KIND_REF] && ref_out)
        CU(cudaMemcpyAsync(ref_out, tab.ref, (size_t)ref.n * P * sizeof(PeakRec), cudaMemcpyDeviceToHost, e->stream));
    if (sharded[TDOA_KIND_TGT] && tgt_out)
        CU(cudaMemcpyAsync(tgt_out, tab.tgt, (size_t)tgt.n * P * sizeof(PeakRec), cudaMemcpyDeviceToHost, e->stream));
    if (retimed && clock_rate)
        CU(cudaMemcpyAsync(clock_rate, tab.rates + S, (size_t)S * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    bool synced = false;
    if ((rc = fix_stage(e, stations_llh, o, T, tab.ref, tab.tgt, ref_fit, range_diffs, pair_used, fix_llh, fix_rms, fix_status,
                        fix_iters, grid, closure, exclusion, &synced)))
        return rc;
    return finish_fix_stage(e, synced);
}

}  // namespace
}  // namespace tdoa

extern "C" {

int tdoa_window_fixes(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o, int64_t win_start, int64_t win_len,
                      int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop, const tdoa_peak *ref_in, const tdoa_peak *tgt_in,
                      double *ref_fit, double *range_diffs, uint8_t *pair_used, double *fix_llh, double *fix_rms,
                      int32_t *fix_status, int32_t *fix_iters)
{
    return window_fixes_impl(e, "tdoa_window_fixes", stations_llh, o, win_start, win_len, n_ref_windows, n_tgt_windows, hop,
                             ref_in, tgt_in, ref_fit, range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters, nullptr);
}

int tdoa_window_fixes_grid(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o, int64_t win_start,
                           int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop, const double *grid_desc,
                           const tdoa_peak *ref_in, const tdoa_peak *tgt_in, double *ref_fit, double *range_diffs,
                           uint8_t *pair_used, double *fix_llh, double *fix_rms, int32_t *fix_status, int32_t *fix_iters,
                           double *seed_llh, double *seed_cost, int64_t *seed_index)
{
    const GridSeed G{grid_desc, seed_llh, seed_cost, seed_index};
    return window_fixes_impl(e, "tdoa_window_fixes_grid", stations_llh, o, win_start, win_len, n_ref_windows, n_tgt_windows,
                             hop, ref_in, tgt_in, ref_fit, range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters, &G);
}

int tdoa_process_windows(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o, int64_t win_start,
                         int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop, tdoa_peak *ref_out,
                         tdoa_peak *tgt_out, double *ref_fit, double *range_diffs, uint8_t *pair_used, double *fix_llh,
                         double *fix_rms, int32_t *fix_status, int32_t *fix_iters)
{
    return process_windows_impl(e, "tdoa_process_windows", stations_llh, o, WinGeom{win_start, win_len, n_ref_windows, hop},
                                WinGeom{win_start, win_len, n_tgt_windows, hop}, ref_out, tgt_out, ref_fit, range_diffs, pair_used,
                                fix_llh, fix_rms, fix_status, fix_iters, nullptr, false, nullptr);
}

int tdoa_process_windows_retimed(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o, int64_t ref_win_start,
                                 int64_t ref_win_len, int32_t n_ref_windows, int64_t ref_hop, int64_t tgt_win_start,
                                 int64_t tgt_win_len, int32_t n_tgt_windows, int64_t tgt_hop, tdoa_peak *ref_out,
                                 tdoa_peak *tgt_out, double *ref_fit, double *range_diffs, uint8_t *pair_used, double *fix_llh,
                                 double *fix_rms, int32_t *fix_status, int32_t *fix_iters, double *clock_rate)
{
    return process_windows_impl(e, "tdoa_process_windows_retimed", stations_llh, o,
                                WinGeom{ref_win_start, ref_win_len, n_ref_windows, ref_hop},
                                WinGeom{tgt_win_start, tgt_win_len, n_tgt_windows, tgt_hop}, ref_out, tgt_out, ref_fit,
                                range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters, nullptr, true, clock_rate);
}

int tdoa_process_windows_grid(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o, int64_t win_start,
                              int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop, const double *grid_desc,
                              tdoa_peak *ref_out, tdoa_peak *tgt_out, double *ref_fit, double *range_diffs, uint8_t *pair_used,
                              double *fix_llh, double *fix_rms, int32_t *fix_status, int32_t *fix_iters, double *seed_llh,
                              double *seed_cost, int64_t *seed_index)
{
    const GridSeed G{grid_desc, seed_llh, seed_cost, seed_index};
    return process_windows_impl(e, "tdoa_process_windows_grid", stations_llh, o, WinGeom{win_start, win_len, n_ref_windows, hop},
                                WinGeom{win_start, win_len, n_tgt_windows, hop}, ref_out, tgt_out, ref_fit, range_diffs, pair_used,
                                fix_llh, fix_rms, fix_status, fix_iters, &G, false, nullptr);
}

int tdoa_process_windows_closure(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                 const tdoa_closure_opts *c, int64_t ref_win_start, int64_t ref_win_len, int32_t n_ref_windows,
                                 int64_t ref_hop, int64_t tgt_win_start, int64_t tgt_win_len, int32_t n_tgt_windows,
                                 int64_t tgt_hop, int32_t retimed, const double *grid_desc, tdoa_peak *ref_out,
                                 tdoa_peak *tgt_out, double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                 double *closure_resid, int32_t *n_dropped, double *fix_llh, double *fix_rms,
                                 int32_t *fix_status, int32_t *fix_iters, double *clock_rate, double *seed_llh,
                                 double *seed_cost, int64_t *seed_index)
{
    static const char *fn = "tdoa_process_windows_closure";
    if (!e) return TDOA_E_INVALID;
    if (!c) return fail(e, TDOA_E_INVALID, "%s: closure options are NULL", fn);
    if (retimed != 0 && retimed != 1) return fail(e, TDOA_E_INVALID, "%s: retimed must be 0 or 1, got %d", fn, retimed);
    const GridSeed G{grid_desc, seed_llh, seed_cost, seed_index};
    return process_windows_impl(e, fn, stations_llh, o, WinGeom{ref_win_start, ref_win_len, n_ref_windows, ref_hop},
                                WinGeom{tgt_win_start, tgt_win_len, n_tgt_windows, tgt_hop}, ref_out, tgt_out, ref_fit,
                                range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters, grid_desc ? &G : nullptr,
                                retimed == 1, clock_rate, Closure{c, closure_resid, n_dropped});
}

int tdoa_window_fixes_closure(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                              const tdoa_closure_opts *c, int64_t win_start, int64_t win_len, int32_t n_ref_windows,
                              int32_t n_tgt_windows, int64_t hop, const double *grid_desc, const tdoa_peak *ref_in,
                              const tdoa_peak *tgt_in, double *ref_fit, double *range_diffs, uint8_t *pair_used,
                              double *closure_resid, int32_t *n_dropped, double *fix_llh, double *fix_rms,
                              int32_t *fix_status, int32_t *fix_iters, double *seed_llh, double *seed_cost,
                              int64_t *seed_index)
{
    static const char *fn = "tdoa_window_fixes_closure";
    if (!e) return TDOA_E_INVALID;
    if (!c) return fail(e, TDOA_E_INVALID, "%s: closure options are NULL", fn);
    const GridSeed G{grid_desc, seed_llh, seed_cost, seed_index};
    return window_fixes_impl(e, fn, stations_llh, o, win_start, win_len, n_ref_windows, n_tgt_windows, hop, ref_in, tgt_in,
                             ref_fit, range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters,
                             grid_desc ? &G : nullptr, Closure{c, closure_resid, n_dropped});
}

int tdoa_process_windows_exclude(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                 const tdoa_closure_opts *c, const tdoa_exclusion_opts *x, int64_t ref_win_start,
                                 int64_t ref_win_len, int32_t n_ref_windows, int64_t ref_hop, int64_t tgt_win_start,
                                 int64_t tgt_win_len, int32_t n_tgt_windows, int64_t tgt_hop, int32_t retimed,
                                 const double *grid_desc, tdoa_peak *ref_out, tdoa_peak *tgt_out, double *ref_fit,
                                 double *range_diffs, uint8_t *pair_used, double *closure_resid, int32_t *n_dropped,
                                 uint8_t *station_round, double *station_rms, int32_t *n_excluded, double *fix_llh,
                                 double *fix_rms, int32_t *fix_status, int32_t *fix_iters, double *clock_rate,
                                 double *seed_llh, double *seed_cost, int64_t *seed_index)
{
    static const char *fn = "tdoa_process_windows_exclude";
    if (!e) return TDOA_E_INVALID;
    if (!x) return fail(e, TDOA_E_INVALID, "%s: exclusion options are NULL", fn);
    if (retimed != 0 && retimed != 1) return fail(e, TDOA_E_INVALID, "%s: retimed must be 0 or 1, got %d", fn, retimed);
    const GridSeed G{grid_desc, seed_llh, seed_cost, seed_index};
    return process_windows_impl(e, fn, stations_llh, o, WinGeom{ref_win_start, ref_win_len, n_ref_windows, ref_hop},
                                WinGeom{tgt_win_start, tgt_win_len, n_tgt_windows, tgt_hop}, ref_out, tgt_out, ref_fit,
                                range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters, grid_desc ? &G : nullptr,
                                retimed == 1, clock_rate, Closure{c, closure_resid, n_dropped},
                                Exclusion{x, station_round, station_rms, n_excluded});
}

int tdoa_window_fixes_exclude(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                              const tdoa_closure_opts *c, const tdoa_exclusion_opts *x, int64_t win_start, int64_t win_len,
                              int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop, const double *grid_desc,
                              const tdoa_peak *ref_in, const tdoa_peak *tgt_in, double *ref_fit, double *range_diffs,
                              uint8_t *pair_used, double *closure_resid, int32_t *n_dropped, uint8_t *station_round,
                              double *station_rms, int32_t *n_excluded, double *fix_llh, double *fix_rms,
                              int32_t *fix_status, int32_t *fix_iters, double *seed_llh, double *seed_cost,
                              int64_t *seed_index)
{
    static const char *fn = "tdoa_window_fixes_exclude";
    if (!e) return TDOA_E_INVALID;
    if (!x) return fail(e, TDOA_E_INVALID, "%s: exclusion options are NULL", fn);
    const GridSeed G{grid_desc, seed_llh, seed_cost, seed_index};
    return window_fixes_impl(e, fn, stations_llh, o, win_start, win_len, n_ref_windows, n_tgt_windows, hop, ref_in, tgt_in,
                             ref_fit, range_diffs, pair_used, fix_llh, fix_rms, fix_status, fix_iters,
                             grid_desc ? &G : nullptr, Closure{c, closure_resid, n_dropped},
                             Exclusion{x, station_round, station_rms, n_excluded});
}

int tdoa_exclude_stations(tdoa_engine *e, const double *stations_llh, int32_t n_stations, const double *range_diffs,
                          const uint8_t *used, int32_t n_sets, int32_t rd_stride, const double *init_llh, int32_t dims,
                          const tdoa_exclusion_opts *x, uint8_t *out_used, uint8_t *station_round, double *station_rms,
                          int32_t *n_excluded, double *out_llh, double *out_rms, int32_t *status, int32_t *iters)
{
    static const char *fn = "tdoa_exclude_stations";
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    const int S = n_stations, P = S * (S - 1) / 2;
    if (!stations_llh || !range_diffs || !used || !out_used || !out_llh || !status)
        return fail(e, TDOA_E_INVALID, "%s: NULL argument", fn);
    if (S < 3 || S > solve_ls_max_stations())
        return fail(e, TDOA_E_INVALID, "%s: 3..%d stations, got %d", fn, solve_ls_max_stations(), S);
    if (dims != 2 && dims != 3) return fail(e, TDOA_E_INVALID, "%s: dims must be 2 or 3, got %d", fn, dims);
    if (n_sets < 0 || rd_stride < P)
        return fail(e, TDOA_E_INVALID, "%s: n_sets >= 0 and rd_stride >= %d, got %d and %d", fn, P, n_sets, rd_stride);
    if ((rc = exclusion_opts_check(e, fn, x))) return rc;
    if (n_sets == 0) return end_call(e, true);
    const size_t n = (size_t)n_sets * rd_stride, ns = (size_t)n_sets;
    double *d_rd = nullptr, *d_init = nullptr, *d_fix = nullptr, *d_rms = nullptr, *d_srms = nullptr;
    const double *d_llh = nullptr;
    uint8_t *d_used = nullptr, *d_round = nullptr;
    int *d_status = nullptr, *d_iters = nullptr, *d_n_excl = nullptr;
    if ((rc = upload(e, std::vector<double>(stations_llh, stations_llh + (size_t)3 * S), &d_llh)) ||
        (rc = alloc_t(e, &d_rd, n)) || (rc = alloc_t(e, &d_used, n)) || (rc = alloc_t(e, &d_fix, 3 * ns)) ||
        (rc = alloc_t(e, &d_rms, ns)) || (rc = alloc_t(e, &d_status, ns)) || (rc = alloc_t(e, &d_iters, ns)) ||
        (rc = alloc_t(e, &d_round, ns * S)) || (rc = alloc_t(e, &d_srms, ns * S)) || (rc = alloc_t(e, &d_n_excl, ns)))
        return rc;
    CU(cudaMemcpyAsync(d_rd, range_diffs, n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_used, used, n, cudaMemcpyHostToDevice, e->stream));
    if (init_llh) {
        if ((rc = alloc_t(e, &d_init, 3 * ns))) return rc;
        CU(cudaMemcpyAsync(d_init, init_llh, 3 * ns * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    }
    // F: the fix without the check; then the check, which marks d_used (the mask it reads) in place
    launch_solve_ls(d_llh, S, d_rd, n_sets, rd_stride, d_init, dims, d_fix, d_rms, d_status, d_iters, e->stream, d_used);
    launch_window_exclude(d_llh, S, d_rd, d_used, d_used, nullptr, n_sets, rd_stride, d_init, dims, x->max_rms, x->max_exclude,
                          d_fix, d_rms, d_status, d_iters, d_round, d_srms, d_n_excl, e->stream);
    count_launch(e, 2);
    CU(cudaGetLastError());
    // the first P slots of each set only: the rest of the caller's rows are left as they are
    CU(cudaMemcpy2DAsync(out_used, rd_stride, d_used, rd_stride, P, n_sets, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(out_llh, d_fix, 3 * ns * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(status, d_status, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    if (out_rms) CU(cudaMemcpyAsync(out_rms, d_rms, ns * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (iters) CU(cudaMemcpyAsync(iters, d_iters, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    if (station_round) CU(cudaMemcpyAsync(station_round, d_round, ns * S, cudaMemcpyDeviceToHost, e->stream));
    if (station_rms) CU(cudaMemcpyAsync(station_rms, d_srms, ns * S * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (n_excluded) CU(cudaMemcpyAsync(n_excluded, d_n_excl, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    return end_call(e, true);
}

int tdoa_closure(tdoa_engine *e, int32_t n_stations, const double *range_diffs, const uint8_t *used, int32_t n_sets,
                 int32_t rd_stride, int32_t dims, const tdoa_closure_opts *c, uint8_t *out_used, double *out_resid,
                 int32_t *out_dropped)
{
    static const char *fn = "tdoa_closure";
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    const int S = n_stations, P = S * (S - 1) / 2;
    if (!range_diffs || !used || !out_used) return fail(e, TDOA_E_INVALID, "%s: NULL argument", fn);
    if (S < 3 || S > kGraphLsMaxStations) return fail(e, TDOA_E_INVALID, "%s: 3..%d stations, got %d", fn, kGraphLsMaxStations, S);
    if (dims != 2 && dims != 3) return fail(e, TDOA_E_INVALID, "%s: dims must be 2 or 3, got %d", fn, dims);
    if (n_sets < 0 || rd_stride < P)
        return fail(e, TDOA_E_INVALID, "%s: n_sets >= 0 and rd_stride >= %d, got %d and %d", fn, P, n_sets, rd_stride);
    if ((rc = closure_opts_check(e, fn, c))) return rc;
    if (n_sets == 0) return end_call(e, true);
    const size_t n = (size_t)n_sets * rd_stride;
    double *d_rd = nullptr, *d_resid = nullptr;
    uint8_t *d_used = nullptr;
    int *d_dropped = nullptr;
    if ((rc = alloc_t(e, &d_rd, n)) || (rc = alloc_t(e, &d_used, n)) || (rc = alloc_t(e, &d_resid, n)) ||
        (rc = alloc_t(e, &d_dropped, (size_t)n_sets)))
        return rc;
    CU(cudaMemcpyAsync(d_rd, range_diffs, n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_used, used, n, cudaMemcpyHostToDevice, e->stream));
    launch_window_closure(d_rd, d_used, nullptr, n_sets, rd_stride, S, dims, c->max_residual, c->max_drop, d_resid, d_dropped,
                          e->stream);
    count_launch(e);
    CU(cudaGetLastError());
    // the first P slots of each set only: the rest of the caller's rows are left as they are
    CU(cudaMemcpy2DAsync(out_used, rd_stride, d_used, rd_stride, P, n_sets, cudaMemcpyDeviceToHost, e->stream));
    if (out_resid)
        CU(cudaMemcpy2DAsync(out_resid, rd_stride * sizeof(double), d_resid, rd_stride * sizeof(double), P * sizeof(double),
                             n_sets, cudaMemcpyDeviceToHost, e->stream));
    if (out_dropped) CU(cudaMemcpyAsync(out_dropped, d_dropped, (size_t)n_sets * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    return end_call(e, true);
}

}  // extern "C"
