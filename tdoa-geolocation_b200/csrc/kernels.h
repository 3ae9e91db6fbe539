// kernels.h -- job descriptors and launchers of the engine's CUDA kernels.
//
// Every launcher is batched: it takes a device array of job descriptors and runs one
// grid whose y (or z) dimension indexes the job.  Reductions are deterministic
// (per-CTA partials added in index order by the last CTA to arrive), so a call gives
// the same bits every time.
#pragma once
#include "common.cuh"
#include "../../include/tdoa_b200.h"

namespace tdoa {

// slots of a signal's device statistics block (doubles)
enum {
    ST_POWER0 = 0,  // calculateSignalPower of the raw signal (processor.go:322-333)
    ST_SUM_RE = 1,  // sum of the signal entering removeDCBias
    ST_SUM_IM = 2,
    ST_DC_RE = 3,   // f32 DC bias (processor.go:309)
    ST_DC_IM = 4,
    ST_POWER1 = 5,  // power before normalizeSignal (processor.go:336-351)
    ST_SCALE = 6,   // f32(1/sqrt(power)), 1 when power <= 0
    ST_COUNT = 8
};

enum { BOX_LP = 0, BOX_HP = 1 };

struct SigJob {
    SigSrc src;        // raw / planar source (kernels that read the capture)
    i64 n;             // samples
    const float *q_re; // input planes (kernels that read planes)
    const float *q_im; // may be nullptr: imaginary part identically zero
    const float *r_re; // second input (notch combine: the band)
    const float *r_im;
    float *p_re;       // output planes
    float *p_im;       // may be nullptr
    double *stats;     // ST_* block of this signal
    double *partials;  // >= 2 * grid.x doubles of scratch for this job
    unsigned *counter; // zeroed ticket counter for this job
    int window;        // box-car window size (processor.go:270)
    int window2;       // k_weak_fused only: the low-pass window that follows the high-pass of `window`
    int mode;          // BOX_LP / BOX_HP
    int sub_dc;        // subtract ST_DC_* from the input while loading
    int want_power;    // accumulate ST_POWER1 / ST_SCALE of the output
    // fused discriminator only: process samples [i_begin, i_end) of the signal (i_end == 0:
    // all of it; i_begin a multiple of 4096) and, when chunk_out is set, leave the two
    // partial sums (power, output sum) there instead of finishing the statistics -- the
    // capture is demodulated chunk by chunk while it is still arriving over PCIe
    i64 i_begin, i_end;
    double *chunk_out;
};

// correlator variants
enum {
    CORR_BINARY = 0,   // real parts only, f32 product, f64 sum, /B per block, mean of blocks
    CORR_SOURCE = 1,   // f32(re*re' + im*im'), same blocking, * sqrt(nb*B)   (processor.go:691-720)
    CORR_EXTENDED = 2  // real parts, exact f64 products, single sum / n
};

struct PairJob {
    const float *t_re, *t_im;  // template planes (pre-normalise) and its stats
    const float *s_re, *s_im;  // signal planes
    const double *t_stats, *s_stats;
    i64 t_off;       // template starts at t_re + t_off
    i64 n_t;         // template samples that take part (nb * block, or n for EXTENDED)
    i64 sl;          // signal length
    i64 block;       // block size B (EXTENDED: partial-sum chunk)
    i64 nb;          // whole blocks
    int lag0;        // first lag of the search (signal index offset)
    int n_lags;      // lags evaluated: lag0 .. lag0+n_lags-1
    int variant;     // CORR_*
    double *blocksums;  // [nb][n_lags]
    double *corr;       // [n_lags] finalised correlation per lag
};

// peak record flags / layout mirror include/tdoa_b200.h
struct PeakRec {
    int32_t lag;
    uint32_t flags;
    double corr;
    float frac;
    float margin;
    int32_t first_lag;
    int32_t n_blocks;
};

struct PeakJob {
    const double *corr;   // first-pass correlations [n_lags]
    const double *corr2;  // sanity re-search correlations [n_lags2] (may alias corr)
    int n_lags;
    int n_lags2;
    int lag_origin;       // lag value of index 0 (EXTENDED: -max_lag)
    int sanity;           // 0 disables the re-search
    int variant;
    int nb;               // blocks of the first pass (0: nothing evaluated)
    uint32_t flags;       // flags or-ed into the record
    PeakRec *out;
    double *first_corr;   // optional: correlation of the first-pass peak (before the sanity re-search)
};

// ---- preprocess.cu
void launch_power(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st);
void launch_unpack(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st);
void launch_demod(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st);
void launch_envelope(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st);
void launch_seqsum(const SigJob *d_jobs, int n_jobs, cudaStream_t st);
// ---- seqsum.cu: the same sequential f32 chain, chunk-parallel and still bit for bit
struct SeqJob {
    const float *x;    // one component plane (nullptr: identically zero, *out = 0)
    i64 n;
    double *out;       // ST_DC_RE or ST_DC_IM slot: f32(sum / n) widened (processor.go:309)
    i64 n_chunks;      // filled by seqsum_carve
    double *csum, *pre;
    void *infos;
};
size_t seqsum_scratch_bytes(i64 n);
void seqsum_carve(SeqJob &J, void *scratch);
void launch_seqsum_chunked(const SeqJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);
void launch_boxcar(const SigJob *d_jobs, int n_jobs, i64 max_n, int max_window, cudaStream_t st);
void launch_boxcar_slide(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);   // EXTENDED: f64 prefix sums
void launch_notch_combine(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);
void launch_normalize(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);
void launch_decimate(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);  // window = D, n = input samples
void launch_interleave(const float *re, const float *im, i64 n, float *out_c64, cudaStream_t st);
void launch_deinterleave(const float *c64, i64 n, float *re, float *im, cudaStream_t st);
int boxcar_grid_x(i64 n);
int stream_grid_x(i64 n);
int unpack_selftest(cudaStream_t st);  // 0 ok: arithmetic unpack == host LUT for all 256 codes

// ---- preprocess_weak.cu (EXTENDED mode, weak branch: two passes over the capture bytes)
void launch_raw_stats(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);    // ST_POWER0 + ST_SUM_* + ST_DC_*
void launch_weak_fused(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);   // bytes -> DC, HP(window), LP(window2), power
int raw_stats_grid_x(i64 n);
int weak_fused_max_half_wide();
int weak_fused_max_half_small();
int weak_unpack_selftest(cudaStream_t st);  // 0 ok: divide-free unpack == unpack_byte for all 256 codes

// ---- preprocess_fast.cu
void launch_demod_fused(const SigJob *d_jobs, int n_jobs, i64 max_n, int fast, cudaStream_t st);
// statistics of a signal demodulated in chunks: adds chunk_sums[c][0..1] in chunk order
void launch_demod_finish(const double *chunk_sums, int n_chunks, i64 n, double *stats, cudaStream_t st);
void launch_boxcar_small(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st);
int boxcar_small_max_half();
long long div_selftest(cudaStream_t st);  // mismatches of the constant-divisor division, 0 = proven
int demod_setup(cudaStream_t st);         // tables + shared-memory opt-in of the lean discriminator; 0 ok
// lean discriminator against the reference statement over all 2^32 (previous, current) byte quads;
// first_bad: [0] = count stored, [1..63] = offending quads (prev I, prev Q, cur I, cur Q from the low byte up)
long long demod_selftest(cudaStream_t st, unsigned *first_bad, int which, long long *extra);
int fast_grid_x(i64 n);

// ---- xcorr_exact.cu
void launch_corr_brute(const PairJob *d_jobs, int n_jobs, i64 max_nb, int max_lags, cudaStream_t st);
void launch_corr_finalize(const PairJob *d_jobs, int n_jobs, int max_lags, cudaStream_t st);
void launch_peak(const PeakJob *d_jobs, int n_jobs, cudaStream_t st);
void launch_lag_units(PeakRec *d_recs, int n, int D, cudaStream_t st);

// ---- analyze.cu (fast_analyzer.go / analyzer.go)
struct QualJob {
    SigSrc src;      // the signal's bytes (REF: first run in block 1, second in block 3)
    i64 n;           // samples
    int fast;        // 1: fast_analyzer.go, 0: analyzer.go
    int m;           // analysed samples of the spectrum (8192 / 16384, or n when shorter)
    void *parts;     // per-CTA partial statistics (quality_part_bytes() each)
    void *out;       // tdoa_signal_quality on the device
    void *fft_a, *fft_b;  // m double2 each
    double *psd;     // m doubles
};
size_t quality_part_bytes();
int quality_setup();
void launch_quality(const QualJob *d_jobs, int n_jobs, int n_stat_cta, int max_m, cudaStream_t st);

// ---- solve.cu
void launch_baselines(const double *d_llh, int n_st, double *d_out, cudaStream_t st);
void launch_solve(const double *d_llh, const double *d_rd, int n_sets, int rd_stride, double *d_out_llh,
                  int *d_status, int *d_iters, cudaStream_t st);
void launch_solve_binary(const double *d_llh, const double *d_rd, int n_rd, double *d_out_llh, int *d_info, double *d_trace,
                         cudaStream_t st);
void launch_solve_ls(const double *d_llh, int n_st, const double *d_rd, int n_sets, int rd_stride, const double *d_init,
                     int dims, double *d_out_llh, double *d_rms, int *d_status, int *d_iters, cudaStream_t st,
                     const uint8_t *d_used = nullptr);   // d_used[set * rd_stride + p]: pair p takes part
int solve_ls_max_stations();
// ---- window_fix.cu (tdoa_process_windows / tdoa_window_fixes): the REF drift fit per pair and the
// range differences per (TGT window, pair); the fix is launch_solve_ls with the used mask
void launch_window_ref_fit(const PeakRec *d_ref, int n_ref, int n_st, const double *d_t_ref, const double *d_t_mid,
                           const double *d_llh, const double *d_ref_tx, float min_margin, double max_resid, double *d_fit,
                           double *d_ref_fit, cudaStream_t st);
void launch_window_rd(const PeakRec *d_tgt, int n_tgt, int n_st, const double *d_t_tgt, const double *d_fit, float min_margin,
                      double fs, double *d_rd, uint8_t *d_used, cudaStream_t st);
constexpr int kWindowFitDoubles = 5;   // per pair: a, beta, t_mean, windows used, geometric term
// ---- retime.cu (tdoa_process_windows_retimed): station clock rates from the REF fits, and the re-timing gather
// rate[S] (0 for a station without a fitted pair) re-times the planes, clock[S] (NaN there) is what the call returns;
// n_st <= 64 (solve_ls_max_stations)
void launch_station_rates(const double *d_fit, int n_st, double *d_rate, double *d_clock, cudaStream_t st);
// the closure check of the windowed fixes (tdoa_closure), one CTA per set, n_st <= 64: d_used[set * stride + p] in u
// (0 / 1), out 0 / 1 / 2 (2: dropped); d_mask (may be nullptr) the final 0 / 1 mask; d_resid (may be nullptr) the
// residuals, NaN where u = 0; d_dropped (may be nullptr) the pairs dropped per set
void launch_window_closure(const double *d_rd, uint8_t *d_used, uint8_t *d_mask, int n_sets, int stride, int n_st, int dims,
                           double max_resid, int max_drop, double *d_resid, int *d_dropped, cudaStream_t st);
// the station check of the windowed fixes (tdoa_exclude_stations; exclude.cu), one CTA per set, n_st <= 64, after
// launch_solve_ls with the same mask and start (d_init may be nullptr: the station mean): d_mask the fix mask (0 /
// nonzero); d_used (may be nullptr, may be d_mask) gets 3 on the pairs of excluded stations; d_final (may be nullptr)
// the final 0 / 1 mask; the fix arrays are overwritten where a station is excluded; d_round[set * n_st + k] (uint8)
// and d_srms[set * n_st + k] (NaN: not a candidate) and d_n_excl may be nullptr
void launch_window_exclude(const double *d_llh, int n_st, const double *d_rd, const uint8_t *d_mask, uint8_t *d_used,
                           uint8_t *d_final, int n_sets, int stride, const double *d_init, int dims, double max_rms,
                           int max_exclude, double *d_out_llh, double *d_rms, int *d_status, int *d_iters, uint8_t *d_round,
                           double *d_srms, int *d_n_excl, cudaStream_t st);
struct RetimeJob {
    const float *x;   // one preprocessed plane, n samples
    float *y;         // its re-timed plane (16-byte aligned)
    i64 n;
    int station;      // index into the rates
};
void launch_retime(const RetimeJob *d_jobs, int n_jobs, i64 max_n, const double *d_rates, cudaStream_t st);
void launch_range_diffs(const PeakRec *d_ref, const PeakRec *d_tgt, int n_pairs, double fs, int mode, double *d_td,
                        double *d_rd, cudaStream_t st);
// the grid arg-min; its one caller, grid_search_queue (engine.cu), chooses the form and checks the ranked one
// d_used (may be nullptr): the masked statement, d_used[set * rd_stride + p]; d_tab then holds the masked rows (their
// "searched" flags); a set without an arg-min gets index -1, cost NaN and leaves d_out_llh as it was
void launch_grid_cells(const double *d_llh, int n_st, const double *d_grid_desc, int nlat, int nlon,
                       const double *d_rd, int n_sets, int rd_stride, double *d_best_cost, i64 *d_best_idx,
                       double *d_out_llh, void *d_scratch, cudaStream_t st, const uint8_t *d_used, const double *d_tab);
size_t grid_scratch_bytes(int nlat, int nlon, int n_sets);
// the same arg-min, ranked by the expanded cost (16 FMA per cell and set) and settled by the statement on the survivors;
// d_count: grid_rank_chunks(n_sets) ints, and grid_rank_overflowed on their host copy means the ranked pass is incomplete
void launch_grid_ranked(const double *d_llh, int n_st, const double *d_grid_desc, int nlat, int nlon, const double *d_tab,
                        const double *d_rd, int n_sets, int rd_stride, double *d_best_cost, i64 *d_best_idx,
                        double *d_out_llh, void *d_scratch, int *d_count, cudaStream_t st, const uint8_t *d_used);
size_t grid_rank_scratch_bytes(int nlat, int nlon, int n_sets);
int grid_rank_chunks(int n_sets);
bool grid_rank_overflowed(const int *h_count, int n_sets);
// one set's row of d_tab on the host (masked when used != nullptr); false: a masked set with no used pair
bool grid_rank_row(const double *rd, const uint8_t *used, int n_st, double *row);
// the masked rows on the device (the windowed seed): a set the least-squares step would refuse (status 2 with dims) is
// not searched
void launch_grid_rows(const double *d_rd, const uint8_t *d_used, int n_sets, int rd_stride, int n_st, int dims, double *d_tab,
                      cudaStream_t st);
int grid_rank_tab_doubles(bool masked = false);

}  // namespace tdoa
