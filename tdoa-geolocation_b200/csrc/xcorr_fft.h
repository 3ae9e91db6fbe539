// xcorr_fft.h -- job descriptors and launchers of the FFT correlation path (xcorr_fft.cu).
#pragma once
#include "kernels.h"

namespace tdoa {

constexpr int kFftN = 8192;               // complex FFT size held in one CTA's shared memory
constexpr int kLagW = 2048;               // lags served by one FFT job
constexpr int kSeg = kFftN - kLagW;       // template samples per segment (6144 = 24 * 256)
constexpr int kMaxCand = 64;              // candidate lags re-evaluated exactly per pair
constexpr int kFftBins = kFftN / 2 + 1;

// The ranking transforms pack two real planes into one complex FFT and split the spectra with Z[k] +- conj Z[N-k],
// so each spectrum carries rounding on the scale of the other plane: with planes of powers P_a, P_b the ranking's
// error in coefficient units grows like eps log N sqrt(P_a / P_b) (a weak-branch station of near-constant bytes
// beside strong ones reaches 2.5e9 and errors up to 1e-2, far over the selection tolerance:
// profiles/r11_ranking.jsonl).  When the scales
// f32(1 / sqrt(power)) of the two planes of a transform differ by more than kRankPackRatio, both are multiplied by
// their scale as the transform loads them -- the very multiply k_corr_candidates applies -- and the finish leaves
// them out; otherwise (stations of similar power: no multiply at all) the finish applies both scales.  Planes
// that share a transform then differ in power by at most kRankPackRatio^2.
constexpr float kRankPackRatio = 16.f;
// a and b: statistics of the two planes of one transform
__device__ __forceinline__ bool rank_scaled(const double *a, const double *b)
{
    const float sa = (float)a[ST_SCALE], sb = (float)b[ST_SCALE];
    return fmaxf(sa, sb) > kRankPackRatio * fminf(sa, sb);
}
// the factor plane a is loaded with (packed with b), and the one the finish applies for it
__device__ __forceinline__ float rank_pre(const double *a, const double *b) { return rank_scaled(a, b) ? (float)a[ST_SCALE] : 1.f; }
__device__ __forceinline__ double rank_post(const double *a, const double *b)
{
    return rank_scaled(a, b) ? 1.0 : (double)(float)a[ST_SCALE];
}

// One (pair, lag chunk): approx[d] ~ corr(lag0 + d), d in [0, n_lags), n_lags <= kLagW.
struct FftJob {
    const float *t, *s;              // real planes, pre-normalise
    const double *t_stats, *s_stats; // ST_SCALE (rank_post in the finish)
    const double *t_pack, *s_pack;   // statistics of the plane t (s) shares its ranking transform with
    i64 t_off;                       // template starts at t + t_off
    i64 n_t;                         // template samples that take part
    i64 sl;                          // signal length
    i64 s_off;                       // signal index matched with template index 0 at lag index 0
    int n_lags;
    int n_seg;                       // ceil(n_t / kSeg)
    int n_cta;                       // CTAs (= partial spectra) of this job
    float2 *partials;                // [n_cta][kFftBins]
    float2 *spectrum;                // [kFftBins] sum of the partials
    float *approx;                   // [n_lags] correlation-coefficient units
};

// A tile of one window's pairs: up to two template signals x two signal-role signals that
// share offsets and lengths.  Product p = 2 a + b is conj(T_a) S_b; partials[p] == nullptr
// where the tile has no such pair.  (xcorr_tile.cu)
struct TileJob {
    const float *t0, *t1;   // template planes (t1 == t0 when the tile has one template)
    const float *s0, *s1;   // signal planes
    const double *t0_stats, *t1_stats, *s0_stats, *s1_stats;   // their statistics (rank_pre as the samples are loaded)
    i64 t_off, n_t, sl, s_off;
    int n_seg, n_cta;
    float2 *partials[4];    // [n_cta][kFftBins] each
};

struct SelJob {
    const float *approx;  // [n_lags] all lag chunks of the pair
    int n_lags;
    int sanity;           // re-search range [0, sanity), 0 = none
    int neighbours;       // also select lag +-1 of every candidate (parabolic vertex)
    int max_cand;
    float tol;
    int *cand;            // [max_cand] ascending lag indices
    int *n_cand;          // candidates found (may exceed max_cand: overflow)
    float *approx_max;
    const double *t_stats, *s_stats;   // per-signal statistics (ST_POWER1): a signal without power is identically zero
    const int2 *bound;    // the record's interval (PeakJob::bound): maximum, candidates and neighbours from its run only
    int lag_origin, decim;
};

struct CandJob {
    const int *cand;
    const int *n_cand;
    int max_cand;
    const float *approx;
    double *blocksums;    // [max_cand][nb]
};

// ---- wide lag searches through a 2^21-point transform in global memory (xcorr_big.cu)
constexpr int kBigN1 = 256;
constexpr i64 kBigN = (i64)kBigN1 * kFftN;     // 2 097 152 complex points
constexpr int kBigMinLags = 8192;              // narrower searches stay with the segment kernel

struct BigColJob {      // forward column pass of one transform: z[n] = x0[base+n] sc0 + i x1[base+n] sc1, lo <= n < hi
    const float *x0, *x1;
    const double *x0_stats, *x1_stats;              // sc0, sc1: rank_pre
    i64 base, lo, hi;
    float2 *out;        // [256][8192]
};
struct BigRowJob {      // row pass, in place
    float2 *buf;
    int inverse;
};
struct BigCrossJob {    // G0 = C00 + i C01, G1 = C10 + i C11 with C_ab = 4 conj(T_a) S_b
    const float2 *A, *B;
    float2 *G0, *G1;
    int accumulate;     // add to what G0 / G1 hold (segments after the first)
};
struct BigOutJob {      // inverse column pass of one packed pair of correlations
    const float2 *G;
    float *approx0, *approx1;                       // [n_lags] each, nullptr: pair absent
    const double *t_stats, *t_pack;                 // the template and the plane it was packed with (rank_post)
    const double *s0_stats, *s1_stats;              // the two signals (packed together)
    i64 n_t;
    int n_lags;
};
int big_setup(cudaStream_t st, float2 **d_fine);
void launch_big_cols(const BigColJob *d_jobs, int n_jobs, const float2 *d_tw, const float2 *d_fine, cudaStream_t st);
void launch_big_rows(const BigRowJob *d_jobs, int n_jobs, const float2 *d_tw, const float2 *d_fine, cudaStream_t st);
void launch_big_cross(const BigCrossJob *d_jobs, int n_jobs, cudaStream_t st);
void launch_big_out(const BigOutJob *d_jobs, int n_jobs, const float2 *d_tw, cudaStream_t st);

// ---- many stations per window: each station-segment transformed once, pairs formed from the
// parked spectra (xcorr_spec.cu)
constexpr int kSpecMaxPacked = 16;   // packed transforms (two stations each) per job: templates + signals
constexpr int kSpecBins = 32;        // frequency bins per accumulation CTA (one warp per register tile)
constexpr int kSpecChunks = 8192 / 2 / kSpecBins + 1;   // 129: the last chunk holds the Nyquist bin alone
constexpr int kSpecMinPairs = 10;    // smaller groups stay with the 2 x 2 tiles
constexpr int kSpecTile = 4;         // register tile: 4 template rows x 4 signal rows per thread
constexpr int kSpecMaxTiles = 10;    // tiles per accumulation job (16 stations, all pairs: 10)

// Parked spectra of one unit: [segment][chunk][row][kSpecBins] float2, row = 2 m + {0, 1} for the two stations of
// packed transform m (templates first): what one accumulation CTA reads per segment is ONE contiguous block.
__host__ __device__ inline size_t spec_seg_elems(int n_rows) { return (size_t)kSpecChunks * n_rows * kSpecBins; }

struct SpecFftJob {     // one packed transform, all its segments
    const float *x0, *x1;   // planes: z = x0 sc0 + i x1 sc1
    const double *x0_stats, *x1_stats;   // sc0, sc1: rank_pre
    i64 base;               // plane index of sample 0 of segment 0
    i64 stride;             // samples between segment starts
    i64 lo, hi;             // plane indices outside [lo, hi) read as zero
    int seg_len;            // samples of a segment that carry data (the rest of the 8192 is zero)
    int n_seg;
    float2 *out;            // parked spectra of the unit
    int row0, n_rows;       // this transform fills rows row0 and row0 + 1 of n_rows
};
struct SpecAccJob {
    const float2 *spec;     // parked spectra of the unit
    int n_rows, n_seg, n_tiles;
    unsigned char t_row[kSpecMaxTiles][kSpecTile];   // rows of the tile's templates / signals (absent slots: any valid row)
    unsigned char s_row[kSpecMaxTiles][kSpecTile];
    float2 *out[kSpecMaxTiles][kSpecTile * kSpecTile];   // [4097] summed cross-spectrum conj(T_a) S_c of slot 4 a + c, or nullptr
};
int spec_setup();
void launch_spec_fft(const SpecFftJob *d_jobs, int n_jobs, int max_seg, const float2 *d_tw, cudaStream_t st);
void launch_spec_acc(const SpecAccJob *d_jobs, int n_jobs, cudaStream_t st);

int fft_setup(cudaStream_t st, float2 **d_tw);
size_t fft_partials_bytes(int n_cta);
void launch_fft_segments(const FftJob *d_jobs, int n_jobs, int max_cta, const float2 *d_tw, cudaStream_t st);
int fft_tile_setup();
void launch_fft_tiles(const TileJob *d_jobs, int n_jobs, int max_cta, const float2 *d_tw, cudaStream_t st);
void launch_fft_reduce(const FftJob *d_jobs, int n_jobs, cudaStream_t st);
void launch_fft_finish(const FftJob *d_jobs, int n_jobs, const float2 *d_tw, cudaStream_t st);
void launch_select_candidates(const SelJob *d_jobs, int n_jobs, cudaStream_t st);
void launch_corr_candidates(const PairJob *d_jobs, const CandJob *d_cjobs, int n_jobs, i64 max_nb, cudaStream_t st);
void launch_peak_candidates(const PairJob *d_jobs, const CandJob *d_cjobs, const PeakJob *d_pjobs, int n_jobs,
                            cudaStream_t st);

}  // namespace tdoa
