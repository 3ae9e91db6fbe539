/*
 * tdoa_b200.h -- C ABI of libtdoa_b200.so, the B200 (sm_100a) TDOA correlation engine.
 *
 * Drop-in boundary for the processing stage of KX0U-Jim/tdoa-geolocation.  The
 * reference has no FFI seam of its own (a single `package main`), so each entry
 * point below names the reference method it replaces (file:line in the reference
 * tree).  Plain pointers and sizes only; the caller owns every host pointer and the
 * library never retains one after a call returns (cgo pointer rules).
 *
 * Error convention: every function returns 0 on success or a negative TDOA_E_* code;
 * tdoa_last_error() returns the message of the last failure on that engine
 * (NULL engine: the last tdoa_create failure of the calling thread).  There is no
 * CPU fallback: without an sm_100 device tdoa_create fails with TDOA_E_NODEVICE.
 *
 * Threading: one caller at a time per engine (the reference is single-threaded);
 * every entry point selects the engine's device itself, so it is safe to call from
 * migrating goroutines/threads without pinning.
 */
#ifndef TDOA_B200_H
#define TDOA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TDOA_API __attribute__((visibility("default")))

/* error codes */
#define TDOA_OK 0
#define TDOA_E_INVALID (-1)   /* bad argument                                      */
#define TDOA_E_NODEVICE (-2)  /* no sm_100 CUDA device / CUDA runtime unusable     */
#define TDOA_E_CUDA (-3)      /* a CUDA call failed (message has the CUDA error)   */
#define TDOA_E_NOMEM (-4)     /* device or pinned-host allocation failed           */
#define TDOA_E_STATE (-5)     /* call sequence error (e.g. station not loaded)     */
#define TDOA_E_SINGULAR (-6)  /* solveTDOA: singular Jacobian (processor.go:997)   */
#define TDOA_E_IO (-7)        /* loadIQData: open / stat / read failed (:170-191)  */

/* processing modes (tdoa_config.mode) */
#define TDOA_MODE_SOURCE 0   /* processor.go as committed: complex64 box-car path,
                                1000-sample blocks, sqrt(N) gain, maxLag 20000      */
#define TDOA_MODE_BINARY 1   /* shipped `processor` ELF: FM discriminator / envelope /
                                weak 3-way preprocess, real correlator over a template
                                shortened by maxLag, 10000-sample blocks, 120-sample
                                sanity re-search                                     */
#define TDOA_MODE_EXTENDED 2 /* BINARY preprocessing + two-sided lag search with
                                parabolic sub-sample refinement (engine-defined)     */

/* signal kinds of the dual-frequency capture (processor.go:208-267) */
#define TDOA_KIND_REF 0 /* blocks 1 and 3 concatenated */
#define TDOA_KIND_TGT 1 /* block 2 */

/* tdoa_peak.flags */
#define TDOA_PEAK_RESEARCHED 0x1u /* sanity re-search replaced the first-pass peak   */
#define TDOA_PEAK_EDGE 0x2u       /* peak on the edge of the lag range (frac = 0)    */
#define TDOA_PEAK_BRUTE 0x4u      /* every lag was evaluated in the time domain      */
#define TDOA_PEAK_EMPTY 0x8u      /* empty input: (0, 0.0) as processor.go:622-625   */
#define TDOA_PEAK_BOUNDED 0x20u   /* lag searched within an interval (tdoa_xcorr_bounded,
                                     tdoa_set_tgt_bounds); EMPTY too: the interval held
                                     no lag of the range                               */
#define TDOA_PEAK_NCAND(f) (((f) >> 16) & 0xffu)   /* lags re-evaluated exactly (FFT path)   */
#define TDOA_PEAK_BRANCH1(f) (((f) >> 8) & 3u)  /* preprocess branch of signal 1      */
#define TDOA_PEAK_BRANCH2(f) (((f) >> 10) & 3u) /* 0 strong/std, 1 moderate, 2 weak   */

typedef struct tdoa_engine tdoa_engine; /* opaque: device memory, streams, plans */

/* One correlation peak; 32 bytes; also the record exchanged between GPUs.
 * margin = (|peak| - |runner-up|) / |peak|, rounded to f32, the runner-up being the largest |corr| over every
 * other lag of the first pass.  On the every-lag path (TDOA_PEAK_BRUTE: use_fft = 0, the candidate-overflow redo)
 * every |corr| is exact.  On the FFT paths the runner-up is the largest |approximate value| of the f32 ranking
 * (exact values exist only for the candidates), so the margin differs from the exact one by at most eps / |peak|
 * plus its rounding, eps (<= 1e-6 in correlation units, measured against an f64 correlation on every FFT path,
 * weak-branch stations beside strong ones included) being the ranking's error.  Two tied peaks: margin 0 exactly
 * on the every-lag path, |margin| <= eps / |peak| on the FFT paths.
 * Which signal is the template: BINARY and SOURCE make the shorter of the two signals the template
 * (processor.go:653-661), so with signal 1 longer the lag is the delay of signal 1.  EXTENDED keeps signal 1 as
 * the template whatever the lengths: with W = min(n1, n2) the search is over the first W samples of both
 * preprocessed signals (each preprocessed over its own full length) and the lag is always the delay of signal 2,
 * i.e. d_j - d_i for pair i < j. */
typedef struct {
    int32_t lag;       /* integer lag of the peak, samples (delay of signal 2; see above) */
    uint32_t flags;    /* TDOA_PEAK_*                                                */
    double corr;       /* correlation at the peak, signed (the Go float64 return)    */
    float frac;        /* sub-sample offset in [-0.5,0.5]; 0 in SOURCE/BINARY modes  */
    float margin;      /* (|peak|-|runner-up|)/|peak|; exact runner-up on BRUTE records,
                          the f32 ranking's on FFT records (see above)                */
    int32_t first_lag; /* first-pass lag before the sanity re-search                 */
    int32_t n_blocks;  /* whole blocks that contributed (processor.go:691-712)       */
} tdoa_peak;

typedef struct {
    double sample_rate;    /* 2e6 (processor.go:821)                                 */
    int32_t mode;          /* TDOA_MODE_*                                            */
    int32_t n_stations;    /* stations the engine holds (>= 2)                       */
    int32_t chunk_samples; /* "test chunk": 2000000 source (processor.go:772),
                              1000000 binary; 0 = whole signal                       */
    int32_t max_lag;       /* 20000 source (processor.go:633), 2000 binary;
                              EXTENDED: lags -max_lag..+max_lag                      */
    int32_t block_size;    /* 1000 source (processor.go:682), 10000 binary           */
    int32_t sanity_lag;    /* 120 (binary re-search window); 0 disables              */
    int32_t fast_demod;    /* 0: f64 products + f64 atan2 as the reference;
                              1: f32 discriminator (<= 2 ulp), EXTENDED only default;
                              2: as 0, every sample through the full-accuracy arctangent
                                 (no fast path; a test switch)                        */
    int32_t use_fft;       /* 1: FFT candidate search + exact re-evaluation (2 x 2 station
                              tiles; station spectra parked once per segment for >= 10
                              pairs per window; a 2^21-point transform for >= 8192 lags);
                              0: evaluate every lag in the time domain;
                              test switches: 2 one transform per pair, 3 no 2^21-point
                              transform, 4 no parked spectra, 5 plain one-add-at-a-
                              time walk for the sequential DC sum, 6 EXTENDED weak
                              branch as four kernels over planes (not the fused pass) */
    int32_t device;        /* CUDA device ordinal                                    */
    int32_t seq_dc_limit;  /* removeDCBias (processor.go:299-319): signals of up to this many
                              samples get the reference's sequential f32 accumulator,
                              bit for bit; longer ones (which the reference never
                              processes: it truncates to its chunk) an exactly rounded
                              sum.  0 = mode default (4194304 SOURCE/BINARY, never in
                              EXTENDED); -1 = never                                   */
    int32_t copy_chunk;    /* tdoa_load_u8_pinned: samples per host->device copy chunk
                              (multiple of 4096); 0 = 16777216 (32 MB of capture)    */
    int32_t guard_samples; /* samples dropped at the start of blocks 2 and 3 (the retune
                              transient, collector.go:85 / rtl_sdr.c:117-135); 0 = the
                              reference's split (processor.go:208-267)                */
    int32_t decimate;      /* EXTENDED mode only: D > 1 appends a decimating box-car
                              (mean of D consecutive samples, rtl_fm.c:302-322 style) to the
                              preprocessing chain; correlation at fs / D over max_lag / D
                              lags, records in samples of the capture (lag + frac)       */
    int32_t serial_kinds;  /* tdoa_process: 0 = the TGT pair loop is queued on a second stream beside
                              the REF pair loop (their kernels share the SMs); 1 = one stream, one
                              kernel at a time (what the per-kernel timings of tdoa_get_stats
                              need to mean anything)                                        */
    int32_t n_devices;     /* 0 or 1: one GPU (`device`).  N > 1: this ONE process drives the N GPUs
                              device .. device + N - 1: every capture is loaded to each of them and
                              tdoa_xcorr over >= 2 windows deals the windows round-robin over them
                              (processor.go:816-850 is the loop being sharded), the peak records
                              meeting in one NCCL all-gather over NVLink; every other call runs on
                              `device`.  One process per GPU instead: tdoa_comm_init            */
    int32_t reserved[1];
} tdoa_config;

/* Fill *cfg with the reference-matching defaults of `mode`. */
TDOA_API int tdoa_default_config(int32_t mode, tdoa_config *cfg);

TDOA_API int tdoa_create(tdoa_engine **out, const tdoa_config *cfg);
TDOA_API void tdoa_destroy(tdoa_engine *e);
TDOA_API const char *tdoa_last_error(const tdoa_engine *e);

/* Pinned host buffers for callers that want full PCIe rate (optional). */
TDOA_API void *tdoa_host_alloc(size_t nbytes);
TDOA_API void tdoa_host_free(void *p);

/* loadIQData + extractReferenceSignal + extractTargetSignal (processor.go:166-267):
 * hands one station's whole .dat capture (interleaved uint8 I,Q) to the engine.
 * The bytes are copied to the device before the call returns. */
TDOA_API int tdoa_load_u8(tdoa_engine *e, int32_t station, const uint8_t *iq, size_t nbytes);
/* loadIQData on a file (processor.go:166-205): streams the .dat capture to the device
 * through two pinned 32 MB staging buffers (disk read of one piece overlaps the PCIe copy
 * of the previous).  *n_samples (may be NULL) = file size / 2 (:183).  Errors carry the
 * reference's messages ("failed to open file: ...", TDOA_E_IO). */
TDOA_API int tdoa_load_file(tdoa_engine *e, int32_t station, const char *path, int64_t *n_samples);
/* Same for a capture in memory obtained from tdoa_host_alloc (C memory, outside the Go
 * heap, so the cgo pointer rules do not apply): returns at once.  The host -> device
 * copies are queued by the next call that needs the capture -- the blocks of the signal
 * kind that call asks for first, across all stations, then the rest -- and the FM
 * discriminator follows them chunk by chunk, so preprocessing overlaps the PCIe
 * transfer.  The buffer must stay unchanged until tdoa_synchronize() returns or both
 * kinds have been correlated.  Captures under 384 KiB are copied synchronously. */
TDOA_API int tdoa_load_u8_pinned(tdoa_engine *e, int32_t station, const uint8_t *pinned_iq, size_t nbytes);
/* Same, capture already resident in device memory; not copied, caller keeps it alive.
 * d_iq must be 16-byte aligned (cudaMalloc memory is; an offset into a buffer may not be):
 * the unpack / discriminator kernels fetch the capture in 16-byte words.  A misaligned
 * pointer is rejected with TDOA_E_INVALID. */
TDOA_API int tdoa_load_u8_device(tdoa_engine *e, int32_t station, const uint8_t *d_iq, size_t nbytes);

/* loadIQData parity probe (processor.go:193-201): complex64 samples
 * [first, first+count) of a station's capture, written to host out_c64[2*count]. */
TDOA_API int tdoa_unpack(tdoa_engine *e, int32_t station, int64_t first, int64_t count, float *out_c64);

/* preprocessSignal probe (processor.go:469-499 / ELF 0x49cd40): preprocesses samples
 * [start, start+len) of `kind` of `station` in the engine's mode and returns the
 * normalised complex64 signal, its initial power and the branch taken.  With
 * decimate = D only the first len / D entries of out_c64 are written. */
TDOA_API int tdoa_preprocess(tdoa_engine *e, int32_t station, int32_t kind, int64_t start, int64_t len,
                             float *out_c64, double *power, int32_t *branch);

/* Channel filter (EXTENDED mode, engine-defined; the reference has none): a complex FIR with the caller's taps,
 * per signal kind, applied to a signal's unpacked samples before preprocessSignal.  An RTL-SDR capture is 2 MHz
 * wide and the discriminator follows the strongest carrier in it, so a stronger station in an adjacent channel
 * (or the wanted one tuned off-centre, away from the DC spike) gives the other programme's lags.  A band-pass
 * around the wanted station recovers it, as any FM receiver does.
 *
 * For one signal -- a REF or TGT view or window, after guard_samples, in view order (a REF view filters across
 * the block 1 | block 3 joint, as the box-car does) -- with x[0..n) its unpacked samples (as loadIQData), the
 * kind's taps h[0..T) (f32 re / im, T odd, 1 <= T <= 127) and c = (T - 1) / 2:
 *   for every i in [0, n): acc_r = acc_i = +0; for k = 0 .. T-1 ascending, v = x[i + c - k] (+0 + 0j outside
 *   [0, n)):  acc_r = fmaf(hr[k], vr, acc_r); acc_r = fmaf(-hi[k], vi, acc_r);
 *             acc_i = fmaf(hr[k], vi, acc_i); acc_i = fmaf(hi[k], vr, acc_i);
 *   y[i] = acc.
 * The signal IS y from then on: BINARY preprocessing runs on it exactly as on unpacked samples, its power picks
 * the branch, and tdoa_xcorr_info reports y's power and DC.  Every other stage (DC, box-car, normalisation,
 * decimator, correlators, fits, re-timing, checks) is unchanged.
 * - The taps are the same for every station of a kind: their delay is common to both stations of every pair and
 *   cancels in every lag; window times are unchanged.
 * - A band-pass centred at f0 adds the constant 2 pi f0 / fs to the discriminator output; the strong branch's DC
 *   removal takes it out.
 * - Co-channel interference (another programme on the same frequency) is not helped; that is the station check's
 *   job (tdoa_exclude_stations).
 * It applies to every signal the engine cuts from its captures: tdoa_xcorr*, tdoa_process, every
 * tdoa_process_windows* (including _retimed, which re-times the filtered chain's plane) and tdoa_preprocess; not to
 * tdoa_cross_correlate or tdoa_analyze.  With no channel set every call runs as before.  taps_im may be NULL (real
 * taps); n_taps = 0 clears the kind's channel.  Setting or clearing resets the kind's remembered branches.  A
 * capture still arriving (tdoa_load_u8_pinned) is waited for as a whole before it is filtered.  An n_devices > 1
 * engine sets every device; with tdoa_comm_init each rank sets its own.  Refused (TDOA_E_INVALID): a mode other
 * than EXTENDED, a kind other than 0 or 1, n_taps < 0, even or > 127, a NULL taps_re with n_taps > 0, a NaN,
 * infinite or subnormal tap. */
TDOA_API int tdoa_set_channel(tdoa_engine *e, int32_t kind, const float *taps_re, const float *taps_im, int32_t n_taps);

/* ProcessTDOA pair loops (processor.go:816-850): correlates every station pair i<j
 * (lexicographic, = argv order) of `kind` over n_windows windows
 * [win_start + w*hop, +win_len).  win_len = 0 means the config's chunk (0 = whole
 * signal).  out[w * P + p], P = S(S-1)/2. */
TDOA_API int tdoa_xcorr(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len,
                        int32_t n_windows, int64_t hop, tdoa_peak *out);
/* Same, peaks left in device memory (e.g. an NCCL send buffer); d_out[n_windows*P]. */
TDOA_API int tdoa_xcorr_device(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len,
                               int32_t n_windows, int64_t hop, tdoa_peak *d_out);
/* Ranking-plane probe (BINARY and EXTENDED): tdoa_xcorr, plus the f32 ranking each FFT record's candidates were
 * chosen from.  out[n_windows * P] is bit for bit what tdoa_xcorr returns; ranking[(w * P + p) * M + d], with M =
 * max_lag (BINARY) or 2 (max_lag / D) + 1 (EXTENDED, D = decimate), is the record's approx at lag index d (lag
 * d in BINARY, d - max_lag / D in EXTENDED, correlation lags before the decimator's scaling).  NaN past the
 * record's lag count and on records that had no ranking (BRUTE without the candidate overflow: use_fft = 0, <= 8
 * lags, BINARY's second template; EMPTY); a record redone lag by lag after the overflow keeps its FFT plane.  The
 * planes are copied out only in this call: tdoa_xcorr runs exactly as before.  Refused (TDOA_E_INVALID): SOURCE
 * mode, an engine over several GPUs (n_devices > 1 or tdoa_comm_init), a NULL out or ranking, and what tdoa_xcorr
 * refuses. */
TDOA_API int tdoa_xcorr_ranking(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows,
                                int64_t hop, tdoa_peak *out, float *ranking);

/* ---- bounded lag search (EXTENDED mode; no reference equivalent; engine-defined): tdoa_xcorr with an interval
 * [lag_lo[k], lag_hi[k]] (int32, capture samples: the units of the records) for each record k = w * P + p.  With
 * D = decimate (1 without the decimator) the searched lags are the correlation's own lags k in -max_lag / D ..
 * +max_lag / D with lo <= D k <= hi: one contiguous run.
 *  - lag: the arg-max of |corr| over the run (ties: the lowest lag); corr its value.
 *  - frac: the 3-point parabola when lags k - 1 and k + 1 are both in the run; otherwise TDOA_PEAK_EDGE and frac 0,
 *    so a maximum pinned to the interval's boundary is unusable in the windowed fixes, as a maximum at +-max_lag is.
 *  - margin: the runner-up over the run without the peak (exact on BRUTE records, the f32 ranking's on FFT records).
 *  - flags: every record carries TDOA_PEAK_BOUNDED; a run without any lag gives EMPTY | BOUNDED, lag 0, corr 0.
 *    The candidate cap's lag-by-lag redo keeps the interval.
 * An interval that covers the whole range gives tdoa_xcorr's record bit for bit, apart from TDOA_PEAK_BOUNDED.
 * It is the primitive for a caller with its own prior on the lags (e.g. a known search area).  On a multi-GPU engine
 * the intervals are dealt with the windows.  Refused (TDOA_E_INVALID): a mode other than EXTENDED, a NULL bound
 * array, lo > hi; and what tdoa_xcorr refuses. */
TDOA_API int tdoa_xcorr_bounded(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows,
                                int64_t hop, const int32_t *lag_lo, const int32_t *lag_hi, tdoa_peak *out);

/* Bounded TGT search in the windowed process calls (EXTENDED mode; engine setting; default off).  Once the REF line
 * of pair p = (i, j) is fitted, physics limits where the target's peak can be: for any transmitter |r_j - r_i| <=
 * d_ij, the baseline, and rd = (y_tgt - y_ref(t_w)) / fs * c + geo, so y_tgt lies within d_ij fs / c of
 * y_ref(t_w) - geo fs / c when the REF transmitter is known (has_ref_tx), within 2 d_ij fs / c of y_ref(t_w)
 * otherwise (|geo| <= d_ij too).  A peak outside is noise, another programme or a repeat of periodic content.
 * While on, every tdoa_process_windows* call (plain, _grid, _retimed, _closure, _exclude) runs the REF pair loop, the
 * REF fit (k_window_ref_fit) and k_tgt_bounds on the REF table, then the TGT pair loop as tdoa_xcorr_bounded with
 * these intervals; the fix stage is unchanged and reads that TGT table.  On a multi-GPU engine the ranks meet twice
 * per call (REF, then TGT), as in the re-timed call.  Per (TGT window w, pair p) with a REF fit (a, beta, t_mean,
 * geo; geo = 0 without has_ref_tx), d = the baseline as tdoa_baselines gives it, t_w = the window time of station i,
 * all in f64 rounded to nearest with no fused multiply-add, in this order:
 *   y_ref  = a + beta * (t_w - t_mean)
 *   centre = y_ref - geo / c * fs                          (c = 299792458, fs = sample_rate)
 *   half   = (has_ref_tx ? d : 2 * d) / c * fs + guard_samples
 *   lo = ceil(centre - half), hi = floor(centre + half), each clamped to [INT32_MIN, INT32_MAX].
 * A pair without a REF fit keeps the unbounded search (no TDOA_PEAK_BOUNDED); it is used in no window anyway.
 * Not affected: tdoa_window_fixes* (their tables are given), tdoa_xcorr* and tdoa_process.  on = 0 launches exactly
 * what the calls launch without the setting.  An n_devices > 1 engine sets every device; with tdoa_comm_init each
 * rank sets its own.  Refused (TDOA_E_INVALID): a mode other than EXTENDED, on not 0 or 1, guard_samples NaN,
 * infinite or negative. */
TDOA_API int tdoa_set_tgt_bounds(tdoa_engine *e, int32_t on, double guard_samples);

/* Both pair loops of ProcessTDOA over windows in ONE call (processor.go:816-830 REF, then :836-850 TGT):
 * ref_out[n_ref_windows * P], tgt_out[n_tgt_windows * P] as tdoa_xcorr(TDOA_KIND_REF, ...) followed by
 * tdoa_xcorr(TDOA_KIND_TGT, ...) would fill them (same win_start / win_len / hop for both kinds; either
 * count may be 0).  On one GPU it is exactly those two calls.  On a multi-GPU engine (n_devices > 1 or
 * tdoa_comm_init) the windows of BOTH kinds are dealt over the ranks as one list and correlated before the
 * first gather, so the ranks meet once per call instead of once per kind -- with 66 + 33 windows on 8 GPUs
 * the busiest rank works 13 window times instead of 9 + 5. */
TDOA_API int tdoa_xcorr_windows(tdoa_engine *e, int64_t win_start, int64_t win_len, int32_t n_ref_windows,
                                int32_t n_tgt_windows, int64_t hop, tdoa_peak *ref_out, tdoa_peak *tgt_out);

/* ---- more than one GPU, one process per GPU (torchrun, MPI, ...).  Rank 0 asks for an id
 * (ncclGetUniqueId), the launcher hands its 128 bytes to every rank, every rank joins with its own
 * engine (ncclCommInitRank on the engine's device).  From then on tdoa_xcorr / tdoa_xcorr_device
 * over >= 2 windows are COLLECTIVE: every rank makes the same call; rank r correlates the windows w
 * with (cursor + w) % world == r -- all pairs of a window on one GPU, so no data-path exchange --
 * its peak kernel writes the records straight into the gather buffer, one ncclAllGather
 * completes the table on every rank, and every rank returns all n_windows * P records.  cursor
 * starts at 0 and advances by n_windows after every sharded call.  Each rank loads the captures it
 * correlates (all of them, or -- tdoa_load_u8_pinned -- only the bytes its windows need).
 * tdoa_xcorr_info afterwards describes the first window this rank processed. */
TDOA_API int tdoa_comm_unique_id(uint8_t id[128]);
TDOA_API int tdoa_comm_init(tdoa_engine *e, const uint8_t id[128], int32_t rank, int32_t world);
TDOA_API int tdoa_comm_rank(tdoa_engine *e, int32_t *rank, int32_t *world);
/* The dealing rule itself (host arithmetic, no GPU): rank's first window and how many it gets. */
TDOA_API int tdoa_shard_windows(int32_t n_windows, int32_t rank, int32_t world, int32_t cursor, int32_t *first,
                                int32_t *count);

/* ProcessTDOA from the pair loops to the fix as ONE call (processor.go:816-929 on window 0
 * with the config's chunk): the REF pair loop, the TGT pair loop, dt = delay / fs, the
 * mode's time differences (SOURCE: target only, :853; binary modes: target - reference,
 * pair by pair), range differences (:899-903) and solveTDOA -- all queued on the device
 * without an intermediate host synchronisation.  ref_out / tgt_out [P]; time_diffs,
 * range_diffs [P] (may be NULL); fix_llh[3]; *fix_status 0 or TDOA_E_SINGULAR.
 * The fix is processor.go's solveTDOA (:932-1020) on rd[0], rd[1] in every mode; the shipped
 * binary's own revision of the solver (filter, exactly-two rule) is tdoa_solve_binary on the
 * range_diffs returned here.  tdoa_xcorr_info() afterwards reports both kinds. */
TDOA_API int tdoa_process(tdoa_engine *e, const double *stations_llh, tdoa_peak *ref_out, tdoa_peak *tgt_out,
                          double *time_diffs, double *range_diffs, double *fix_llh, int32_t *fix_status,
                          int32_t *fix_iters);

/* ---- windowed ProcessTDOA: one fix per TGT window (no reference equivalent; engine-defined).
 * BINARY and EXTENDED modes (SOURCE has no REF correction, processor.go:853).  Window arguments as
 * tdoa_xcorr_windows; P = S(S-1)/2 pairs i<j.
 *  - Window time: the capture-sample index of the window's centre, start + (len - 1) / 2 mapped into the
 *    capture of the pair's FIRST station i (b = nsamp_i / 3, g = guard_samples): REF sample k is at k when
 *    k < b, else at 2b + g + (k - b); TGT sample k at b + g + k.  A REF window with samples in both block 1
 *    and block 3 has no single time and takes no part in the fit.
 *  - A record is usable unless it is EMPTY or EDGE, or margin < min_margin (min_margin = 0: no margin
 *    test).  Its value y = lag + frac, in capture samples.
 *  - REF fit per pair: least-squares line y = a + beta (t - t_mean) through the usable REF windows, sums in
 *    f64 in window order; one window: beta = 0; none: the pair is used in no TGT window.  ref_max_residual
 *    > 0: one refit without the windows whose |residual| from the first line exceeds it (none left: no fit).
 *    ref_fit[p] = {REF lag at the centre of station i's block 2 (b + (b - 1) / 2; 0 without a fit), beta
 *    (samples per sample = ppm * 1e-6), windows used}.
 *  - Range difference of (TGT window w, pair p): (y_tgt / fs - (a + beta (t_w - t_mean)) / fs) * c, plus
 *    |x_ref - s_j| - |x_ref - s_i| when has_ref_tx (the REF transmitter is not equidistant from i and j);
 *    NaN and pair_used = 0 unless the TGT record is usable and the pair has a fit.  With whole blocks as
 *    windows (win_len = hop = b, guard 0), no drift and no REF position this is tdoa_process's range
 *    difference with chunk_samples = 0: exactly in BINARY, within 1e-3 samples in EXTENDED (the whole-signal
 *    frac and the mean of two block fracs need not agree).
 *  - Fix per TGT window: tdoa_solve_ls over the used pairs only (dims 2 or 3; start init_llh, or the mean
 *    of the stations); rms over the used pairs.  fix_status 0 ok, 1 degenerate, 2 too few measurements
 *    (fewer than dims used pairs, or used pairs touching fewer than dims + 1 stations; no iteration, the
 *    start point is returned). */
typedef struct {
    int32_t dims;              /* 2 or 3 (3 needs >= 4 stations)                                  */
    float min_margin;          /* records below this margin are not used; 0 = off                 */
    double ref_max_residual;   /* samples; > 0: one refit without REF outliers; 0 = off           */
    int32_t has_ref_tx;        /* 1: ref_tx_llh is the REF transmitter (geometric term)           */
    int32_t has_init;          /* 1: init_llh is the least-squares start of every window          */
    double ref_tx_llh[3];
    double init_llh[3];
} tdoa_window_opts;

/* Captures -> REF and TGT tables -> range differences -> one fix per TGT window.  The tables are those
 * tdoa_xcorr_windows gives for the same arguments, bit for bit (on a multi-GPU engine dealt and gathered
 * the same way); the fix stage reads them where the pair loops left them in device memory.  On one GPU the
 * pair loops make their checks as tdoa_xcorr_windows does; on a multi-GPU engine the call is collective and
 * every rank runs the fix stage on its own gathered tables (no second collective), so every rank returns
 * everything.  ref_out[n_ref * P], tgt_out[n_tgt * P], ref_fit[P][3], range_diffs[n_tgt][P],
 * pair_used[n_tgt][P], fix_rms[n_tgt], fix_iters[n_tgt] may be NULL; fix_llh[n_tgt][3], fix_status[n_tgt]
 * may not.  Refused (TDOA_E_INVALID): SOURCE mode, S < 3 or S > 64, dims not 2 or 3, dims 3 with S < 4,
 * n_ref_windows < 1, n_tgt_windows < 1, bad window arguments. */
TDOA_API int tdoa_process_windows(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                  int64_t win_start, int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows,
                                  int64_t hop, tdoa_peak *ref_out, tdoa_peak *tgt_out, double *ref_fit,
                                  double *range_diffs, uint8_t *pair_used, double *fix_llh, double *fix_rms,
                                  int32_t *fix_status, int32_t *fix_iters);
/* The same fix stage from host tables (e.g. kept from earlier tdoa_xcorr_windows calls); the window times
 * come from the captures the engine holds.  Same arguments and refusals; ref_in / tgt_in may not be NULL. */
TDOA_API int tdoa_window_fixes(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                               int64_t win_start, int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows,
                               int64_t hop, const tdoa_peak *ref_in, const tdoa_peak *tgt_in, double *ref_fit,
                               double *range_diffs, uint8_t *pair_used, double *fix_llh, double *fix_rms,
                               int32_t *fix_status, int32_t *fix_iters);
/* ---- re-timed target correlation (no reference equivalent; engine-defined): tdoa_process_windows with every
 * station's TGT planes re-timed by that station's clock rate, so that a TGT window may be as long as block 2.
 * 1 ppm of relative rate moves the lag 2 samples per second; tdoa_process_windows corrects the OFFSET of each TGT
 * lag but not the drift inside a window, which smears a long window's peak.  Clock error belongs to a station:
 * the REF fit's slopes satisfy beta_ij = c_j - c_i.
 *  - Station rates: the pairs whose REF fit used at least 2 windows (ref_fit[p][2] >= 2) enter the fit.  c[S]
 *    minimises the sum over those pairs of (c_j - c_i - beta_ij)^2, and sums to zero within each connected
 *    component of those pairs.  Computed in f64, every operation rounded to nearest (no fused multiply-add), in
 *    this order: A = the normal matrix of the pairs plus, for each component, 1 at every (i, j) of its stations;
 *    b[i] -= beta and b[j] += beta pair by pair in pair order; A = L L^T by Cholesky, right-looking (L_kk =
 *    sqrt(A_kk), L_ik = A_ik / L_kk, then A_ij -= L_ik L_jk for k < j <= i, k ascending); L y = b and L^T c = y
 *    column by column (y_k = b_k / L_kk, then b_i -= L_ik y_k for i > k; c_k = y_k / L_kk, then y_i -= L_ki c_k
 *    for i < k, k descending).  A station with no fitted pair gets rate 0 (it re-times nothing) and NaN in
 *    clock_rate; its pairs are used in no TGT window anyway.
 *  - Re-timing: x[0..len) is station k's preprocessed plane of one TGT window, the plane the correlator reads, in
 *    that plane's own samples (n / decimate with the decimator).  Its re-timed plane is x~[n] = x[n + delta(n)]
 *    where 0 <= n + delta(n) < len, and 0 elsewhere; delta(n) = floor(c_k * (n - n_c) + 0.5), n_c = (len - 1) / 2,
 *    in f64 rounded to nearest with no fused multiply-add.  Length, statistics and normalisation scale stay
 *    those of x.  delta(n_c) = 0, so a record's lag + frac is the lag at the window's centre: the time the range
 *    differences already take.
 *  - The call: the REF pair loop over the REF windows (records as tdoa_xcorr gives them), the REF fit, the
 *    station rates, the TGT pair loop over the TGT windows on re-timed planes, then the range differences and
 *    fixes of tdoa_process_windows.  REF and TGT windows have separate geometry (e.g. short REF windows and one
 *    TGT window of the whole block); tgt_win_len = 0 follows tdoa_xcorr's rule.  Outputs are those of
 *    tdoa_process_windows plus clock_rate[S] (samples per sample), which may be NULL.  With rates so small that
 *    |c| (len - 1) / 2 < 0.5 for every station, delta is 0 everywhere and the results are tdoa_process_windows'.
 *  - On a multi-GPU engine the call is collective.  The REF windows are dealt and gathered as tdoa_xcorr deals
 *    them, every rank fits the rates from its gathered table (the fit is deterministic: the same bits on every
 *    rank), then the TGT windows are dealt and gathered the same way.  The TGT pass depends on the fit, so the
 *    ranks meet twice per call instead of once.
 * Refused (TDOA_E_INVALID): what tdoa_process_windows refuses, for either geometry. */
TDOA_API int tdoa_process_windows_retimed(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                          int64_t ref_win_start, int64_t ref_win_len, int32_t n_ref_windows,
                                          int64_t ref_hop, int64_t tgt_win_start, int64_t tgt_win_len,
                                          int32_t n_tgt_windows, int64_t tgt_hop, tdoa_peak *ref_out, tdoa_peak *tgt_out,
                                          double *ref_fit, double *range_diffs, uint8_t *pair_used, double *fix_llh,
                                          double *fix_rms, int32_t *fix_status, int32_t *fix_iters, double *clock_rate);

/* Grid-seeded windowed fixes: as tdoa_process_windows / tdoa_window_fixes, with each TGT window's
 * least-squares fix started from the arg-min of tdoa_grid_masked over grid_desc (7 doubles, as
 * tdoa_grid) with that window's range differences and used pairs -- computed on the device between the
 * range differences and the fix, in the same stream and without another host synchronisation.  A window
 * the least-squares step refuses (status 2) is not searched: seed_index -1, seed_cost NaN, and it keeps
 * the start it has without a grid.  Every other window starts at its arg-min cell (lat, lon, the grid's
 * elevation); dims 3 solves the height from there.  The ranked arg-min is checked after the call's one
 * synchronisation; a candidate table that overflowed, or a searched window without a survivor, reruns the
 * grid on every cell and the fixes before anything is returned, so the results are those of evaluating
 * every cell.  seed_llh[n_tgt][3], seed_cost[n_tgt], seed_index[n_tgt] may be NULL.  Refused
 * (TDOA_E_INVALID): what the base calls refuse, a NULL grid_desc, more than 16 stations, an empty or too
 * large grid.  ms_fix covers the grid. */
TDOA_API int tdoa_process_windows_grid(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                       int64_t win_start, int64_t win_len, int32_t n_ref_windows,
                                       int32_t n_tgt_windows, int64_t hop, const double *grid_desc, tdoa_peak *ref_out,
                                       tdoa_peak *tgt_out, double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                       double *fix_llh, double *fix_rms, int32_t *fix_status, int32_t *fix_iters,
                                       double *seed_llh, double *seed_cost, int64_t *seed_index);
TDOA_API int tdoa_window_fixes_grid(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                    int64_t win_start, int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows,
                                    int64_t hop, const double *grid_desc, const tdoa_peak *ref_in,
                                    const tdoa_peak *tgt_in, double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                    double *fix_llh, double *fix_rms, int32_t *fix_status, int32_t *fix_iters,
                                    double *seed_llh, double *seed_cost, int64_t *seed_index);

/* ---- closure-checked windowed fixes (no reference equivalent; engine-defined).  A range difference is a
 * difference of two station ranges, rd_ij = r_j - r_i, so the P pairs of a window hold only S - 1 independent
 * numbers and every cycle of pairs closes (rd_ij + rd_jk - rd_ik = 0; the REF correction keeps this, clock offsets
 * belong to stations).  One wrong TGT lag (a noise peak, an interferer, one of several equal peaks of periodic
 * content) enters the fix at full weight; the check drops the pairs the rest of the window contradicts.
 * Per set (one TGT window): rd[P] in metres, the usable mask u[P] in {0, 1} (pair_used of tdoa_process_windows),
 * dims, max_residual (metres, > 0, may be +inf) and max_drop (>= 0, 0 = no limit).  m = u, 0 drops; then repeat:
 *  1. Station values: on the graph of the pairs with m = 1, components labelled with their smallest station
 *     index, tau[S] (metres) minimises sum (tau_j - tau_i - rd_ij)^2 over those pairs and sums to zero in each
 *     component; a station with no pair is its own component and gets tau = 0.  Solved exactly as the station
 *     rates of tdoa_process_windows_retimed, with rd in place of beta (b[i] -= rd, b[j] += rd in pair order; the
 *     same Cholesky and solves, every f64 operation rounded to nearest, no contraction).
 *  2. Residuals: e_p = rd_p - (tau_j - tau_i) (that rounding order) for every pair with u = 1, dropped ones
 *     included; NaN for the others.
 *  3. Stop if the redundancy of m (used pairs - stations they touch + components among those stations) is below
 *     2 (a single cycle shows an inconsistency but cannot say which pair caused it), or max_drop > 0 and the
 *     drops have reached max_drop, or q = the m-pair with the largest |e_p| (ties: the lowest p) has
 *     |e_q| <= max_residual.
 *  4. Tentative drop: m' = m without q; then, repeatedly, a station that lost a pair in this step and has exactly
 *     one m'-pair left loses that pair too (a station seen through one pair cannot be checked).
 *  5. If m' fails the least-squares step's status-2 rule (fewer than dims pairs, or pairs touching fewer than
 *     dims + 1 stations), stop and keep m; else m = m', add the pairs removed to the drops and go to 1.
 * Outputs: the final m (which the grid seed and the fix read in place of u), e from the last solve (the one on
 * the final m) and the number of drops.  When nothing exceeds max_residual in the first pass, m = u and every
 * output of the fix stage is, bit for bit, that of the call without the check: max_residual = INFINITY turns it
 * off.  The check sees errors of single pairs only: an error common to all of one station's pairs is a station
 * value, which tau absorbs.  A station that hears another programme, or only its own noise, in block 2 gives such
 * an error (the peak of pair (i, s) moves with station i's own delay), so the check does not find that station.
 * In BINARY mode lags are integers, so consistent pairs can already disagree by about 1 sample (150 m at
 * 2 Msps); set max_residual above that. */
typedef struct {
    double max_residual;   /* metres; > 0, may be INFINITY                                     */
    int32_t max_drop;      /* pairs per set; 0 = no limit                                      */
    int32_t reserved;
} tdoa_closure_opts;

/* The check alone over host sets: range_diffs[set * rd_stride + p], used[...] in {0, 1} (an unused slot is never
 * read); out_used[...] in {0, 1, 2} (2: usable but dropped), out_resid[...] (may be NULL), out_dropped[n_sets]
 * (may be NULL).  Only the first P slots of each set are read or written.  Refused (TDOA_E_INVALID): a NULL
 * range_diffs, used, out_used or c, S outside 3..64, dims not 2 or 3, n_sets < 0, rd_stride < P, max_residual
 * NaN or <= 0, max_drop < 0. */
TDOA_API int tdoa_closure(tdoa_engine *e, int32_t n_stations, const double *range_diffs, const uint8_t *used,
                          int32_t n_sets, int32_t rd_stride, int32_t dims, const tdoa_closure_opts *c,
                          uint8_t *out_used, double *out_resid, int32_t *out_dropped);
/* One process call for every combination: REF and TGT window geometry as tdoa_process_windows_retimed; retimed 1
 * re-times the TGT planes as that call does, 0 correlates them as tdoa_process_windows does (with two different
 * geometries the tables are those tdoa_xcorr gives for each kind's geometry); grid_desc (may be NULL) seeds the
 * fixes as tdoa_process_windows_grid.  The check runs on the device between the range differences and the grid
 * seed / fix, in the same stream, with no other host synchronisation; on a multi-GPU engine every rank runs it on
 * its own gathered tables and returns the same bits.  pair_used[n_tgt][P]: 0 not usable, 1 used by the fix, 2
 * usable but dropped by the check.  closure_resid[n_tgt][P], n_dropped[n_tgt], clock_rate[S] (retimed 1 only),
 * seed_llh, seed_cost and seed_index may be NULL.  ms_fix covers the check.  Refused (TDOA_E_INVALID): what the
 * base calls refuse, a NULL c, max_residual NaN or <= 0, max_drop < 0, retimed not 0 or 1. */
TDOA_API int tdoa_process_windows_closure(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                          const tdoa_closure_opts *c, int64_t ref_win_start, int64_t ref_win_len,
                                          int32_t n_ref_windows, int64_t ref_hop, int64_t tgt_win_start,
                                          int64_t tgt_win_len, int32_t n_tgt_windows, int64_t tgt_hop, int32_t retimed,
                                          const double *grid_desc, tdoa_peak *ref_out, tdoa_peak *tgt_out,
                                          double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                          double *closure_resid, int32_t *n_dropped, double *fix_llh, double *fix_rms,
                                          int32_t *fix_status, int32_t *fix_iters, double *clock_rate,
                                          double *seed_llh, double *seed_cost, int64_t *seed_index);
/* The same on host tables, as tdoa_window_fixes_grid (grid_desc may be NULL). */
TDOA_API int tdoa_window_fixes_closure(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                       const tdoa_closure_opts *c, int64_t win_start, int64_t win_len,
                                       int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop,
                                       const double *grid_desc, const tdoa_peak *ref_in, const tdoa_peak *tgt_in,
                                       double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                       double *closure_resid, int32_t *n_dropped, double *fix_llh, double *fix_rms,
                                       int32_t *fix_status, int32_t *fix_iters, double *seed_llh, double *seed_cost,
                                       int64_t *seed_index);

/* ---- station-checked windowed fixes (no reference equivalent; engine-defined).  An error common to all of one
 * station's pairs (a collector tuned to another programme, overloaded by one, or with its antenna down) is a
 * station value: the closure check cannot see it.  The range differences must also agree with ONE position: with
 * S stations the used pairs carry S - 1 independent numbers and the position takes dims of them, so S - 1 - dims
 * are left to check with.  As a GNSS receiver's fault detection and exclusion does, the check detects the fault
 * from the fix's rms, identifies the station by solving again without each station in turn, and keeps the solve
 * that fits.  Per set (one TGT window): rd[P] in metres; the fix mask m[P] in {0, 1} (the used mask, or the
 * closure check's output when both checks run); the start x0 (init_llh, the station mean, or with a grid the grid
 * arg-min over m); dims; max_rms (metres, > 0, may be +inf) and max_exclude (>= 0, 0 = no limit).  LS(mask, x) is
 * exactly what tdoa_solve_ls's least-squares step returns for that mask from start x (position, rms, status,
 * iterations).
 *  1. F = LS(m, x0) (the fix without the check); E = {}.
 *  2. Stop if F.status != 0, or F.rms <= max_rms, or max_exclude > 0 and |E| = max_exclude.
 *  3. Station k is a candidate if it touches an m-pair, m_k (m without every pair that touches k) passes the
 *     status-2 rule, and m_k has redundancy >= 1: (stations m_k touches) - (components of m_k's pair graph) - dims.
 *     (Without that rule an exclusion that leaves an exactly determined fix would win with rms 0; one exclusion
 *     needs dims + 3 stations: 5 for dims 2, 6 for dims 3.)  No candidate: stop.
 *  4. F_k = LS(m_k, x0) for every candidate; a candidate with F_k.status != 0 is not eligible.
 *  5. k* = the eligible candidate with the least F_k.rms (ties: the lowest k).  Stop if there is none or
 *     F_k*.rms >= F.rms; else m = m_k*, E = E + {k*}, F = F_k*, go to 2.
 * With a grid and E not empty, the window is seeded again from the grid arg-min over the final m (a wrong station
 * can have pulled the first arg-min into a trap) and F = LS(m, that seed); the seed outputs report that seed.
 * Outputs per set: the final m; station_round[S] (0: not excluded, else the round, from 1, that excluded it);
 * station_rms[S] (F_k.rms of the FIRST round for every candidate, NaN for the others or when no round ran: how far
 * the bad station stands apart); the number excluded; F.  When the first F.rms <= max_rms every output of the fix
 * stage is, bit for bit, that of the call without the check: max_rms = INFINITY turns it off.  Decisions rest on
 * the unweighted rms, as the fix does.  The check does not see an error that a shift of the position can absorb
 * (near-collinear stations, a station whose error moves the fix along its own gradient).  In BINARY mode integer
 * lags already give rms of order 100 m; set max_rms above that. */
typedef struct {
    double max_rms;        /* metres; > 0, may be INFINITY                                     */
    int32_t max_exclude;   /* stations per set; 0 = no limit                                   */
    int32_t reserved;
} tdoa_exclusion_opts;

/* The check alone over host sets (no grid): range_diffs[set * rd_stride + p], used[...] in {0, 1} (an unused slot is
 * never read), init_llh[n_sets][3] (NULL: the station mean).  out_used[...] in {0, 1, 3} (3: used, excluded with
 * its station); station_round[n_sets][S], station_rms[n_sets][S], n_excluded[n_sets], out_llh[n_sets][3],
 * out_rms[n_sets], status[n_sets] and iters[n_sets] (F, as tdoa_solve_ls gives it).  Only the first P slots of each
 * set are read or written.  Every output but out_used, out_llh and status may be NULL.  Refused (TDOA_E_INVALID): a
 * NULL stations_llh, range_diffs, used, out_used, out_llh, status or x, S outside 3..64, dims not 2 or 3,
 * n_sets < 0, rd_stride < P, max_rms NaN or <= 0, max_exclude < 0. */
TDOA_API int tdoa_exclude_stations(tdoa_engine *e, const double *stations_llh, int32_t n_stations,
                                   const double *range_diffs, const uint8_t *used, int32_t n_sets, int32_t rd_stride,
                                   const double *init_llh, int32_t dims, const tdoa_exclusion_opts *x,
                                   uint8_t *out_used, uint8_t *station_round, double *station_rms,
                                   int32_t *n_excluded, double *out_llh, double *out_rms, int32_t *status,
                                   int32_t *iters);
/* tdoa_process_windows_closure with the station check after the first fix: c may be NULL (no closure check); with
 * both, the closure check runs first, so pair outliers are dropped before a station outlier is looked for.  The
 * check runs on the device after the first grid seed and fix, on the same stream, with no other host
 * synchronisation; on a multi-GPU engine every rank runs it on its own gathered tables.  pair_used[n_tgt][P]: 0
 * not usable, 1 used by the fix, 2 dropped by the closure check, 3 excluded with its station.  station_round,
 * station_rms and n_excluded may be NULL; ms_fix covers the check.  Refused (TDOA_E_INVALID): what
 * tdoa_process_windows_closure refuses (but c may be NULL), a NULL x, max_rms NaN or <= 0, max_exclude < 0. */
TDOA_API int tdoa_process_windows_exclude(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                          const tdoa_closure_opts *c, const tdoa_exclusion_opts *x,
                                          int64_t ref_win_start, int64_t ref_win_len, int32_t n_ref_windows,
                                          int64_t ref_hop, int64_t tgt_win_start, int64_t tgt_win_len,
                                          int32_t n_tgt_windows, int64_t tgt_hop, int32_t retimed,
                                          const double *grid_desc, tdoa_peak *ref_out, tdoa_peak *tgt_out,
                                          double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                          double *closure_resid, int32_t *n_dropped, uint8_t *station_round,
                                          double *station_rms, int32_t *n_excluded, double *fix_llh, double *fix_rms,
                                          int32_t *fix_status, int32_t *fix_iters, double *clock_rate,
                                          double *seed_llh, double *seed_cost, int64_t *seed_index);
/* The same on host tables, as tdoa_window_fixes_closure (c and grid_desc may be NULL). */
TDOA_API int tdoa_window_fixes_exclude(tdoa_engine *e, const double *stations_llh, const tdoa_window_opts *o,
                                       const tdoa_closure_opts *c, const tdoa_exclusion_opts *x, int64_t win_start,
                                       int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows, int64_t hop,
                                       const double *grid_desc, const tdoa_peak *ref_in, const tdoa_peak *tgt_in,
                                       double *ref_fit, double *range_diffs, uint8_t *pair_used,
                                       double *closure_resid, int32_t *n_dropped, uint8_t *station_round,
                                       double *station_rms, int32_t *n_excluded, double *fix_llh, double *fix_rms,
                                       int32_t *fix_status, int32_t *fix_iters, double *seed_llh, double *seed_cost,
                                       int64_t *seed_index);

/* crossCorrelate seam (processor.go:619-643): two host complex64 slices
 * (interleaved re,im), returns (delay, correlation).  Empty input -> (0, 0.0). */
TDOA_API int tdoa_cross_correlate(tdoa_engine *e, const float *sig1_c64, int64_t n1,
                                  const float *sig2_c64, int64_t n2, tdoa_peak *out);

/* latLonToECEF / calculateBaseline (processor.go:125-163): baselines[p] in metres
 * for pairs i<j of stations_llh[S][3] (lat deg, lon deg, elev m). */
TDOA_API int tdoa_baselines(tdoa_engine *e, const double *stations_llh, int32_t n_stations, double *baselines);

/* solveTDOA (processor.go:932-1020) batched: n_sets range-difference sets,
 * range_diffs[set * rd_stride + p].  out_llh[set][3]; status[set] = 0 ok,
 * TDOA_E_SINGULAR singular Jacobian; iters[set] (may be NULL). */
TDOA_API int tdoa_solve(tdoa_engine *e, const double *stations_llh, int32_t n_stations,
                        const double *range_diffs, int32_t n_sets, int32_t rd_stride,
                        double *out_llh, int32_t *status, int32_t *iters);

/* solveTDOA of the SHIPPED BINARY (ELF 0x4a0360; a later revision than processor.go:932-1020,
 * restated from its disassembly and pinned by the iteration traces it prints): the range
 * differences with |rd| <= 20400 m are kept in order; the binary solves only when exactly
 * two remain (res1 = (r2 - r1) - valid[0], res2 = (r3 - r1) - valid[1]; Newton step times 0.7,
 * steps over 1000 m scaled to 1000 m first; single-equation fall-back when |det| < 1e-12;
 * converged when both residuals < 1 m; at most 10 iterations; Z frozen).
 * *status: 0 a fix in out_llh[3]; 1 fewer than two valid ("insufficient valid measurements: only
 * %d of %d range differences are reliable"); 2 more than two valid ("no valid range difference
 * measurements remain"); 3 "singular Jacobian matrix at iteration %d (det=%.2e)".
 * n_valid, n_iter (iterations whose trace line the binary prints), converged, and
 * trace[10][5] = {det, res1, res2, step length, code: 0 plain step, 1 step limited, 2 / 3
 * single equation 1 / 2} may each be NULL. */
TDOA_API int tdoa_solve_binary(tdoa_engine *e, const double *stations_llh, int32_t n_stations,
                               const double *range_diffs, int32_t n_rd, double *out_llh, int32_t *status,
                               int32_t *n_valid, int32_t *n_iter, int32_t *converged, double *trace);

/* Dense lat-lon grid multilateration (no reference equivalent): for each set the
 * cell minimising sum_{i<j} ((r_j - r_i) - rd_ij)^2, the terms added pair by pair in
 * that order; ties go to the lowest linear index lat_index * nlon + lon_index.
 * grid_desc = {lat0, lon0, dlat, dlon, nlat, nlon, elev}.
 * The cells are RANKED by an expanded form of the cost (16 multiply-adds per cell and
 * set) whose rounding error is bounded; only cells within that bound of the minimum are
 * evaluated by the sum above, and the arg-min is taken over those values -- index and
 * cost are what evaluating every cell gives, bit for bit (use_fft = 0 does evaluate
 * every cell; a set holding a NaN, or a plateau of more than 64 ties per set, falls
 * back to that).  range_diffs is read on the host as well (one pass, n_sets * pairs). */
TDOA_API int tdoa_grid(tdoa_engine *e, const double *stations_llh, int32_t n_stations,
                       const double *grid_desc, const double *range_diffs, int32_t n_sets,
                       int32_t rd_stride, double *out_llh, double *out_cost, int64_t *out_index);
/* The same arg-min over a subset of the pairs of each set (no reference equivalent): the
 * cost is the sum above over the pairs with used[set * rd_stride + p] != 0 only, in the
 * same order; an unused slot is never read (NaN there is fine).  A set with no used pair
 * has no arg-min: out_index -1, out_cost NaN, out_llh NaN.  used == NULL is tdoa_grid
 * exactly.  Ranked as tdoa_grid (the bracket of the expanded cost loses the unused pairs'
 * terms), with the same fall-back to evaluating every cell; same refusals as tdoa_grid. */
TDOA_API int tdoa_grid_masked(tdoa_engine *e, const double *stations_llh, int32_t n_stations,
                              const double *grid_desc, const double *range_diffs, const uint8_t *used,
                              int32_t n_sets, int32_t rd_stride, double *out_llh, double *out_cost,
                              int64_t *out_index);

/* Least-squares fix over ALL S(S-1)/2 range differences (SURVEY.md 8f rank 4; no reference
 * equivalent -- solveTDOA uses two of three measurements, freezes Z and stops after ten
 * half steps, processor.go:932-1020).  Levenberg-Marquardt in the local east/north/up
 * frame; dims = 2 keeps the start elevation (what 3 stations support), dims = 3 solves
 * it too (>= 4 stations).  init_llh[set][3] = start points (e.g. the tdoa_grid arg-min),
 * NULL: mean of the station coordinates.  out_rms[set] = sqrt(sum f^2 / P) in metres
 * (may be NULL); status[set] = 0 ok, 1 degenerate geometry. */
TDOA_API int tdoa_solve_ls(tdoa_engine *e, const double *stations_llh, int32_t n_stations,
                           const double *range_diffs, int32_t n_sets, int32_t rd_stride,
                           const double *init_llh, int32_t dims, double *out_llh, double *out_rms,
                           int32_t *status, int32_t *iters);

/* Per-capture signal quality (fast_analyzer.go:15-24 FastAnalysis, analyzer.go:18-42
 * SignalAnalysis): the numbers the reference's analyzers print and base their gain
 * recommendations on.  fast != 0 follows fast_analyzer.go (first 32768 samples of each
 * block, 8192-point Hanning spectrum, top 10 % vs bottom 40 %); fast == 0 follows
 * analyzer.go (whole blocks, dead-zone scan, 16384-point DC-corrected Blackman-Harris
 * spectrum, top 10 % vs lowest 50 %).  ref = blocks 1 + 3, tgt = block 2 of `station`. */
typedef struct {
    int64_t total_samples;
    double i_avg, q_avg, i_std, q_std;
    int32_t i_min, i_max, q_min, q_max;
    double snr_db, power_db;
    double dc_offset, iq_imbalance;            /* analyzer.go only */
    int32_t has_clipping, has_overload;
    int32_t has_dead_zones, has_noise;         /* analyzer.go only */
} tdoa_signal_quality;
TDOA_API int tdoa_analyze(tdoa_engine *e, int32_t station, int32_t fast, tdoa_signal_quality *ref,
                          tdoa_signal_quality *tgt);

/* What the reference prints while it works on a pair (shipped binary: "Initial signal
 * power", "Removed DC bias", "Normalized signal power", "Time domain correlation ... at
 * delay" before the sanity re-search; processor.go:474-497 prints the same quantities).
 * Values of window 0 of the last tdoa_xcorr(kind) call; signals in station order,
 * first_corr in pair order. */
typedef struct {
    double power0;        /* calculateSignalPower of the raw signal (processor.go:322)   */
    double dc_re, dc_im;  /* removeDCBias mean (processor.go:309)                         */
    double power1;        /* power entering normalizeSignal (processor.go:336)            */
    int32_t branch;       /* 0 strong FM / standard, 1 moderate (envelope), 2 weak        */
    int32_t reserved;
    int64_t n;            /* samples of the signal                                        */
} tdoa_signal_info;
TDOA_API int tdoa_xcorr_info(tdoa_engine *e, int32_t kind, tdoa_signal_info *signals, double *first_corr);

/* Introspection for the benchmark: kernels launched and device time of the last
 * tdoa_xcorr call, per stage (CUDA events on the engine's stream). */
typedef struct {
    int64_t launches_total;   /* kernels launched by this engine since creation   */
    int64_t launches_last;    /* ... by the last xcorr / cross_correlate call     */
    float ms_preprocess;      /* stats + demod + box-car of the last call         */
    float ms_fft;             /* segmented FFT cross-spectrum + inverse           */
    float ms_exact;           /* exact time-domain re-evaluation + peak select    */
    float ms_total;
    int64_t fft_launches;     /* launches of the segmented FFT kernel, last call  */
    float ms_fft_seg;         /* device time of those launches                    */
    int64_t fft_pair_samples; /* template samples they covered                    */
    int64_t brute_pairs;      /* pair-windows that fell back to every-lag search  */
    /* per-kernel device time of the last call (CUDA events around each launch) and the
     * units each kernel covered -- what the benchmark's per-kernel roofline is made of */
    float ms_demod;           /* fused unpack + power + FM discriminator launches */
    float ms_boxcar;          /* small box-car (DC subtract + low-pass + power)   */
    float ms_cand;            /* exact re-evaluation of the candidate lags        */
    float ms_fix;             /* fix stage of the last tdoa_process_windows / tdoa_window_fixes
                                 (REF fit, range differences, grid seed of the _grid
                                 calls, least-squares fixes)                        */
    int64_t demod_launches, demod_samples;
    int64_t boxcar_launches, boxcar_samples;
    int64_t cand_launches, cand_pair_samples;
} tdoa_stats;
TDOA_API int tdoa_get_stats(tdoa_engine *e, tdoa_stats *out);

/* Device self-tests of arithmetic shortcuts the kernels rely on.  which = 0: the
 * box-car's constant-divisor division equals a correctly rounded f32 divide for every
 * float input (exhaustive, ~10 ms); *mismatches = 0 means proven.  which = 1: the
 * production FM discriminator (fast arctangent + full-accuracy fall-back where the f32
 * rounding is not decided) against the reference statement of it over all 2^32
 * (previous, current) byte quads; tdoa_last_error then carries the counts and the
 * differing quads.  which = 2: *mismatches = how many of the 2^32 quads take the
 * fall-back.  which = 3: as 1 for the full-accuracy arctangent on every sample
 * (fast_demod = 2). */
TDOA_API int tdoa_selftest(tdoa_engine *e, int32_t which, int64_t *mismatches);

/* Raw CUDA stream of the engine (cudaStream_t as void*), for callers that time or
 * chain work on it. */
TDOA_API void *tdoa_stream(tdoa_engine *e);
/* Run on a caller-owned stream instead (cudaStream_t as void*; NULL: a fresh private
 * stream).  The benchmark uses this so that its CUDA events bracket the engine's work. */
TDOA_API int tdoa_set_stream(tdoa_engine *e, void *stream);
/* Block until everything queued on the engine's stream is done. */
TDOA_API int tdoa_synchronize(tdoa_engine *e);

#ifdef __cplusplus
}
#endif
#endif /* TDOA_B200_H */
