// engine_internal.h -- what the translation units of the engine share: the engine object, the
// per-call scratch / descriptor / timing helpers, and the entry points of the pipeline that the C
// ABI wrappers (engine.cu), the per-signal and per-pair orchestration (engine_pipeline.cu) and the
// multi-GPU layer (engine_multi.cu) call across files.  Not part of the ABI.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/tdoa_b200.h"
#include "kernels.h"
#include "xcorr_fft.h"

namespace tdoa {

// one piece of a capture on its way to the device (tdoa_load_u8_pinned): samples
// [q_begin, q_end) of the REF or TGT signal; `landed` is recorded on the copy stream
struct CopyChunk {
    i64 q_begin = 0, q_end = 0;
    cudaEvent_t landed = nullptr;
};

struct Station {
    const uint8_t *d_raw = nullptr;
    uint8_t *owned = nullptr;
    size_t owned_cap = 0;
    size_t nbytes = 0;
    i64 nsamp = 0;
    bool loaded = false;
    // lazy load from pinned host memory: the copies are queued by the first call that
    // needs the capture, the needed signal kind first, in chunks the discriminator follows
    const uint8_t *h_lazy = nullptr;
    bool lazy_queued = false;
    std::vector<CopyChunk> chunks[2];
    std::vector<cudaEvent_t> event_pool;
    size_t events_used = 0;
};

constexpr i64 kCopyChunkDefault = (i64)16 << 20;  // samples per copy chunk (32 MB of capture)

// one signal (station-window) moving through preprocessing
struct Sig {
    SigSrc src{};
    i64 n = 0;
    i64 n_out = -1;       // samples of the preprocessed signal (n / decimate); -1: n
    float *plane[4][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};
    float *out_re = nullptr, *out_im = nullptr;  // pre-normalise result (scale in stats)
    double *stats = nullptr;
    double *partials = nullptr;
    unsigned *counter = nullptr;
    double power0 = 0.0;
    int branch = 0;
    int memo = -1;        // slot of the branch memo (station * 2 + kind), -1: none
    int station = -1;     // station and kind the view was cut from (-1: not a capture view)
    int kind = 0;
    i64 q0 = 0;           // first sample of the view within that station's REF / TGT signal
    bool fused = false;   // stage 0 ran the fused power + discriminator kernel
    bool deferred = false;  // branch 0 was assumed without reading the power back; the caller verifies
    bool raw_sums = false;  // the power pass was k_raw_stats: ST_SUM_* / ST_DC_* of the raw signal are in place
    bool need_im = false;   // a consumer reads out_im of a BINARY / EXTENDED signal (the tdoa_preprocess probe)
    bool filtered = false;  // the kind's channel filter wrote the signal to planes: ysrc is its source from then on
    SigSrc ysrc{};
};

struct Pair {
    int a, b;  // indices into the Sig array: signal 1, signal 2 (argv order, processor.go:816-817)
    int group = 0;  // window the pair belongs to
};

constexpr size_t kFrameBytes = 8u << 20;  // descriptor staging per call

struct Pending;      // engine_pipeline.cu: what an optimistic (queue-only) pass leaves to be checked
struct MultiState;   // engine_multi.cu: communicator, shard cursor, child engines

}  // namespace tdoa

struct tdoa_engine {
    tdoa_config cfg{};
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;   // host -> device copies of lazily loaded captures
    cudaStream_t side_stream = nullptr;   // tdoa_process: the TGT pair loop runs beside the REF pair loop
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    void *h_stage[2] = {nullptr, nullptr};        // tdoa_load_file: pinned staging, double buffered
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};
    cudaEvent_t ev_reload = nullptr;
    std::vector<tdoa::Station> stations;
    std::string error;
    // descriptor staging
    uint8_t *h_frame = nullptr, *d_frame = nullptr;
    const uint8_t *h_frame_dev = nullptr;  // device-side address of the pinned frame
    size_t frame_used = 0;
    cudaEvent_t frame_done = nullptr;
    bool frame_pending = false;
    // allocations of the current call (stream-ordered)
    std::vector<void *> call_allocs;
    // stats
    tdoa_stats st{};
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool ev_valid = false;
    int64_t launches_at_call = 0;
    float2 *d_tw = nullptr;  // FFT twiddle table
    float2 *d_tw_fine = nullptr;  // W_N^k, k < 2048, of the 2^21-point transform
    std::vector<int8_t> branch_memo;  // last preprocess branch per (station, kind); -1 unknown
    tdoa::ChannelTaps channel[2] = {};   // per kind (tdoa_set_channel); n = 0: no channel filter
    bool channel_cplx[2] = {false, false};
    std::vector<tdoa_signal_info> info_sig[2];  // window 0 of the last xcorr per kind
    std::vector<double> info_first[2];
    int sm_count = 148;
    // per-kernel timing spans of the current call (events are created once and reused)
    struct Span { cudaEvent_t a = nullptr, b = nullptr; int tag = 0; };
    std::vector<Span> spans;
    size_t spans_used = 0;
    float ms_corr = 0.f;   // correlation stage of the current call (ms_exact = ms_corr - ms_fft)
    tdoa::MultiState *multi = nullptr;   // engine_multi.cu; nullptr: one process, one GPU
    bool tgt_bounds = false;             // tdoa_set_tgt_bounds: the windowed calls bound their TGT lag search
    double tgt_guard = 0.0;              // samples added to each side of those intervals
    // tdoa_xcorr_ranking: while rank_dump is set, run_fft copies each record's ranking plane to
    // rank_dump + (record - rank_base) * rank_stride (device)
    float *rank_dump = nullptr;
    const tdoa::PeakRec *rank_base = nullptr;
    int rank_stride = 0;
};

namespace tdoa {

int fail(tdoa_engine *e, int code, const char *fmt, ...);

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t err__ = (call);                                                                \
        if (err__ != cudaSuccess)                                                                  \
            return fail(e, err__ == cudaErrorMemoryAllocation ? TDOA_E_NOMEM : TDOA_E_CUDA,        \
                        "%s failed: %s", #call, cudaGetErrorString(err__));                        \
    } while (0)

int begin_call(tdoa_engine *e);
int end_call(tdoa_engine *e, bool sync);
int alloc(tdoa_engine *e, void **out, size_t bytes);   // stream-ordered scratch that lives until end_call
template <class T>
int alloc_t(tdoa_engine *e, T **out, size_t count)
{
    return alloc(e, reinterpret_cast<void **>(out), count * sizeof(T));
}

void launch_fetch_descriptors(uint8_t *d_dst, const uint8_t *mapped_src, int n16, cudaStream_t st);

// copy a descriptor array to the device through the pinned frame
template <class T>
int upload(tdoa_engine *e, const std::vector<T> &v, const T **d_out)
{
    const size_t bytes = v.size() * sizeof(T);
    const size_t off = (e->frame_used + 255) & ~size_t(255);
    if (off + bytes > kFrameBytes) return fail(e, TDOA_E_NOMEM, "descriptor frame overflow (%zu bytes)", off + bytes);
    std::memcpy(e->h_frame + off, v.data(), bytes);
    const int n16 = (int)((bytes + 15) / 16);
    if (n16 > 0) {
        launch_fetch_descriptors(e->d_frame + off, e->h_frame_dev + off, n16, e->stream);
        CU(cudaGetLastError());
    }
    e->frame_used = off + bytes;
    *d_out = reinterpret_cast<const T *>(e->d_frame + off);
    return TDOA_OK;
}

inline void count_launch(tdoa_engine *e, int n = 1) { e->st.launches_total += n; }

// ---- per-kernel device time: an event pair around a launch, read back at the call's sync
enum { SPAN_DEMOD = 0, SPAN_BOXCAR = 1, SPAN_CAND = 2, SPAN_STAGE_PRE = 3, SPAN_STAGE_CORR = 4, SPAN_FFT = 5, SPAN_FFT_SEG = 6 };
int span_begin(tdoa_engine *e, int tag);
void span_end(tdoa_engine *e, int idx);
void spans_collect(tdoa_engine *e);   // the stream must be idle

// ---- grid multilateration (engine.cu): the argument checks every grid entry point shares
int grid_check(tdoa_engine *e, const char *fn, int n_stations, const double *grid_desc);
// The arg-min search of the grid entry points: the ranked pass and, where it is incomplete or use_fft = 0, every cell
struct GridSearch {
    const double *d_llh = nullptr, *d_desc = nullptr, *d_tab = nullptr, *d_rd = nullptr;   // d_tab: the ranked rows
    const uint8_t *d_used = nullptr;   // nullptr: unmasked
    int n_sets = 0, rd_stride = 0, n_st = 0, nlat = 0, nlon = 0;
    double *d_cost = nullptr, *d_out = nullptr;
    i64 *d_idx = nullptr;
    bool ranked = false;   // the last queued pass was the ranked one
    int *d_count = nullptr;
    std::vector<int> h_count;
    std::vector<i64> h_idx;
};
int grid_search_queue(tdoa_engine *e, GridSearch &g, bool every_cell);
int grid_search_fetch(tdoa_engine *e, GridSearch &g);   // the ranked pass's read-back, before the caller's sync
// after the sync: false if the ranked pass overflowed or a searched set found no cell
bool grid_search_complete(const GridSearch &g, const std::vector<char> &searched);

// ---- signal views and lazy loads (engine_pipeline.cu)
i64 signal_length(const Station &s, int kind, i64 guard);
SigSrc make_view(const Station &s, int kind, i64 start, i64 len, i64 guard);
int queue_lazy_copies(tdoa_engine *e, int first_kind);
int wait_kind(tdoa_engine *e, Station &s, int kind);
void retire_lazy(tdoa_engine *e);
int capture_ready(tdoa_engine *e, Station &s);

// ---- the pair loops over windows (engine_pipeline.cu)
void stats_reset(tdoa_engine *e);
int window_lengths(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows, int64_t hop,
                   std::vector<i64> &len);
// d_rates (device, S doubles, may be nullptr): every plane re-timed by its station's rate (tdoa_process_windows_retimed)
// d_bounds (device, n_windows * P intervals, may be nullptr): the bounded search of tdoa_xcorr_bounded, record by record
int xcorr_core(tdoa_engine *e, int32_t kind, int64_t win_start, const std::vector<i64> &len, int32_t n_windows,
               int64_t hop, PeakRec *d_out, Pending *pend, const double *d_rates = nullptr, const int2 *d_bounds = nullptr);
// tdoa_xcorr / tdoa_xcorr_device as one call; d_table (device, n_windows * P, out may then be nullptr): the
// records are also left there, past the call's end (tdoa_process_windows); d_rates, d_bounds as xcorr_core.
// h_bounds: the same intervals on the host -- what a multi-GPU engine deals with the windows; on one GPU they are
// copied to the device when d_bounds is nullptr
int xcorr_impl(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows, int64_t hop,
               tdoa_peak *out, bool out_is_device, PeakRec *d_table = nullptr, const double *d_rates = nullptr,
               const int2 *d_bounds = nullptr, const int2 *h_bounds = nullptr);

// ---- more than one GPU (engine_multi.cu)
// windows dealt over the ranks of the engine's communicator, records gathered: true if it took the call
bool multi_wants(const tdoa_engine *e, int32_t n_windows);
int xcorr_sharded(tdoa_engine *e, int32_t kind, int64_t win_start, const std::vector<i64> &len, int32_t n_windows, int64_t hop,
                  tdoa_peak *out, bool out_is_device, const int2 *h_bounds = nullptr);
// several signal kinds' windows in one collective call (tdoa_xcorr_windows): one meeting of the ranks
struct ShardPart {
    int32_t kind = 0;
    int64_t win_start = 0;
    std::vector<i64> len;       // per-station window lengths (window_lengths)
    int32_t n_windows = 0;
    int64_t hop = 0;
    tdoa_peak *out = nullptr;   // host or device table of n_windows * P records, or nullptr
    bool out_is_device = false;
    const double *rates = nullptr;   // station rates on the calling rank's device: the planes are re-timed (xcorr_core)
    const int2 *bounds = nullptr;    // host intervals [n_windows * P] (tdoa_xcorr_bounded): each rank takes its windows'
};
int xcorr_sharded(tdoa_engine *e, const std::vector<ShardPart> &parts);
void multi_destroy(tdoa_engine *e);
int multi_create_peers(tdoa_engine *e, const tdoa_config *cfg);   // tdoa_create with n_devices > 1
// which: 0 tdoa_load_u8, 1 tdoa_load_u8_pinned, 2 tdoa_load_file (p = path)
int multi_forward_load(tdoa_engine *e, int which, int32_t station, const void *p, size_t nbytes, int64_t *n_samples);
int multi_forward_channel(tdoa_engine *e, int32_t kind, const float *taps_re, const float *taps_im, int32_t n_taps);
int multi_forward_tgt_bounds(tdoa_engine *e, int32_t on, double guard_samples);

}  // namespace tdoa
