// engine.cu -- the C ABI of libtdoa_b200.so (include/tdoa_b200.h): engine lifetime, the capture
// loaders, and the entry points that are one kernel deep (baselines, solvers, grid, analyzers,
// self-tests).  The per-signal / per-pair orchestration of the path is engine_pipeline.cu, more than
// one GPU is engine_multi.cu; engine_internal.h is what they share.
//
// There is no CPU fallback anywhere in the engine: every numeric result is produced
// by a kernel on the engine's device, and tdoa_create fails without an sm_100 GPU.
#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "engine_internal.h"

using namespace tdoa;

static_assert(sizeof(tdoa_peak) == 32, "tdoa_peak is a 32-byte wire record");
static_assert(sizeof(PeakRec) == sizeof(tdoa_peak), "device and ABI peak records must match");

namespace {
thread_local std::string g_create_error;
}

namespace tdoa {

int fail(tdoa_engine *e, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (e) e->error = buf; else g_create_error = buf;
    return code;
}

int begin_call(tdoa_engine *e)
{
    CU(cudaSetDevice(e->device));
    if (e->frame_pending) {
        CU(cudaEventSynchronize(e->frame_done));
        e->frame_pending = false;
    }
    e->frame_used = 0;
    e->spans_used = 0;
    e->launches_at_call = e->st.launches_total;
    return TDOA_OK;
}

int end_call(tdoa_engine *e, bool sync)
{
    for (void *p : e->call_allocs) cudaFreeAsync(p, e->stream);
    e->call_allocs.clear();
    CU(cudaEventRecord(e->frame_done, e->stream));
    e->frame_pending = true;
    if (sync) {
        CU(cudaStreamSynchronize(e->stream));
        e->frame_pending = false;
    }
    CU(cudaGetLastError());
    return TDOA_OK;
}

// stream-ordered scratch that lives until end_call
int alloc(tdoa_engine *e, void **out, size_t bytes)
{
    *out = nullptr;
    if (bytes == 0) bytes = 16;
    CU(cudaMallocAsync(out, bytes, e->stream));
    e->call_allocs.push_back(*out);
    return TDOA_OK;
}

// Descriptors travel host -> device inside a kernel that reads the pinned (mapped) frame,
// not through the copy engine: while a lazily loaded capture is arriving, the engine's
// host -> device queue holds hundreds of MB of bulk copies, and a cudaMemcpyAsync of a
// few hundred bytes on the compute stream would wait behind all of them.
__global__ void k_fetch_descriptors(uint4 *__restrict__ dst, const uint4 *__restrict__ src, int n16)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

void launch_fetch_descriptors(uint8_t *d_dst, const uint8_t *mapped_src, int n16, cudaStream_t st)
{
    k_fetch_descriptors<<<std::min(32, (n16 + 255) / 256), 256, 0, st>>>(reinterpret_cast<uint4 *>(d_dst),
                                                                         reinterpret_cast<const uint4 *>(mapped_src), n16);
}

// ---- per-kernel device time: an event pair around a launch, read back at the call's sync

int span_begin(tdoa_engine *e, int tag)
{
    if (e->spans_used == e->spans.size()) {
        tdoa_engine::Span sp;
        if (cudaEventCreate(&sp.a) != cudaSuccess || cudaEventCreate(&sp.b) != cudaSuccess) return -1;
        e->spans.push_back(sp);
    }
    const int idx = (int)e->spans_used++;
    e->spans[idx].tag = tag;
    cudaEventRecord(e->spans[idx].a, e->stream);
    return idx;
}

void span_end(tdoa_engine *e, int idx)
{
    if (idx >= 0) cudaEventRecord(e->spans[idx].b, e->stream);
}

// the stream must be idle
void spans_collect(tdoa_engine *e)
{
    for (size_t i = 0; i < e->spans_used; i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e->spans[i].a, e->spans[i].b) != cudaSuccess) { cudaGetLastError(); continue; }
        switch (e->spans[i].tag) {
            case SPAN_DEMOD: e->st.ms_demod += ms; e->st.demod_launches++; break;
            case SPAN_BOXCAR: e->st.ms_boxcar += ms; e->st.boxcar_launches++; break;
            case SPAN_CAND: e->st.ms_cand += ms; e->st.cand_launches++; break;
            case SPAN_STAGE_PRE: e->st.ms_preprocess += ms; break;
            case SPAN_STAGE_CORR: e->ms_corr += ms; break;
            case SPAN_FFT: e->st.ms_fft += ms; break;
            case SPAN_FFT_SEG: e->st.ms_fft_seg += ms; break;
        }
    }
    e->spans_used = 0;
}

// the checks of every grid entry point: 2..16 stations, a grid descriptor, a non-empty grid whose CTA count fits an int
int grid_check(tdoa_engine *e, const char *fn, int n_stations, const double *grid_desc)
{
    if (!grid_desc || n_stations < 2 || n_stations > 16)
        return fail(e, TDOA_E_INVALID, "%s: bad arguments (2..16 stations, rd_stride >= pairs)", fn);
    if (!(grid_desc[4] >= 1.0 && grid_desc[5] >= 1.0)) return fail(e, TDOA_E_INVALID, "%s: empty grid", fn);
    // one CTA per 128 cells, gridDim.x is an int: reject what would wrap
    if (grid_desc[4] > 2147483647.0 || grid_desc[5] > 2147483647.0 || grid_desc[4] * grid_desc[5] / 128.0 > 2147483647.0)
        return fail(e, TDOA_E_INVALID, "%s: grid of %.0f x %.0f cells is too large", fn, grid_desc[4], grid_desc[5]);
    return TDOA_OK;
}

int grid_search_queue(tdoa_engine *e, GridSearch &g, bool every_cell)
{
    int rc;
    void *d_scratch = nullptr;
    // use_fft = 0 evaluates every cell by the statement (SOURCE mode's default)
    g.ranked = !every_cell && e->cfg.use_fft != 0;
    if (!g.ranked) {
        if ((rc = alloc(e, &d_scratch, grid_scratch_bytes(g.nlat, g.nlon, g.n_sets)))) return rc;
        launch_grid_cells(g.d_llh, g.n_st, g.d_desc, g.nlat, g.nlon, g.d_rd, g.n_sets, g.rd_stride, g.d_cost, g.d_idx, g.d_out,
                          d_scratch, e->stream, g.d_used, g.d_tab);
        count_launch(e, 2);
        return TDOA_OK;
    }
    // ranked: the expanded cost (16 FMA per cell and set) finds the cells that can hold the minimum, the statement
    // settles them (solve.cu)
    if ((rc = alloc_t(e, &g.d_count, (size_t)grid_rank_chunks(g.n_sets))) ||
        (rc = alloc(e, &d_scratch, grid_rank_scratch_bytes(g.nlat, g.nlon, g.n_sets))))
        return rc;
    launch_grid_ranked(g.d_llh, g.n_st, g.d_desc, g.nlat, g.nlon, g.d_tab, g.d_rd, g.n_sets, g.rd_stride, g.d_cost, g.d_idx,
                       g.d_out, d_scratch, g.d_count, e->stream, g.d_used);
    count_launch(e, 5 * grid_rank_chunks(g.n_sets));
    return TDOA_OK;
}

int grid_search_fetch(tdoa_engine *e, GridSearch &g)
{
    if (!g.ranked) return TDOA_OK;
    g.h_count.resize((size_t)grid_rank_chunks(g.n_sets));
    g.h_idx.resize((size_t)g.n_sets);
    CU(cudaMemcpyAsync(g.h_count.data(), g.d_count, g.h_count.size() * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(g.h_idx.data(), g.d_idx, g.h_idx.size() * sizeof(i64), cudaMemcpyDeviceToHost, e->stream));
    return TDOA_OK;
}

bool grid_search_complete(const GridSearch &g, const std::vector<char> &searched)
{
    if (!g.ranked) return true;
    if (grid_rank_overflowed(g.h_count.data(), g.n_sets)) return false;   // a plateau of ties
    // a searched set without a survivor (range differences that are not numbers: every comparison of the bound
    // fails): the statement decides such sets too
    for (int s = 0; s < g.n_sets; s++)
        if (g.h_idx[s] < 0 && searched[s]) return false;
    return true;
}

// tdoa_grid (used == nullptr) and tdoa_grid_masked
int grid_impl(tdoa_engine *e, const char *fn, const double *stations_llh, int32_t n_stations, const double *grid_desc,
              const double *range_diffs, const uint8_t *used, int32_t n_sets, int32_t rd_stride, double *out_llh,
              double *out_cost, int64_t *out_index)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    const int P = n_stations * (n_stations - 1) / 2;
    if (!stations_llh || !range_diffs || !out_llh || n_sets < 0 || rd_stride < P)
        return fail(e, TDOA_E_INVALID, "%s: bad arguments (2..16 stations, rd_stride >= pairs)", fn);
    if ((rc = grid_check(e, fn, n_stations, grid_desc))) return rc;
    if (n_sets == 0) return end_call(e, true);
    GridSearch g;
    g.n_sets = n_sets; g.rd_stride = rd_stride; g.n_st = n_stations; g.nlat = (int)grid_desc[4]; g.nlon = (int)grid_desc[5];
    double *d_llh = nullptr, *d_desc = nullptr, *d_rd = nullptr, *d_tab = nullptr;
    uint8_t *d_used = nullptr;
    // the host's share: the table of c_k per set (masked: also which sets are searched, which every cell reads)
    const int T = grid_rank_tab_doubles(used != nullptr);
    std::vector<double> tab((size_t)n_sets * T, 0.0);
    std::vector<char> searched((size_t)n_sets);
    for (int s = 0; s < n_sets; s++)
        searched[s] = grid_rank_row(range_diffs + (size_t)s * rd_stride, used ? used + (size_t)s * rd_stride : nullptr,
                                    n_stations, tab.data() + (size_t)s * T);
    if ((rc = alloc_t(e, &d_llh, (size_t)3 * n_stations)) || (rc = alloc_t(e, &d_desc, 8)) ||
        (rc = alloc_t(e, &d_rd, (size_t)n_sets * rd_stride)) || (rc = alloc_t(e, &d_tab, tab.size())) ||
        (rc = alloc_t(e, &g.d_cost, (size_t)n_sets)) || (rc = alloc_t(e, &g.d_idx, (size_t)n_sets)) ||
        (rc = alloc_t(e, &g.d_out, (size_t)3 * n_sets)))
        return rc;
    CU(cudaMemcpyAsync(d_llh, stations_llh, (size_t)3 * n_stations * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_desc, grid_desc, 7 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_rd, range_diffs, (size_t)n_sets * rd_stride * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    if (used) {
        if ((rc = alloc_t(e, &d_used, (size_t)n_sets * rd_stride))) return rc;
        CU(cudaMemcpyAsync(d_used, used, (size_t)n_sets * rd_stride, cudaMemcpyHostToDevice, e->stream));
        CU(cudaMemsetAsync(g.d_out, 0xff, (size_t)3 * n_sets * sizeof(double), e->stream));   // NaN where no arg-min
    }
    g.d_llh = d_llh; g.d_desc = d_desc; g.d_rd = d_rd; g.d_tab = d_tab; g.d_used = d_used;
    if ((rc = grid_search_queue(e, g, false)) || (rc = grid_search_fetch(e, g))) return rc;
    CU(cudaStreamSynchronize(e->stream));   // tab and the read-back are this frame's
    if (!grid_search_complete(g, searched) && (rc = grid_search_queue(e, g, true))) return rc;
    CU(cudaMemcpyAsync(out_llh, g.d_out, (size_t)3 * n_sets * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (out_cost) CU(cudaMemcpyAsync(out_cost, g.d_cost, (size_t)n_sets * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (out_index) CU(cudaMemcpyAsync(out_index, g.d_idx, (size_t)n_sets * sizeof(i64), cudaMemcpyDeviceToHost, e->stream));
    return end_call(e, true);
}

}  // namespace tdoa

// =========================================================================== C ABI

extern "C" {

int tdoa_default_config(int32_t mode, tdoa_config *cfg)
{
    if (!cfg) return TDOA_E_INVALID;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->sample_rate = 2000000.0;  // processor.go:821
    cfg->mode = mode;
    cfg->n_stations = 3;
    cfg->device = 0;
    switch (mode) {
        case TDOA_MODE_SOURCE:
            cfg->chunk_samples = 2000000;  // processor.go:772
            cfg->max_lag = 20000;          // processor.go:633
            cfg->block_size = 1000;        // processor.go:682
            cfg->sanity_lag = 0;
            cfg->use_fft = 0;
            break;
        case TDOA_MODE_BINARY:
            cfg->chunk_samples = 1000000;
            cfg->max_lag = 2000;
            cfg->block_size = 10000;
            cfg->sanity_lag = 120;
            cfg->use_fft = 1;
            break;
        case TDOA_MODE_EXTENDED:
            cfg->chunk_samples = 0;
            cfg->max_lag = 2000;
            cfg->block_size = 10000;
            cfg->sanity_lag = 0;
            cfg->use_fft = 1;
            break;
        default:
            return TDOA_E_INVALID;
    }
    return TDOA_OK;
}

int tdoa_create(tdoa_engine **out, const tdoa_config *cfg)
{
    tdoa_engine *e = nullptr;  // CU() reports into the thread-local create error
    if (!out || !cfg) return fail(nullptr, TDOA_E_INVALID, "tdoa_create: NULL argument");
    *out = nullptr;
    if (cfg->mode < TDOA_MODE_SOURCE || cfg->mode > TDOA_MODE_EXTENDED)
        return fail(nullptr, TDOA_E_INVALID, "tdoa_create: bad mode %d", cfg->mode);
    if (cfg->n_stations < 2 || cfg->n_stations > 64)
        return fail(nullptr, TDOA_E_INVALID, "tdoa_create: n_stations must be 2..64, got %d", cfg->n_stations);
    if (cfg->decimate < 0 || cfg->decimate > 4096 || (cfg->decimate > 1 && cfg->mode != TDOA_MODE_EXTENDED))
        return fail(nullptr, TDOA_E_INVALID, "tdoa_create: decimate is an EXTENDED-mode option (1..4096), got %d", cfg->decimate);
    if (cfg->n_devices < 0 || cfg->n_devices > 64)
        return fail(nullptr, TDOA_E_INVALID, "tdoa_create: n_devices must be 0..64, got %d", cfg->n_devices);
    if (cfg->max_lag < 0 || cfg->block_size < 1 || cfg->chunk_samples < 0 || cfg->sanity_lag < 0 || cfg->guard_samples < 0 ||
        cfg->copy_chunk < 0)
        return fail(nullptr, TDOA_E_INVALID, "tdoa_create: negative size in config");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) {
        cudaGetLastError();
        return fail(nullptr, TDOA_E_NODEVICE, "tdoa_create: no CUDA device (this engine has no CPU path)");
    }
    if (cfg->device < 0 || cfg->device >= n_dev)
        return fail(nullptr, TDOA_E_NODEVICE, "tdoa_create: device %d of %d does not exist", cfg->device, n_dev);
    cudaDeviceProp prop{};
    CU(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return fail(nullptr, TDOA_E_NODEVICE, "tdoa_create: device %d is sm_%d%d; this library is built for sm_100a only",
                    cfg->device, prop.major, prop.minor);
    CU(cudaSetDevice(cfg->device));
    e = new tdoa_engine();
    e->cfg = *cfg;
    e->device = cfg->device;
    e->stations.resize(cfg->n_stations);
    e->branch_memo.assign((size_t)cfg->n_stations * 2, (int8_t)-1);
    cudaError_t err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
    if (err == cudaSuccess) { e->own_stream = true; err = cudaMallocHost(&e->h_frame, kFrameBytes); }
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_reload, cudaEventDisableTiming);
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->side_stream, cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming);
    if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming);
    if (err == cudaSuccess) {
        void *dp = nullptr;
        err = cudaHostGetDevicePointer(&dp, e->h_frame, 0);
        e->h_frame_dev = static_cast<const uint8_t *>(dp);
    }
    if (err == cudaSuccess) err = cudaMalloc(&e->d_frame, kFrameBytes);
    if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->frame_done, cudaEventDisableTiming);
    for (int i = 0; i < 6 && err == cudaSuccess; i++) err = cudaEventCreate(&e->ev[i]);
    if (err == cudaSuccess) {
        // keep freed stream-ordered scratch cached in the pool between calls
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, cfg->device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    if (err != cudaSuccess) {
        g_create_error = std::string("tdoa_create: ") + cudaGetErrorString(err);
        tdoa_destroy(e);
        return err == cudaErrorMemoryAllocation ? TDOA_E_NOMEM : TDOA_E_CUDA;
    }
    e->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    if (err == cudaSuccess && fft_setup(e->stream, &e->d_tw) != 0) err = cudaErrorUnknown;
    if (err == cudaSuccess && demod_setup(e->stream) != 0) err = cudaErrorUnknown;
    if (err == cudaSuccess && fft_tile_setup() != 0) err = cudaErrorUnknown;
    if (err == cudaSuccess && big_setup(e->stream, &e->d_tw_fine) != 0) err = cudaErrorUnknown;
    if (err == cudaSuccess && spec_setup() != 0) err = cudaErrorUnknown;
    if (err == cudaSuccess && quality_setup() != 0) err = cudaErrorUnknown;
    if (err != cudaSuccess) {
        g_create_error = std::string("tdoa_create: ") + cudaGetErrorString(err);
        tdoa_destroy(e);
        return TDOA_E_CUDA;
    }
    int bad = unpack_selftest(e->stream);
    if (bad == 0 && e->cfg.mode == TDOA_MODE_EXTENDED) bad = weak_unpack_selftest(e->stream);   // k_weak_fused's divide-free unpack
    if (bad != 0) {
        g_create_error = "tdoa_create: device unpack self-test failed (kernel image not runnable on this GPU?)";
        tdoa_destroy(e);
        return TDOA_E_CUDA;
    }
    e->st.launches_total = e->cfg.mode == TDOA_MODE_EXTENDED ? 2 : 1;
    if (cfg->n_devices > 1) {
        e->cfg.n_devices = cfg->n_devices;
        const int rc = multi_create_peers(e, cfg);
        if (rc) {
            g_create_error = "tdoa_create: " + e->error;
            tdoa_destroy(e);
            return rc;
        }
    }
    *out = e;
    return TDOA_OK;
}

void tdoa_destroy(tdoa_engine *e)
{
    if (!e) return;
    multi_destroy(e);   // peers of a multi-device engine, the communicator
    cudaSetDevice(e->device);
    if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (void *p : e->call_allocs) cudaFreeAsync(p, e->stream);
    for (auto &s : e->stations) {
        if (s.owned) cudaFree(s.owned);
        for (cudaEvent_t ev : s.event_pool) cudaEventDestroy(ev);
    }
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->side_stream) { cudaStreamSynchronize(e->side_stream); cudaStreamDestroy(e->side_stream); }
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    for (int k = 0; k < 2; k++) {
        if (e->h_stage[k]) cudaFreeHost(e->h_stage[k]);
        if (e->ev_stage[k]) cudaEventDestroy(e->ev_stage[k]);
    }
    if (e->ev_reload) cudaEventDestroy(e->ev_reload);
    if (e->h_frame) cudaFreeHost(e->h_frame);
    if (e->d_frame) cudaFree(e->d_frame);
    if (e->d_tw) cudaFree(e->d_tw);
    if (e->d_tw_fine) cudaFree(e->d_tw_fine);
    for (auto &sp : e->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    if (e->frame_done) cudaEventDestroy(e->frame_done);
    for (auto &ev : e->ev)
        if (ev) cudaEventDestroy(ev);
    if (e->stream && e->own_stream) { cudaStreamSynchronize(e->stream); cudaStreamDestroy(e->stream); }
    delete e;
}

const char *tdoa_last_error(const tdoa_engine *e) { return e ? e->error.c_str() : g_create_error.c_str(); }

void *tdoa_host_alloc(size_t nbytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, nbytes ? nbytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void tdoa_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

int tdoa_set_stream(tdoa_engine *e, void *stream)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    CU(cudaStreamSynchronize(e->stream));
    if (e->own_stream) { cudaStreamDestroy(e->stream); e->own_stream = false; }
    if (stream) {
        e->stream = reinterpret_cast<cudaStream_t>(stream);
    } else {
        CU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
        e->own_stream = true;
    }
    return TDOA_OK;
}

// device buffer of a station for a capture of nbytes; forgets any lazy load in progress
static int station_buffer(tdoa_engine *e, Station &s, size_t nbytes)
{
    if (s.h_lazy || !s.chunks[0].empty() || !s.chunks[1].empty()) {
        CU(cudaStreamSynchronize(e->copy_stream));  // copies of the previous capture still target this buffer
        s.h_lazy = nullptr; s.lazy_queued = false;
        s.chunks[0].clear(); s.chunks[1].clear();
        s.events_used = 0;
    }
    if (s.owned_cap < nbytes || !s.owned) {
        CU(cudaStreamSynchronize(e->stream));
        if (s.owned) cudaFree(s.owned);
        s.owned = nullptr; s.owned_cap = 0;
        const size_t cap = std::max<size_t>((nbytes + 255) & ~size_t(255), 256);
        CU(cudaMalloc(&s.owned, cap));
        s.owned_cap = cap;
    }
    return TDOA_OK;
}

int tdoa_load_u8_pinned(tdoa_engine *e, int32_t station, const uint8_t *pinned_iq, size_t nbytes)
{
    if (!e) return TDOA_E_INVALID;
    // small captures gain nothing from following the copy
    // (and the chunk map below is written for the reference's split: no guard)
    if (nbytes < (size_t)12 * 4096 * 8 || e->cfg.guard_samples > 0) return tdoa_load_u8(e, station, pinned_iq, nbytes);
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations)
        return fail(e, TDOA_E_INVALID, "tdoa_load_u8_pinned: bad station %d", station);
    if (!pinned_iq) return fail(e, TDOA_E_INVALID, "tdoa_load_u8_pinned: NULL capture");
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, pinned_iq) != cudaSuccess || attr.type != cudaMemoryTypeHost) {
        cudaGetLastError();
        return fail(e, TDOA_E_INVALID, "tdoa_load_u8_pinned: the capture must live in tdoa_host_alloc memory");
    }
    Station &s = e->stations[station];
    if ((rc = station_buffer(e, s, nbytes))) return rc;
    s.h_lazy = pinned_iq;
    s.lazy_queued = false;
    s.d_raw = s.owned;
    s.nbytes = nbytes;
    s.nsamp = (i64)(nbytes / 2);
    s.loaded = true;
    return multi_forward_load(e, 1, station, pinned_iq, nbytes, nullptr);
}

// loadIQData for a file (processor.go:166-191): the capture is read in 32 MB pieces into two
// pinned staging buffers and copied to the device from there, the read of one piece
// overlapping the PCIe copy of the previous one; nothing of the file stays in host memory.
// Go's text for an errno (os.PathError: "open <path>: no such file or directory"): the C
// library's message with a lower-case first letter
static std::string go_errno(int err)
{
    std::string m = strerror(err);
    if (!m.empty() && m[0] >= 'A' && m[0] <= 'Z') m[0] = (char)(m[0] - 'A' + 'a');
    return m;
}

int tdoa_load_file(tdoa_engine *e, int32_t station, const char *path, int64_t *n_samples)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations) return fail(e, TDOA_E_INVALID, "tdoa_load_file: bad station %d", station);
    if (!path) return fail(e, TDOA_E_INVALID, "tdoa_load_file: NULL path");
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(e, TDOA_E_IO, "failed to open file: open %s: %s", path, go_errno(errno).c_str());  // processor.go:170-172
    struct stat sb;
    if (fstat(fd, &sb) != 0) {
        const int err = errno;
        close(fd);
        return fail(e, TDOA_E_IO, "failed to get file size: stat %s: %s", path, go_errno(err).c_str());  // processor.go:177-179
    }
    const size_t nbytes = (size_t)sb.st_size;
    Station &s = e->stations[station];
    if ((rc = station_buffer(e, s, nbytes))) { close(fd); return rc; }
    constexpr size_t kPiece = (size_t)32 << 20;
    for (int k = 0; k < 2; k++) {
        if (!e->h_stage[k]) {
            if (cudaMallocHost(&e->h_stage[k], kPiece) != cudaSuccess ||
                cudaEventCreateWithFlags(&e->ev_stage[k], cudaEventDisableTiming) != cudaSuccess) {
                close(fd);
                return fail(e, TDOA_E_NOMEM, "tdoa_load_file: pinned staging allocation failed");
            }
        }
    }
    // kernels queued earlier may still read the station's previous capture
    cudaEventRecord(e->ev_reload, e->stream);
    cudaStreamWaitEvent(e->copy_stream, e->ev_reload, 0);
    size_t off = 0;
    int piece = 0;
    bool used[2] = {false, false};
    while (off < nbytes) {
        const int k = piece & 1;
        if (used[k]) cudaEventSynchronize(e->ev_stage[k]);  // the copy out of this buffer has finished
        const size_t want = std::min(kPiece, nbytes - off);
        size_t got = 0;
        while (got < want) {
            const ssize_t r = read(fd, static_cast<uint8_t *>(e->h_stage[k]) + got, want - got);
            if (r < 0 && errno == EINTR) continue;
            if (r <= 0) {
                const int err = errno;
                close(fd);
                cudaStreamSynchronize(e->copy_stream);
                if (r == 0) return fail(e, TDOA_E_IO, "failed to read data: unexpected end of file");
                return fail(e, TDOA_E_IO, "failed to read data: read %s: %s", path, go_errno(err).c_str());  // :189-191
            }
            got += (size_t)r;
        }
        cudaError_t ce = cudaMemcpyAsync(s.owned + off, e->h_stage[k], want, cudaMemcpyHostToDevice, e->copy_stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(e->ev_stage[k], e->copy_stream);
        if (ce != cudaSuccess) {
            close(fd);
            return fail(e, TDOA_E_CUDA, "tdoa_load_file: copy failed: %s", cudaGetErrorString(ce));
        }
        used[k] = true;
        off += want;
        piece++;
    }
    close(fd);
    CU(cudaStreamSynchronize(e->copy_stream));
    s.d_raw = s.owned;
    s.nbytes = nbytes;
    s.nsamp = (i64)(nbytes / 2);  // processor.go:183  numSamples = fileSize / 2
    s.loaded = true;
    if (n_samples) *n_samples = s.nsamp;
    return multi_forward_load(e, 2, station, path, 0, nullptr);
}

int tdoa_load_u8(tdoa_engine *e, int32_t station, const uint8_t *iq, size_t nbytes)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations) return fail(e, TDOA_E_INVALID, "tdoa_load_u8: bad station %d", station);
    if (!iq && nbytes) return fail(e, TDOA_E_INVALID, "tdoa_load_u8: NULL capture");
    Station &s = e->stations[station];
    if ((rc = station_buffer(e, s, nbytes))) return rc;
    if (nbytes) CU(cudaMemcpyAsync(s.owned, iq, nbytes, cudaMemcpyHostToDevice, e->stream));
    // the caller's buffer may be Go memory: do not return before the copy has left it
    CU(cudaStreamSynchronize(e->stream));
    s.d_raw = s.owned;
    s.nbytes = nbytes;
    s.nsamp = (i64)(nbytes / 2);  // processor.go:187  numSamples = fileSize / 2
    s.loaded = true;
    return multi_forward_load(e, 0, station, iq, nbytes, nullptr);
}

int tdoa_load_u8_device(tdoa_engine *e, int32_t station, const uint8_t *d_iq, size_t nbytes)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations)
        return fail(e, TDOA_E_INVALID, "tdoa_load_u8_device: bad station %d", station);
    if (!d_iq && nbytes) return fail(e, TDOA_E_INVALID, "tdoa_load_u8_device: NULL capture");
    if (reinterpret_cast<uintptr_t>(d_iq) & 15u)
        return fail(e, TDOA_E_INVALID, "tdoa_load_u8_device: capture must be 16-byte aligned");
    if (e->cfg.n_devices > 1)
        return fail(e, TDOA_E_STATE, "tdoa_load_u8_device: a capture in one device's memory cannot feed n_devices = %d", e->cfg.n_devices);
    Station &s = e->stations[station];
    if (s.h_lazy || !s.chunks[0].empty() || !s.chunks[1].empty()) {
        CU(cudaStreamSynchronize(e->copy_stream));
        s.h_lazy = nullptr; s.lazy_queued = false;
        s.chunks[0].clear(); s.chunks[1].clear();
        s.events_used = 0;
    }
    s.d_raw = d_iq;
    s.nbytes = nbytes;
    s.nsamp = (i64)(nbytes / 2);
    s.loaded = true;
    return TDOA_OK;
}

int tdoa_baselines(tdoa_engine *e, const double *stations_llh, int32_t n_stations, double *baselines)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (!stations_llh || !baselines || n_stations < 2)
        return fail(e, TDOA_E_INVALID, "tdoa_baselines: bad arguments");
    const int P = n_stations * (n_stations - 1) / 2;
    double *d_llh = nullptr, *d_out = nullptr;
    if ((rc = alloc_t(e, &d_llh, (size_t)3 * n_stations)) || (rc = alloc_t(e, &d_out, (size_t)P))) return rc;
    CU(cudaMemcpyAsync(d_llh, stations_llh, (size_t)3 * n_stations * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    launch_baselines(d_llh, n_stations, d_out, e->stream);
    count_launch(e);
    CU(cudaMemcpyAsync(baselines, d_out, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    return end_call(e, true);
}

int tdoa_solve(tdoa_engine *e, const double *stations_llh, int32_t n_stations, const double *range_diffs,
               int32_t n_sets, int32_t rd_stride, double *out_llh, int32_t *status, int32_t *iters)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    // processor.go:933-935 needs at least 3 stations and 2 range differences
    if (!stations_llh || !range_diffs || !out_llh || !status || n_stations < 3 || n_sets < 0 || rd_stride < 2)
        return fail(e, TDOA_E_INVALID, "tdoa_solve: bad arguments (need >= 3 stations, rd_stride >= 2)");
    if (n_sets == 0) return end_call(e, true);
    double *d_llh = nullptr, *d_rd = nullptr, *d_out = nullptr;
    int *d_status = nullptr, *d_iters = nullptr;
    if ((rc = alloc_t(e, &d_llh, (size_t)3 * n_stations)) || (rc = alloc_t(e, &d_rd, (size_t)n_sets * rd_stride)) ||
        (rc = alloc_t(e, &d_out, (size_t)3 * n_sets)) || (rc = alloc_t(e, &d_status, (size_t)n_sets)) ||
        (rc = alloc_t(e, &d_iters, (size_t)n_sets)))
        return rc;
    CU(cudaMemcpyAsync(d_llh, stations_llh, (size_t)3 * n_stations * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_rd, range_diffs, (size_t)n_sets * rd_stride * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    launch_solve(d_llh, d_rd, n_sets, rd_stride, d_out, d_status, d_iters, e->stream);
    count_launch(e);
    std::vector<int> h_status(n_sets);
    CU(cudaMemcpyAsync(out_llh, d_out, (size_t)3 * n_sets * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(h_status.data(), d_status, (size_t)n_sets * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    if (iters) CU(cudaMemcpyAsync(iters, d_iters, (size_t)n_sets * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    rc = end_call(e, true);
    if (rc) return rc;
    for (int i = 0; i < n_sets; i++) status[i] = h_status[i] ? TDOA_E_SINGULAR : TDOA_OK;
    return TDOA_OK;
}

int tdoa_solve_binary(tdoa_engine *e, const double *stations_llh, int32_t n_stations, const double *range_diffs, int32_t n_rd,
                      double *out_llh, int32_t *status, int32_t *n_valid, int32_t *n_iter, int32_t *converged, double *trace)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (!stations_llh || !range_diffs || !out_llh || !status || n_stations < 3 || n_rd < 0)
        return fail(e, TDOA_E_INVALID, "tdoa_solve_binary: bad arguments (need >= 3 stations)");
    double *d_llh = nullptr, *d_rd = nullptr, *d_out = nullptr, *d_trace = nullptr;
    int *d_info = nullptr;
    if ((rc = alloc_t(e, &d_llh, (size_t)3 * n_stations)) || (rc = alloc_t(e, &d_rd, (size_t)std::max(n_rd, 1))) ||
        (rc = alloc_t(e, &d_out, 3)) || (rc = alloc_t(e, &d_trace, 50)) || (rc = alloc_t(e, &d_info, 4)))
        return rc;
    CU(cudaMemcpyAsync(d_llh, stations_llh, (size_t)3 * n_stations * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    if (n_rd > 0) CU(cudaMemcpyAsync(d_rd, range_diffs, (size_t)n_rd * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemsetAsync(d_trace, 0, 50 * sizeof(double), e->stream));
    launch_solve_binary(d_llh, d_rd, n_rd, d_out, d_info, d_trace, e->stream);
    count_launch(e);
    int h_info[4] = {0, 0, 0, 0};
    double h_trace[50];
    CU(cudaMemcpyAsync(out_llh, d_out, 3 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(h_info, d_info, sizeof(h_info), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(h_trace, d_trace, sizeof(h_trace), cudaMemcpyDeviceToHost, e->stream));
    rc = end_call(e, true);
    if (rc) return rc;
    *status = h_info[0];
    if (n_valid) *n_valid = h_info[1];
    if (n_iter) *n_iter = h_info[2];
    if (converged) *converged = h_info[3];
    if (trace) std::memcpy(trace, h_trace, sizeof(h_trace));
    return TDOA_OK;
}

int tdoa_grid(tdoa_engine *e, const double *stations_llh, int32_t n_stations, const double *grid_desc,
              const double *range_diffs, int32_t n_sets, int32_t rd_stride, double *out_llh, double *out_cost,
              int64_t *out_index)
{
    return tdoa::grid_impl(e, "tdoa_grid", stations_llh, n_stations, grid_desc, range_diffs, nullptr, n_sets, rd_stride,
                           out_llh, out_cost, out_index);
}

int tdoa_grid_masked(tdoa_engine *e, const double *stations_llh, int32_t n_stations, const double *grid_desc,
                     const double *range_diffs, const uint8_t *used, int32_t n_sets, int32_t rd_stride, double *out_llh,
                     double *out_cost, int64_t *out_index)
{
    return tdoa::grid_impl(e, "tdoa_grid_masked", stations_llh, n_stations, grid_desc, range_diffs, used, n_sets, rd_stride,
                           out_llh, out_cost, out_index);
}

int tdoa_solve_ls(tdoa_engine *e, const double *stations_llh, int32_t n_stations, const double *range_diffs,
                  int32_t n_sets, int32_t rd_stride, const double *init_llh, int32_t dims, double *out_llh,
                  double *out_rms, int32_t *status, int32_t *iters)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    const int P = n_stations * (n_stations - 1) / 2;
    if (!stations_llh || !range_diffs || !out_llh || !status || n_sets < 0 || rd_stride < P)
        return fail(e, TDOA_E_INVALID, "tdoa_solve_ls: bad arguments");
    if (n_stations < 3 || n_stations > solve_ls_max_stations())
        return fail(e, TDOA_E_INVALID, "tdoa_solve_ls: 3..%d stations, got %d", solve_ls_max_stations(), n_stations);
    if (dims != 2 && dims != 3) return fail(e, TDOA_E_INVALID, "tdoa_solve_ls: dims must be 2 or 3");
    if (dims == 3 && n_stations < 4)
        return fail(e, TDOA_E_INVALID, "tdoa_solve_ls: elevation needs at least 4 stations (3 range differences)");
    if (n_sets == 0) return end_call(e, true);
    double *d_llh = nullptr, *d_rd = nullptr, *d_init = nullptr, *d_out = nullptr, *d_rms = nullptr;
    int *d_status = nullptr, *d_iters = nullptr;
    if ((rc = alloc_t(e, &d_llh, (size_t)3 * n_stations)) || (rc = alloc_t(e, &d_rd, (size_t)n_sets * rd_stride)) ||
        (rc = alloc_t(e, &d_out, (size_t)3 * n_sets)) || (rc = alloc_t(e, &d_rms, (size_t)n_sets)) ||
        (rc = alloc_t(e, &d_status, (size_t)n_sets)) || (rc = alloc_t(e, &d_iters, (size_t)n_sets)))
        return rc;
    CU(cudaMemcpyAsync(d_llh, stations_llh, (size_t)3 * n_stations * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(d_rd, range_diffs, (size_t)n_sets * rd_stride * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    if (init_llh) {
        if ((rc = alloc_t(e, &d_init, (size_t)3 * n_sets))) return rc;
        CU(cudaMemcpyAsync(d_init, init_llh, (size_t)3 * n_sets * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    }
    launch_solve_ls(d_llh, n_stations, d_rd, n_sets, rd_stride, d_init, dims, d_out, d_rms, d_status, d_iters, e->stream);
    count_launch(e);
    CU(cudaMemcpyAsync(out_llh, d_out, (size_t)3 * n_sets * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (out_rms) CU(cudaMemcpyAsync(out_rms, d_rms, (size_t)n_sets * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(status, d_status, (size_t)n_sets * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    if (iters) CU(cudaMemcpyAsync(iters, d_iters, (size_t)n_sets * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    return end_call(e, true);
}

int tdoa_analyze(tdoa_engine *e, int32_t station, int32_t fast, tdoa_signal_quality *ref, tdoa_signal_quality *tgt)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations || !e->stations[station].loaded)
        return fail(e, TDOA_E_STATE, "tdoa_analyze: station %d not loaded", station);
    if (!ref || !tgt) return fail(e, TDOA_E_INVALID, "tdoa_analyze: NULL output");
    Station &s = e->stations[station];
    if ((rc = capture_ready(e, s))) return rc;
    const i64 block = s.nsamp / 3;
    // fast_analyzer.go:71-73
    if (block == 0) return fail(e, TDOA_E_INVALID, "file too small for dual-frequency analysis");
    std::vector<QualJob> jobs(2);
    const int n_cta = 4 * e->sm_count;
    tdoa_signal_quality *d_out = nullptr;
    if ((rc = alloc_t(e, &d_out, 2))) return rc;
    int max_m = 0;
    for (int k = 0; k < 2; k++) {
        QualJob &J = jobs[k];
        J.fast = fast ? 1 : 0;
        if (fast) {
            // fast_analyzer.go:76-103: the first min(32768, block) samples of each block
            const i64 a = std::min<i64>(32768, block);
            if (k == 0) { J.src.raw = s.d_raw; J.src.run0_start = 0; J.src.run0_len = a; J.src.run1_start = 2 * block; J.n = 2 * a; }
            else { J.src.raw = s.d_raw; J.src.run0_start = block; J.src.run0_len = a; J.src.run1_start = 0; J.n = a; }
        } else {
            // analyzer.go:111-121: whole blocks
            J.n = k == 0 ? 2 * block : block;
            J.src = make_view(s, k == 0 ? TDOA_KIND_REF : TDOA_KIND_TGT, 0, J.n, 0);
        }
        const i64 msz = fast ? 8192 : 16384;
        J.m = (int)std::min<i64>(msz, J.n);
        max_m = std::max(max_m, J.m);
        J.out = d_out + k;
        if ((rc = alloc(e, &J.parts, quality_part_bytes() * (size_t)n_cta)) ||
            (rc = alloc(e, &J.fft_a, sizeof(double) * 2 * (size_t)std::max(J.m, 1))) ||
            (rc = alloc(e, &J.fft_b, sizeof(double) * 2 * (size_t)std::max(J.m, 1))) ||
            (rc = alloc_t(e, &J.psd, (size_t)std::max(J.m, 1))))
            return rc;
    }
    const QualJob *d_jobs = nullptr;
    if ((rc = upload(e, jobs, &d_jobs))) return rc;
    launch_quality(d_jobs, 2, n_cta, max_m, e->stream);
    count_launch(e, 2);
    tdoa_signal_quality h[2];
    CU(cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, e->stream));
    rc = end_call(e, true);
    if (rc) return rc;
    *ref = h[0];
    *tgt = h[1];
    return TDOA_OK;
}

int tdoa_xcorr_info(tdoa_engine *e, int32_t kind, tdoa_signal_info *signals, double *first_corr)
{
    if (!e) return TDOA_E_INVALID;
    if (kind != TDOA_KIND_REF && kind != TDOA_KIND_TGT) return fail(e, TDOA_E_INVALID, "tdoa_xcorr_info: bad kind %d", kind);
    if (e->info_sig[kind].empty()) return fail(e, TDOA_E_STATE, "tdoa_xcorr_info: no tdoa_xcorr call of this kind yet");
    if (signals) std::copy(e->info_sig[kind].begin(), e->info_sig[kind].end(), signals);
    if (first_corr) std::copy(e->info_first[kind].begin(), e->info_first[kind].end(), first_corr);
    return TDOA_OK;
}

int tdoa_get_stats(tdoa_engine *e, tdoa_stats *out)
{
    if (!e || !out) return TDOA_E_INVALID;
    *out = e->st;
    return TDOA_OK;
}

int tdoa_selftest(tdoa_engine *e, int32_t which, int64_t *mismatches)
{
    if (!e || !mismatches) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (which < 0 || which > 3) return fail(e, TDOA_E_INVALID, "tdoa_selftest: unknown test %d", which);
    unsigned first_bad[64] = {0};
    long long extra[2] = {0, 0};
    const long long bad = which == 0 ? div_selftest(e->stream) : demod_selftest(e->stream, first_bad, which == 3 ? 3 : 1, extra);
    if (bad < 0) return fail(e, TDOA_E_CUDA, "tdoa_selftest: kernel failed");
    if (which == 2) { *mismatches = extra[0]; return TDOA_OK; }   // fall-backs taken over the 2^32 quads
    if (which != 0) {
        char buf[400];
        int off = snprintf(buf, sizeof(buf), "demod selftest: %lld differing quads, %lld fall-backs to the full-accuracy arctangent "
                           "(%lld of them changed the value)%s", bad, extra[0], extra[1], bad ? "; first:" : "");
        for (unsigned k = 0; k < first_bad[0] && k < 12 && off < (int)sizeof(buf) - 12; k++)
            off += snprintf(buf + off, sizeof(buf) - off, " %08x", first_bad[1 + k]);
        e->error = buf;
    }
    *mismatches = bad;
    return TDOA_OK;
}

void *tdoa_stream(tdoa_engine *e) { return e ? reinterpret_cast<void *>(e->stream) : nullptr; }

int tdoa_synchronize(tdoa_engine *e)
{
    if (!e) return TDOA_E_INVALID;
    CU(cudaSetDevice(e->device));
    int rc = queue_lazy_copies(e, TDOA_KIND_REF);  // a lazily loaded capture is on the device after this call
    if (rc) return rc;
    CU(cudaStreamSynchronize(e->copy_stream));
    CU(cudaStreamSynchronize(e->stream));
    retire_lazy(e);
    return TDOA_OK;
}

}  // extern "C"
