// engine_pipeline.cu -- host-side orchestration of the processing stage: which kernels run, on
// which buffers, in which order.  Mirrors ProcessTDOA's data flow (processor.go:739-929): per
// station load -> split ref/target -> window -> preprocess once per station-window -> all
// station pairs i<j -> peak records; then the fix.  Entry points: tdoa_unpack, tdoa_preprocess,
// tdoa_xcorr, tdoa_xcorr_device, tdoa_process, tdoa_cross_correlate.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "engine_internal.h"

using namespace tdoa;

namespace tdoa {

// ---------------------------------------------------------------- signal views

// processor.go:208-267: block = N/3; REF = blocks 1 and 3 concatenated, TGT = block 2;
// fewer than 3 samples: the data is returned unchanged.
// guard = samples dropped at the start of blocks 2 and 3 (0: the reference's split).  The
// retune of the dual-frequency recorder is issued from the USB callback while up to 15
// buffers of 262144 bytes are in flight (rtl_sdr.c:117-135, librtlsdr.c:358), so the first
// samples of a block after a retune still carry the other frequency ("contamination
// dilution", collector.go:85); an engine-defined option, not reference behaviour.
i64 signal_length(const Station &s, int kind, i64 guard)
{
    const i64 b = s.nsamp / 3;
    if (b == 0) return s.nsamp;
    const i64 g = std::min(guard, b);
    return kind == TDOA_KIND_REF ? 2 * b - g : b - g;
}

SigSrc make_view(const Station &s, int kind, i64 start, i64 len, i64 guard)
{
    SigSrc v{};
    v.raw = s.d_raw;
    const i64 b = s.nsamp / 3;
    const i64 g = std::min(guard, b);
    if (b == 0) {
        v.run0_start = start; v.run0_len = len; v.run1_start = 0;
    } else if (kind == TDOA_KIND_TGT) {
        v.run0_start = b + g + start; v.run0_len = len; v.run1_start = 0;
    } else if (start < b) {
        v.run0_start = start; v.run0_len = std::min(len, b - start); v.run1_start = 2 * b + g;
    } else {
        v.run0_start = 2 * b + g + (start - b); v.run0_len = len; v.run1_start = 0;
    }
    return v;
}

// processor.go:397-409: window = int(fs / (2 fc)) clamped to [3, 1000]; the reference
// hard-codes fs = 2e6 in every call site (:440, :488; binary likewise).
int cutoff_window(double fc)
{
    int w = (int)(2000000.0 / (2 * fc));
    if (w < 3) w = 3;
    if (w > 1000) w = 1000;
    return w;
}

// ---------------------------------------------------------------- lazy loads

// Queue the host -> device copies of every lazily loaded capture that is not on its way
// yet: first the chunks of `first_kind` of all stations, then the other kind, so the
// pipeline of the signal that was asked for first starts as early as PCIe allows.
int queue_lazy_copies(tdoa_engine *e, int first_kind)
{
    bool any = false;
    for (auto &s : e->stations) any |= s.h_lazy && !s.lazy_queued;
    if (!any) return TDOA_OK;
    // the device buffers may still be read by kernels queued earlier on the compute stream
    CU(cudaEventRecord(e->ev_reload, e->stream));
    CU(cudaStreamWaitEvent(e->copy_stream, e->ev_reload, 0));
    for (int pass = 0; pass < 2; pass++) {
        const int kind = pass == 0 ? first_kind : 1 - first_kind;
        for (auto &s : e->stations) {
            if (!s.h_lazy || s.lazy_queued) continue;
            const i64 b = s.nsamp / 3;
            const i64 L = kind == TDOA_KIND_REF ? 2 * b : b;
            s.chunks[kind].clear();
            const i64 chunk = e->cfg.copy_chunk > 0 ? std::max<i64>(4096, (i64)e->cfg.copy_chunk / 4096 * 4096) : kCopyChunkDefault;
            for (i64 q0 = 0; q0 < L; q0 += chunk) {
                const i64 q1 = std::min(L, q0 + chunk);
                // raw sample ranges of [q0, q1): REF = blocks 1 and 3, TGT = block 2
                i64 r0[2], r1[2];
                int nr = 0;
                if (kind == TDOA_KIND_TGT) { r0[0] = b + q0; r1[0] = b + q1; nr = 1; }
                else {
                    if (q0 < b) { r0[nr] = q0; r1[nr] = std::min(q1, b); nr++; }
                    if (q1 > b) { r0[nr] = 2 * b + std::max<i64>(q0, b) - b; r1[nr] = 2 * b + q1 - b; nr++; }
                }
                for (int k = 0; k < nr; k++) {
                    size_t off = (size_t)r0[k] * 2, len = (size_t)(r1[k] - r0[k]) * 2;
                    // the 0..2 samples after block 3 (N not a multiple of 3) travel with its last chunk
                    if (kind == TDOA_KIND_REF && r1[k] == 3 * b) len = s.nbytes - off;
                    CU(cudaMemcpyAsync(s.owned + off, s.h_lazy + off, len, cudaMemcpyHostToDevice, e->copy_stream));
                }
                if (s.events_used == s.event_pool.size()) {
                    cudaEvent_t ev = nullptr;
                    CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                    s.event_pool.push_back(ev);
                }
                CopyChunk c;
                c.q_begin = q0; c.q_end = q1; c.landed = s.event_pool[s.events_used++];
                CU(cudaEventRecord(c.landed, e->copy_stream));
                s.chunks[kind].push_back(c);
            }
        }
    }
    for (auto &s : e->stations)
        if (s.h_lazy) s.lazy_queued = true;
    return TDOA_OK;
}

// the compute stream waits until `kind` of the station has landed completely
int wait_kind(tdoa_engine *e, Station &s, int kind)
{
    if (!s.chunks[kind].empty()) CU(cudaStreamWaitEvent(e->stream, s.chunks[kind].back().landed, 0));
    return TDOA_OK;
}

// Once every queued copy has landed the chunk lists have served their purpose: later calls on the
// same capture then take the batched path (one fused launch per kind) instead of one launch and
// one event wait per chunk.  Called after a call's final synchronisation.
void retire_lazy(tdoa_engine *e)
{
    bool any = false;
    for (auto &s : e->stations) any |= s.lazy_queued;
    if (!any) return;
    if (cudaStreamQuery(e->copy_stream) != cudaSuccess) { cudaGetLastError(); return; }
    for (auto &s : e->stations) {
        if (!s.lazy_queued) continue;
        s.h_lazy = nullptr; s.lazy_queued = false;
        s.chunks[0].clear(); s.chunks[1].clear();
        s.events_used = 0;
    }
}

// for entry points that read a capture outside the chunk-following discriminator
int capture_ready(tdoa_engine *e, Station &s)
{
    int rc = queue_lazy_copies(e, TDOA_KIND_REF);
    if (rc) return rc;
    if ((rc = wait_kind(e, s, TDOA_KIND_REF))) return rc;
    return wait_kind(e, s, TDOA_KIND_TGT);
}

// ---------------------------------------------------------------- preprocessing

struct Step {  // one batched kernel over a set of signals
    std::vector<SigJob> jobs;
    i64 max_n = 0;
};

SigJob base_job(const Sig &s)
{
    SigJob j{};
    j.src = s.src;
    j.n = s.n;
    j.stats = s.stats;
    j.partials = s.partials;
    j.counter = s.counter;
    return j;
}

int ensure_plane(tdoa_engine *e, Sig &s, int idx, bool cplx)
{
    if (!s.plane[idx][0]) {
        int rc = alloc_t(e, &s.plane[idx][0], (size_t)s.n);
        if (rc) return rc;
    }
    if (cplx && !s.plane[idx][1]) {
        int rc = alloc_t(e, &s.plane[idx][1], (size_t)s.n);
        if (rc) return rc;
    }
    return TDOA_OK;
}

enum Kern { K_UNPACK, K_DEMOD, K_ENVELOPE, K_SEQSUM, K_BOXCAR, K_BOXCAR_SMALL, K_BOXCAR_SLIDE, K_NOTCH, K_DECIMATE, K_WEAK_FUSED };

// queue of (stage, kernel) steps: step k of every signal that runs the same kernel at
// that stage is batched into one launch; stages run in order
struct Pipeline {
    struct Entry { Kern kern; Step step; };
    std::vector<std::vector<Entry>> stages;
    void add(size_t stage, Kern k, const SigJob &j)
    {
        if (stages.size() <= stage) stages.resize(stage + 1);
        Entry *en = nullptr;
        for (auto &x : stages[stage])
            if (x.kern == k) en = &x;
        if (!en) { stages[stage].push_back(Entry{k, Step{}}); en = &stages[stage].back(); }
        en->step.jobs.push_back(j);
        en->step.max_n = std::max(en->step.max_n, j.n);
    }
};

SigJob box_job(const Sig &s, int in, int out, bool cplx, int window, int mode, bool sub_dc, bool power)
{
    SigJob j = base_job(s);
    j.q_re = s.plane[in][0];
    j.q_im = cplx ? s.plane[in][1] : nullptr;
    j.p_re = s.plane[out][0];
    j.p_im = cplx ? s.plane[out][1] : nullptr;
    j.window = window;
    j.mode = mode;
    j.sub_dc = sub_dc;
    j.want_power = power;
    return j;
}

// removeDCBias with the reference's sequential f32 accumulator (see seq_dc_limit)
SigJob seqsum_job(const Sig &s, int in, bool cplx)
{
    SigJob j = base_job(s);
    j.q_re = s.plane[in][0];
    j.q_im = cplx ? s.plane[in][1] : nullptr;
    return j;
}

bool wants_seq_dc(const tdoa_engine *e, i64 n)
{
    i64 lim = e->cfg.seq_dc_limit;
    if (lim == 0) lim = e->cfg.mode == TDOA_MODE_EXTENDED ? -1 : 4194304;
    return lim > 0 && n <= lim;
}

SigJob notch_job(const Sig &s, int in, int band, int out)
{
    SigJob j = base_job(s);
    j.q_re = s.plane[in][0]; j.q_im = s.plane[in][1];
    j.r_re = s.plane[band][0]; j.r_im = s.plane[band][1];
    j.p_re = s.plane[out][0]; j.p_im = s.plane[out][1];
    return j;
}

int run_pipeline(tdoa_engine *e, Pipeline &pl)
{
    for (auto &stage : pl.stages) {
        for (auto &en : stage) {
            Step &st = en.step;
            if (st.jobs.empty()) continue;
            const SigJob *d_jobs = nullptr;
            int rc = upload(e, st.jobs, &d_jobs);
            if (rc) return rc;
            const int nj = (int)st.jobs.size();
            switch (en.kern) {
                case K_UNPACK: launch_unpack(d_jobs, nj, st.max_n, stream_grid_x(st.max_n), e->stream); break;
                case K_DEMOD: launch_demod(d_jobs, nj, st.max_n, stream_grid_x(st.max_n), e->stream); break;
                case K_ENVELOPE: launch_envelope(d_jobs, nj, st.max_n, stream_grid_x(st.max_n), e->stream); break;
                case K_SEQSUM:
                    if (st.max_n < 32768 || e->cfg.use_fft == 5) {   // short chains (5: test switch): the plain walk
                        launch_seqsum(d_jobs, nj, e->stream);
                    } else {
                        // chunk-parallel evaluation of the same chain (seqsum.cu), one job per component
                        std::vector<SeqJob> sq;
                        for (const SigJob &j : st.jobs) {
                            const float *planes[2] = {j.q_re, j.q_im};
                            for (int c = 0; c < 2; c++) {
                                SeqJob q{};
                                q.x = planes[c]; q.n = j.n; q.out = j.stats + (c == 0 ? ST_DC_RE : ST_DC_IM);
                                if (q.x) {
                                    void *scratch = nullptr;
                                    if ((rc = alloc(e, &scratch, seqsum_scratch_bytes(j.n)))) return rc;
                                    seqsum_carve(q, scratch);
                                }
                                sq.push_back(q);
                            }
                        }
                        const SeqJob *d_sq = nullptr;
                        if ((rc = upload(e, sq, &d_sq))) return rc;
                        launch_seqsum_chunked(d_sq, (int)sq.size(), st.max_n, e->stream);
                        count_launch(e, 3);
                    }
                    break;
                case K_BOXCAR: launch_boxcar(d_jobs, nj, st.max_n, 0, e->stream); break;
                case K_BOXCAR_SMALL: {
                    const int sp = span_begin(e, SPAN_BOXCAR);
                    launch_boxcar_small(d_jobs, nj, st.max_n, e->stream);
                    span_end(e, sp);
                    for (const SigJob &j : st.jobs) e->st.boxcar_samples += j.n;
                    break;
                }
                case K_BOXCAR_SLIDE: launch_boxcar_slide(d_jobs, nj, st.max_n, e->stream); break;
                case K_NOTCH: launch_notch_combine(d_jobs, nj, st.max_n, e->stream); break;
                case K_DECIMATE: launch_decimate(d_jobs, nj, st.max_n, e->stream); break;
                case K_WEAK_FUSED: launch_weak_fused(d_jobs, nj, st.max_n, e->stream); break;
            }
            count_launch(e);
        }
    }
    return TDOA_OK;
}

inline int decimation(const tdoa_engine *e) { return e->cfg.mode == TDOA_MODE_EXTENDED && e->cfg.decimate > 1 ? e->cfg.decimate : 1; }

// shipped binary (ELF 0x49cd40): > 0.01 strong, > 0.001 moderate, else weak
inline int binary_branch(double power0) { return power0 > 0.01 ? 0 : (power0 > 0.001 ? 1 : 2); }

// Preprocess every signal (preprocessSignal, processor.go:469-499 / ELF 0x49cd40).
// On return out_re/out_im/stats of each signal are valid on the stream.
// allow_defer: when every signal runs the speculative fused kernel, do not wait for the
// powers at all -- assume the "strong FM" branch, queue the whole pipeline, and leave
// the check to the caller (verify_deferred), which reads the statistics back at the
// call's final synchronisation and redoes the group if a guess was wrong.
int preprocess(tdoa_engine *e, std::vector<Sig> &sigs, bool allow_defer = false)
{
    if (sigs.empty()) return TDOA_OK;
    const int ns = (int)sigs.size();
    i64 max_n = 0;
    for (auto &s : sigs) max_n = std::max(max_n, s.n);
    const int gx = stream_grid_x(max_n);
    const int gmax = std::max(std::max(gx, boxcar_grid_x(max_n)), fast_grid_x(max_n));
    double *d_stats = nullptr, *d_partials = nullptr;
    unsigned *d_counters = nullptr;
    int rc;
    if ((rc = alloc_t(e, &d_stats, (size_t)ns * ST_COUNT))) return rc;
    if ((rc = alloc_t(e, &d_partials, (size_t)ns * 3 * gmax))) return rc;   // k_raw_stats reduces three sums
    if ((rc = alloc_t(e, &d_counters, (size_t)ns))) return rc;
    CU(cudaMemsetAsync(d_stats, 0, (size_t)ns * ST_COUNT * sizeof(double), e->stream));
    CU(cudaMemsetAsync(d_counters, 0, (size_t)ns * sizeof(unsigned), e->stream));
    for (int i = 0; i < ns; i++) {
        sigs[i].stats = d_stats + (size_t)i * ST_COUNT;
        sigs[i].partials = d_partials + (size_t)i * 3 * gmax;
        sigs[i].counter = d_counters + i;
    }
    // ---- initial power (selects the branch).  In the shipped binary's modes a capture
    // that was "strong FM" last time is assumed to be so again: its power pass is fused
    // with the discriminator (one read of the raw bytes); a wrong guess only costs the
    // discarded demod output.
    const int gmax2 = std::max(gmax, fast_grid_x(max_n));
    (void)gmax2;
    {
        std::vector<SigJob> pjobs, fjobs;
        const bool mode_raw_stats = e->cfg.mode == TDOA_MODE_EXTENDED && e->cfg.use_fft != 6;   // 6: test switch, the four-kernel chain
        // signals whose capture is still arriving (tdoa_load_u8_pinned): the discriminator
        // follows the copy chunk by chunk, every launch waiting for one chunk only
        struct Follow { SigJob job; cudaEvent_t wait; i64 len; int sig; bool last; int n_sub; double *sums; };
        std::vector<Follow> follow;
        for (size_t si = 0; si < sigs.size(); si++) {
            Sig &s = sigs[si];
            const bool spec = e->cfg.mode != TDOA_MODE_SOURCE && s.src.raw && s.n >= 2 &&
                              (s.memo < 0 || e->branch_memo[s.memo] <= 0);
            s.fused = spec;
            Station *stn = s.station >= 0 ? &e->stations[s.station] : nullptr;
            const bool arriving = stn && !stn->chunks[s.kind].empty();
            if (spec) {
                if ((rc = ensure_plane(e, s, 0, false))) return rc;
                SigJob j = base_job(s);
                j.p_re = s.plane[0][0];
                if (arriving && !e->cfg.fast_demod) {
                    const auto &ch = stn->chunks[s.kind];
                    double *sums = nullptr;
                    if ((rc = alloc_t(e, &sums, 2 * ch.size()))) return rc;
                    i64 done = 0;
                    int n_sub = 0;
                    const size_t first = follow.size();
                    for (const CopyChunk &c : ch) {
                        const i64 avail = std::max<i64>(0, std::min<i64>(s.n, c.q_end - s.q0));
                        // a tile reads one 32-bit word past its end: stay 8 samples behind the copy
                        const i64 upto = avail == s.n ? s.n : std::max<i64>(0, (avail - 8) / 4096 * 4096);
                        if (upto <= done) continue;
                        Follow f{j, c.landed, upto - done, (int)si, false, 0, sums};
                        f.job.i_begin = done; f.job.i_end = upto; f.job.chunk_out = sums + 2 * n_sub;
                        follow.push_back(f);
                        done = upto;
                        n_sub++;
                        if (done == s.n) break;
                    }
                    follow.back().last = true;
                    for (size_t k = first; k < follow.size(); k++) follow[k].n_sub = n_sub;
                } else {
                    if (arriving && (rc = wait_kind(e, *stn, s.kind))) return rc;
                    fjobs.push_back(j);
                }
            } else {
                if (arriving && (rc = wait_kind(e, *stn, s.kind))) return rc;
                pjobs.push_back(base_job(s));
                s.raw_sums = mode_raw_stats;
            }
        }
        if (!follow.empty()) {
            std::vector<SigJob> jobs;
            for (const Follow &f : follow) jobs.push_back(f.job);
            const SigJob *d_jobs = nullptr;
            if ((rc = upload(e, jobs, &d_jobs))) return rc;
            for (size_t k = 0; k < follow.size(); k++) {
                const Follow &f = follow[k];
                CU(cudaStreamWaitEvent(e->stream, f.wait, 0));
                const int sp = span_begin(e, SPAN_DEMOD);
                launch_demod_fused(d_jobs + k, 1, f.len, 0, e->stream);
                span_end(e, sp);
                e->st.demod_samples += f.len;
                count_launch(e);
                if (f.last) {
                    launch_demod_finish(f.sums, f.n_sub, sigs[f.sig].n, sigs[f.sig].stats, e->stream);
                    count_launch(e);
                }
            }
        }
        if (!pjobs.empty()) {
            const SigJob *d_jobs = nullptr;
            if ((rc = upload(e, pjobs, &d_jobs))) return rc;
            // EXTENDED: power and both DC sums from one vectorised read of the bytes (k_weak_fused then needs
            // no unpacked planes); the other modes keep k_power, whose partition the golden digits were taken with
            if (mode_raw_stats) launch_raw_stats(d_jobs, (int)pjobs.size(), max_n, e->stream);
            else launch_power(d_jobs, (int)pjobs.size(), max_n, gx, e->stream);
            count_launch(e);
        }
        if (!fjobs.empty()) {
            const SigJob *d_jobs = nullptr;
            if ((rc = upload(e, fjobs, &d_jobs))) return rc;
            const int sp = span_begin(e, SPAN_DEMOD);
            launch_demod_fused(d_jobs, (int)fjobs.size(), max_n, e->cfg.fast_demod, e->stream);
            span_end(e, sp);
            for (const SigJob &j : fjobs) e->st.demod_samples += j.n;
            count_launch(e);
        }
        const bool defer = allow_defer && pjobs.empty();
        (void)follow;
        if (defer) {
            for (auto &s : sigs) s.deferred = true;
        } else {
            std::vector<double> h_stats((size_t)ns * ST_COUNT);
            CU(cudaMemcpyAsync(h_stats.data(), d_stats, h_stats.size() * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            CU(cudaStreamSynchronize(e->stream));
            for (int i = 0; i < ns; i++) sigs[i].power0 = h_stats[(size_t)i * ST_COUNT + ST_POWER0];
        }
    }
    // ---- per-branch pipelines
    const int mode = e->cfg.mode;
    Pipeline pl;
    for (auto &s : sigs) {
        if (s.n == 0) { s.branch = 0; continue; }
        if (mode == TDOA_MODE_SOURCE) {
            const bool weak = s.power0 < 0.001;  // processor.go:476
            s.branch = weak ? 2 : 0;
            for (int k = 0; k < (weak ? 4 : 2); k++)
                if ((rc = ensure_plane(e, s, k, true))) return rc;
            SigJob u = base_job(s);
            u.p_re = s.plane[0][0]; u.p_im = s.plane[0][1];
            size_t g = 0;
            pl.add(g++, K_UNPACK, u);
            if (wants_seq_dc(e, s.n)) pl.add(g, K_SEQSUM, seqsum_job(s, 0, true));
            g++;
            if (!weak) {
                // processor.go:485-495  DC -> BP(500, 50k) -> LP(100) -> normalise
                pl.add(g++, K_BOXCAR, box_job(s, 0, 1, true, cutoff_window(500.0), BOX_HP, true, false));
                pl.add(g++, K_BOXCAR, box_job(s, 1, 0, true, cutoff_window(50000.0), BOX_LP, false, false));
                pl.add(g++, K_BOXCAR, box_job(s, 0, 1, true, 100, BOX_LP, false, true));
                s.out_re = s.plane[1][0]; s.out_im = s.plane[1][1];
            } else {
                // processor.go:437-466  enhanceWeakSignal; planes: 0 = scratch T1, 1 = X, 2 = Y, 3 = T2
                pl.add(g++, K_BOXCAR, box_job(s, 0, 1, true, 1, BOX_LP, true, false));  // X = s - dc
                // notch 60 Hz / 5 Hz: band = LP(62.5)(HP(57.5)(X)); Y = X - 0.8 band
                pl.add(g++, K_BOXCAR, box_job(s, 1, 0, true, cutoff_window(57.5), BOX_HP, false, false));
                pl.add(g++, K_BOXCAR, box_job(s, 0, 3, true, cutoff_window(62.5), BOX_LP, false, false));
                pl.add(g++, K_NOTCH, notch_job(s, 1, 3, 2));
                // notch 120 Hz / 5 Hz: X = Y - 0.8 band
                pl.add(g++, K_BOXCAR, box_job(s, 2, 0, true, cutoff_window(117.5), BOX_HP, false, false));
                pl.add(g++, K_BOXCAR, box_job(s, 0, 3, true, cutoff_window(122.5), BOX_LP, false, false));
                pl.add(g++, K_NOTCH, notch_job(s, 2, 3, 1));
                // notch 1 MHz / 50 kHz: hi clamps to fs/2 so only HP(975 kHz) applies; Y = X - 0.8 band
                pl.add(g++, K_BOXCAR, box_job(s, 1, 0, true, cutoff_window(975000.0), BOX_HP, false, false));
                pl.add(g++, K_NOTCH, notch_job(s, 1, 0, 2));
                // BP(100, 40k): X = LP(40k)(HP(100)(Y))
                pl.add(g++, K_BOXCAR, box_job(s, 2, 0, true, cutoff_window(100.0), BOX_HP, false, false));
                pl.add(g++, K_BOXCAR, box_job(s, 0, 1, true, cutoff_window(40000.0), BOX_LP, false, false));
                // LP(window 50) + power: Y
                pl.add(g++, K_BOXCAR, box_job(s, 1, 2, true, 50, BOX_LP, false, true));
                s.out_re = s.plane[2][0]; s.out_im = s.plane[2][1];
            }
        } else {
            // shipped binary (ELF 0x49cd40): > 0.01 strong, > 0.001 moderate, else weak
            s.branch = s.deferred ? 0 : binary_branch(s.power0);
            size_t g = 0;
            if (s.memo >= 0 && !s.deferred) e->branch_memo[s.memo] = (int8_t)s.branch;
            if (s.branch == 0) {
                const bool cplx = s.n < 2;  // convertToInstantaneousFrequency returns its input for n < 2
                if ((rc = ensure_plane(e, s, 0, cplx)) || (rc = ensure_plane(e, s, 1, cplx))) return rc;
                if (!s.fused) {
                    SigJob u = base_job(s);
                    u.p_re = s.plane[0][0]; u.p_im = s.plane[0][1];
                    pl.add(g, cplx ? K_UNPACK : K_DEMOD, u);
                }
                g++;
                if (wants_seq_dc(e, s.n)) pl.add(g, K_SEQSUM, seqsum_job(s, 0, cplx));
                g++;
                pl.add(g++, cplx ? K_BOXCAR : K_BOXCAR_SMALL, box_job(s, 0, 1, cplx, 10, BOX_LP, true, true));
                s.out_re = s.plane[1][0]; s.out_im = s.plane[1][1];
            } else if (s.branch == 1) {
                if ((rc = ensure_plane(e, s, 0, false)) || (rc = ensure_plane(e, s, 1, false))) return rc;
                SigJob u = base_job(s);
                u.p_re = s.plane[0][0];
                pl.add(g++, K_ENVELOPE, u);
                if (wants_seq_dc(e, s.n)) pl.add(g, K_SEQSUM, seqsum_job(s, 0, false));
                g++;
                pl.add(g++, K_BOXCAR, box_job(s, 0, 1, false, 1, BOX_LP, true, true));
                s.out_re = s.plane[1][0]; s.out_im = nullptr;
            } else {
                const int w_hp = cutoff_window(100.0), w_lp = cutoff_window(200000.0);
                if (mode == TDOA_MODE_EXTENDED && s.raw_sums && s.src.raw && !wants_seq_dc(e, s.n) && w_hp >= 3 && w_lp >= 3 &&
                    w_hp / 2 <= weak_fused_max_half_wide() && w_lp / 2 <= weak_fused_max_half_small()) {
                    // the whole chain in one pass over the bytes (preprocess_weak.cu); the imaginary plane only
                    // where somebody reads it (the correlators of this revision take real parts only)
                    const bool im = s.need_im || decimation(e) > 1;
                    if ((rc = ensure_plane(e, s, 0, im))) return rc;
                    SigJob u = base_job(s);
                    u.p_re = s.plane[0][0]; u.p_im = im ? s.plane[0][1] : nullptr;
                    u.window = w_hp; u.window2 = w_lp;
                    pl.add(g++, K_WEAK_FUSED, u);
                    s.out_re = s.plane[0][0]; s.out_im = u.p_im;
                    continue;
                }
                if ((rc = ensure_plane(e, s, 0, true)) || (rc = ensure_plane(e, s, 1, true))) return rc;
                SigJob u = base_job(s);
                u.p_re = s.plane[0][0]; u.p_im = s.plane[0][1];
                pl.add(g++, K_UNPACK, u);
                if (wants_seq_dc(e, s.n)) pl.add(g, K_SEQSUM, seqsum_job(s, 0, true));
                g++;
                // removeDC -> bandpass(100 Hz, 200 kHz) -> normalise.  The 1001-tap high-pass: tap by tap
                // in the reference's f32 order where its digits are at stake (BINARY); EXTENDED, whose
                // arithmetic is the engine's own, takes the window sums from an f64 prefix sum
                pl.add(g++, mode == TDOA_MODE_EXTENDED ? K_BOXCAR_SLIDE : K_BOXCAR,
                       box_job(s, 0, 1, true, cutoff_window(100.0), BOX_HP, true, false));
                pl.add(g++, K_BOXCAR, box_job(s, 1, 0, true, cutoff_window(200000.0), BOX_LP, false, true));
                s.out_re = s.plane[0][0]; s.out_im = s.plane[0][1];
            }
        }
    }
    // EXTENDED mode, decimate = D > 1: the mode's chain, then the decimating box-car; the
    // correlators see n / D samples at fs / D
    const int D = decimation(e);
    if (D > 1) {
        const size_t last = pl.stages.size();
        for (auto &s : sigs) {
            s.n_out = s.n / D;
            if (s.n == 0) continue;
            SigJob j = base_job(s);
            j.q_re = s.out_re; j.q_im = s.out_im;
            float *dre = nullptr, *dim = nullptr;
            if ((rc = alloc_t(e, &dre, (size_t)std::max<i64>(s.n_out, 1)))) return rc;
            if (s.out_im && (rc = alloc_t(e, &dim, (size_t)std::max<i64>(s.n_out, 1)))) return rc;
            j.p_re = dre; j.p_im = dim;
            j.window = D; j.want_power = 1;
            pl.add(last, K_DECIMATE, j);
            s.out_re = dre; s.out_im = dim;
        }
    }
    return run_pipeline(e, pl);
}

// ---------------------------------------------------------------- correlation

struct CorrPlan {
    int group = 0;   // pairs of one group (window) may share transforms in a tile
    PairJob job{};
    PairJob job2{};  // sanity re-search with a different template length (rare)
    bool need2 = false;
    PeakJob peak{};
};

// whole blocks of the reference's loop `for bs = 0; bs < tl - B; bs += B`
i64 whole_blocks(i64 tl, i64 B)
{
    if (B <= 0 || tl <= B) return 0;
    return (tl - B + B - 1) / B;
}

// exact time-domain evaluation of every lag (reference order), then the peak scan
int run_brute(tdoa_engine *e, std::vector<CorrPlan *> &plans)
{
    if (plans.empty()) return TDOA_OK;
    int rc;
    std::vector<PairJob> jobs, jobs2;
    std::vector<PeakJob> peaks;
    i64 max_nb = 0, max_nb2 = 0;
    int max_lags = 0, max_lags2 = 0;
    for (CorrPlan *pl : plans) {
        PairJob &J = pl->job;
        PeakJob &K = pl->peak;
        K.flags |= TDOA_PEAK_BRUTE;
        if (K.n_lags > 0) {
            if ((rc = alloc_t(e, &J.blocksums, (size_t)std::max<i64>(J.nb, 1) * J.n_lags))) return rc;
            if ((rc = alloc_t(e, &J.corr, (size_t)J.n_lags))) return rc;
            K.corr = J.corr; K.corr2 = J.corr;
            K.n_lags2 = J.n_lags;
            max_nb = std::max(max_nb, J.nb);
            max_lags = std::max(max_lags, J.n_lags);
            if (pl->need2) {
                PairJob &J2 = pl->job2;
                if ((rc = alloc_t(e, &J2.blocksums, (size_t)std::max<i64>(J2.nb, 1) * J2.n_lags))) return rc;
                if ((rc = alloc_t(e, &J2.corr, (size_t)J2.n_lags))) return rc;
                K.corr2 = J2.corr; K.n_lags2 = J2.nb > 0 ? J2.n_lags : 0;
                max_nb2 = std::max(max_nb2, J2.nb);
                max_lags2 = std::max(max_lags2, J2.n_lags);
                jobs2.push_back(J2);
            }
            jobs.push_back(J);
        }
        peaks.push_back(K);
    }
    if (!jobs.empty()) {
        const PairJob *d_jobs = nullptr;
        if ((rc = upload(e, jobs, &d_jobs))) return rc;
        if (max_nb > 0) { launch_corr_brute(d_jobs, (int)jobs.size(), max_nb, max_lags, e->stream); count_launch(e); }
        launch_corr_finalize(d_jobs, (int)jobs.size(), max_lags, e->stream);
        count_launch(e);
        e->st.brute_pairs += (int64_t)jobs.size();
    }
    if (!jobs2.empty()) {
        const PairJob *d_jobs = nullptr;
        if ((rc = upload(e, jobs2, &d_jobs))) return rc;
        if (max_nb2 > 0) { launch_corr_brute(d_jobs, (int)jobs2.size(), max_nb2, max_lags2, e->stream); count_launch(e); }
        launch_corr_finalize(d_jobs, (int)jobs2.size(), max_lags2, e->stream);
        count_launch(e);
    }
    const PeakJob *d_peaks = nullptr;
    if ((rc = upload(e, peaks, &d_peaks))) return rc;
    launch_peak(d_peaks, (int)peaks.size(), e->stream);
    count_launch(e);
    return TDOA_OK;
}

// FFT candidate search + exact evaluation of the candidates (xcorr_fft.cu)
int run_fft(tdoa_engine *e, std::vector<CorrPlan *> &plans)
{
    if (plans.empty()) return TDOA_OK;
    int rc;
    const int np = (int)plans.size();
    std::vector<FftJob> fjobs;
    std::vector<SelJob> sjobs(np);
    std::vector<CandJob> cjobs(np);
    std::vector<PairJob> pjobs(np);
    std::vector<PeakJob> kjobs(np);
    // ---- tiles: pairs of one group with identical geometry share transforms.  Rows are
    // the distinct template planes, columns the distinct signal planes; rows and columns
    // are taken two at a time, and a tile carries the (<= 4) pairs that exist among them.
    struct Tile { int plan[4]; const float *t[2]; const float *s[2]; };
    std::vector<Tile> tiles;
    struct SpecGroup { std::vector<int> plans; std::vector<const float *> rows, cols; };
    std::vector<SpecGroup> spec_groups;
    std::vector<char> spec_plan(np, 0);
    const bool tiled = e->cfg.use_fft != 2;
    {
        std::vector<char> done(np, 0);
        for (int p0 = 0; p0 < np; p0++) {
            if (done[p0]) continue;
            const PairJob &K0 = plans[p0]->job;
            std::vector<int> grp;  // plans with the geometry of p0
            for (int p = p0; p < np; p++) {
                const PairJob &K = plans[p]->job;
                if (!done[p] && plans[p]->group == plans[p0]->group && K.t_off == K0.t_off && K.n_t == K0.n_t &&
                    K.sl == K0.sl && K.lag0 == K0.lag0 && K.n_lags == K0.n_lags) {
                    grp.push_back(p);
                    done[p] = 1;
                }
            }
            if (!tiled) {
                for (int p : grp) tiles.push_back(Tile{{p, -1, -1, -1}, {plans[p]->job.t_re, plans[p]->job.t_re},
                                                       {plans[p]->job.s_re, plans[p]->job.s_re}});
                continue;
            }
            std::vector<const float *> rows;
            for (int p : grp)
                if (std::find(rows.begin(), rows.end(), plans[p]->job.t_re) == rows.end()) rows.push_back(plans[p]->job.t_re);
            // many pairs on few stations: transform each station once and form the pairs from
            // the parked spectra (xcorr_spec.cu) instead of 2 x 2 tiles
            if ((int)grp.size() >= kSpecMinPairs && K0.n_lags < kBigMinLags && e->cfg.use_fft != 4) {
                std::vector<const float *> cols;
                for (int p : grp)
                    if (std::find(cols.begin(), cols.end(), plans[p]->job.s_re) == cols.end()) cols.push_back(plans[p]->job.s_re);
                if ((rows.size() + 1) / 2 + (cols.size() + 1) / 2 <= (size_t)kSpecMaxPacked) {
                    SpecGroup G;
                    G.plans = grp; G.rows = rows; G.cols = cols;
                    spec_groups.push_back(G);
                    for (int p : grp) spec_plan[p] = 1;
                    continue;
                }
            }
            for (size_t r = 0; r < rows.size(); r += 2) {
                const float *tr[2] = {rows[r], r + 1 < rows.size() ? rows[r + 1] : rows[r]};
                std::vector<const float *> cols;
                for (int p : grp) {
                    const PairJob &K = plans[p]->job;
                    if ((K.t_re == tr[0] || K.t_re == tr[1]) && std::find(cols.begin(), cols.end(), K.s_re) == cols.end())
                        cols.push_back(K.s_re);
                }
                for (size_t c = 0; c < cols.size(); c += 2) {
                    Tile T{{-1, -1, -1, -1}, {tr[0], tr[1]}, {cols[c], c + 1 < cols.size() ? cols[c + 1] : cols[c]}};
                    bool any = false;
                    for (int p : grp) {
                        const PairJob &K = plans[p]->job;
                        for (int a = 0; a < 2; a++)
                            for (int b = 0; b < 2; b++)
                                if (K.t_re == T.t[a] && K.s_re == T.s[b] && T.plan[2 * a + b] < 0 &&
                                    !(a == 1 && T.t[1] == T.t[0]) && !(b == 1 && T.s[1] == T.s[0])) {
                                    T.plan[2 * a + b] = p;
                                    any = true;
                                }
                    }
                    if (any) tiles.push_back(T);
                }
            }
        }
    }
    // wide lag ranges go through the 2^21-point transform in global memory (xcorr_big.cu)
    std::vector<char> big_plan(np, 0), big_tile(tiles.size(), 0);
    if (tiled && e->cfg.use_fft != 3) {
        for (size_t ti = 0; ti < tiles.size(); ti++) {
            int lead = -1;
            for (int q = 0; q < 4; q++) if (tiles[ti].plan[q] >= 0) lead = tiles[ti].plan[q];
            const PairJob &K = plans[lead]->job;
            if (K.n_lags >= kBigMinLags && (i64)K.n_lags <= kBigN / 2) {
                big_tile[ti] = 1;
                for (int q = 0; q < 4; q++) if (tiles[ti].plan[q] >= 0) big_plan[tiles[ti].plan[q]] = 1;
            }
        }
    }
    // lag chunks
    int n_fft_jobs = 0, n_tile_jobs = 0;
    for (int p = 0; p < np; p++)
        if (!big_plan[p] && !spec_plan[p]) n_fft_jobs += (plans[p]->job.n_lags + kLagW - 1) / kLagW;
    for (size_t ti = 0; ti < tiles.size(); ti++) {
        if (big_tile[ti]) continue;
        const Tile &T = tiles[ti];
        int p = -1;
        for (int q = 0; q < 4; q++) if (T.plan[q] >= 0) p = T.plan[q];
        n_tile_jobs += (plans[p]->job.n_lags + kLagW - 1) / kLagW;
    }
    // per-pair kernel: 2 CTAs per SM; tile kernel: 1 CTA (512 threads) per SM
    const int cta_budget = tiled ? std::max(1, e->sm_count / std::max(1, n_tile_jobs))
                                 : std::max(1, 2 * e->sm_count / std::max(1, n_fft_jobs));
    int max_cta = 0;
    i64 max_nb = 0;
    std::vector<int> first_job(np, 0);  // index into fjobs of the plan's first lag chunk
    // one arena for the per-pair scratch (16 stations x 33 windows = 3960 pairs: tens of
    // thousands of separate stream-ordered allocations would cost more host time than the kernels)
    auto up256 = [](size_t b) { return (b + 255) & ~size_t(255); };
    size_t arena_bytes = 0;
    for (int p = 0; p < np; p++) {
        const PairJob &J = plans[p]->job;
        arena_bytes += up256((size_t)J.n_lags * sizeof(float)) + up256(sizeof(float)) + up256(kMaxCand * sizeof(int)) +
                       up256(sizeof(int)) + up256((size_t)kMaxCand * std::max<i64>(J.nb, 1) * sizeof(double));
        if (spec_plan[p]) {
            arena_bytes += (size_t)((J.n_lags + 2047) / 2048) * up256((size_t)kFftBins * sizeof(float2));
        } else if (!big_plan[p]) {
            const int n_chunks = (J.n_lags + kLagW - 1) / kLagW;
            const int n_seg = (int)((J.n_t + kSeg - 1) / kSeg);
            const int n_cta = std::max(1, std::min(n_seg, cta_budget));
            arena_bytes += (size_t)n_chunks * (up256(fft_partials_bytes(n_cta)) + up256((size_t)kFftBins * sizeof(float2)));
        }
    }
    char *arena = nullptr;
    if ((rc = alloc(e, reinterpret_cast<void **>(&arena), arena_bytes))) return rc;
    size_t arena_off = 0;
    auto take = [&](size_t bytes) { void *q = arena + arena_off; arena_off += up256(bytes); return q; };
    for (int p = 0; p < np; p++) {
        CorrPlan *pl = plans[p];
        PairJob &J = pl->job;
        PeakJob &K = pl->peak;
        float *d_approx = static_cast<float *>(take((size_t)J.n_lags * sizeof(float)));
        float *d_amax = static_cast<float *>(take(sizeof(float)));
        int *d_cand = static_cast<int *>(take(kMaxCand * sizeof(int)));
        int *d_ncand = static_cast<int *>(take(sizeof(int)));
        J.blocksums = static_cast<double *>(take((size_t)kMaxCand * std::max<i64>(J.nb, 1) * sizeof(double)));
        first_job[p] = (int)fjobs.size();
        for (int c0 = 0; c0 < J.n_lags && !big_plan[p] && !spec_plan[p]; c0 += kLagW) {
            FftJob F{};
            F.t = J.t_re; F.s = J.s_re; F.t_stats = J.t_stats; F.s_stats = J.s_stats;
            F.t_off = J.t_off; F.n_t = J.n_t; F.sl = J.sl;
            F.s_off = (i64)J.lag0 + c0;
            F.n_lags = std::min(kLagW, J.n_lags - c0);
            F.n_seg = (int)((J.n_t + kSeg - 1) / kSeg);
            F.n_cta = std::max(1, std::min(F.n_seg, cta_budget));
            F.partials = static_cast<float2 *>(take(fft_partials_bytes(F.n_cta)));
            F.spectrum = static_cast<float2 *>(take((size_t)kFftBins * sizeof(float2)));
            F.approx = d_approx + c0;
            max_cta = std::max(max_cta, F.n_cta);
            fjobs.push_back(F);
            e->st.fft_pair_samples += J.n_t;
        }
        SelJob &S = sjobs[p];
        S.approx = d_approx; S.n_lags = J.n_lags; S.sanity = K.sanity;
        S.neighbours = J.variant == CORR_EXTENDED; S.max_cand = kMaxCand;
        S.tol = 2e-5f;
        S.cand = d_cand; S.n_cand = d_ncand; S.approx_max = d_amax;
        S.t_stats = J.t_stats; S.s_stats = J.s_stats;
        CandJob &C = cjobs[p];
        C.cand = d_cand; C.n_cand = d_ncand; C.max_cand = kMaxCand; C.approx = d_approx; C.blocksums = J.blocksums;
        pjobs[p] = J;
        kjobs[p] = K;
        max_nb = std::max(max_nb, J.nb);
    }
    std::vector<TileJob> tjobs;
    if (tiled) {
        for (size_t ti = 0; ti < tiles.size(); ti++) {
            if (big_tile[ti]) continue;
            const Tile &T = tiles[ti];
            int lead = -1;
            for (int q = 0; q < 4; q++) if (T.plan[q] >= 0) lead = T.plan[q];
            const PairJob &K = plans[lead]->job;
            const int n_chunks = (K.n_lags + kLagW - 1) / kLagW;
            for (int ci = 0; ci < n_chunks; ci++) {
                const FftJob &F0 = fjobs[first_job[lead] + ci];
                TileJob TJ{};
                TJ.t0 = T.t[0]; TJ.t1 = T.t[1]; TJ.s0 = T.s[0]; TJ.s1 = T.s[1];
                TJ.t_off = F0.t_off; TJ.n_t = F0.n_t; TJ.sl = F0.sl; TJ.s_off = F0.s_off;
                TJ.n_seg = F0.n_seg; TJ.n_cta = F0.n_cta;
                for (int q = 0; q < 4; q++) TJ.partials[q] = T.plan[q] >= 0 ? fjobs[first_job[T.plan[q]] + ci].partials : nullptr;
                tjobs.push_back(TJ);
            }
        }
    }
    const FftJob *d_f = nullptr;
    const SelJob *d_s = nullptr;
    const CandJob *d_c = nullptr;
    const PairJob *d_p = nullptr;
    const PeakJob *d_k = nullptr;
    if ((rc = upload(e, fjobs, &d_f)) || (rc = upload(e, sjobs, &d_s)) || (rc = upload(e, cjobs, &d_c)) ||
        (rc = upload(e, pjobs, &d_p)) || (rc = upload(e, kjobs, &d_k)))
        return rc;
    const TileJob *d_t = nullptr;
    if (tiled && (rc = upload(e, tjobs, &d_t))) return rc;
    const int sp_fft = span_begin(e, SPAN_FFT);
    {
        const int sp_seg = span_begin(e, SPAN_FFT_SEG);
        if (tiled) launch_fft_tiles(d_t, (int)tjobs.size(), max_cta, e->d_tw, e->stream);
        else launch_fft_segments(d_f, (int)fjobs.size(), max_cta, e->d_tw, e->stream);
        span_end(e, sp_seg);
    }
    launch_fft_reduce(d_f, (int)fjobs.size(), e->stream);
    launch_fft_finish(d_f, (int)fjobs.size(), e->d_tw, e->stream);
    // ---- station-spectra groups: units of (group, lag chunk), in batches that share one
    // spectra buffer; the pair spectra go straight to the finish kernel
    if (!spec_groups.empty()) {
        struct Unit { int grp; int c0, lw, seg, n_seg; size_t spec_elems; };
        std::vector<Unit> units;
        std::vector<FftJob> sf;                       // finish jobs of the spec plans, unit by unit
        std::vector<std::vector<int>> unit_fjob;      // per unit: index into sf of each plan of the group
        for (size_t gi = 0; gi < spec_groups.size(); gi++) {
            const SpecGroup &G = spec_groups[gi];
            const PairJob &K = plans[G.plans[0]]->job;
            const int lw = K.n_lags <= 2048 ? 2048 : 4096;   // lags per chunk; segment = 8192 - lw samples
            const int n_pk = (int)((G.rows.size() + 1) / 2 + (G.cols.size() + 1) / 2);
            for (int c0 = 0; c0 < K.n_lags; c0 += lw) {
                Unit U;
                U.grp = (int)gi; U.c0 = c0; U.lw = std::min(lw, K.n_lags - c0); U.seg = kFftN - lw;
                U.n_seg = (int)std::max<i64>(1, (K.n_t + U.seg - 1) / U.seg);
                U.spec_elems = (size_t)U.n_seg * spec_seg_elems(2 * n_pk);
                std::vector<int> idx;
                for (int p : G.plans) {
                    const PairJob &J = plans[p]->job;
                    FftJob F{};
                    F.t = J.t_re; F.s = J.s_re; F.t_stats = J.t_stats; F.s_stats = J.s_stats;
                    F.t_off = J.t_off; F.n_t = J.n_t; F.sl = J.sl; F.s_off = (i64)J.lag0 + c0;
                    F.n_lags = U.lw; F.n_seg = U.n_seg; F.n_cta = 0; F.partials = nullptr;
                    F.spectrum = static_cast<float2 *>(take((size_t)kFftBins * sizeof(float2)));
                    F.approx = const_cast<float *>(sjobs[p].approx) + c0;
                    idx.push_back((int)sf.size());
                    sf.push_back(F);
                }
                unit_fjob.push_back(idx);
                units.push_back(U);
            }
        }
        size_t max_unit = 0;
        for (const Unit &U : units) max_unit = std::max(max_unit, U.spec_elems);
        const size_t budget_elems = std::max<size_t>(max_unit, ((size_t)18 << 30) / sizeof(float2));  // 18 GiB of parked spectra per batch
        float2 *spec_buf = nullptr;
        {
            size_t total = 0;
            for (const Unit &U : units) total += U.spec_elems;
            if ((rc = alloc_t(e, &spec_buf, std::min(total, budget_elems)))) return rc;
        }
        for (size_t u0 = 0; u0 < units.size();) {
            std::vector<SpecFftJob> fj;
            std::vector<SpecAccJob> aj;
            size_t used = 0;
            int max_seg = 0;
            size_t u1 = u0;
            while (u1 < units.size() && (u1 == u0 || used + units[u1].spec_elems <= budget_elems)) {
                const Unit &U = units[u1];
                const SpecGroup &G = spec_groups[U.grp];
                const PairJob &K = plans[G.plans[0]]->job;
                const int n_pk_t = (int)((G.rows.size() + 1) / 2), n_pk_s = (int)((G.cols.size() + 1) / 2);
                const int n_pk = n_pk_t + n_pk_s;
                float2 *spec = spec_buf + used;
                for (int m = 0; m < n_pk; m++) {
                    SpecFftJob F{};
                    const bool tpl = m < n_pk_t;
                    const std::vector<const float *> &src = tpl ? G.rows : G.cols;
                    const size_t a = (size_t)2 * (tpl ? m : m - n_pk_t);
                    F.x0 = src[a]; F.x1 = a + 1 < src.size() ? src[a + 1] : src[a];
                    F.stride = U.seg; F.n_seg = U.n_seg;
                    if (tpl) { F.base = K.t_off; F.lo = K.t_off; F.hi = K.t_off + K.n_t; F.seg_len = U.seg; }
                    else { F.base = (i64)K.lag0 + U.c0; F.lo = 0; F.hi = K.sl; F.seg_len = kFftN; }
                    F.out = spec; F.row0 = 2 * m; F.n_rows = 2 * n_pk;
                    fj.push_back(F);
                }
                // the pairs of the group as 4 x 4 register tiles over (template row, signal row); <= kSpecMaxTiles per job
                {
                    struct TileOut { int I, J; float2 *out[kSpecTile * kSpecTile]; };
                    std::vector<TileOut> tl;
                    for (size_t q = 0; q < G.plans.size(); q++) {
                        const PairJob &J = plans[G.plans[q]]->job;
                        const int tr = (int)(std::find(G.rows.begin(), G.rows.end(), J.t_re) - G.rows.begin());
                        const int sc = (int)(std::find(G.cols.begin(), G.cols.end(), J.s_re) - G.cols.begin());
                        const int I = tr / kSpecTile, Jb = sc / kSpecTile;
                        TileOut *T = nullptr;
                        for (auto &x : tl)
                            if (x.I == I && x.J == Jb) T = &x;
                        if (!T) {
                            tl.push_back(TileOut{I, Jb, {}});
                            T = &tl.back();
                            for (auto &o : T->out) o = nullptr;
                        }
                        T->out[kSpecTile * (tr % kSpecTile) + sc % kSpecTile] = sf[unit_fjob[u1][q]].spectrum;
                    }
                    for (size_t t0 = 0; t0 < tl.size(); t0 += kSpecMaxTiles) {
                        SpecAccJob A{};
                        A.spec = spec; A.n_rows = 2 * n_pk; A.n_seg = U.n_seg;
                        A.n_tiles = (int)std::min<size_t>(kSpecMaxTiles, tl.size() - t0);
                        for (int t = 0; t < A.n_tiles; t++) {
                            const TileOut &T = tl[t0 + t];
                            for (int a = 0; a < kSpecTile; a++) {
                                // rows beyond the group's stations: any valid row (their products have no output)
                                const int tr = std::min<int>(T.I * kSpecTile + a, (int)G.rows.size() - 1);
                                const int sc = std::min<int>(T.J * kSpecTile + a, (int)G.cols.size() - 1);
                                A.t_row[t][a] = (unsigned char)tr;
                                A.s_row[t][a] = (unsigned char)(2 * n_pk_t + sc);
                            }
                            for (int q = 0; q < kSpecTile * kSpecTile; q++) A.out[t][q] = T.out[q];
                        }
                        aj.push_back(A);
                    }
                }
                used += U.spec_elems;
                max_seg = std::max(max_seg, U.n_seg);
                u1++;
            }
            const SpecFftJob *d_fj = nullptr;
            const SpecAccJob *d_aj = nullptr;
            if ((rc = upload(e, fj, &d_fj)) || (rc = upload(e, aj, &d_aj))) return rc;
            launch_spec_fft(d_fj, (int)fj.size(), max_seg, e->d_tw, e->stream);
            launch_spec_acc(d_aj, (int)aj.size(), e->stream);
            count_launch(e, 2);
            u0 = u1;
        }
        const FftJob *d_sf = nullptr;
        if ((rc = upload(e, sf, &d_sf))) return rc;
        launch_fft_finish(d_sf, (int)sf.size(), e->d_tw, e->stream);
        count_launch(e);
    }
    // ---- big tiles, in batches that share four 16 MiB buffers per tile
    {
        std::vector<int> bt;
        for (size_t ti = 0; ti < tiles.size(); ti++) if (big_tile[ti]) bt.push_back((int)ti);
        const int kBatch = 48;
        const size_t buf_elems = (size_t)kBigN;
        float2 *pool = nullptr;
        if (!bt.empty() && (rc = alloc_t(e, &pool, (size_t)std::min<int>(kBatch, (int)bt.size()) * 4 * buf_elems))) return rc;
        for (size_t b0 = 0; b0 < bt.size(); b0 += kBatch) {
            const int nb_t = (int)std::min<size_t>(kBatch, bt.size() - b0);
            struct Geo { i64 t_off, n_t, sl, lag0, Ts; int n_lags, n_seg; };
            std::vector<Geo> geo(nb_t);
            int max_seg = 0;
            for (int k = 0; k < nb_t; k++) {
                const Tile &T = tiles[bt[b0 + k]];
                int lead = -1;
                for (int q = 0; q < 4; q++) if (T.plan[q] >= 0) lead = T.plan[q];
                const PairJob &K = plans[lead]->job;
                Geo &G = geo[k];
                G.t_off = K.t_off; G.n_t = K.n_t; G.sl = K.sl; G.lag0 = K.lag0; G.n_lags = K.n_lags;
                G.Ts = (kBigN - K.n_lags) & ~(i64)3;
                G.n_seg = (int)std::max<i64>(1, (K.n_t + G.Ts - 1) / G.Ts);
                max_seg = std::max(max_seg, G.n_seg);
            }
            auto buf = [&](int k, int which) { return pool + ((size_t)k * 4 + which) * buf_elems; };  // A, B, G0, G1
            for (int g = 0; g < max_seg; g++) {
                std::vector<BigColJob> cj;
                std::vector<BigRowJob> rj;
                std::vector<BigCrossJob> xj;
                for (int k = 0; k < nb_t; k++) {
                    const Geo &G = geo[k];
                    if (g >= G.n_seg) continue;
                    const Tile &T = tiles[bt[b0 + k]];
                    const i64 first = (i64)g * G.Ts;
                    BigColJob a{};
                    a.x0 = T.t[0]; a.x1 = T.t[1]; a.base = G.t_off + first; a.lo = 0;
                    a.hi = std::max<i64>(0, std::min<i64>(G.Ts, G.n_t - first)); a.out = buf(k, 0);
                    BigColJob b{};
                    b.x0 = T.s[0]; b.x1 = T.s[1]; b.base = G.lag0 + first;
                    b.lo = std::max<i64>(0, -b.base); b.hi = std::max<i64>(b.lo, std::min<i64>(kBigN, G.sl - b.base));
                    b.out = buf(k, 1);
                    cj.push_back(a); cj.push_back(b);
                    rj.push_back(BigRowJob{buf(k, 0), 0});
                    rj.push_back(BigRowJob{buf(k, 1), 0});
                    xj.push_back(BigCrossJob{buf(k, 0), buf(k, 1), buf(k, 2), buf(k, 3), g > 0 ? 1 : 0});
                }
                const BigColJob *d_cj = nullptr;
                const BigRowJob *d_rj = nullptr;
                const BigCrossJob *d_xj = nullptr;
                if ((rc = upload(e, cj, &d_cj)) || (rc = upload(e, rj, &d_rj)) || (rc = upload(e, xj, &d_xj))) return rc;
                launch_big_cols(d_cj, (int)cj.size(), e->d_tw, e->d_tw_fine, e->stream);
                launch_big_rows(d_rj, (int)rj.size(), e->d_tw, e->d_tw_fine, e->stream);
                launch_big_cross(d_xj, (int)xj.size(), e->stream);
                count_launch(e, 3);
            }
            std::vector<BigRowJob> irj;
            std::vector<BigOutJob> oj;
            for (int k = 0; k < nb_t; k++) {
                const Tile &T = tiles[bt[b0 + k]];
                for (int a = 0; a < 2; a++) {
                    const int q0 = T.plan[2 * a], q1 = T.plan[2 * a + 1];
                    if (q0 < 0 && q1 < 0) continue;
                    const int any = q0 >= 0 ? q0 : q1;
                    BigOutJob O{};
                    O.G = buf(k, 2 + a);
                    O.approx0 = q0 >= 0 ? const_cast<float *>(sjobs[q0].approx) : nullptr;
                    O.approx1 = q1 >= 0 ? const_cast<float *>(sjobs[q1].approx) : nullptr;
                    O.t_stats = plans[any]->job.t_stats;
                    O.s0_stats = q0 >= 0 ? plans[q0]->job.s_stats : plans[any]->job.s_stats;
                    O.s1_stats = q1 >= 0 ? plans[q1]->job.s_stats : plans[any]->job.s_stats;
                    O.n_t = geo[k].n_t; O.n_lags = geo[k].n_lags;
                    irj.push_back(BigRowJob{buf(k, 2 + a), 1});
                    oj.push_back(O);
                }
            }
            const BigRowJob *d_irj = nullptr;
            const BigOutJob *d_oj = nullptr;
            if ((rc = upload(e, irj, &d_irj)) || (rc = upload(e, oj, &d_oj))) return rc;
            launch_big_rows(d_irj, (int)irj.size(), e->d_tw, e->d_tw_fine, e->stream);
            launch_big_out(d_oj, (int)oj.size(), e->d_tw, e->stream);
            count_launch(e, 2);
        }
    }
    launch_select_candidates(d_s, np, e->stream);
    span_end(e, sp_fft);
    {
        const int sp = span_begin(e, SPAN_CAND);
        launch_corr_candidates(d_p, d_c, np, max_nb, e->stream);
        span_end(e, sp);
        for (const PairJob &J : pjobs) e->st.cand_pair_samples += J.n_t;
    }
    launch_peak_candidates(d_p, d_c, d_k, np, e->stream);
    count_launch(e, 6);
    e->st.fft_launches += 1;
    return TDOA_OK;
}

// optimistic = true: queue only -- the candidate-overflow check (and the lag-by-lag redo it may
// ask for) is left to the caller, who looks at the records' flags after its own synchronisation
int correlate(tdoa_engine *e, const std::vector<Sig> &sigs, const std::vector<Pair> &pairs, PeakRec *d_out,
              double *d_first = nullptr, bool optimistic = false)
{
    if (pairs.empty()) return TDOA_OK;
    const tdoa_config &cfg = e->cfg;
    const int np = (int)pairs.size();
    std::vector<CorrPlan> plans(np);
    std::vector<CorrPlan *> brute, viafft;
    for (int p = 0; p < np; p++) {
        const Sig &s1 = sigs[pairs[p].a], &s2 = sigs[pairs[p].b];
        CorrPlan &pl = plans[p];
        pl.group = pairs[p].group;
        PairJob &J = pl.job;
        PeakJob &K = pl.peak;
        K.out = d_out + p;
        K.first_corr = d_first ? d_first + p : nullptr;
        K.flags = ((uint32_t)s1.branch << 8) | ((uint32_t)s2.branch << 10);
        K.sanity = 0;
        K.lag_origin = 0;
        const i64 n1 = s1.n_out >= 0 ? s1.n_out : s1.n, n2 = s2.n_out >= 0 ? s2.n_out : s2.n;
        if (n1 == 0 || n2 == 0) {  // processor.go:622-625
            K.flags |= TDOA_PEAK_EMPTY;
            K.nb = 0; K.n_lags = 0; K.n_lags2 = 0; K.corr = K.corr2 = nullptr;
            K.variant = CORR_BINARY;
            brute.push_back(&pl);
            continue;
        }
        // processor.go:653-661: the shorter input is the template
        const Sig *tp = &s1, *sg = &s2;
        if (n1 > n2) { tp = &s2; sg = &s1; }
        const i64 tl = std::min(n1, n2), sl = std::max(n1, n2);
        J.t_re = tp->out_re; J.t_im = tp->out_im; J.t_stats = tp->stats;
        J.s_re = sg->out_re; J.s_im = sg->out_im; J.s_stats = sg->stats;
        J.sl = sl;
        J.lag0 = 0;
        J.t_off = 0;
        if (cfg.mode == TDOA_MODE_EXTENDED) {
            const i64 W = std::min(tl, sl), L = cfg.max_lag / decimation(e);
            const i64 n = W - 2 * L;
            J.variant = CORR_EXTENDED;
            J.t_off = L;
            J.n_t = n > 0 ? n : 0;
            J.block = 65536;   // partial-sum chunk of the exact evaluation (engine-defined mode: any grouping)
            J.nb = n > 0 ? (n + J.block - 1) / J.block : 0;
            J.n_lags = (int)(2 * L + 1);
            K.lag_origin = (int)-L;
        } else if (cfg.mode == TDOA_MODE_BINARY) {
            // ELF 0x49d6a0: equal lengths -> template shortened by maxLag
            const i64 tl_eff = (sl == tl) ? tl - cfg.max_lag : tl;
            i64 ml = std::min<i64>(cfg.max_lag, sl - tl_eff);
            if (ml <= 0) ml = 1;
            J.variant = CORR_BINARY;
            J.block = cfg.block_size;
            J.nb = whole_blocks(tl_eff, J.block);
            J.n_t = J.nb * J.block;
            J.n_lags = (int)ml;
            K.sanity = cfg.sanity_lag;
            if (K.sanity > 0 && ml > K.sanity + 1) {
                // ELF 0x49dda7: the re-search template is tl-2000 (hard-coded) for equal lengths
                const i64 tl2 = (sl == tl) ? tl - 2000 : tl;
                const i64 nb2 = whole_blocks(tl2, J.block);
                if (nb2 != J.nb) {
                    pl.need2 = true;
                    pl.job2 = J;
                    pl.job2.nb = nb2;
                    pl.job2.n_t = nb2 * J.block;
                    pl.job2.n_lags = K.sanity;
                }
            }
        } else {
            // processor.go:668-675
            i64 ml = std::min<i64>(cfg.max_lag, sl - tl);
            if (ml < 1) ml = 1;
            J.variant = CORR_SOURCE;
            J.block = cfg.block_size;
            J.nb = whole_blocks(tl, J.block);
            J.n_t = J.nb * J.block;
            J.n_lags = (int)ml;
        }
        K.n_lags = J.n_lags;
        K.n_lags2 = J.n_lags;
        K.nb = (int)J.nb;
        K.variant = J.variant;
        // the FFT path serves the real-valued correlators; a handful of lags is cheaper exactly
        const bool fft_ok = cfg.use_fft && J.variant != CORR_SOURCE && J.nb > 0 && J.n_lags > 8 && !pl.need2;
        (fft_ok ? viafft : brute).push_back(&pl);
    }
    int rc;
    if ((rc = run_brute(e, brute))) return rc;
    if (!viafft.empty()) {
        if ((rc = run_fft(e, viafft))) return rc;
        if (optimistic) return TDOA_OK;
        // candidate overflow (a flat correlation surface): redo those pairs lag by lag
        std::vector<PeakRec> h(np);
        CU(cudaMemcpyAsync(h.data(), d_out, (size_t)np * sizeof(PeakRec), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        std::vector<CorrPlan *> redo;
        for (CorrPlan *pl : viafft)
            if (h[pl->peak.out - d_out].flags & 0x10u) redo.push_back(pl);
        if ((rc = run_brute(e, redo))) return rc;
    }
    return TDOA_OK;
}

// ---------------------------------------------------------------- xcorr over windows

// What an optimistic (host-sync-free) pass over one signal kind leaves to be checked once
// the caller has synchronised: the statistics of its signals (branch guesses, the
// reference's diagnostics) and the first-pass correlations.
struct Pending {
    int kind = 0;
    std::vector<Sig> sigs;       // window 0 (the only window of an optimistic pass)
    double *d_first = nullptr;
    bool valid = false;
};

void stats_reset(tdoa_engine *e)
{
    e->st.ms_preprocess = e->st.ms_fft = e->st.ms_fft_seg = e->st.ms_exact = e->st.ms_total = 0.f;
    e->st.fft_launches = 0; e->st.fft_pair_samples = 0;
    e->st.ms_demod = e->st.ms_boxcar = e->st.ms_cand = 0.f;
    e->st.demod_launches = e->st.demod_samples = e->st.boxcar_launches = e->st.boxcar_samples = 0;
    e->st.cand_launches = e->st.cand_pair_samples = 0;
    e->ms_corr = 0.f;
    e->spans_used = 0;
}

// window 0 of the last pass over `kind`: what the reference prints (tdoa_xcorr_info)
void fill_info(tdoa_engine *e, int kind, const std::vector<Sig> &sigs, const double *h_stats, int S)
{
    e->info_sig[kind].assign(S, tdoa_signal_info{});
    for (int s = 0; s < S; s++) {
        tdoa_signal_info &I = e->info_sig[kind][s];
        const double *st = h_stats + (size_t)s * ST_COUNT;
        I.power0 = st[ST_POWER0]; I.dc_re = st[ST_DC_RE]; I.dc_im = st[ST_DC_IM]; I.power1 = st[ST_POWER1];
        I.branch = sigs[s].branch; I.n = sigs[s].n;
    }
}

// true: every speculated signal really was on the "strong FM" branch (memo updated either way)
bool verify_deferred(tdoa_engine *e, std::vector<Sig> &sigs, const double *h_stats)
{
    bool ok = true;
    for (size_t i = 0; i < sigs.size(); i++) {
        Sig &sg = sigs[i];
        if (!sg.deferred) continue;
        sg.power0 = h_stats[i * ST_COUNT + ST_POWER0];
        const int actual = sg.n == 0 ? 0 : binary_branch(sg.power0);
        if (sg.memo >= 0) e->branch_memo[sg.memo] = (int8_t)actual;
        ok &= actual == 0;
    }
    return ok;
}

// Validates the window arguments and fills the per-station window length.
int window_lengths(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows, int64_t hop,
                   std::vector<i64> &len)
{
    if (kind != TDOA_KIND_REF && kind != TDOA_KIND_TGT) return fail(e, TDOA_E_INVALID, "tdoa_xcorr: bad kind %d", kind);
    if (n_windows < 1 || win_start < 0 || win_len < 0 || (n_windows > 1 && hop <= 0))
        return fail(e, TDOA_E_INVALID, "tdoa_xcorr: bad window arguments");
    const int S = e->cfg.n_stations;
    for (int s = 0; s < S; s++)
        if (!e->stations[s].loaded) return fail(e, TDOA_E_STATE, "tdoa_xcorr: station %d has no capture loaded", s);
    len.assign(S, 0);
    for (int s = 0; s < S; s++) {
        const i64 n = signal_length(e->stations[s], kind, e->cfg.guard_samples);
        if (win_len == 0) {
            // processor.go:772-780: truncate to the test chunk when longer
            i64 l = n - win_start;
            if (l < 0) l = 0;
            if (e->cfg.chunk_samples > 0 && l > e->cfg.chunk_samples) l = e->cfg.chunk_samples;
            len[s] = l;
            if (n_windows > 1) return fail(e, TDOA_E_INVALID, "tdoa_xcorr: win_len = 0 needs n_windows = 1");
        } else {
            const i64 last = win_start + (i64)(n_windows - 1) * hop + win_len;
            if (last > n)
                return fail(e, TDOA_E_INVALID, "tdoa_xcorr: windows end at %lld but station %d has %lld samples",
                            (long long)last, s, (long long)n);
            len[s] = win_len;
        }
    }
    return TDOA_OK;
}

// windows per group: the planes of a group stay under 24 GiB (retimed: one more plane per signal)
int window_group(const tdoa_engine *e, const std::vector<i64> &len, int n_windows, bool retimed)
{
    i64 per_window_bytes = 0;
    for (int s = 0; s < e->cfg.n_stations; s++) per_window_bytes += len[s] * 4 * (retimed ? 5 : 4);
    const i64 budget = (i64)24 << 30;
    const int group = (int)std::max<i64>(1, std::min<i64>(n_windows, budget / std::max<i64>(per_window_bytes, 1)));
    return std::min(group, 64);
}

// Every preprocessed plane re-timed by its station's rate (k_retime): the correlators read the re-timed plane with
// the statistics block (normalisation scale) of the original.  The imaginary plane is dropped: the BINARY and
// EXTENDED correlators read real parts only, and SOURCE mode has no re-timed call.
int retime(tdoa_engine *e, std::vector<Sig> &sigs, const double *d_rates)
{
    std::vector<RetimeJob> jobs;
    i64 max_n = 0;
    for (Sig &sg : sigs) {
        const i64 n = sg.n_out >= 0 ? sg.n_out : sg.n;
        if (n == 0) continue;
        RetimeJob j{sg.out_re, nullptr, n, sg.station};
        if (const int rc = alloc_t(e, &j.y, (size_t)n)) return rc;
        sg.out_re = j.y;
        sg.out_im = nullptr;
        jobs.push_back(j);
        max_n = std::max(max_n, n);
    }
    if (jobs.empty()) return TDOA_OK;
    const RetimeJob *d_jobs = nullptr;
    if (const int rc = upload(e, jobs, &d_jobs)) return rc;
    launch_retime(d_jobs, (int)jobs.size(), max_n, d_rates, e->stream);
    count_launch(e);
    return TDOA_OK;
}

// The pair loops of one signal kind over the windows, records to d_out (device).
// pend == nullptr: every check is made here (the stream is synchronised as needed).
// pend != nullptr: one window, everything only QUEUED -- branch guesses and candidate
// overflow are the caller's to check after its synchronisation (tdoa_process).
// d_rates != nullptr: station rates on the device; every plane is re-timed between preprocessing and correlation.
int xcorr_core(tdoa_engine *e, int32_t kind, int64_t win_start, const std::vector<i64> &len, int32_t n_windows,
               int64_t hop, PeakRec *d_out, Pending *pend, const double *d_rates)
{
    int rc;
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    if ((rc = queue_lazy_copies(e, kind))) return rc;
    // windows are processed in groups that keep the working set bounded
    const int group = window_group(e, len, n_windows, d_rates != nullptr);
    for (int w0 = 0; w0 < n_windows; w0 += group) {
        const int gw = std::min(group, n_windows - w0);
        std::vector<Sig> sigs((size_t)gw * S);
        std::vector<Pair> pairs;
        for (int w = 0; w < gw; w++) {
            for (int s = 0; s < S; s++) {
                Sig &sg = sigs[(size_t)w * S + s];
                sg.n = len[s];
                sg.src = make_view(e->stations[s], kind, win_start + (i64)(w0 + w) * hop, len[s], e->cfg.guard_samples);
                sg.memo = s * 2 + kind;
                sg.station = s; sg.kind = kind; sg.q0 = win_start + (i64)(w0 + w) * hop;
            }
            for (int i = 0; i < S; i++)
                for (int j = i + 1; j < S; j++) pairs.push_back({w * S + i, w * S + j, w});
        }
        double *d_first = nullptr;
        std::vector<double> h_stats;
        // scratch of this group: everything allocated / staged from here on (what the caller
        // allocated before -- record buffers, the other kind's planes -- is not ours to free)
        const size_t alloc_mark = e->call_allocs.size(), frame_mark = e->frame_used;
        auto drop_group_scratch = [&]() {
            for (size_t k = alloc_mark; k < e->call_allocs.size(); k++) cudaFreeAsync(e->call_allocs[k], e->stream);
            e->call_allocs.resize(alloc_mark);
            e->frame_used = frame_mark;  // the stream is idle: descriptor staging can be reused
        };
        for (int attempt = 0; attempt < 2; attempt++) {
            const int sp_pre = span_begin(e, SPAN_STAGE_PRE);
            if ((rc = preprocess(e, sigs, attempt == 0))) return rc;
            if (d_rates && (rc = retime(e, sigs, d_rates))) return rc;
            span_end(e, sp_pre);
            const int sp_corr = span_begin(e, SPAN_STAGE_CORR);
            d_first = nullptr;
            if (w0 == 0 && (rc = alloc_t(e, &d_first, pairs.size()))) return rc;
            if ((rc = correlate(e, sigs, pairs, d_out + (size_t)w0 * P, d_first, pend != nullptr))) return rc;
            if (decimation(e) > 1) {
                launch_lag_units(d_out + (size_t)w0 * P, (int)pairs.size(), decimation(e), e->stream);
                count_launch(e);
            }
            span_end(e, sp_corr);
            if (pend) {
                pend->kind = kind; pend->sigs = sigs; pend->d_first = d_first; pend->valid = true;
                return TDOA_OK;
            }
            bool any_deferred = false;
            for (auto &sg : sigs) any_deferred |= sg.deferred;
            if (!any_deferred && w0 != 0) break;
            // statistics of the group: the branch check of the speculated signals and
            // (window 0) what the reference prints.  One read-back; it waits for the stream.
            h_stats.resize(sigs.size() * ST_COUNT);
            CU(cudaMemcpyAsync(h_stats.data(), sigs[0].stats, h_stats.size() * sizeof(double), cudaMemcpyDeviceToHost,
                               e->stream));
            CU(cudaStreamSynchronize(e->stream));
            if (verify_deferred(e, sigs, h_stats.data())) break;
            // a guess was wrong (the capture is not "strong FM"): drop the group's scratch and
            // redo it with the powers read first; the memo now keeps those signals off the fused path
            spans_collect(e);
            drop_group_scratch();
            for (auto &sg : sigs) {
                Sig fresh;
                fresh.n = sg.n; fresh.src = sg.src; fresh.memo = sg.memo;
                fresh.station = sg.station; fresh.kind = sg.kind; fresh.q0 = sg.q0;
                sg = fresh;
            }
        }
        if (w0 == 0) {
            // what the reference prints about window 0 (tdoa_xcorr_info)
            e->info_first[kind].assign(P, 0.0);
            CU(cudaMemcpyAsync(e->info_first[kind].data(), d_first, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            CU(cudaStreamSynchronize(e->stream));
            fill_info(e, kind, sigs, h_stats.data(), S);
        }
        // free this group's planes before the next group allocates
        if (w0 + group < n_windows) {
            CU(cudaStreamSynchronize(e->stream));
            spans_collect(e);
            drop_group_scratch();
        }
    }
    return TDOA_OK;
}

int xcorr_impl(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows, int64_t hop,
               tdoa_peak *out, bool out_is_device, PeakRec *d_table, const double *d_rates)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (!out && !d_table) return fail(e, TDOA_E_INVALID, "tdoa_xcorr: out is NULL");
    std::vector<i64> len;
    if ((rc = window_lengths(e, kind, win_start, win_len, n_windows, hop, len))) return rc;
    // more than one GPU: windows dealt over the ranks, records gathered (engine_multi.cu)
    if (multi_wants(e, n_windows)) return xcorr_sharded(e, kind, win_start, len, n_windows, hop, out, out_is_device);
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    PeakRec *d_out = nullptr;
    if (out_is_device) d_out = reinterpret_cast<PeakRec *>(out);
    else if (d_table) d_out = d_table;
    else if ((rc = alloc_t(e, &d_out, (size_t)n_windows * P))) return rc;
    stats_reset(e);
    cudaEventRecord(e->ev[0], e->stream);
    // Two halves of the windows side by side on two streams (as tdoa_process does with the two
    // signal kinds): one half's compute-bound kernels share the SMs with the other half's
    // memory-bound ones.  Both halves are only queued; branch guesses and candidate overflow are
    // checked after the one synchronisation, and any failure falls back to the checked pass.
    const int nA = (n_windows + 1) / 2, nB = n_windows - nA;
    bool done = false;
    if (!e->cfg.serial_kinds && !out_is_device && nB >= 1 && window_group(e, len, nA, d_rates != nullptr) >= nA) {
        Pending pend[2];
        cudaStream_t main_stream = e->stream;
        CU(cudaEventRecord(e->ev_fork, main_stream));
        CU(cudaStreamWaitEvent(e->side_stream, e->ev_fork, 0));
        if ((rc = xcorr_core(e, kind, win_start, len, nA, hop, d_out, &pend[0], d_rates))) return rc;
        e->stream = e->side_stream;
        rc = xcorr_core(e, kind, win_start + (i64)nA * hop, len, nB, hop, d_out + (size_t)nA * P, &pend[1], d_rates);
        e->stream = main_stream;
        CU(cudaEventRecord(e->ev_join, e->side_stream));
        CU(cudaStreamWaitEvent(main_stream, e->ev_join, 0));
        if (rc) { cudaStreamSynchronize(e->side_stream); return rc; }
        cudaEventRecord(e->ev[4], e->stream);
        std::vector<PeakRec> h_pk((size_t)n_windows * P);
        std::vector<double> h_stats[2], h_first(P, 0.0);
        CU(cudaMemcpyAsync(h_pk.data(), d_out, h_pk.size() * sizeof(PeakRec), cudaMemcpyDeviceToHost, e->stream));
        for (int k = 0; k < 2; k++) {
            if (!pend[k].valid) continue;
            h_stats[k].resize(pend[k].sigs.size() * ST_COUNT);
            CU(cudaMemcpyAsync(h_stats[k].data(), pend[k].sigs[0].stats, h_stats[k].size() * sizeof(double), cudaMemcpyDeviceToHost,
                               e->stream));
        }
        if (pend[0].valid)
            CU(cudaMemcpyAsync(h_first.data(), pend[0].d_first, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        bool ok = pend[0].valid && pend[1].valid;
        for (int k = 0; k < 2 && ok; k++) ok &= verify_deferred(e, pend[k].sigs, h_stats[k].data());
        for (size_t i = 0; i < h_pk.size() && ok; i++) ok &= (h_pk[i].flags & 0x10u) == 0;   // candidate overflow
        if (ok) {
            e->info_first[kind] = h_first;
            fill_info(e, kind, pend[0].sigs, h_stats[0].data(), S);
            if (out) std::memcpy(out, h_pk.data(), h_pk.size() * sizeof(PeakRec));
            done = true;
        } else {
            spans_collect(e);
        }
    }
    if (!done) {
        if ((rc = xcorr_core(e, kind, win_start, len, n_windows, hop, d_out, nullptr, d_rates))) return rc;
        cudaEventRecord(e->ev[4], e->stream);
        if (!out_is_device && out)
            CU(cudaMemcpyAsync(out, d_out, (size_t)n_windows * P * sizeof(tdoa_peak), cudaMemcpyDeviceToHost, e->stream));
    }
    rc = end_call(e, !out_is_device);
    if (rc) return rc;
    e->st.launches_last = e->st.launches_total - e->launches_at_call;
    if (!out_is_device) {
        float t = 0.f;
        retire_lazy(e);
        spans_collect(e);
        cudaEventElapsedTime(&t, e->ev[0], e->ev[4]);
        e->st.ms_exact = e->ms_corr - e->st.ms_fft;
        e->st.ms_total = t;
    }
    return TDOA_OK;
}

}  // namespace tdoa

extern "C" {

int tdoa_unpack(tdoa_engine *e, int32_t station, int64_t first, int64_t count, float *out_c64)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations || !e->stations[station].loaded)
        return fail(e, TDOA_E_STATE, "tdoa_unpack: station %d not loaded", station);
    Station &s = e->stations[station];
    if ((rc = capture_ready(e, s))) return rc;
    if (first < 0 || count < 0 || first + count > s.nsamp || (!out_c64 && count))
        return fail(e, TDOA_E_INVALID, "tdoa_unpack: range [%lld,+%lld) outside %lld samples", (long long)first,
                    (long long)count, (long long)s.nsamp);
    if (count == 0) return end_call(e, true);
    std::vector<Sig> sigs(1);
    Sig &sg = sigs[0];
    sg.n = count;
    sg.src.raw = s.d_raw; sg.src.run0_start = first; sg.src.run0_len = count;
    float *d_c64 = nullptr;
    if ((rc = ensure_plane(e, sg, 0, true))) return rc;
    if ((rc = alloc_t(e, &sg.stats, ST_COUNT)) || (rc = alloc_t(e, &sg.partials, (size_t)2 * stream_grid_x(count))) ||
        (rc = alloc_t(e, &sg.counter, 1)) || (rc = alloc_t(e, &d_c64, (size_t)2 * count)))
        return rc;
    CU(cudaMemsetAsync(sg.counter, 0, sizeof(unsigned), e->stream));
    std::vector<SigJob> jobs(1, base_job(sg));
    jobs[0].p_re = sg.plane[0][0]; jobs[0].p_im = sg.plane[0][1];
    const SigJob *d_jobs = nullptr;
    if ((rc = upload(e, jobs, &d_jobs))) return rc;
    launch_unpack(d_jobs, 1, count, stream_grid_x(count), e->stream);
    launch_interleave(sg.plane[0][0], sg.plane[0][1], count, d_c64, e->stream);
    count_launch(e, 2);
    CU(cudaMemcpyAsync(out_c64, d_c64, (size_t)2 * count * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    return end_call(e, true);
}

int tdoa_preprocess(tdoa_engine *e, int32_t station, int32_t kind, int64_t start, int64_t len, float *out_c64,
                    double *power, int32_t *branch)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (station < 0 || station >= e->cfg.n_stations || !e->stations[station].loaded)
        return fail(e, TDOA_E_STATE, "tdoa_preprocess: station %d not loaded", station);
    if (kind != TDOA_KIND_REF && kind != TDOA_KIND_TGT) return fail(e, TDOA_E_INVALID, "tdoa_preprocess: bad kind");
    const Station &s = e->stations[station];
    const i64 n = signal_length(s, kind, e->cfg.guard_samples);
    if (start < 0 || len < 0 || start + len > n || (!out_c64 && len))
        return fail(e, TDOA_E_INVALID, "tdoa_preprocess: range [%lld,+%lld) outside %lld samples", (long long)start,
                    (long long)len, (long long)n);
    std::vector<Sig> sigs(1);
    sigs[0].n = len;
    sigs[0].src = make_view(s, kind, start, len, e->cfg.guard_samples);
    sigs[0].station = station; sigs[0].kind = kind; sigs[0].q0 = start;
    sigs[0].need_im = true;   // the probe returns complex samples
    sigs[0].memo = station * 2 + kind;   // a branch seen before is not guessed again
    if ((rc = queue_lazy_copies(e, kind))) return rc;
    if ((rc = preprocess(e, sigs))) return rc;
    if (power) *power = sigs[0].power0;
    if (branch) *branch = sigs[0].branch;
    if (decimation(e) > 1) len = sigs[0].n_out;  // the first len / D entries of out_c64 are written
    if (len > 0) {
        Sig &sg = sigs[0];
        float *d_nre = nullptr, *d_nim = nullptr, *d_c64 = nullptr;
        if ((rc = alloc_t(e, &d_nre, (size_t)len)) || (rc = alloc_t(e, &d_nim, (size_t)len)) ||
            (rc = alloc_t(e, &d_c64, (size_t)2 * len)))
            return rc;
        SigJob j = base_job(sg);
        j.n = len;  // the preprocessed signal's length (n / D with the decimator)
        j.q_re = sg.out_re; j.q_im = sg.out_im; j.p_re = d_nre; j.p_im = d_nim;
        std::vector<SigJob> jobs(1, j);
        const SigJob *d_jobs = nullptr;
        if ((rc = upload(e, jobs, &d_jobs))) return rc;
        launch_normalize(d_jobs, 1, len, e->stream);
        launch_interleave(d_nre, d_nim, len, d_c64, e->stream);
        count_launch(e, 2);
        CU(cudaMemcpyAsync(out_c64, d_c64, (size_t)2 * len * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    }
    return end_call(e, true);
}

int tdoa_xcorr(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows, int64_t hop,
               tdoa_peak *out)
{
    return xcorr_impl(e, kind, win_start, win_len, n_windows, hop, out, false);
}

int tdoa_xcorr_device(tdoa_engine *e, int32_t kind, int64_t win_start, int64_t win_len, int32_t n_windows,
                      int64_t hop, tdoa_peak *d_out)
{
    return xcorr_impl(e, kind, win_start, win_len, n_windows, hop, d_out, true);
}

int tdoa_xcorr_windows(tdoa_engine *e, int64_t win_start, int64_t win_len, int32_t n_ref_windows, int32_t n_tgt_windows,
                       int64_t hop, tdoa_peak *ref_out, tdoa_peak *tgt_out)
{
    if (!e) return TDOA_E_INVALID;
    if (n_ref_windows < 0 || n_tgt_windows < 0 || (n_ref_windows && !ref_out) || (n_tgt_windows && !tgt_out))
        return fail(e, TDOA_E_INVALID, "tdoa_xcorr_windows: a table is NULL");
    const bool sharded = multi_wants(e, n_ref_windows + n_tgt_windows);
    if (!sharded) {   // one GPU: the two pair loops one after the other (processor.go:816-830, then :836-850)
        int rc = TDOA_OK;
        if (n_ref_windows) rc = xcorr_impl(e, TDOA_KIND_REF, win_start, win_len, n_ref_windows, hop, ref_out, false);
        if (!rc && n_tgt_windows) rc = xcorr_impl(e, TDOA_KIND_TGT, win_start, win_len, n_tgt_windows, hop, tgt_out, false);
        return rc;
    }
    int rc = begin_call(e);
    if (rc) return rc;
    std::vector<ShardPart> parts;
    for (int kind = 0; kind < 2; kind++) {
        const int32_t nw = kind == TDOA_KIND_REF ? n_ref_windows : n_tgt_windows;
        if (!nw) continue;
        ShardPart Q;
        Q.kind = kind; Q.win_start = win_start; Q.n_windows = nw; Q.hop = hop;
        Q.out = kind == TDOA_KIND_REF ? ref_out : tgt_out;
        if ((rc = window_lengths(e, kind, win_start, win_len, nw, hop, Q.len))) return rc;
        parts.push_back(Q);
    }
    return xcorr_sharded(e, parts);
}

int tdoa_process(tdoa_engine *e, const double *stations_llh, tdoa_peak *ref_out, tdoa_peak *tgt_out, double *time_diffs,
                 double *range_diffs, double *fix_llh, int32_t *fix_status, int32_t *fix_iters)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (!stations_llh || !ref_out || !tgt_out || !fix_llh || !fix_status)
        return fail(e, TDOA_E_INVALID, "tdoa_process: NULL argument");
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    if (S < 3) return fail(e, TDOA_E_INVALID, "need at least 3 collector stations, got %d", S);  // processor.go:740-742
    std::vector<i64> len_ref, len_tgt;
    if ((rc = window_lengths(e, TDOA_KIND_REF, 0, 0, 1, 0, len_ref)) || (rc = window_lengths(e, TDOA_KIND_TGT, 0, 0, 1, 0, len_tgt)))
        return rc;
    PeakRec *d_ref = nullptr, *d_tgt = nullptr;
    double *d_td = nullptr, *d_rd = nullptr, *d_fix = nullptr;
    int *d_status = nullptr, *d_iters = nullptr;
    if ((rc = alloc_t(e, &d_ref, (size_t)P)) || (rc = alloc_t(e, &d_tgt, (size_t)P)) || (rc = alloc_t(e, &d_td, (size_t)P)) ||
        (rc = alloc_t(e, &d_rd, (size_t)P)) || (rc = alloc_t(e, &d_fix, 3)) || (rc = alloc_t(e, &d_status, 1)) ||
        (rc = alloc_t(e, &d_iters, 1)))
        return rc;
    // the station table rides with the descriptors (a kernel fetches it): a copy-engine
    // transfer would wait behind the bulk copies of a lazily loaded capture
    const double *d_llh = nullptr;
    {
        std::vector<double> llh(stations_llh, stations_llh + (size_t)3 * S);
        if ((rc = upload(e, llh, &d_llh))) return rc;
    }
    stats_reset(e);
    cudaEventRecord(e->ev[0], e->stream);
    auto fix_chain = [&]() {
        launch_range_diffs(d_ref, d_tgt, P, e->cfg.sample_rate, e->cfg.mode, d_td, d_rd, e->stream);
        launch_solve(d_llh, d_rd, 1, P, d_fix, d_status, d_iters, e->stream);
        count_launch(e, 2);
    };
    // optimistic pass: both pair loops and the fix are only queued; one synchronisation
    // The two pair loops do not depend on each other: the TGT loop is queued on a second stream,
    // so its compute-bound discriminator shares the SMs with the REF loop's memory-bound kernels
    // (and vice versa) instead of every kernel waiting for the previous one's tail.
    Pending pend[2];
    cudaStream_t main_stream = e->stream;
    CU(cudaEventRecord(e->ev_fork, main_stream));
    CU(cudaStreamWaitEvent(e->side_stream, e->ev_fork, 0));
    if ((rc = xcorr_core(e, TDOA_KIND_REF, 0, len_ref, 1, 0, d_ref, &pend[0]))) return rc;
    if (!e->cfg.serial_kinds) e->stream = e->side_stream;
    rc = xcorr_core(e, TDOA_KIND_TGT, 0, len_tgt, 1, 0, d_tgt, &pend[1]);
    e->stream = main_stream;
    CU(cudaEventRecord(e->ev_join, e->side_stream));
    CU(cudaStreamWaitEvent(main_stream, e->ev_join, 0));
    if (rc) { cudaStreamSynchronize(e->side_stream); return rc; }
    fix_chain();
    cudaEventRecord(e->ev[4], e->stream);
    std::vector<PeakRec> h_pk((size_t)2 * P);
    std::vector<double> h_stats[2], h_first[2];
    // Everything comes back through the top of the pinned frame (the descriptors grow from its
    // bottom): a device->host copy into pageable memory blocks the caller once per copy, into
    // pinned memory it is just queued -- ten small copies, one synchronisation.
    struct Back { void *dst; const void *pinned; size_t bytes; };
    std::vector<Back> backs;
    size_t back_top = kFrameBytes;
    auto fetch = [&](void *dst, const void *d_src, size_t bytes) -> int {
        const size_t need = (bytes + 63) & ~size_t(63);
        if (back_top < need || back_top - need < e->frame_used + 4096) {   // no room: the plain (blocking) copy
            CU(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, e->stream));
            return TDOA_OK;
        }
        back_top -= need;
        CU(cudaMemcpyAsync(e->h_frame + back_top, d_src, bytes, cudaMemcpyDeviceToHost, e->stream));
        backs.push_back(Back{dst, e->h_frame + back_top, bytes});
        return TDOA_OK;
    };
    auto deliver = [&]() {
        for (const Back &b : backs) std::memcpy(b.dst, b.pinned, b.bytes);
        backs.clear();
        back_top = kFrameBytes;
    };
    auto read_back = [&]() -> int {
        int r;
        if ((r = fetch(h_pk.data(), d_ref, (size_t)P * sizeof(PeakRec))) || (r = fetch(h_pk.data() + P, d_tgt, (size_t)P * sizeof(PeakRec))))
            return r;
        if (time_diffs && (r = fetch(time_diffs, d_td, (size_t)P * sizeof(double)))) return r;
        if (range_diffs && (r = fetch(range_diffs, d_rd, (size_t)P * sizeof(double)))) return r;
        if ((r = fetch(fix_llh, d_fix, 3 * sizeof(double))) || (r = fetch(fix_status, d_status, sizeof(int32_t)))) return r;
        if (fix_iters && (r = fetch(fix_iters, d_iters, sizeof(int32_t)))) return r;
        return TDOA_OK;
    };
    if ((rc = read_back())) return rc;
    bool ok = true;
    for (int k = 0; k < 2; k++) {
        if (!pend[k].valid) continue;   // the pass ran with its own checks (not speculated)
        h_stats[k].resize(pend[k].sigs.size() * ST_COUNT);
        h_first[k].assign(P, 0.0);
        if ((rc = fetch(h_stats[k].data(), pend[k].sigs[0].stats, h_stats[k].size() * sizeof(double))) ||
            (rc = fetch(h_first[k].data(), pend[k].d_first, (size_t)P * sizeof(double))))
            return rc;
    }
    CU(cudaStreamSynchronize(e->stream));
    deliver();
    for (int k = 0; k < 2; k++) {
        if (!pend[k].valid) continue;
        ok &= verify_deferred(e, pend[k].sigs, h_stats[k].data());
        for (int p = 0; p < P; p++) ok &= (h_pk[(size_t)k * P + p].flags & 0x10u) == 0;   // candidate overflow
    }
    if (ok) {
        for (int k = 0; k < 2; k++) {
            if (!pend[k].valid) continue;
            e->info_first[k] = h_first[k];
            fill_info(e, k, pend[k].sigs, h_stats[k].data(), S);
        }
    } else {
        // a branch guess was wrong or a pair overflowed its candidate list: run the pair
        // loops again with every check made on the way (the memo keeps the guesses off)
        spans_collect(e);
        if ((rc = xcorr_core(e, TDOA_KIND_REF, 0, len_ref, 1, 0, d_ref, nullptr)) ||
            (rc = xcorr_core(e, TDOA_KIND_TGT, 0, len_tgt, 1, 0, d_tgt, nullptr)))
            return rc;
        fix_chain();
        cudaEventRecord(e->ev[4], e->stream);
        if ((rc = read_back())) return rc;
        CU(cudaStreamSynchronize(e->stream));
        deliver();
    }
    std::memcpy(ref_out, h_pk.data(), (size_t)P * sizeof(tdoa_peak));
    std::memcpy(tgt_out, h_pk.data() + P, (size_t)P * sizeof(tdoa_peak));
    if (*fix_status != 0) *fix_status = TDOA_E_SINGULAR;
    rc = end_call(e, true);
    if (rc) return rc;
    e->st.launches_last = e->st.launches_total - e->launches_at_call;
    float t = 0.f;
    retire_lazy(e);
    spans_collect(e);
    cudaEventElapsedTime(&t, e->ev[0], e->ev[4]);
    e->st.ms_exact = e->ms_corr - e->st.ms_fft;
    e->st.ms_total = t;
    return TDOA_OK;
}

int tdoa_cross_correlate(tdoa_engine *e, const float *sig1_c64, int64_t n1, const float *sig2_c64, int64_t n2,
                         tdoa_peak *out)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (!out || n1 < 0 || n2 < 0 || (n1 && !sig1_c64) || (n2 && !sig2_c64))
        return fail(e, TDOA_E_INVALID, "tdoa_cross_correlate: bad arguments");
    std::vector<Sig> sigs(2);
    const float *h[2] = {sig1_c64, sig2_c64};
    const i64 n[2] = {n1, n2};
    for (int k = 0; k < 2; k++) {
        Sig &sg = sigs[k];
        sg.n = n[k];
        if (n[k] == 0) continue;
        float *d_c64 = nullptr, *d_re = nullptr, *d_im = nullptr;
        if ((rc = alloc_t(e, &d_c64, (size_t)2 * n[k])) || (rc = alloc_t(e, &d_re, (size_t)n[k])) ||
            (rc = alloc_t(e, &d_im, (size_t)n[k])))
            return rc;
        CU(cudaMemcpyAsync(d_c64, h[k], (size_t)2 * n[k] * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        launch_deinterleave(d_c64, n[k], d_re, d_im, e->stream);
        count_launch(e);
        sg.src.raw = nullptr; sg.src.re = d_re; sg.src.im = d_im;
        sg.src.run0_len = n[k];
    }
    // the host slices may be Go memory: they have been read once the copies complete,
    // which preprocess() guarantees (it synchronises after the power pass)
    PeakRec *d_out = nullptr;
    if ((rc = alloc_t(e, &d_out, 1))) return rc;
    if ((rc = preprocess(e, sigs))) return rc;
    std::vector<Pair> pairs(1, Pair{0, 1, 0});
    if ((rc = correlate(e, sigs, pairs, d_out))) return rc;
    CU(cudaMemcpyAsync(out, d_out, sizeof(tdoa_peak), cudaMemcpyDeviceToHost, e->stream));
    rc = end_call(e, true);
    e->st.launches_last = e->st.launches_total - e->launches_at_call;
    return rc;
}

}  // extern "C"
