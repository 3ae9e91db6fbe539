// xcorr_fft.cu -- FFT cross-correlation over station pairs: candidate search in the
// frequency domain, then the reference's own arithmetic on the few candidate lags.
//
// The reference evaluates corr(lag) = (1/n) sum_i t[i] s[i+lag] for every lag in the
// time domain (processor.go:689-727, O(lags * n)).  Here the template is cut into
// segments of kSeg samples; each CTA transforms one segment of the template (zero
// padded) and the matching kN-sample span of the signal as ONE complex FFT
// (z = t + i s), forms the segment's cross-spectrum conj(T) S from Z[k] and Z[N-k], and
// accumulates it in registers across its segments -- the inverse transform is linear,
// so it is done once per pair on the summed spectrum (k_fft_finish), not per segment.
// One pass over the data: 4 B/sample of template + 4 B/sample of signal (x kN/kSeg).
//
// The f32 spectrum path only has to rank lags: every lag whose approximate |corr| is
// within `tol` of the maximum is re-evaluated by k_corr_candidates with f32 products
// and f64 accumulation exactly as the reference, and the peak logic runs on those
// exact values -- so the integer lag is the reference's, bit for bit.
#include "fft_core.cuh"
#include "kernels.h"
#include "xcorr_fft.h"

namespace tdoa {

using namespace fft;

namespace {

constexpr int kBins = kN / 2 + 1;          // 4097 cross-spectrum bins kept (Hermitian)
constexpr int kTabLen = 16 * 32;                                // pass-2 twiddles per lane
constexpr int kSmemBytes = (kPad + kTabLen) * (int)sizeof(float2);

// ---------------------------------------------------------------- segment accumulate
__global__ void __launch_bounds__(kThreads, 2) k_fft_segments(const FftJob *jobs, const float2 *__restrict__ tw)
{
    extern __shared__ float2 sm[];
    const FftJob &J = jobs[blockIdx.y];
    const int cta = blockIdx.x;
    if (cta >= J.n_cta) return;
    const int tid = threadIdx.x;
    const float *__restrict__ tp = J.t + J.t_off;
    const float *__restrict__ sp = J.s;
    // xcorr_fft.h: 1 unless the two planes' powers differ widely
    const float sc_t = rank_pre(J.t_stats, J.s_stats), sc_s = rank_pre(J.s_stats, J.t_stats);
    const bool pre = sc_t != 1.f || sc_s != 1.f;
    float2 *tab = sm + kPad;
    for (int idx = tid; idx < kTabLen; idx += kThreads) tab[idx] = tw[(16 * (idx & 31) * (idx >> 5)) & (kN - 1)];
    // (the first barrier inside the segment loop orders these writes before their use)

    float acc_re[16], acc_im[16];
    float acc_nyq = 0.f;
#pragma unroll
    for (int u = 0; u < 16; u++) { acc_re[u] = 0.f; acc_im[u] = 0.f; }

    for (int seg = cta; seg < J.n_seg; seg += J.n_cta) {
        const i64 t0 = (i64)seg * kSeg;       // template index of m = 0
        const i64 s0 = J.s_off + t0;          // signal index of m = 0
        const i64 t_left = J.n_t - t0;        // template samples left (>= 1)
        {
            float2 v[32];
            {
                // pull the next segment of this CTA towards L2 while this one is transformed:
                // 448 lines of 128 B per segment, two per thread
                const i64 nt0 = t0 + (i64)J.n_cta * kSeg, ns0 = s0 + (i64)J.n_cta * kSeg;
                const i64 pt = nt0 + 32 * tid, ps = ns0 + 32 * tid;
                if (tid < kSeg / 32 && pt < J.n_t) asm volatile("prefetch.global.L2 [%0];" ::"l"(tp + pt));
                if (ps >= 0 && ps < J.sl) asm volatile("prefetch.global.L2 [%0];" ::"l"(sp + ps));
            }
            if (t_left >= kSeg && s0 >= 0 && s0 + kN <= J.sl) {
                // interior segment: one base pointer each, immediate offsets, no bounds tests
                const float *__restrict__ tq = tp + t0 + tid;
                const float *__restrict__ sq = sp + s0 + tid;
#pragma unroll
                for (int r = 0; r < 32; r++) v[r] = make_float2(r < kSeg / 256 ? tq[256 * r] : 0.f, sq[256 * r]);
            } else {
#pragma unroll
                for (int r = 0; r < 32; r++) {
                    const int m = tid + 256 * r;
                    float a = 0.f, b = 0.f;
                    if (r < kSeg / 256 && m < t_left) a = tp[t0 + m];
                    const i64 g = s0 + m;
                    if (g >= 0 && g < J.sl) b = sp[g];
                    v[r] = make_float2(a, b);
                }
            }
            if (pre) {
#pragma unroll
                for (int r = 0; r < 32; r++) v[r] = make_float2(__fmul_rn(v[r].x, sc_t), __fmul_rn(v[r].y, sc_s));
            }
            pass1_store(v, tid, sm);
        }
        __syncthreads();
        float2 u0[16], u1[16];
        pass_load16(sm, tid, u0);
        pass_load16(sm, tid + 256, u1);
        __syncthreads();
        pass2_store_tab(u0, tid, tab, sm);
        pass2_store_tab(u1, tid + 256, tab, sm);
        __syncthreads();
        pass_load16(sm, tid, u0);
        pass_load16(sm, tid + 256, u1);
        __syncthreads();
        pass3_compute(u0, tid, tw);
        pass3_compute(u1, tid + 256, tw);
        // u0[r] = Z[tid + 512 r], u1[r] = Z[tid + 256 + 512 r]: bins tid + 256 w, w = 2r (+1)
        // upper half (k >= 4096 <=> r >= 8) goes to shared memory for the partner lookup
#pragma unroll
        for (int r = 8; r < 16; r++) {
            sm[tid + 512 * r - 4096] = u0[r];
            sm[tid + 256 + 512 * r - 4096] = u1[r];
        }
        __syncthreads();
        // C[k] = conj(T[k]) S[k] = (a d + b c)/2 - i (|Z[k]|^2 - |Z[N-k]|^2)/4,
        // Z[k] = a + i b, Z[N-k] = c + i d; the 1/2 and 1/4 are applied in k_fft_finish
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int k = tid + 256 * h + 512 * r;
                const float2 z = h ? u1[r] : u0[r];
                const float2 p = k == 0 ? z : sm[4096 - k];  // Z[N-k] at index (N-k) - 4096
                const int w = 2 * r + h;
                acc_re[w] += z.x * p.y + z.y * p.x;
                acc_im[w] += (p.x * p.x + p.y * p.y) - (z.x * z.x + z.y * z.y);
            }
        }
        if (tid == 0) acc_nyq += 2.f * u0[8].x * u0[8].y;  // k = 4096 is its own partner
        __syncthreads();
    }
    float2 *out = J.partials + (size_t)cta * kBins;
#pragma unroll
    for (int w = 0; w < 16; w++) out[tid + 256 * w] = make_float2(acc_re[w], acc_im[w]);
    if (tid == 0) out[4096] = make_float2(acc_nyq, 0.f);
}

// ---------------------------------------------------------------- reduce the partial spectra
__global__ void __launch_bounds__(256) k_fft_reduce(const FftJob *jobs)
{
    const FftJob &J = jobs[blockIdx.y];
    const int k = blockIdx.x * 256 + threadIdx.x;
    if (k >= kBins) return;
    double sr = 0.0, si = 0.0;
#pragma unroll 8
    for (int c = 0; c < J.n_cta; c++) {
        const float2 p = J.partials[(size_t)c * kBins + k];
        sr += (double)p.x;
        si += (double)p.y;
    }
    // C[k] = (sum re / 2, sum im / 4), see k_fft_segments
    J.spectrum[k] = make_float2((float)(0.5 * sr), (float)(0.25 * si));
}

// ---------------------------------------------------------------- finish: inverse FFT, scale
// fft(conj(C))[d] = N * corr_raw[d] for real corr, so the forward transform is reused.
__global__ void __launch_bounds__(kThreads, 1) k_fft_finish(const FftJob *jobs, const float2 *__restrict__ tw)
{
    extern __shared__ float2 sm[];
    const FftJob &J = jobs[blockIdx.x];
    const int tid = threadIdx.x;
    {
        float2 v[32];
#pragma unroll
        for (int r = 0; r < 32; r++) {
            const int k = tid + 256 * r;
            // C[N-k] = conj(C[k]); the transform input is conj(C[k])
            const float2 c = J.spectrum[k <= 4096 ? k : kN - k];
            v[r] = make_float2(c.x, k <= 4096 ? -c.y : c.y);
        }
        pass1_store(v, tid, sm);
    }
    __syncthreads();
    float2 u0[16], u1[16];
    pass_load16(sm, tid, u0);
    pass_load16(sm, tid + 256, u1);
    __syncthreads();
    pass2_store(u0, tid, tw, sm);
    pass2_store(u1, tid + 256, tw, sm);
    __syncthreads();
    pass_load16(sm, tid, u0);
    pass_load16(sm, tid + 256, u1);
    pass3_compute(u0, tid, tw);
    pass3_compute(u1, tid + 256, tw);
    // correlation coefficient units: scale_t * scale_s / n_t (processor.go:347-349, :709-717), less the scales the
    // transforms applied as they loaded the planes (rank_pre)
    const double sc = J.n_t > 0 ? rank_post(J.t_stats, J.t_pack) * rank_post(J.s_stats, J.s_pack) /
                                      ((double)J.n_t * (double)kN)
                                : 0.0;
#pragma unroll
    for (int r = 0; r < 16; r++) {
        const int d0 = tid + 512 * r, d1 = tid + 256 + 512 * r;
        if (d0 < J.n_lags) J.approx[d0] = (float)((double)u0[r].x * sc);
        if (d1 < J.n_lags) J.approx[d1] = (float)((double)u1[r].x * sc);
    }
}

// ---------------------------------------------------------------- candidate selection
// One CTA per pair.  Candidates = lags whose approximate |corr| is within tol of the
// maximum over the whole search, plus (sanity > 0) the same for the re-search range
// [0, sanity), plus (neighbours) the lags either side for the parabolic vertex.  A bounded
// record (EXTENDED) takes all three from its run [i0, i1] only.
__global__ void __launch_bounds__(256) k_select_candidates(const SelJob *jobs)
{
    __shared__ float s_red[256];
    __shared__ int s_base;
    const SelJob &J = jobs[blockIdx.x];
    const int tid = threadIdx.x;
    const int n = J.n_lags;
    int i0, i1;
    bound_run(J.bound, J.lag_origin, J.decim, n, &i0, &i1);
    if (i0 > i1) {   // n <= 0, or an empty run: k_peak_candidates writes the record
        if (tid == 0) *J.n_cand = 0;
        return;
    }
    float m1 = 0.f, m2 = 0.f;
    for (int i = i0 + tid; i <= i1; i += 256) {
        const float a = fabsf(J.approx[i]);
        m1 = fmaxf(m1, a);
        if (i < J.sanity) m2 = fmaxf(m2, a);
    }
    s_red[tid] = m1;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (tid < o) s_red[tid] = fmaxf(s_red[tid], s_red[tid + o]); __syncthreads(); }
    m1 = s_red[0];
    __syncthreads();
    s_red[tid] = m2;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (tid < o) s_red[tid] = fmaxf(s_red[tid], s_red[tid + o]); __syncthreads(); }
    m2 = s_red[0];
    __syncthreads();
    // A signal whose power before normalisation is zero is identically zero (the weak simulator's
    // reference blocks quantise to a constant byte): every product is +-0, every lag's correlation
    // is exactly 0, and the reference's strict `>` keeps its initial (first lag, 0.0).  One
    // candidate says the same; without this the flat surface makes every lag a candidate.
    if (m1 == 0.f && ((J.t_stats && J.t_stats[ST_POWER1] == 0.0) || (J.s_stats && J.s_stats[ST_POWER1] == 0.0))) {
        if (tid == 0) { J.cand[0] = i0; *J.n_cand = 1; *J.approx_max = 0.f; }
        return;
    }
    const float thr1 = m1 - J.tol, thr2 = m2 - J.tol;
    // candidates are few: collect them with a shared-memory ticket, then order them by rank
    // (ascending lag, as the reference scans).  More than 256 means overflow anyway.
    __shared__ int s_list[256];
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int i = i0 + tid; i <= i1; i += 256) {
        const float a = fabsf(J.approx[i]);
        bool take = a >= thr1 || (i < J.sanity && a >= thr2);
        if (!take && J.neighbours) {
            if (i > i0 && fabsf(J.approx[i - 1]) >= thr1) take = true;
            if (i < i1 && fabsf(J.approx[i + 1]) >= thr1) take = true;
        }
        if (take) {
            const int pos = atomicAdd(&s_base, 1);
            if (pos < 256) s_list[pos] = i;
        }
    }
    __syncthreads();
    const int found = s_base;
    if (found <= 256 && tid < found) {
        const int mine = s_list[tid];
        int rank = 0;
        for (int k = 0; k < found; k++) rank += s_list[k] < mine ? 1 : 0;
        if (rank < J.max_cand) J.cand[rank] = mine;
    }
    if (tid == 0) {
        *J.n_cand = s_base;  // may exceed max_cand: the peak kernel raises the overflow flag
        *J.approx_max = m1;
    }
}

// ---------------------------------------------------------------- exact evaluation of the candidates
constexpr int kCandThreads = 256;
constexpr int kCandChunk = 2048;   // template samples staged per step
constexpr int kCandSpan = 2048;    // lag span served from shared memory
constexpr int kCandGroup = 8;      // candidates evaluated per sweep

// f32 x f32 widened to f64 is an exact product (48 significant bits), so one fused multiply-add rounds
// exactly as the separate multiply and add of the statement (acc + (double)t * (double)s) would: bit-identical,
// and one FP64-pipe instruction per (sample, candidate) instead of two.
__device__ __forceinline__ double fma_exact(float t, float s, double acc) { return __fma_rn((double)t, (double)s, acc); }

// Inner sweep over one staged chunk for NG candidates (NG = 1, 2, 4, 8: no wasted lanes
// of FP64 work when the peak is sharp and only one lag needs the exact treatment).
template <int NG, bool STAGED, bool F64>
__device__ __forceinline__ void cand_sweep(const float *s_t, const float *s_s, const PairJob &J, float sc_s, i64 sbase,
                                           int clen, const int (&off)[kCandGroup], double (&acc)[kCandGroup])
{
    for (int i = threadIdx.x; i < clen; i += kCandThreads) {
        const float tv = s_t[i];
#pragma unroll
        for (int c = 0; c < NG; c++) {
            float sv;
            if (STAGED) {
                sv = s_s[i + off[c]];
            } else {
                const i64 q = sbase + i + off[c];
                sv = (q >= 0 && q < J.sl) ? __fmul_rn(J.s_re[q], sc_s) : 0.f;
            }
            if (F64) acc[c] = fma_exact(tv, sv, acc[c]);
            else acc[c] = __dadd_rn(acc[c], (double)__fmul_rn(tv, sv));
        }
    }
}

template <bool STAGED, bool F64>
__device__ __forceinline__ void cand_sweep_ng(int ng, const float *s_t, const float *s_s, const PairJob &J, float sc_s,
                                              i64 sbase, int clen, const int (&off)[kCandGroup],
                                              double (&acc)[kCandGroup])
{
    if (ng == 1) cand_sweep<1, STAGED, F64>(s_t, s_s, J, sc_s, sbase, clen, off, acc);
    else if (ng == 2) cand_sweep<2, STAGED, F64>(s_t, s_s, J, sc_s, sbase, clen, off, acc);
    else if (ng <= 4) cand_sweep<4, STAGED, F64>(s_t, s_s, J, sc_s, sbase, clen, off, acc);
    else cand_sweep<8, STAGED, F64>(s_t, s_s, J, sc_s, sbase, clen, off, acc);
}

// Single candidate, vector path: the template block is 16-byte aligned, the signal starts A
// floats past an aligned address.  Each thread takes 4 consecutive samples per step from
// 128-bit loads (two for the signal, picked apart by the compile-time shift A), 4 steps in
// flight: 192 bytes of loads per thread instead of 48, which is what this latency-bound
// sweep needs.  Returns the thread's partial sum over samples [0, 4 * (len / 4)).
template <int A, int NC, bool F64>
__device__ __forceinline__ void cand_sweep_vec(const float *__restrict__ tp, const float *__restrict__ sp, int len,
                                               float sc_t, float sc_s, double (&acc)[NC])
{
    constexpr int NV = (A + NC + 2) / 4 + 1;   // 128-bit signal loads that cover samples A .. A + NC + 2
    const float4 *__restrict__ tp4 = reinterpret_cast<const float4 *>(tp);
    const float4 *__restrict__ sp4 = reinterpret_cast<const float4 *>(sp - A);
    const int n4 = len >> 2;
#pragma unroll
    for (int c = 0; c < NC; c++) acc[c] = 0.0;
    auto mac = [&](const float4 &t, const float4 (&s)[NV]) {
        float w[4 * NV];
#pragma unroll
        for (int v = 0; v < NV; v++) { w[4 * v] = s[v].x; w[4 * v + 1] = s[v].y; w[4 * v + 2] = s[v].z; w[4 * v + 3] = s[v].w; }
#pragma unroll
        for (int i = 0; i < 4 * NV; i++) w[i] = __fmul_rn(w[i], sc_s);
        const float tv[4] = {__fmul_rn(t.x, sc_t), __fmul_rn(t.y, sc_t), __fmul_rn(t.z, sc_t), __fmul_rn(t.w, sc_t)};
#pragma unroll
        for (int k = 0; k < 4; k++) {
#pragma unroll
            for (int c = 0; c < NC; c++) {
                if (F64) acc[c] = fma_exact(tv[k], w[A + k + c], acc[c]);
                else acc[c] = __dadd_rn(acc[c], (double)__fmul_rn(tv[k], w[A + k + c]));
            }
        }
    };
    constexpr int U = NC == 1 ? 4 : 2;   // steps in flight
    int j = threadIdx.x;
    for (; j + (U - 1) * kCandThreads < n4; j += U * kCandThreads) {
        float4 t[U], sv[U][NV];
#pragma unroll
        for (int u = 0; u < U; u++) {
            t[u] = tp4[j + u * kCandThreads];
#pragma unroll
            for (int v = 0; v < NV; v++) sv[u][v] = sp4[j + u * kCandThreads + v];
        }
#pragma unroll
        for (int u = 0; u < U; u++) mac(t[u], sv[u]);
    }
    for (; j < n4; j += kCandThreads) {
        float4 sv[NV];
#pragma unroll
        for (int v = 0; v < NV; v++) sv[v] = sp4[j + v];
        mac(tp4[j], sv);
    }
}

template <int NC, bool F64>
__device__ __forceinline__ void cand_sweep_vec_a(int a, const float *__restrict__ tp, const float *__restrict__ sp, int len,
                                                 float sc_t, float sc_s, double (&acc)[NC])
{
    if (a == 0) cand_sweep_vec<0, NC, F64>(tp, sp, len, sc_t, sc_s, acc);
    else if (a == 1) cand_sweep_vec<1, NC, F64>(tp, sp, len, sc_t, sc_s, acc);
    else if (a == 2) cand_sweep_vec<2, NC, F64>(tp, sp, len, sc_t, sc_s, acc);
    else cand_sweep_vec<3, NC, F64>(tp, sp, len, sc_t, sc_s, acc);
}

// One CTA: block b of the template (B samples) of one pair, every candidate.
// f32 product, widened, f64 accumulate (processor.go:703-705); per-thread partial sums in
// ascending i, then a fixed reduction tree -- deterministic, not the reference's order
// (differences ~1e-16 relative; the brute-force kernel keeps the reference's order).
__global__ void __launch_bounds__(kCandThreads) k_corr_candidates(const PairJob *jobs, const CandJob *cjobs, int n_jobs)
{
    __shared__ float s_t[kCandChunk];
    __shared__ float s_s[kCandChunk + kCandSpan];
    __shared__ double s_red[kCandGroup][kCandThreads / 32];
    // pair fastest: the CTAs that work on block b of every pair of a window are launched
    // side by side, so the planes the pairs share (3 stations: each plane serves 2 pairs)
    // come out of L2 for all but the first reader
    const int pair = (int)(blockIdx.x % (unsigned)n_jobs);
    const PairJob &J = jobs[pair];
    const CandJob &C = cjobs[pair];
    const i64 b = blockIdx.x / (unsigned)n_jobs;
    if (b >= J.nb) return;
    const int n_cand = min(*C.n_cand, C.max_cand);
    if (n_cand <= 0) return;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const float sc_t = (float)J.t_stats[ST_SCALE], sc_s = (float)J.s_stats[ST_SCALE];
    const i64 B = J.block;
    const i64 blk_start = b * B;
    const i64 blk_len = min(B, J.n_t - blk_start);
    const bool exact_f64 = J.variant == CORR_EXTENDED;

    for (int g0 = 0; g0 < n_cand; g0 += kCandGroup) {
        const int ng = min(kCandGroup, n_cand - g0);
        int off[kCandGroup];  // lag offsets from the group's first (lowest) candidate
        const int dmin = C.cand[g0];
#pragma unroll
        for (int c = 0; c < kCandGroup; c++) off[c] = C.cand[g0 + min(c, ng - 1)] - dmin;
        const int span = C.cand[g0 + ng - 1] - dmin;  // candidates are ascending
        const bool staged = span <= kCandSpan;
        double acc[kCandGroup];
#pragma unroll
        for (int c = 0; c < kCandGroup; c++) acc[c] = 0.0;
        const i64 s_first = blk_start + J.lag0 + dmin;
        const bool run3 = ng == 3 && off[1] == 1 && off[2] == 2;   // a peak and its two neighbours (EXTENDED)
        if ((ng == 1 || run3) && s_first >= 0 && s_first + blk_len + 12 <= J.sl && ((J.t_off + blk_start) & 3) == 0 &&
            (reinterpret_cast<uintptr_t>(J.t_re) & 15) == 0 && (reinterpret_cast<uintptr_t>(J.s_re) & 15) == 0) {
            const float *__restrict__ tp = J.t_re + J.t_off + blk_start;
            const float *__restrict__ sp = J.s_re + s_first;
            const int len = (int)blk_len;
            const int a = (int)(s_first & 3);
            if (run3) {
                double v[3];
                if (exact_f64) cand_sweep_vec_a<3, true>(a, tp, sp, len, sc_t, sc_s, v);
                else cand_sweep_vec_a<3, false>(a, tp, sp, len, sc_t, sc_s, v);
                acc[0] = v[0]; acc[1] = v[1]; acc[2] = v[2];
            } else {
                double v[1];
                if (exact_f64) cand_sweep_vec_a<1, true>(a, tp, sp, len, sc_t, sc_s, v);
                else cand_sweep_vec_a<1, false>(a, tp, sp, len, sc_t, sc_s, v);
                acc[0] = v[0];
            }
            for (int i = (len & ~3) + tid; i < len; i += kCandThreads) {  // the block's last len % 4 samples
                const float t = __fmul_rn(tp[i], sc_t);
                for (int c = 0; c < ng; c++) {
                    const float q = __fmul_rn(sp[i + c], sc_s);
                    acc[c] = exact_f64 ? fma_exact(t, q, acc[c]) : __dadd_rn(acc[c], (double)__fmul_rn(t, q));
                }
            }
        } else if (ng <= 2 && s_first >= 0 && s_first + blk_len + span <= J.sl) {
            // sharp peak (the common case): stream both signals straight from global
            // memory, 4 independent strides in flight per thread, no staging, no barriers
            const float *__restrict__ tp = J.t_re + J.t_off + blk_start;
            const float *__restrict__ sp = J.s_re + s_first;
            const int o1 = off[1];
            const int len = (int)blk_len;
            int i = tid;
            for (; i + 3 * kCandThreads < len; i += 4 * kCandThreads) {
                float tv[4], s0[4], s1[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    tv[u] = tp[i + u * kCandThreads];
                    s0[u] = sp[i + u * kCandThreads];
                    s1[u] = ng == 2 ? sp[i + u * kCandThreads + o1] : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const float t = __fmul_rn(tv[u], sc_t), a = __fmul_rn(s0[u], sc_s), bb = __fmul_rn(s1[u], sc_s);
                    if (exact_f64) {
                        acc[0] = fma_exact(t, a, acc[0]);
                        if (ng == 2) acc[1] = fma_exact(t, bb, acc[1]);
                    } else {
                        acc[0] = __dadd_rn(acc[0], (double)__fmul_rn(t, a));
                        if (ng == 2) acc[1] = __dadd_rn(acc[1], (double)__fmul_rn(t, bb));
                    }
                }
            }
            for (; i < len; i += kCandThreads) {
                const float t = __fmul_rn(tp[i], sc_t), a = __fmul_rn(sp[i], sc_s);
                const float bb = ng == 2 ? __fmul_rn(sp[i + o1], sc_s) : 0.f;
                if (exact_f64) {
                    acc[0] = fma_exact(t, a, acc[0]);
                    if (ng == 2) acc[1] = fma_exact(t, bb, acc[1]);
                } else {
                    acc[0] = __dadd_rn(acc[0], (double)__fmul_rn(t, a));
                    if (ng == 2) acc[1] = __dadd_rn(acc[1], (double)__fmul_rn(t, bb));
                }
            }
        } else
        for (i64 c0 = 0; c0 < blk_len; c0 += kCandChunk) {
            const int clen = (int)min((i64)kCandChunk, blk_len - c0);
            __syncthreads();
            const i64 tbase = J.t_off + blk_start + c0;
            for (int i = tid; i < clen; i += kCandThreads) s_t[i] = __fmul_rn(J.t_re[tbase + i], sc_t);
            const i64 sbase = blk_start + c0 + J.lag0 + dmin;
            if (staged) {
                for (int i = tid; i < clen + span; i += kCandThreads) {
                    const i64 q = sbase + i;
                    s_s[i] = (q >= 0 && q < J.sl) ? __fmul_rn(J.s_re[q], sc_s) : 0.f;
                }
            }
            __syncthreads();
            if (staged) {
                if (exact_f64) cand_sweep_ng<true, true>(ng, s_t, s_s, J, sc_s, sbase, clen, off, acc);
                else cand_sweep_ng<true, false>(ng, s_t, s_s, J, sc_s, sbase, clen, off, acc);
            } else {
                if (exact_f64) cand_sweep_ng<false, true>(ng, s_t, s_s, J, sc_s, sbase, clen, off, acc);
                else cand_sweep_ng<false, false>(ng, s_t, s_s, J, sc_s, sbase, clen, off, acc);
            }
        }
        // block reduction, fixed order
#pragma unroll
        for (int c = 0; c < kCandGroup; c++) {
            if (c < ng) {   // ng is uniform: a sharp peak reduces one value, not eight
                const double w = warp_sum(acc[c]);
                if (lane == 0) s_red[c][wid] = w;
            }
        }
        __syncthreads();
        if (tid < ng) {
            double v = 0.0;
#pragma unroll
            for (int w = 0; w < kCandThreads / 32; w++) v += s_red[tid][w];
            // processor.go:709  blockCorr /= blockSize  (EXTENDED keeps the raw sum)
            if (!exact_f64) v = v / (double)B;
            C.blocksums[(size_t)(g0 + tid) * J.nb + b] = v;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- peak from the exact candidate values
// One CTA (8 warps) per pair: warp w adds the blocks of candidates w, w+8, ...; then
// thread 0 runs the reference's selection (strict >, ascending lag; sanity re-search).
// A bounded record's candidates all lie in its run (k_select_candidates), so only the
// runner-up, the BOUNDED flag and an empty run's EMPTY flag need the run here.
__global__ void __launch_bounds__(256) k_peak_candidates(const PairJob *jobs, const CandJob *cjobs, const PeakJob *pjobs)
{
    __shared__ double s_val[kMaxCand];
    __shared__ float s_red[256];
    const PairJob &J = jobs[blockIdx.x];
    const CandJob &C = cjobs[blockIdx.x];
    const PeakJob &K = pjobs[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n_all = *C.n_cand;
    const int n_cand = min(n_all, C.max_cand);
    // few candidates and many blocks (the sharp-peak, long-signal case): the whole CTA adds
    // one candidate's blocks -- thread t takes blocks t, t + 256, ...; then the fixed tree
    __shared__ double s_part[8];
    const bool wide = n_cand < 8 && J.nb > 1024;
    for (int c = wide ? 0 : wid; c < n_cand; c += wide ? 1 : 8) {
        double v = 0.0;
        if (wide) {
            for (i64 b = tid; b < J.nb; b += 256) v += C.blocksums[(size_t)c * J.nb + b];
            v = warp_sum(v);
            __syncthreads();
            if (lane == 0) s_part[wid] = v;
            __syncthreads();
            v = 0.0;
            if (tid == 0)
                for (int w = 0; w < 8; w++) v += s_part[w];
        } else {
            for (i64 b = lane; b < J.nb; b += 32) v += C.blocksums[(size_t)c * J.nb + b];
            v = warp_sum(v);
        }
        if (wide ? tid == 0 : lane == 0) {
            if (J.variant == CORR_EXTENDED) v = J.n_t > 0 ? v / (double)J.n_t : 0.0;
            else {
                v = J.nb > 0 ? v / (double)J.nb : 0.0;
                if (J.variant == CORR_SOURCE) v = v * sqrt((double)(J.nb * J.block));
            }
            s_val[c] = v;
        }
    }
    __syncthreads();
    // first pass over the candidates (ascending lag)
    int best = -1, rbest = -1;
    double bv = 0.0, rv = 0.0;
    if (tid == 0) {
        for (int c = 0; c < n_cand; c++)
            if (fabs(s_val[c]) > fabs(bv)) { bv = s_val[c]; best = c; }
    }
    // runner-up magnitude from the approximate search (for the margin field)
    __shared__ int s_best_idx;
    if (tid == 0) s_best_idx = best >= 0 ? C.cand[best] : -1;
    __syncthreads();
    int i0, i1;
    const bool bounded = bound_run(K.bound, K.lag_origin, K.decim, K.n_lags, &i0, &i1);
    float ru = 0.f;
    for (int i = i0 + tid; i <= i1; i += 256)
        if (i != s_best_idx) ru = fmaxf(ru, fabsf(C.approx[i]));
    s_red[tid] = ru;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (tid < o) s_red[tid] = fmaxf(s_red[tid], s_red[tid + o]); __syncthreads(); }
    if (tid != 0) return;
    PeakRec r;
    r.lag = 0; r.flags = K.flags; r.corr = 0.0; r.frac = 0.f; r.margin = 0.f; r.first_lag = 0; r.n_blocks = K.nb;
    if (n_all > C.max_cand) r.flags |= 0x10u;  // TDOA_PEAK_OVERFLOW: the host re-runs this pair brute force
    r.flags |= (uint32_t)min(n_all, 255) << 16;  // TDOA_PEAK_NCAND: exactly evaluated lags
    if (bounded) r.flags |= i0 > i1 ? TDOA_PEAK_BOUNDED | TDOA_PEAK_EMPTY : TDOA_PEAK_BOUNDED;
    if (K.nb > 0 && best >= 0) {
        const int bi = C.cand[best];
        r.lag = bi + K.lag_origin;
        r.first_lag = r.lag;
        r.corr = bv;
        r.margin = (float)((fabs(bv) - (double)s_red[0]) / fabs(bv));
        if (K.variant == CORR_BINARY && K.sanity > 0 && bi > K.sanity) {
            for (int c = 0; c < n_cand && C.cand[c] < K.sanity; c++)
                if (fabs(s_val[c]) > fabs(rv)) { rv = s_val[c]; rbest = c; }
            if (rbest >= 0 && fabs(rv) > 0.5 * fabs(bv)) {
                r.lag = C.cand[rbest];
                r.corr = rv;
                r.flags |= 0x1u;  // TDOA_PEAK_RESEARCHED
            }
        }
        if (K.variant == CORR_EXTENDED) {
            // neighbours were selected as candidates, so they sit next to `best`
            const bool has_l = best > 0 && C.cand[best - 1] == bi - 1;
            const bool has_r = best + 1 < n_cand && C.cand[best + 1] == bi + 1;
            if (has_l && has_r) {
                const double a = fabs(s_val[best - 1]), m = fabs(bv), d = fabs(s_val[best + 1]);
                const double den = a - 2.0 * m + d;
                r.frac = den != 0.0 ? (float)(0.5 * (a - d) / den) : 0.f;
            } else {
                r.flags |= 0x2u;  // TDOA_PEAK_EDGE
            }
        }
    }
    *K.out = r;
    if (K.first_corr) *K.first_corr = (K.nb > 0 && best >= 0) ? bv : 0.0;
}

}  // namespace

size_t fft_partials_bytes(int n_cta) { return (size_t)n_cta * kBins * sizeof(float2); }

int fft_setup(cudaStream_t st, float2 **d_tw)
{
    // twiddles W_8192^k, computed in double on the host
    static float2 h_tw[kN];
    for (int k = 0; k < kN; k++) {
        const double a = -2.0 * 3.14159265358979323846 * (double)k / (double)kN;
        h_tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    if (cudaMalloc(d_tw, sizeof(h_tw)) != cudaSuccess) return -1;
    if (cudaMemcpyAsync(*d_tw, h_tw, sizeof(h_tw), cudaMemcpyHostToDevice, st) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_fft_segments, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_fft_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) != cudaSuccess) return -1;
    return 0;
}

void launch_fft_segments(const FftJob *d_jobs, int n_jobs, int max_cta, const float2 *d_tw, cudaStream_t st)
{
    if (n_jobs <= 0 || max_cta <= 0) return;
    k_fft_segments<<<dim3(max_cta, n_jobs), kThreads, kSmemBytes, st>>>(d_jobs, d_tw);
}

void launch_fft_reduce(const FftJob *d_jobs, int n_jobs, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_fft_reduce<<<dim3((kBins + 255) / 256, n_jobs), 256, 0, st>>>(d_jobs);
}

void launch_fft_finish(const FftJob *d_jobs, int n_jobs, const float2 *d_tw, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_fft_finish<<<n_jobs, kThreads, kSmemBytes, st>>>(d_jobs, d_tw);
}

void launch_select_candidates(const SelJob *d_jobs, int n_jobs, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_select_candidates<<<n_jobs, 256, 0, st>>>(d_jobs);
}

void launch_corr_candidates(const PairJob *d_jobs, const CandJob *d_cjobs, int n_jobs, i64 max_nb, cudaStream_t st)
{
    if (n_jobs <= 0 || max_nb <= 0) return;
    k_corr_candidates<<<(unsigned)(max_nb * n_jobs), kCandThreads, 0, st>>>(d_jobs, d_cjobs, n_jobs);
}

void launch_peak_candidates(const PairJob *d_jobs, const CandJob *d_cjobs, const PeakJob *d_pjobs, int n_jobs,
                            cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_peak_candidates<<<n_jobs, 256, 0, st>>>(d_jobs, d_cjobs, d_pjobs);
}

}  // namespace tdoa
