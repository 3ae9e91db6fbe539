// preprocess.cu -- per-signal stage of the path: uint8 IQ unpack, power, DC, the FM
// discriminator / envelope, the edge-normalised box-car filters and normalisation.
//
// Replaces, per signal:  loadIQData (processor.go:193-201), calculateSignalPower
// (:322-333), removeDCBias (:299-319), applyLowPassFilter (:270-296) and its HP/BP/
// notch compositions (:354-434), normalizeSignal (:336-351), and the shipped binary's
// convertToInstantaneousFrequency / envelope (ELF 0x49d120 / 0x49d021).
//
// Layout: signals are planar f32 (re[], im[]); im == nullptr means "identically 0",
// which is what the discriminator and envelope branches produce.
#include "discriminate.cuh"
#include "kernels.h"

namespace tdoa {

namespace {

constexpr int kThreads = 256;
constexpr int kBoxTile = 2048;   // outputs per CTA of the box-car kernel
constexpr int kBoxHalfMax = 500; // processor.go:404 clamps the window to 1000

__device__ __forceinline__ float dc_from_sum(double sum, i64 n)
{
    // processor.go:309  dcBias /= complex(float32(len), 0): f32 accumulator divided by
    // f32(n), correctly rounded.  The accumulator here is the exactly rounded sum.
    return __fdiv_rn((float)sum, (float)n);
}

// ---------------------------------------------------------------- power
__global__ void __launch_bounds__(kThreads) k_power(const SigJob *jobs)
{
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    double acc = 0.0;
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < J.n; i += stride) {
        const float2 v = load_sample(J.src, i);
        acc += (double)mag2_f32(v.x, v.y);
    }
    double part[1] = {block_sum(acc, scratch)}, total[1];
    if (grid_sum_last<1>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total))
        J.stats[ST_POWER0] = J.n > 0 ? total[0] / (double)J.n : 0.0;
}

// ---------------------------------------------------------------- unpack to planes (+ DC sums)
__global__ void __launch_bounds__(kThreads) k_unpack(const SigJob *jobs)
{
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    double sr = 0.0, si = 0.0;
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < J.n; i += stride) {
        const float2 v = load_sample(J.src, i);
        J.p_re[i] = v.x;
        J.p_im[i] = v.y;
        sr += (double)v.x;
        si += (double)v.y;
    }
    double part[2], total[2];
    part[0] = block_sum(sr, scratch);
    part[1] = block_sum(si, scratch);
    if (grid_sum_last<2>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
        J.stats[ST_SUM_RE] = total[0];
        J.stats[ST_SUM_IM] = total[1];
        J.stats[ST_DC_RE] = J.n > 0 ? (double)dc_from_sum(total[0], J.n) : 0.0;
        J.stats[ST_DC_IM] = J.n > 0 ? (double)dc_from_sum(total[1], J.n) : 0.0;
    }
}

// ---------------------------------------------------------------- FM discriminator (discriminate.cuh)
__global__ void __launch_bounds__(kThreads) k_demod(const SigJob *jobs)
{
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    double sr = 0.0;
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < J.n; i += stride) {
        const i64 k = i == 0 ? 1 : i;  // out[0] = out[1]
        const float y = discriminate(load_sample(J.src, k - 1), load_sample(J.src, k));
        J.p_re[i] = y;
        sr += (double)y;
    }
    double part[1] = {block_sum(sr, scratch)}, total[1];
    if (grid_sum_last<1>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
        J.stats[ST_SUM_RE] = total[0];
        J.stats[ST_SUM_IM] = 0.0;
        J.stats[ST_DC_RE] = J.n > 0 ? (double)dc_from_sum(total[0], J.n) : 0.0;
        J.stats[ST_DC_IM] = 0.0;
    }
}

// ---------------------------------------------------------------- envelope (ELF 0x49d021)
__global__ void __launch_bounds__(kThreads) k_envelope(const SigJob *jobs)
{
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    double sr = 0.0;
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < J.n; i += stride) {
        const float2 v = load_sample(J.src, i);
        const float y = __fsqrt_rn(mag2_f32(v.x, v.y));
        J.p_re[i] = y;
        sr += (double)y;
    }
    double part[1] = {block_sum(sr, scratch)}, total[1];
    if (grid_sum_last<1>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
        J.stats[ST_SUM_RE] = total[0];
        J.stats[ST_SUM_IM] = 0.0;
        J.stats[ST_DC_RE] = J.n > 0 ? (double)dc_from_sum(total[0], J.n) : 0.0;
        J.stats[ST_DC_IM] = 0.0;
    }
}

// ---------------------------------------------------------------- sequential f32 DC sum
// processor.go:304-309 accumulates the DC bias in a complex64, i.e. two sequential f32
// chains; their rounding error is far from negligible on DC-heavy signals (the
// envelope branch), so parity of the printed correlation needs the same chain.  One
// warp per (signal, component): lanes fetch 32 consecutive samples at a time (next
// batch prefetched), every lane then walks the same 32 dependent adds.
__global__ void __launch_bounds__(32) k_seqsum(const SigJob *jobs)
{
    const SigJob &J = jobs[blockIdx.x];
    const float *x = blockIdx.y == 0 ? J.q_re : J.q_im;
    const int lane = threadIdx.x;
    if (!x) {
        if (lane == 0) J.stats[blockIdx.y == 0 ? ST_DC_RE : ST_DC_IM] = 0.0;
        return;
    }
    const i64 n = J.n;
    float s = 0.f;
    constexpr int U = 4;
    float cur[U], nxt[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
        const i64 i = (i64)u * 32 + lane;
        cur[u] = i < n ? x[i] : 0.f;
    }
    for (i64 base = 0; base < n; base += 32 * U) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const i64 i = base + 32 * U + (i64)u * 32 + lane;
            nxt[u] = i < n ? x[i] : 0.f;
        }
        const i64 left = n - base;
        if (left >= 32 * U) {
#pragma unroll
            for (int u = 0; u < U; u++)
#pragma unroll
                for (int k = 0; k < 32; k++) s = __fadd_rn(s, __shfl_sync(0xffffffffu, cur[u], k));
        } else {
#pragma unroll
            for (int u = 0; u < U; u++)
#pragma unroll
                for (int k = 0; k < 32; k++) {
                    const float v = __shfl_sync(0xffffffffu, cur[u], k);
                    if ((i64)u * 32 + k < left) s = __fadd_rn(s, v);
                }
        }
#pragma unroll
        for (int u = 0; u < U; u++) cur[u] = nxt[u];
    }
    if (lane == 0) J.stats[blockIdx.y == 0 ? ST_DC_RE : ST_DC_IM] = n > 0 ? (double)__fdiv_rn(s, (float)n) : 0.0;
}

// ---------------------------------------------------------------- box-car
// processor.go:270-296: out[i] = (sum_{j=i-h..i+h, in range} in[j]) / count, the sum
// taken in ascending j from a zero f32 accumulator (so every output is an independent
// sequential sum and the result is bit-identical to the reference's).
// mode BOX_HP gives in[i] - LP(in)[i] (processor.go:384-394).  sub_dc folds
// removeDCBias (in[j] - dc) into the tile load.  window <= 1 is the identity (:271).
__global__ void __launch_bounds__(kThreads) k_boxcar(const SigJob *jobs)
{
    __shared__ float s_re[kBoxTile + 2 * kBoxHalfMax];
    __shared__ float s_im[kBoxTile + 2 * kBoxHalfMax];
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    const i64 n = J.n;
    const bool has_im = J.q_im != nullptr;
    const int h = J.window <= 1 ? 0 : J.window / 2;
    const i64 i0 = (i64)blockIdx.x * kBoxTile;
    double pacc = 0.0;
    if (i0 < n) {
        const i64 lo = max((i64)0, i0 - h);
        const i64 hi = min(n, i0 + kBoxTile + h);  // exclusive
        const float dcr = J.sub_dc ? (float)J.stats[ST_DC_RE] : 0.f;
        const float dci = J.sub_dc ? (float)J.stats[ST_DC_IM] : 0.f;
        for (i64 j = lo + threadIdx.x; j < hi; j += kThreads) {
            float vr = J.q_re[j];
            if (J.sub_dc) vr = __fsub_rn(vr, dcr);
            s_re[j - lo] = vr;
            if (has_im) {
                float vi = J.q_im[j];
                if (J.sub_dc) vi = __fsub_rn(vi, dci);
                s_im[j - lo] = vi;
            }
        }
        __syncthreads();
        const i64 iend = min(n, i0 + kBoxTile);
        for (i64 i = i0 + threadIdx.x; i < iend; i += kThreads) {
            float outr, outi = 0.f;
            if (h == 0) {
                outr = s_re[i - lo];
                if (has_im) outi = s_im[i - lo];
            } else {
                const i64 a = max((i64)0, i - h), b = min(n - 1, i + h);
                const int ja = (int)(a - lo), cnt = (int)(b - a + 1);
                const float fc = (float)cnt;
                float ar = 0.f;
#pragma unroll 4
                for (int j = 0; j < cnt; j++) ar = __fadd_rn(ar, s_re[ja + j]);
                outr = __fdiv_rn(ar, fc);
                if (J.mode == BOX_HP) outr = __fsub_rn(s_re[i - lo], outr);
                if (has_im) {
                    float ai = 0.f;
#pragma unroll 4
                    for (int j = 0; j < cnt; j++) ai = __fadd_rn(ai, s_im[ja + j]);
                    outi = __fdiv_rn(ai, fc);
                    if (J.mode == BOX_HP) outi = __fsub_rn(s_im[i - lo], outi);
                }
            }
            J.p_re[i] = outr;
            if (has_im) J.p_im[i] = outi;
            pacc += (double)mag2_f32(outr, outi);
        }
    }
    if (J.want_power) {
        double part[1] = {block_sum(pacc, scratch)}, total[1];
        if (grid_sum_last<1>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
            const double p = n > 0 ? total[0] / (double)n : 0.0;
            J.stats[ST_POWER1] = p;
            // processor.go:343-345  scale = f32(1/sqrt(power)); power <= 0 leaves the signal alone
            J.stats[ST_SCALE] = p > 0.0 ? (double)(float)(1.0 / sqrt(p)) : 1.0;
        }
    }
}

// ---------------------------------------------------------------- wide box-car, O(1) per sample
// EXTENDED mode only (engine-defined arithmetic; oracle: orc_lowpass_wide).  The reference's
// box-car (processor.go:270-296) spends one f32 addition per tap and output -- 1001 per sample in
// the weak branch's 100 Hz high-pass -- and only that brute-force walk reproduces its f32 rounding
// chain bit for bit, so SOURCE and BINARY keep it (k_boxcar).  Here the window sum is the
// difference of two entries of an f64 prefix sum over the staged tile: the same taps, the same edge
// normalisation (divisor = taps in range), one rounding to f32 at the divide.  It differs from the
// reference's chain by that chain's own f32 rounding (~1e-6 relative), which the mode does not promise.
// Tiles of 6144 outputs (round 1: 2048, where the 1000-sample halo was half of what a CTA staged and scanned:
// 0.22 of the HBM roofline), 512 threads, the staged samples and their prefix sums in 86 KB of dynamic shared memory.
constexpr int kSlideTile = 6144;
constexpr int kSlideThreads = 512;
constexpr int kSlideLen = kSlideTile + 2 * kBoxHalfMax;
constexpr int kSlideSmem = kSlideLen * (int)(sizeof(float) + sizeof(double));

__global__ void __launch_bounds__(kSlideThreads, 2) k_boxcar_slide(const SigJob *jobs)
{
    constexpr int kBoxTile = kSlideTile, kThreads = kSlideThreads;   // this kernel's own tile and CTA size
    constexpr int kLen = kSlideLen;
    constexpr int kPer = (kLen + kThreads - 1) / kThreads;   // 14 consecutive entries per thread
    extern __shared__ __align__(16) unsigned char slide_raw[];
    double *s_p = reinterpret_cast<double *>(slide_raw);      // inclusive prefix sums of s_x
    float *s_x = reinterpret_cast<float *>(s_p + kLen);
    __shared__ double s_w[kThreads / 32];
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    const i64 n = J.n;
    const int h = J.window <= 1 ? 0 : J.window / 2;
    const i64 i0 = (i64)blockIdx.x * kBoxTile;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    double pacc = 0.0;
    if (i0 < n) {   // uniform per CTA
        const i64 lo = max((i64)0, i0 - h);
        const i64 hi = min(n, i0 + kBoxTile + h);  // exclusive
        const int len = (int)(hi - lo);
        const i64 iend = min(n, i0 + kBoxTile);
        for (int comp = 0; comp < 2; comp++) {
            const float *__restrict__ q = comp == 0 ? J.q_re : J.q_im;
            float *__restrict__ p = comp == 0 ? J.p_re : J.p_im;
            if (!q) break;
            const float dc = J.sub_dc ? (float)J.stats[comp == 0 ? ST_DC_RE : ST_DC_IM] : 0.f;
            __syncthreads();
            for (int j = tid; j < len; j += kThreads) s_x[j] = J.sub_dc ? __fsub_rn(q[lo + j], dc) : q[lo + j];
            __syncthreads();
            // block-wide inclusive scan: a thread's 12 entries, then warps, then the warp totals
            const int j0 = tid * kPer;
            double loc[kPer], run = 0.0;
#pragma unroll
            for (int k = 0; k < kPer; k++) { run += j0 + k < len ? (double)s_x[j0 + k] : 0.0; loc[k] = run; }
            double inc = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const double t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
            if (lane == 31) s_w[wid] = inc;
            __syncthreads();
            double base = inc - run;                       // exclusive within the warp
            for (int w = 0; w < wid; w++) base += s_w[w];  // fixed order
#pragma unroll
            for (int k = 0; k < kPer; k++) if (j0 + k < len) s_p[j0 + k] = base + loc[k];
            __syncthreads();
            for (i64 i = i0 + tid; i < iend; i += kThreads) {
                float out = s_x[i - lo];
                if (h > 0) {
                    const i64 a = max((i64)0, i - h), b = min(n - 1, i + h);
                    const int ja = (int)(a - lo), jb = (int)(b - lo);
                    const double sum = s_p[jb] - (ja > 0 ? s_p[ja - 1] : 0.0);
                    const float lp = (float)(sum / (double)(int)(b - a + 1));
                    out = J.mode == BOX_HP ? __fsub_rn(out, lp) : lp;
                }
                p[i] = out;
                pacc += (double)__fmul_rn(out, out);
            }
        }
    }
    if (J.want_power) {
        // f32 re^2 + im^2 per sample in the reference (processor.go:328); here the two squares are
        // added in f64 (the mode's own arithmetic, as above)
        double part[1] = {block_sum(pacc, scratch)}, total[1];
        if (grid_sum_last<1>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
            const double pw = n > 0 ? total[0] / (double)n : 0.0;
            J.stats[ST_POWER1] = pw;
            J.stats[ST_SCALE] = pw > 0.0 ? (double)(float)(1.0 / sqrt(pw)) : 1.0;
        }
    }
}

// ---------------------------------------------------------------- notch combine
// processor.go:428-431  out = s - 0.8 * band  (complex64 constant: one f32 rounding)
__global__ void __launch_bounds__(kThreads) k_notch_combine(const SigJob *jobs)
{
    const SigJob &J = jobs[blockIdx.y];
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < J.n; i += stride) {
        J.p_re[i] = __fsub_rn(J.q_re[i], __fmul_rn(J.r_re[i], 0.8f));
        if (J.q_im) J.p_im[i] = __fsub_rn(J.q_im[i], __fmul_rn(J.r_im[i], 0.8f));
    }
}

// ---------------------------------------------------------------- normalise (materialised)
// processor.go:347-349  out = in * scale.  The correlators fold this multiply into
// their loads; this kernel only serves the tdoa_preprocess probe.
__global__ void __launch_bounds__(kThreads) k_normalize(const SigJob *jobs)
{
    const SigJob &J = jobs[blockIdx.y];
    const float sc = (float)J.stats[ST_SCALE];
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < J.n; i += stride) {
        J.p_re[i] = __fmul_rn(J.q_re[i], sc);
        if (J.p_im) J.p_im[i] = J.q_im ? __fmul_rn(J.q_im[i], sc) : 0.f;
    }
}

// ---------------------------------------------------------------- decimating box-car
// Engine-defined (EXTENDED mode, cfg.decimate = D > 1; the reference's processor never
// decimates -- the integrate-and-dump low-pass of the vendored rtl_fm.c:302-322 is the
// model): y[m] = (x[mD] + ... + x[mD + D-1]) / D, m < n / D, sums sequential f32 in
// ascending order, one f32 divide; plus the power of y for normalizeSignal.
// One thread per output: a warp reads 32 D consecutive floats.
__global__ void __launch_bounds__(kThreads) k_decimate(const SigJob *jobs)
{
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    const int D = J.window;
    const i64 m_out = J.n / D;
    const float fd = (float)D;
    double pacc = 0.0;
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 m = (i64)blockIdx.x * kThreads + threadIdx.x; m < m_out; m += stride) {
        const float *__restrict__ qr = J.q_re + m * D;
        float ar = qr[0];
        for (int k = 1; k < D; k++) ar = __fadd_rn(ar, qr[k]);
        ar = __fdiv_rn(ar, fd);
        float ai = 0.f;
        if (J.q_im) {
            const float *__restrict__ qi = J.q_im + m * D;
            ai = qi[0];
            for (int k = 1; k < D; k++) ai = __fadd_rn(ai, qi[k]);
            ai = __fdiv_rn(ai, fd);
        }
        J.p_re[m] = ar;
        if (J.p_im) J.p_im[m] = ai;
        pacc += (double)mag2_f32(ar, ai);
    }
    double part[1] = {block_sum(pacc, scratch)}, total[1];
    if (grid_sum_last<1>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
        const double pw = m_out > 0 ? total[0] / (double)m_out : 0.0;
        J.stats[ST_POWER1] = pw;
        J.stats[ST_SCALE] = pw > 0.0 ? (double)(float)(1.0 / sqrt(pw)) : 1.0;
    }
}

__global__ void __launch_bounds__(kThreads) k_interleave(const float *re, const float *im, i64 n, float2 *out)
{
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride)
        out[i] = make_float2(re[i], im ? im[i] : 0.f);
}

__global__ void __launch_bounds__(kThreads) k_deinterleave(const float2 *in, i64 n, float *re, float *im)
{
    const i64 stride = (i64)gridDim.x * kThreads;
    for (i64 i = (i64)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
        const float2 v = in[i];
        re[i] = v.x;
        im[i] = v.y;
    }
}

__global__ void k_unpack_selftest(const float *lut, int *bad)
{
    const unsigned b = threadIdx.x;
    if (unpack_byte(b) != lut[b]) atomicAdd(bad, 1);
}

}  // namespace

int stream_grid_x(i64 n)
{
    const i64 want = (n + kThreads * 4 - 1) / (kThreads * 4);
    const i64 cap = 148 * 8;
    return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

int boxcar_grid_x(i64 n)
{
    const i64 g = (n + kBoxTile - 1) / kBoxTile;
    return (int)(g < 1 ? 1 : g);
}

void launch_power(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st)
{
    (void)max_n;
    k_power<<<dim3(grid_x, n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_unpack(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st)
{
    (void)max_n;
    k_unpack<<<dim3(grid_x, n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_demod(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st)
{
    (void)max_n;
    k_demod<<<dim3(grid_x, n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_envelope(const SigJob *d_jobs, int n_jobs, i64 max_n, int grid_x, cudaStream_t st)
{
    (void)max_n;
    k_envelope<<<dim3(grid_x, n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_seqsum(const SigJob *d_jobs, int n_jobs, cudaStream_t st)
{
    k_seqsum<<<dim3(n_jobs, 2), 32, 0, st>>>(d_jobs);
}
void launch_boxcar(const SigJob *d_jobs, int n_jobs, i64 max_n, int max_window, cudaStream_t st)
{
    (void)max_window;
    k_boxcar<<<dim3(boxcar_grid_x(max_n), n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_boxcar_slide(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st)
{
    static bool opted_in[64] = {false};   // per device: more than 48 KB of dynamic shared memory
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !opted_in[dev]) {
        cudaFuncSetAttribute(k_boxcar_slide, cudaFuncAttributeMaxDynamicSharedMemorySize, kSlideSmem);
        opted_in[dev] = true;
    }
    const i64 g = (max_n + kSlideTile - 1) / kSlideTile;   // <= boxcar_grid_x(max_n): the partial-sum slots suffice
    k_boxcar_slide<<<dim3((unsigned)(g < 1 ? 1 : g), n_jobs), kSlideThreads, kSlideSmem, st>>>(d_jobs);
}
void launch_notch_combine(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st)
{
    k_notch_combine<<<dim3(stream_grid_x(max_n), n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_decimate(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st)
{
    k_decimate<<<dim3(stream_grid_x(max_n), n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_normalize(const SigJob *d_jobs, int n_jobs, i64 max_n, cudaStream_t st)
{
    k_normalize<<<dim3(stream_grid_x(max_n), n_jobs), kThreads, 0, st>>>(d_jobs);
}
void launch_interleave(const float *re, const float *im, i64 n, float *out_c64, cudaStream_t st)
{
    k_interleave<<<stream_grid_x(n), kThreads, 0, st>>>(re, im, n, reinterpret_cast<float2 *>(out_c64));
}
void launch_deinterleave(const float *c64, i64 n, float *re, float *im, cudaStream_t st)
{
    k_deinterleave<<<stream_grid_x(n), kThreads, 0, st>>>(reinterpret_cast<const float2 *>(c64), n, re, im);
}

int unpack_selftest(cudaStream_t st)
{
    float h_lut[256];
    for (int b = 0; b < 256; b++) {
        volatile float x = (float)b - 127.5f;  // processor.go:198, host IEEE arithmetic
        volatile float y = x / 127.5f;
        h_lut[b] = y;
    }
    float *d_lut = nullptr;
    int *d_bad = nullptr, h_bad = -1;
    if (cudaMalloc(&d_lut, sizeof(h_lut)) != cudaSuccess) return -1;
    if (cudaMalloc(&d_bad, sizeof(int)) != cudaSuccess) { cudaFree(d_lut); return -1; }
    cudaMemcpyAsync(d_lut, h_lut, sizeof(h_lut), cudaMemcpyHostToDevice, st);
    cudaMemsetAsync(d_bad, 0, sizeof(int), st);
    k_unpack_selftest<<<1, 256, 0, st>>>(d_lut, d_bad);
    cudaMemcpyAsync(&h_bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaError_t err = cudaStreamSynchronize(st);
    cudaFree(d_lut);
    cudaFree(d_bad);
    return err == cudaSuccess ? h_bad : -1;
}

}  // namespace tdoa
