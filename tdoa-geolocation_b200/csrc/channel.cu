// channel.cu -- the channel filter of EXTENDED mode (tdoa_set_channel): a complex FIR over a signal's unpacked
// samples, ahead of preprocessSignal, so that the discriminator follows the station the collector is tuned to and
// not a stronger one elsewhere in the 2 MHz capture (include/tdoa_b200.h states it).
//
//   k_channel       : capture bytes -> the filtered signal y as planar f32 (re, im), 2 B in, 8 B out per sample.
//                     The plane kernels then read y through SigSrc (raw == nullptr).
//   k_channel_demod : the same FIR, then discriminate() on y (k_demod's statement): 2 B in, 4 B out, with the
//                     power of y and the sum of the output in the statistics block.  The strong branch's path.
//
// Both cost 4 T FMA per sample (2 T with real taps), so they are FP32-bound.  A CTA stages a tile of unpacked
// samples plus the 2c halo once in shared memory; each thread keeps 8 consecutive outputs in registers and a
// window of 8 samples that slides by one per tap, so one 64-bit shared load feeds 32 FMA (complex taps).  The taps
// are a __grid_constant__ parameter.  Every output is the sequential fmaf chain of the statement, k ascending.
#include "discriminate.cuh"
#include "kernels.h"

namespace tdoa {

namespace {

constexpr int kThreads = 256;
constexpr int kPer = 8;                                  // consecutive outputs per thread
constexpr int kTile = kThreads * kPer;                   // filter outputs per CTA tile
constexpr int kHalf = (kChannelMaxTaps - 1) / 2;          // c <= 63
constexpr int kStage = kTile + 2 * kHalf;                // samples staged per tile
// thread t reads element 8 t + m: one pad slot every 8 elements makes that a stride of 9 float2 across the
// lanes, which no two of 16 lanes share a bank in (the minimum of two wavefronts for a 64-bit load)
__device__ __forceinline__ int slot(int j) { return j + (j >> 3); }
constexpr int kStageSlots = kStage + kStage / 8 + 1;
constexpr int kOutSlots = kTile + kTile / 8;

__device__ __forceinline__ float dc_from_sum(double sum, i64 n) { return __fdiv_rn((float)sum, (float)n); }

// FIR outputs f0 .. f0 + kTile - 1 of the job into s_y (padded layout); s_x is the staging buffer
template <bool CPLX>
__device__ __forceinline__ void fir_tile(const SigJob &J, const ChannelTaps &taps, const float *lut, float2 *s_x,
                                         float2 *s_y, i64 f0)
{
    const int tid = threadIdx.x;
    const int T = taps.n, c = (T - 1) >> 1;
    const i64 n = J.n;
    const uchar2 *__restrict__ raw = reinterpret_cast<const uchar2 *>(J.src.raw);
    __syncthreads();   // the previous tile's readers of s_x / s_y are done
    // s_x[j] = x[f0 - c + j], +0 + 0j outside [0, n)
    const int len = kTile + 2 * c;
    for (int j = tid; j < len; j += kThreads) {
        const i64 q = f0 - c + j;
        float2 v = make_float2(0.f, 0.f);
        if (q >= 0 && q < n) {
            const uchar2 b = raw[raw_index(J.src, q)];
            v = make_float2(lut[b.x], lut[b.y]);
        }
        s_x[slot(j)] = v;
    }
    __syncthreads();
    // output f0 + t0 + r takes x[f0 + t0 + r + c - k] = s_x[j0 + r - k], j0 = t0 + 2c.  Window slot (r - k) mod 8
    // holds that sample at tap k: going to tap k + 1 drops the sample of r = 7 and loads the one of r = 0.
    const int j0 = tid * kPer + 2 * c;
    float ar[kPer], ai[kPer];
    float2 w[kPer];
#pragma unroll
    for (int r = 0; r < kPer; r++) { ar[r] = 0.f; ai[r] = 0.f; }
#pragma unroll
    for (int r = 1; r < kPer; r++) w[r] = s_x[slot(j0 + r)];
    auto tap = [&](int k, int kk) {   // kk = k mod 8, a compile-time constant in every call
        w[(kPer - kk) & (kPer - 1)] = s_x[slot(j0 - k)];
        const float hr = taps.re[k];
        const float hi = taps.im[k];
#pragma unroll
        for (int r = 0; r < kPer; r++) {
            const float2 v = w[(r - kk) & (kPer - 1)];
            ar[r] = __fmaf_rn(hr, v.x, ar[r]);
            if (CPLX) ar[r] = __fmaf_rn(-hi, v.y, ar[r]);
            ai[r] = __fmaf_rn(hr, v.y, ai[r]);
            if (CPLX) ai[r] = __fmaf_rn(hi, v.x, ai[r]);
        }
    };
    int k = 0;
    for (; k + kPer <= T; k += kPer) {
#pragma unroll
        for (int kk = 0; kk < kPer; kk++) tap(k + kk, kk);
    }
#pragma unroll
    for (int kk = 0; kk < kPer - 1; kk++)
        if (k + kk < T) tap(k + kk, kk);
#pragma unroll
    for (int r = 0; r < kPer; r++) s_y[slot(tid * kPer + r)] = make_float2(ar[r], ai[r]);
    __syncthreads();
}

template <bool CPLX>
__global__ void __launch_bounds__(kThreads) k_channel(const SigJob *jobs, const __grid_constant__ ChannelTaps taps)
{
    __shared__ float lut[256];
    __shared__ float2 s_x[kStageSlots];
    __shared__ float2 s_y[kOutSlots];
    const SigJob &J = jobs[blockIdx.y];
    lut[threadIdx.x] = unpack_byte(threadIdx.x);   // processor.go:198-199, exact per code
    const i64 n = J.n;
    for (i64 f0 = (i64)blockIdx.x * kTile; f0 < n; f0 += (i64)gridDim.x * kTile) {
        fir_tile<CPLX>(J, taps, lut, s_x, s_y, f0);
        for (int t = threadIdx.x; t < kTile; t += kThreads) {
            const i64 i = f0 + t;
            if (i >= n) break;
            const float2 y = s_y[slot(t)];
            J.p_re[i] = y.x;
            J.p_im[i] = y.y;
        }
    }
}

// A tile's first filter output is the previous sample of its first discriminator output, so tiles step by
// kTile - 1 outputs and each recomputes one filter output of its neighbour.
template <bool CPLX>
__global__ void __launch_bounds__(kThreads) k_channel_demod(const SigJob *jobs, const __grid_constant__ ChannelTaps taps)
{
    constexpr int kStep = kTile - 1;
    __shared__ float lut[256];
    __shared__ float2 s_x[kStageSlots];
    __shared__ float2 s_y[kOutSlots];
    __shared__ double scratch[32];
    const SigJob &J = jobs[blockIdx.y];
    lut[threadIdx.x] = unpack_byte(threadIdx.x);
    const i64 n = J.n;
    double pw = 0.0, sr = 0.0;
    for (i64 o0 = (i64)blockIdx.x * kStep; o0 < n; o0 += (i64)gridDim.x * kStep) {
        fir_tile<CPLX>(J, taps, lut, s_x, s_y, o0 - 1);   // s_y[slot(u + 1)] = y[o0 + u]
        for (int u = threadIdx.x; u < kStep; u += kThreads) {
            const i64 i = o0 + u;
            if (i >= n) break;
            const float2 cur = s_y[slot(u + 1)];
            // out[0] = out[1]: the pair (y[0], y[1])
            const float o = i == 0 ? discriminate(cur, s_y[slot(2)]) : discriminate(s_y[slot(u)], cur);
            J.p_re[i] = o;
            pw += (double)mag2_f32(cur.x, cur.y);   // calculateSignalPower of the filtered signal
            sr += (double)o;
        }
    }
    double part[2], total[2];
    part[0] = block_sum(pw, scratch);
    part[1] = block_sum(sr, scratch);
    if (grid_sum_last<2>(part, J.partials, J.counter, gridDim.x, blockIdx.x, scratch, total)) {
        J.stats[ST_POWER0] = n > 0 ? total[0] / (double)n : 0.0;
        J.stats[ST_SUM_RE] = total[1];
        J.stats[ST_SUM_IM] = 0.0;
        J.stats[ST_DC_RE] = n > 0 ? (double)dc_from_sum(total[1], n) : 0.0;
        J.stats[ST_DC_IM] = 0.0;
    }
}

}  // namespace

void launch_channel(const SigJob *d_jobs, int n_jobs, i64 max_n, const ChannelTaps &taps, bool cplx, cudaStream_t st)
{
    const dim3 grid(stream_grid_x(max_n), n_jobs);
    if (cplx) k_channel<true><<<grid, kThreads, 0, st>>>(d_jobs, taps);
    else k_channel<false><<<grid, kThreads, 0, st>>>(d_jobs, taps);
}

// stream_grid_x(max_n) CTAs: the partial-sum slots the engine gives every signal suffice
void launch_channel_demod(const SigJob *d_jobs, int n_jobs, i64 max_n, const ChannelTaps &taps, bool cplx, cudaStream_t st)
{
    const dim3 grid(stream_grid_x(max_n), n_jobs);
    if (cplx) k_channel_demod<true><<<grid, kThreads, 0, st>>>(d_jobs, taps);
    else k_channel_demod<false><<<grid, kThreads, 0, st>>>(d_jobs, taps);
}

}  // namespace tdoa
