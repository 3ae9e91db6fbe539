// xcorr_exact.cu -- time-domain correlator with the reference's own arithmetic, and
// the peak selection.
//
// Replaces timeDomainCorrelation (processor.go:646-736; shipped binary ELF 0x49d6a0):
//   corr(lag) = mean over whole blocks b of ( sum_{i in block b} f32(t[i]*s[lag+i]) / B )
// with f32 products widened to f64 and summed in ascending i, exactly as the
// reference does, so the per-block sums are bit-identical to the CPU oracle's.
// Parallelism is (block, lag): every thread owns one lag of one block and walks the
// block sequentially; a second kernel adds the blocks in ascending order per lag.
#include "kernels.h"

namespace tdoa {

namespace {

constexpr int kCorrThreads = 256;
constexpr int kLagsPerThread = 4;
constexpr int kLagTile = kCorrThreads * kLagsPerThread;  // 1024 lags per CTA
constexpr int kChunk = 2048;                             // template samples staged per step

// One CTA: block blockIdx.x of the template, lag tile blockIdx.y, pair blockIdx.z.
__global__ void __launch_bounds__(kCorrThreads) k_corr_brute(const PairJob *jobs)
{
    __shared__ float s_t[kChunk];
    __shared__ float s_s[kChunk + kLagTile];
    __shared__ float s_ti[kChunk];             // imaginary planes (CORR_SOURCE only)
    __shared__ float s_si[kChunk + kLagTile];
    const PairJob &J = jobs[blockIdx.z];
    const i64 b = blockIdx.x;
    const int lag_base = blockIdx.y * kLagTile;
    if (b >= J.nb || lag_base >= J.n_lags) return;
    const int variant = J.variant;
    const bool cplx = variant == CORR_SOURCE && J.t_im != nullptr && J.s_im != nullptr;
    const float sc_t = (float)J.t_stats[ST_SCALE], sc_s = (float)J.s_stats[ST_SCALE];
    const i64 B = J.block;
    const i64 blk_start = b * B;
    const i64 blk_len = min(B, J.n_t - blk_start);
    double acc[kLagsPerThread];
#pragma unroll
    for (int k = 0; k < kLagsPerThread; k++) acc[k] = 0.0;

    for (i64 c0 = 0; c0 < blk_len; c0 += kChunk) {
        const int clen = (int)min((i64)kChunk, blk_len - c0);
        __syncthreads();
        // template chunk, normalised on the fly (processor.go:347-349: in * scale)
        const i64 tbase = J.t_off + blk_start + c0;
        for (int i = threadIdx.x; i < clen; i += kCorrThreads) {
            s_t[i] = __fmul_rn(J.t_re[tbase + i], sc_t);
            if (cplx) s_ti[i] = __fmul_rn(J.t_im[tbase + i], sc_t);
        }
        // signal span for this chunk and lag tile
        const i64 sbase = blk_start + c0 + J.lag0 + lag_base;
        const int slen = clen + kLagTile;
        for (int i = threadIdx.x; i < slen; i += kCorrThreads) {
            const i64 g = sbase + i;
            const bool in = g >= 0 && g < J.sl;
            s_s[i] = in ? __fmul_rn(J.s_re[g], sc_s) : 0.f;
            if (cplx) s_si[i] = in ? __fmul_rn(J.s_im[g], sc_s) : 0.f;
        }
        __syncthreads();
        if (variant == CORR_BINARY || (variant == CORR_SOURCE && !cplx)) {
            for (int i = 0; i < clen; i++) {
                const float tv = s_t[i];
#pragma unroll
                for (int k = 0; k < kLagsPerThread; k++) {
                    float p = __fmul_rn(tv, s_s[i + threadIdx.x + k * kCorrThreads]);
                    // CORR_SOURCE with a zero imaginary plane: f32(re*re' + 0*0) == p
                    acc[k] = __dadd_rn(acc[k], (double)p);
                }
            }
        } else if (variant == CORR_SOURCE) {
            for (int i = 0; i < clen; i++) {
                const float tr = s_t[i], ti = s_ti[i];
#pragma unroll
                for (int k = 0; k < kLagsPerThread; k++) {
                    const int j = i + threadIdx.x + k * kCorrThreads;
                    // processor.go:703  real(t)*real(s) + imag(t)*imag(s), f32
                    const float p = __fadd_rn(__fmul_rn(tr, s_s[j]), __fmul_rn(ti, s_si[j]));
                    acc[k] = __dadd_rn(acc[k], (double)p);
                }
            }
        } else {  // CORR_EXTENDED: exact f64 product of the two f32 values
            for (int i = 0; i < clen; i++) {
                const double tv = (double)s_t[i];
#pragma unroll
                for (int k = 0; k < kLagsPerThread; k++)
                    acc[k] = __fma_rn(tv, (double)s_s[i + threadIdx.x + k * kCorrThreads], acc[k]);   // the product is exact: one rounding either way
            }
        }
    }
#pragma unroll
    for (int k = 0; k < kLagsPerThread; k++) {
        const int lag = lag_base + threadIdx.x + k * kCorrThreads;
        if (lag < J.n_lags) {
            // processor.go:709  blockCorr /= blockSize   (EXTENDED keeps the raw sum)
            const double v = variant == CORR_EXTENDED ? acc[k] : acc[k] / (double)B;
            J.blocksums[(size_t)b * J.n_lags + lag] = v;
        }
    }
}

// processor.go:710-720: corr = sum of block means (ascending b) / nb [* sqrt(nb*B)].
__global__ void __launch_bounds__(kCorrThreads) k_corr_finalize(const PairJob *jobs)
{
    const PairJob &J = jobs[blockIdx.y];
    const int lag = blockIdx.x * kCorrThreads + threadIdx.x;
    if (lag >= J.n_lags) return;
    double corr = 0.0;
    for (i64 b = 0; b < J.nb; b++) corr = __dadd_rn(corr, J.blocksums[(size_t)b * J.n_lags + lag]);
    if (J.nb > 0) {
        if (J.variant == CORR_EXTENDED) {
            corr = corr / (double)J.n_t;
        } else {
            corr = corr / (double)J.nb;
            if (J.variant == CORR_SOURCE) corr = __dmul_rn(corr, sqrt((double)(J.nb * J.block)));
        }
    }
    J.corr[lag] = corr;
}

// ---------------------------------------------------------------- peak selection
// processor.go:722-725: scan lags ascending, keep when |c| > |best| (strict): the
// first maximum wins and the correlation keeps its sign.
struct Best {
    double v;  // signed value
    int idx;   // index, INT_MAX when none
};

__device__ __forceinline__ Best better(Best a, Best b)
{
    // the earlier index wins ties; "none" (idx = INT_MAX, v = 0) loses to any |v| > 0
    const double fa = fabs(a.v), fb = fabs(b.v);
    if (fb > fa || (fb == fa && b.idx < a.idx)) return b;
    return a;
}

__device__ Best warp_argmax_abs(const double *c, int n)
{
    const int lane = threadIdx.x & 31;
    Best m = {0.0, 0x7fffffff};
    for (int i = lane; i < n; i += 32) {
        const double v = c[i];
        if (fabs(v) > fabs(m.v)) { m.v = v; m.idx = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Best other;
        other.v = __shfl_xor_sync(0xffffffffu, m.v, o);
        other.idx = __shfl_xor_sync(0xffffffffu, m.idx, o);
        m = better(m, other);
    }
    // |v| == 0 everywhere: the reference never updates best (0 > 0 is false) -> lag 0, corr 0
    if (m.v == 0.0) { m.idx = 0; }
    if (m.idx == 0x7fffffff) m.idx = 0;
    return m;
}

// runner-up magnitude: largest |c| over indices other than `skip`
__device__ double warp_second_abs(const double *c, int n, int skip)
{
    const int lane = threadIdx.x & 31;
    double m = 0.0;
    for (int i = lane; i < n; i += 32)
        if (i != skip) m = fmax(m, fabs(c[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    return m;
}

// A bounded record (EXTENDED) scans its run [i0, i1] only: arg-max, runner-up and the parabola's neighbours.
__global__ void __launch_bounds__(32) k_peak(const PeakJob *jobs)
{
    const PeakJob &J = jobs[blockIdx.x];
    PeakRec r;
    r.lag = 0; r.flags = J.flags; r.corr = 0.0; r.frac = 0.f; r.margin = 0.f; r.first_lag = 0; r.n_blocks = J.nb;
    int i0, i1;
    if (bound_run(J.bound, J.lag_origin, J.decim, J.n_lags, &i0, &i1))
        r.flags |= i0 > i1 ? TDOA_PEAK_BOUNDED | TDOA_PEAK_EMPTY : TDOA_PEAK_BOUNDED;
    double first = 0.0;
    if (J.nb > 0 && i0 <= i1) {
        const double *c = J.corr + i0;
        const int n = i1 - i0 + 1;
        Best b = warp_argmax_abs(c, n);
        const double second = warp_second_abs(c, n, b.idx);
        b.idx += i0;
        first = b.v;
        r.lag = b.idx + J.lag_origin;
        r.first_lag = r.lag;
        r.corr = b.v;
        r.margin = b.v != 0.0 ? (float)((fabs(b.v) - second) / fabs(b.v)) : 0.f;
        if (J.variant == CORR_BINARY && J.sanity > 0 && b.idx > J.sanity && J.n_lags2 > 0) {
            // ELF 0x49dda7: re-search [0, sanity); accept when |c| > 0.5 |best|
            const Best rb = warp_argmax_abs(J.corr2, min(J.n_lags2, J.sanity));
            if (fabs(rb.v) > 0.5 * fabs(b.v)) {
                r.lag = rb.idx;
                r.corr = rb.v;
                r.flags |= 0x1u;  // TDOA_PEAK_RESEARCHED
            }
        }
        if (J.variant == CORR_EXTENDED) {
            // 3-point parabolic vertex on |c| (engine-defined; oracle orc_peak_parabolic)
            if (b.idx > i0 && b.idx < i1) {
                const double a = fabs(J.corr[b.idx - 1]), m = fabs(J.corr[b.idx]), d = fabs(J.corr[b.idx + 1]);
                const double den = a - 2.0 * m + d;
                r.frac = den != 0.0 ? (float)(0.5 * (a - d) / den) : 0.f;
            } else {
                r.flags |= 0x2u;  // TDOA_PEAK_EDGE
            }
        }
    }
    if ((threadIdx.x & 31) == 0) {
        *J.out = r;
        if (J.first_corr) *J.first_corr = first;
    }
}

}  // namespace

void launch_corr_brute(const PairJob *d_jobs, int n_jobs, i64 max_nb, int max_lags, cudaStream_t st)
{
    if (n_jobs <= 0 || max_nb <= 0 || max_lags <= 0) return;
    const dim3 grid((unsigned)max_nb, (unsigned)((max_lags + kLagTile - 1) / kLagTile), (unsigned)n_jobs);
    k_corr_brute<<<grid, kCorrThreads, 0, st>>>(d_jobs);
}

void launch_corr_finalize(const PairJob *d_jobs, int n_jobs, int max_lags, cudaStream_t st)
{
    if (n_jobs <= 0 || max_lags <= 0) return;
    const dim3 grid((unsigned)((max_lags + kCorrThreads - 1) / kCorrThreads), (unsigned)n_jobs);
    k_corr_finalize<<<grid, kCorrThreads, 0, st>>>(d_jobs);
}

// lags found on decimated signals, back in samples of the capture: lag + frac -> D (lag + frac)
__global__ void k_lag_units(PeakRec *recs, int n, int D)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PeakRec r = recs[i];
    const double total = (double)D * ((double)r.lag + (double)r.frac);
    const double whole = rint(total);
    r.lag = (int32_t)whole;
    r.frac = (float)(total - whole);
    r.first_lag *= D;
    recs[i] = r;
}

void launch_lag_units(PeakRec *d_recs, int n, int D, cudaStream_t st)
{
    if (n > 0 && D > 1) k_lag_units<<<(n + 127) / 128, 128, 0, st>>>(d_recs, n, D);
}

void launch_peak(const PeakJob *d_jobs, int n_jobs, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_peak<<<n_jobs, 32, 0, st>>>(d_jobs);
}

}  // namespace tdoa
