// xcorr_big.cu -- wide lag searches: cross-correlation through a 2^21-point FFT that lives
// in global memory (four-step, 256 x 8192), for lag ranges the 8192-point segment kernel
// (xcorr_tile.cu) would have to sweep in dozens of 2048-lag chunks -- BASELINE config 3:
// 1 s windows, +-50 000 lags.
//
// A tile is, as in xcorr_tile.cu, up to 2 template stations x 2 signal stations of one
// window: A = FFT(t0 + i t1), B = FFT(s0 + i s1), four cross-spectra conj(T_a) S_b, of
// which two real correlations ride in one complex inverse transform (G = C_a0 + i C_a1).
// Long templates are cut into segments of N - n_lags samples whose cross-spectra are
// added in place before the one inverse.
//
// With n = 8192 n1 + n2 and k = k1 + 256 k2:
//   X[k1 + 256 k2] = sum_n2 W_8192^(n2 k2) [ W_N^(n2 k1) sum_n1 x[8192 n1 + n2] W_256^(n1 k1) ]
//   k_big_cols : 256-point transforms down the columns (two radix-16 stages in shared
//                memory, 32 columns per CTA, coalesced rows)
//   k_big_rows : times W_N^(n2 k1) while loading, then 8192-point transforms along the
//                rows (fft_tile_core.cuh); the spectrum stays in the [k1][k2] layout -- a
//                pointwise product does not care
//   k_big_cross: T, S from Z[k], Z[N-k] (the mirror of [k1][k2] is [256-k1][8191-k2]), the
//                four products, packed in pairs
//   k_big_rows (inverse) and k_big_out: the same two passes backwards; only the rows
//                n1 < ceil(n_lags / 8192) of the result are formed and written
// Every pass is a streaming kernel over 16 MiB buffers: the path is HBM/L2 bound, not
// issue bound like the segment kernel.  The result only RANKS lags (f32); the candidates
// are then re-evaluated exactly (k_corr_candidates), as everywhere else.
#include "fft_tile_core.cuh"
#include "kernels.h"
#include "xcorr_fft.h"

namespace tdoa {

using namespace fft2;

namespace {

constexpr int kN1 = kBigN1;          // 256 column points
constexpr int kN2 = kN;              // 8192 row points
constexpr int kCols = 32;            // columns per CTA of the column passes
constexpr int kColThreads = 256;
constexpr int kColSmem = kN1 * kCols * (int)sizeof(float2);          // 64 KB
constexpr int kRowSmem = (kBuf + kTab) * (int)sizeof(float2);        // 73.6 KB

static_assert(kBigN == (i64)kN1 * kN2, "big transform is 256 x 8192");

// W_N^m, m < 2^21, from W_1024^(m >> 11) (every 8th entry of the 8192-entry table) and the
// fine table W_N^(m & 2047)
__device__ __forceinline__ float2 big_twiddle(unsigned m, const float2 *__restrict__ tw, const float2 *__restrict__ fine)
{
    return cmul(tw[8u * (m >> 11)], fine[m & 2047u]);
}

// W_N^(k1 j) for the row elements j = t + 256 r a thread touches: W_N^(k1 t) once per thread
// (two table loads), times W_N^(256 k1 r) = W_8192^(k1 r), a warp-uniform table entry
struct RowTwiddle {
    float2 base;
    unsigned k1;
    const float2 *tw;
    __device__ __forceinline__ RowTwiddle(unsigned k1_, unsigned t, const float2 *__restrict__ tw_, const float2 *__restrict__ fine)
        : base(big_twiddle(k1_ * t, tw_, fine)), k1(k1_), tw(tw_) {}
    __device__ __forceinline__ float2 at(int r) const { return cmul(base, tw[(k1 * (unsigned)r) & (kN - 1)]); }
};

// 256-point transform of every column of the [256][32] strip in shared memory, in place:
// on return row r = 16 p + q holds X[p + 16 q].  Two radix-16 stages, items (column, b) and
// (column, p): lanes run along the columns (conflict free).
__device__ __forceinline__ void strip_fft256(float2 *sm, int tid, const float2 *__restrict__ tw)
{
    const int c = tid & 31;
#pragma unroll 1
    for (int it = 0; it < 2; it++) {
        const int b = (tid >> 5) + 8 * it;
        float2 u[16];
#pragma unroll
        for (int a = 0; a < 16; a++) u[a] = sm[(16 * a + b) * kCols + c];
        dft<16>(u);
#pragma unroll
        for (int p = 1; p < 16; p++) u[p] = cmul(u[p], tw[(32 * b * p) & (kN - 1)]);  // W_256^(b p)
#pragma unroll
        for (int p = 0; p < 16; p++) sm[(16 * p + b) * kCols + c] = u[p];
    }
    __syncthreads();
#pragma unroll 1
    for (int it = 0; it < 2; it++) {
        const int p = (tid >> 5) + 8 * it;
        float2 v[16];
#pragma unroll
        for (int b = 0; b < 16; b++) v[b] = sm[(16 * p + b) * kCols + c];
        dft<16>(v);
#pragma unroll
        for (int q = 0; q < 16; q++) sm[(16 * p + q) * kCols + c] = v[q];
    }
    __syncthreads();
}

// ---------------------------------------------------------------- forward column pass
__global__ void __launch_bounds__(kColThreads) k_big_cols(const BigColJob *jobs, const float2 *__restrict__ tw,
                                                          const float2 *__restrict__ fine)
{
    extern __shared__ __align__(16) float2 sm[];
    const BigColJob &J = jobs[blockIdx.y];
    const int tid = threadIdx.x, c = tid & 31;
    const int n2 = blockIdx.x * kCols + c;
    // z[n] = x0[base + n] sc0 + i x1[base + n] sc1 for lo <= n < hi, else 0; sc = rank_pre (xcorr_fft.h), 1 unless
    // the two planes' powers differ widely
    const float *__restrict__ x0 = J.x0 + J.base, *__restrict__ x1 = J.x1 + J.base;
    const float sc0 = rank_pre(J.x0_stats, J.x1_stats), sc1 = rank_pre(J.x1_stats, J.x0_stats);
    const i64 lo = J.lo, hi = J.hi;
#pragma unroll 1
    for (int g = 0; g < 4; g++) {   // 8 rows per thread in flight
        float2 z[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int n1 = (tid >> 5) + 8 * (8 * g + u);
            const i64 n = (i64)n1 * kN2 + n2;
            z[u] = (n >= lo && n < hi) ? make_float2(x0[n], x1[n]) : make_float2(0.f, 0.f);
        }
        if (sc0 != 1.f || sc1 != 1.f) {
#pragma unroll
            for (int u = 0; u < 8; u++) z[u] = make_float2(__fmul_rn(z[u].x, sc0), __fmul_rn(z[u].y, sc1));
        }
#pragma unroll
        for (int u = 0; u < 8; u++) sm[((tid >> 5) + 8 * (8 * g + u)) * kCols + c] = z[u];
    }
    __syncthreads();
    strip_fft256(sm, tid, tw);
    (void)fine;
#pragma unroll 8
    for (int i = 0; i < 32; i++) {
        const int r = (tid >> 5) + 8 * i;
        const int k1 = (r >> 4) + 16 * (r & 15);
        J.out[(size_t)k1 * kN2 + n2] = sm[r * kCols + c];
    }
}

// ---------------------------------------------------------------- row pass (forward / inverse)
__global__ void __launch_bounds__(kT, 2) k_big_rows(const BigRowJob *jobs, const float2 *__restrict__ tw,
                                                    const float2 *__restrict__ fine)
{
    extern __shared__ __align__(16) float2 sm[];
    const BigRowJob &J = jobs[blockIdx.y];
    const int t = threadIdx.x, k1 = blockIdx.x;
    float2 *buf = sm, *tab = sm + kBuf;
    float2 *row = J.buf + (size_t)k1 * kN2;
    for (int idx = t; idx < kTab; idx += kT) tab[idx] = tw[(16 * (idx & 31) * (idx >> 5)) & (kN - 1)];
    const float2 w1a = tw[2 * t], w1b = tw[2 * t + 1];
    const RowTwiddle W((unsigned)k1, (unsigned)t, tw, fine);
    {
        float2 v[32];
#pragma unroll
        for (int r = 0; r < 32; r++) v[r] = row[t + 256 * r];
        if (J.inverse) {
#pragma unroll
            for (int r = 0; r < 32; r++) v[r].y = -v[r].y;   // IFFT(g) = conj(FFT(conj g))
        } else {
#pragma unroll
            for (int r = 0; r < 32; r++) v[r] = cmul(v[r], W.at(r));   // the twiddle between the two passes
        }
        pass1_store(v, t, buf);
    }
    __syncthreads();
    {
        float2 u0[16], u1[16];
        pass_load(buf, t, u0, u1);
        __syncthreads();
        pass2_twiddle(u0, u1, t, tab);
        pass2_store(u0, u1, t, buf);
        __syncthreads();
        pass_load(buf, t, u0, u1);
        __syncthreads();
        pass3_compute(u0, w1a);
        pass3_compute(u1, w1b);
        spectrum_store(u0, u1, t, buf);
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < 32; r++) {
        const int j = t + 256 * r;
        float2 x = buf[j];
        if (J.inverse) {
            // back through the twiddle between the passes: conj(X) conj(W_N^(n2 k1))
            const float2 w = W.at(r);
            x = cmul(make_float2(x.x, -x.y), make_float2(w.x, -w.y));
        }
        row[j] = x;
    }
}

// ---------------------------------------------------------------- cross-spectra of the tile
__global__ void __launch_bounds__(256) k_big_cross(const BigCrossJob *jobs)
{
    const BigCrossJob &J = jobs[blockIdx.y];
    const unsigned idx = blockIdx.x * 256u + threadIdx.x;   // k1 * 8192 + k2
    const unsigned k1 = idx >> 13, k2 = idx & (kN2 - 1);
    const unsigned m1 = (kN1 - k1) & (kN1 - 1);
    const unsigned m2 = k1 == 0 ? ((kN2 - k2) & (kN2 - 1)) : (kN2 - 1 - k2);
    const size_t mid = (size_t)m1 * kN2 + m2;
    const float2 a = J.A[idx], c = J.A[mid], b = J.B[idx], d = J.B[mid];
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    cross_accumulate(a, c, b, d, acc);   // acc[2 (2 ta + sb) + {0, 1}] = 4 conj(T_ta) S_sb
    // two real correlations per complex inverse: G = C_a0 + i C_a1
    float2 g0 = make_float2(acc[0] - acc[3], acc[1] + acc[2]);
    float2 g1 = make_float2(acc[4] - acc[7], acc[5] + acc[6]);
    if (J.accumulate) {
        const float2 p0 = J.G0[idx], p1 = J.G1[idx];
        g0.x += p0.x; g0.y += p0.y; g1.x += p1.x; g1.y += p1.y;
    }
    J.G0[idx] = g0;
    J.G1[idx] = g1;
}

// ---------------------------------------------------------------- inverse column pass + output
// G already went through the inverse row pass ([k1][n2], conjugated).  Only the rows
// n1 = d / 8192 that hold lags d < n_lags are written.
__global__ void __launch_bounds__(kColThreads) k_big_out(const BigOutJob *jobs, const float2 *__restrict__ tw)
{
    extern __shared__ __align__(16) float2 sm[];
    const BigOutJob &J = jobs[blockIdx.y];
    const int tid = threadIdx.x, c = tid & 31;
    const int n2 = blockIdx.x * kCols + c;
    const float2 *__restrict__ G = J.G + n2;
#pragma unroll 1
    for (int g4 = 0; g4 < 4; g4++) {
        float2 z[8];
#pragma unroll
        for (int u = 0; u < 8; u++) z[u] = G[(size_t)((tid >> 5) + 8 * (8 * g4 + u)) * kN2];
#pragma unroll
        for (int u = 0; u < 8; u++) sm[((tid >> 5) + 8 * (8 * g4 + u)) * kCols + c] = make_float2(z[u].x, -z[u].y);
    }
    __syncthreads();
    strip_fft256(sm, tid, tw);
    // c[n] = conj(X): real part -> pair (a, 0), imaginary part -> pair (a, 1); coefficient units:
    // scale_t scale_s / n_t (processor.go:347-349, :709-717) less what k_big_cols applied (rank_pre), 1/N of the
    // inverse, 1/4 of 2T 2S
    const double k = J.n_t > 0 ? 0.25 / ((double)J.n_t * (double)kBigN) : 0.0;
    const double st = rank_post(J.t_stats, J.t_pack);
    const double sc0 = J.approx0 ? st * rank_post(J.s0_stats, J.s1_stats) * k : 0.0;
    const double sc1 = J.approx1 ? st * rank_post(J.s1_stats, J.s0_stats) * k : 0.0;
    const int rows = (J.n_lags + kN2 - 1) / kN2;
    for (int r = tid >> 5; r < kN1; r += 8) {
        const int n1 = (r >> 4) + 16 * (r & 15);
        if (n1 >= rows) continue;
        const int dlag = n1 * kN2 + n2;
        if (dlag >= J.n_lags) continue;
        const float2 x = sm[r * kCols + c];
        if (J.approx0) J.approx0[dlag] = (float)((double)x.x * sc0);
        if (J.approx1) J.approx1[dlag] = (float)(-(double)x.y * sc1);
    }
}

}  // namespace

int big_setup(cudaStream_t st, float2 **d_fine)
{
    static float2 h[2048];
    for (int k = 0; k < 2048; k++) {
        const double a = -2.0 * 3.14159265358979323846 * (double)k / (double)kBigN;
        h[k] = make_float2((float)cos(a), (float)sin(a));
    }
    if (cudaMalloc(d_fine, sizeof(h)) != cudaSuccess) return -1;
    if (cudaMemcpyAsync(*d_fine, h, sizeof(h), cudaMemcpyHostToDevice, st) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_big_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, kColSmem) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_big_out, cudaFuncAttributeMaxDynamicSharedMemorySize, kColSmem) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_big_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, kRowSmem) != cudaSuccess) return -1;
    return 0;
}

void launch_big_cols(const BigColJob *d_jobs, int n_jobs, const float2 *d_tw, const float2 *d_fine, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_big_cols<<<dim3(kN2 / kCols, n_jobs), kColThreads, kColSmem, st>>>(d_jobs, d_tw, d_fine);
}

void launch_big_rows(const BigRowJob *d_jobs, int n_jobs, const float2 *d_tw, const float2 *d_fine, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_big_rows<<<dim3(kN1, n_jobs), kT, kRowSmem, st>>>(d_jobs, d_tw, d_fine);
}

void launch_big_cross(const BigCrossJob *d_jobs, int n_jobs, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_big_cross<<<dim3((unsigned)(kBigN / 256), n_jobs), 256, 0, st>>>(d_jobs);
}

void launch_big_out(const BigOutJob *d_jobs, int n_jobs, const float2 *d_tw, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_big_out<<<dim3(kN2 / kCols, n_jobs), kColThreads, kColSmem, st>>>(d_jobs, d_tw);
}

}  // namespace tdoa
