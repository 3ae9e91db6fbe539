// xcorr_tile.cu -- segmented-FFT cross-spectra of a TILE of station pairs in one pass.
//
// The per-pair kernel (xcorr_fft.cu, k_fft_segments) spends one 8192-point complex
// transform per pair and segment: z = t + i s.  Pairs of one window share stations, so a
// tile of up to 2 template stations x 2 signal stations needs only TWO transforms per
// segment -- A = FFT(t0 + i t1), B = FFT(s0 + i s1) -- for up to four cross-spectra
// conj(T_a) S_b (three for the reference's 3-station case: (0,1), (0,2), (1,2)).
//
// One CTA of 512 threads per SM: threads 0..255 run transform A, threads 256..511
// transform B, concurrently, each in its own shared-memory buffer with its own named
// barrier (fft_tile_core.cuh).  The accumulated cross-spectra -- 4 products x 4097 bins
// x (re, im) = 128 KB per CTA, 64 floats per thread -- do not fit in the register file
// next to a 32-point-per-thread transform, and shared memory is taken by the two
// buffers; they live in the SM's TENSOR MEMORY (256 KB, otherwise idle on this path):
// each thread owns 72 columns of its TMEM lane and does tcgen05.ld -> FMA -> tcgen05.st
// around the bins it is responsible for (measured: a full read-modify-write of all
// 128 KB takes ~400 cycles, tools/micro/tmem_rw.cu).  No tensor-core instruction is
// involved: the FFT is not a dense contraction.
//
// The next segment's samples are loaded into registers before the cross phase, so the
// HBM latency hides behind it.
#include <cstdlib>
#include "fft_tile_core.cuh"
#include "fft_tile16_core.cuh"
#include "kernels.h"
#include "xcorr_fft.h"

namespace tdoa {

using namespace fft2;

namespace {

constexpr int kBins = kN / 2 + 1;
constexpr int kTileThreads = 2 * kT;
constexpr int kTileSmem = (2 * kBuf + kTab) * (int)sizeof(float2);   // 143 360 B: one CTA per SM
constexpr int kTmemCols = 512;

static_assert(kSeg == 6144 && kFftN == kN, "tile kernel is written for 6144-sample segments of an 8192-point transform");

__device__ __forceinline__ void tmem_st16(unsigned taddr, const float *v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 :: "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                    "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                    "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])),
                    "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
                    "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
                    "r"(__float_as_uint(v[15]))
                 : "memory");
}

__device__ __forceinline__ void tmem_ld8(unsigned taddr, float *v)
{
    unsigned r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_st8(unsigned taddr, const float *v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                    "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                    "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}

__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// barrier over the 256 threads of transform g (ids 1 and 2; 0 is __syncthreads)
__device__ __forceinline__ void bar_transform(int g) { asm volatile("bar.sync %0, 256;" ::"r"(g + 1) : "memory"); }

// samples m = t + 256 r of one segment as complex points (x0[m] sc0, x1[m] sc1); CNT rows carry data.  sc0, sc1:
// rank_pre (xcorr_fft.h), 1 unless the two planes' powers differ widely: no multiply at all then.
template <int CNT>
__device__ __forceinline__ void load_rows(const float *__restrict__ x0, const float *__restrict__ x1, float sc0,
                                          float sc1, i64 base, i64 lo, i64 hi, int t, float2 (&v)[32])
{
    if (lo <= 0 && hi >= 256 * CNT) {
        const float *__restrict__ p0 = x0 + base + t;
        const float *__restrict__ p1 = x1 + base + t;
#pragma unroll
        for (int r = 0; r < 32; r++) v[r] = r < CNT ? make_float2(__ldg(p0 + 256 * r), __ldg(p1 + 256 * r)) : make_float2(0.f, 0.f);
    } else {
#pragma unroll
        for (int r = 0; r < 32; r++) {
            const i64 m = t + 256 * r;
            const bool ok = r < CNT && m >= lo && m < hi;
            v[r] = ok ? make_float2(__ldg(x0 + base + m), __ldg(x1 + base + m)) : make_float2(0.f, 0.f);
        }
    }
    if (sc0 != 1.f || sc1 != 1.f) {
#pragma unroll
        for (int r = 0; r < CNT; r++) v[r] = make_float2(__fmul_rn(v[r].x, sc0), __fmul_rn(v[r].y, sc1));
    }
}

__global__ void __launch_bounds__(kTileThreads, 1) k_fft_tiles(const TileJob *jobs, const float2 *__restrict__ tw)
{
    extern __shared__ __align__(16) float2 sm[];
    __shared__ unsigned s_tmem;
    const TileJob &J = jobs[blockIdx.y];
    const int cta = blockIdx.x;
    if (cta >= J.n_cta) return;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int g = tid >> 8, t = tid & (kT - 1);
    // the scales first: their two dependent loads overlap the table fill and the tensor-memory set-up
    const double *st0 = g ? J.s0_stats : J.t0_stats, *st1 = g ? J.s1_stats : J.t1_stats;
    const float sc0 = rank_pre(st0, st1), sc1 = rank_pre(st1, st0);
    float2 *buf = sm + g * kBuf;
    float2 *tab = sm + 2 * kBuf;
    for (int idx = tid; idx < kTab; idx += kTileThreads) tab[idx] = tw[(16 * (idx & 31) * (idx >> 5)) & (kN - 1)];
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (unsigned)__cvta_generic_to_shared(&s_tmem)), "n"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const unsigned tmem_base = s_tmem;
    // this thread's accumulators: lane 32 (warp % 4) + lane id, columns 128 (warp / 4) + [0, 72)
    const unsigned tmem = tmem_base + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)(128 * (warp >> 2));
    {
        float z[16];
#pragma unroll
        for (int i = 0; i < 16; i++) z[i] = 0.f;
#pragma unroll
        for (int c = 0; c < 5; c++) tmem_st16(tmem + 16 * c, z);
        tmem_wait_st();
    }
    const float2 w1a = tw[2 * t], w1b = tw[2 * t + 1];
    const float *__restrict__ x0 = g ? J.s0 : J.t0;
    const float *__restrict__ x1 = g ? J.s1 : J.t1;

    auto load_segment = [&](int seg, float2 (&v)[32]) {
        const i64 first = (i64)seg * kSeg;
        if (g == 0) {
            load_rows<kSeg / 256>(x0, x1, sc0, sc1, J.t_off + first, 0, J.n_t - first, t, v);
        } else {
            const i64 base = J.s_off + first;
            load_rows<32>(x0, x1, sc0, sc1, base, -base, J.sl - base, t, v);
        }
    };

    const int n_seg = J.n_seg, stride = J.n_cta;
    float2 v[32];
    load_segment(cta, v);
    const float2 *ZA = sm, *ZB = sm + kBuf;
    const float2 *ZO = g ? ZA : ZB;   // the other transform's spectrum
    const int q = tile_bin_parity(g, t);
    for (int seg = cta; seg < n_seg; seg += stride) {
        pass1_store(v, t, buf);
        bar_transform(g);
        float2 own[8];   // X_g[2t + q + 512 c], c = 0..7: this thread's own operand of its bins
        {
            float2 u0[16], u1[16];
            pass_load(buf, t, u0, u1);
            bar_transform(g);
            pass2_twiddle(u0, u1, t, tab);
            pass2_store(u0, u1, t, buf);
            bar_transform(g);
            pass_load(buf, t, u0, u1);
            bar_transform(g);
            pass3_compute(u0, w1a);
            pass3_compute(u1, w1b);
            spectrum_store(u0, u1, t, buf);  // natural order, into the (free again) buffer
#pragma unroll
            for (int c = 0; c < 8; c++) own[c] = q ? u1[c] : u0[c];
        }
        // the next segment's samples travel while the cross-spectra are formed (the fence
        // keeps the loads from being hoisted into the transform, where registers are full)
        asm volatile("" ::: "memory");
        // pass 1 transformed v in place: without the else, the last segment's spectrum (64 registers) would stay
        // live through passes 2 and 3 for an iteration the compiler cannot rule out, and the transform would spill
        if (seg + stride < n_seg) load_segment(seg + stride, v);
        else
#pragma unroll
            for (int r = 0; r < 32; r++) v[r] = make_float2(0.f, 0.f);
        __syncthreads();
        // bins k = 2t + q + 512 c, c = 0..7: X_g[k] is in a register, three operands come from shared memory
#pragma unroll
        for (int c = 0; c < 8; c++) {
            float acc[8];
            tmem_ld8(tmem + 8 * c, acc);
            const int k = 2 * t + q + 512 * c;
            const int nk = (kN - k) & (kN - 1);
            const float2 o = ZO[k];
            if (g == 0) cross_accumulate(own[c], ZA[nk], o, ZB[nk], acc);
            else cross_accumulate(o, ZA[nk], own[c], ZB[nk], acc);
            tmem_st8(tmem + 8 * c, acc);
        }
        if (warp == 8) {  // Nyquist bin: thread 0 of transform B; the whole warp moves its columns
            float acc[8];
            tmem_ld8(tmem + 64, acc);
            if (t == 0) cross_accumulate(ZA[kN / 2], ZA[kN / 2], ZB[kN / 2], ZB[kN / 2], acc);
            tmem_st8(tmem + 64, acc);
        }
        tmem_wait_st();
        __syncthreads();
    }
    // partial cross-spectra of this CTA, in the convention k_fft_reduce expects (re / 2, im / 4 applied there)
#pragma unroll
    for (int c = 0; c < 8; c++) {
        float acc[8];
        tmem_ld8(tmem + 8 * c, acc);
        const int k = 2 * t + q + 512 * c;
#pragma unroll
        for (int p = 0; p < 4; p++)
            if (J.partials[p]) J.partials[p][(size_t)cta * kBins + k] = make_float2(0.5f * acc[2 * p], acc[2 * p + 1]);
    }
    if (warp == 8) {
        float acc[8];
        tmem_ld8(tmem + 64, acc);
        if (t == 0) {
#pragma unroll
            for (int p = 0; p < 4; p++)
                if (J.partials[p]) J.partials[p][(size_t)cta * kBins + kN / 2] = make_float2(0.5f * acc[2 * p], acc[2 * p + 1]);
        }
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
}

// ---------------------------------------------------------------- 1024 threads, 16 points per thread
// The same tile, transform and accumulators with twice the warps: fft_tile16_core.cuh splits the 8192 points
// as 16 x 16 x 32 over 512 threads per transform (the radix-32 step by pairs of lanes through a shuffle), so a
// thread needs 64 registers and a CTA of 1024 threads fits the register file -- eight warps per scheduler
// instead of four to cover the shared-memory bursts and barriers between the arithmetic.
constexpr int kTile16Threads = 2 * fft16::kT16;

__device__ __forceinline__ void bar_transform16(int g) { asm volatile("bar.sync %0, 512;" ::"r"(g + 1) : "memory"); }

template <int CNT>
__device__ __forceinline__ void load_rows16(const float *__restrict__ x0, const float *__restrict__ x1, float sc0,
                                            float sc1, i64 base, i64 lo, i64 hi, int t, float2 (&v)[16])
{
    if (lo <= 0 && hi >= 512 * CNT) {
        const float *__restrict__ p0 = x0 + base + t;
        const float *__restrict__ p1 = x1 + base + t;
#pragma unroll
        for (int r = 0; r < 16; r++) v[r] = r < CNT ? make_float2(__ldg(p0 + 512 * r), __ldg(p1 + 512 * r)) : make_float2(0.f, 0.f);
    } else {
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const i64 m = t + 512 * r;
            const bool ok = r < CNT && m >= lo && m < hi;
            v[r] = ok ? make_float2(__ldg(x0 + base + m), __ldg(x1 + base + m)) : make_float2(0.f, 0.f);
        }
    }
    if (sc0 != 1.f || sc1 != 1.f) {
#pragma unroll
        for (int r = 0; r < CNT; r++) v[r] = make_float2(__fmul_rn(v[r].x, sc0), __fmul_rn(v[r].y, sc1));
    }
}

__global__ void __launch_bounds__(kTile16Threads, 1) k_fft_tiles16(const TileJob *jobs, const float2 *__restrict__ tw)
{
    using namespace fft16;
    extern __shared__ __align__(16) float2 sm[];
    __shared__ unsigned s_tmem;
    const TileJob &J = jobs[blockIdx.y];
    const int cta = blockIdx.x;
    if (cta >= J.n_cta) return;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int g = tid >> 9, t = tid & (kT16 - 1);
    // the scales first: their two dependent loads overlap the table fill and the tensor-memory set-up
    const double *st0 = g ? J.s0_stats : J.t0_stats, *st1 = g ? J.s1_stats : J.t1_stats;
    const float sc0 = rank_pre(st0, st1), sc1 = rank_pre(st1, st0);
    float2 *buf = sm + g * kBuf;
    float2 *tab = sm + 2 * kBuf;
    for (int idx = tid; idx < kTab; idx += kTile16Threads) tab[idx] = tw[(16 * (idx & 31) * (idx >> 5)) & (kN - 1)];
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (unsigned)__cvta_generic_to_shared(&s_tmem)), "n"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const unsigned tmem_base = s_tmem;
    // this thread's accumulators: lane 32 (warp % 4) + lane id, columns 64 (warp / 4) + [0, 40): four bins x
    // four products x (re, im), and the Nyquist bin's eight in the columns of warp 0
    const unsigned tmem = tmem_base + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)(64 * (warp >> 2));
    {
        float z[16];
#pragma unroll
        for (int i = 0; i < 16; i++) z[i] = 0.f;
#pragma unroll
        for (int c = 0; c < 3; c++) tmem_st16(tmem + 16 * c, z);
        tmem_wait_st();
    }
    const float2 w1 = tw[t];
    const float *__restrict__ x0 = g ? J.s0 : J.t0;
    const float *__restrict__ x1 = g ? J.s1 : J.t1;

    auto load_segment = [&](int seg, float2 (&v)[16]) {
        const i64 first = (i64)seg * kSeg;
        if (g == 0) {
            load_rows16<kSeg / 512>(x0, x1, sc0, sc1, J.t_off + first, 0, J.n_t - first, t, v);
        } else {
            const i64 base = J.s_off + first;
            load_rows16<16>(x0, x1, sc0, sc1, base, -base, J.sl - base, t, v);
        }
    };

    float2 v[16];
    int seg = cta;
    load_segment(seg, v);
    const float2 *ZA = sm, *ZB = sm + kBuf;
    for (; seg < J.n_seg; seg += J.n_cta) {
        pass1(v, t, w1, buf);
        bar_transform16(g);
        {
            float2 u[16];
            pass2_load(buf, t, u);
            bar_transform16(g);
            pass2_store(u, t, tab, buf);
        }
        bar_transform16(g);
        {
            float2 p[16], recv[8], lo[8], hi[8];
            pass3_first(buf, t, p);
#pragma unroll
            for (int i = 0; i < 8; i++)
                recv[i] = make_float2(__shfl_xor_sync(0xffffffffu, p[8 + i].x, 16), __shfl_xor_sync(0xffffffffu, p[8 + i].y, 16));
            bar_transform16(g);   // every thread of the transform has read its pass-3 inputs: the buffer takes the spectrum
            pass3_combine(p, recv, t, lo, hi);
            spectrum_store16(lo, hi, t, buf);
        }
        asm volatile("" ::: "memory");
        if (seg + J.n_cta < J.n_seg) load_segment(seg + J.n_cta, v);
        __syncthreads();
        // bins k = tid + 1024 c, c = 0..3: four products per 8-column chunk
#pragma unroll
        for (int c = 0; c < 4; c++) {
            float acc[8];
            tmem_ld8(tmem + 8 * c, acc);
            const int k = tid + 1024 * c;
            const int nk = (kN - k) & (kN - 1);
            cross_accumulate(ZA[k], ZA[nk], ZB[k], ZB[nk], acc);
            tmem_st8(tmem + 8 * c, acc);
        }
        if (warp == 0) {  // Nyquist bin: thread 0; the whole warp moves its columns
            float acc[8];
            tmem_ld8(tmem + 32, acc);
            if (tid == 0) cross_accumulate(ZA[kN / 2], ZA[kN / 2], ZB[kN / 2], ZB[kN / 2], acc);
            tmem_st8(tmem + 32, acc);
        }
        tmem_wait_st();
        __syncthreads();
    }
    // partial cross-spectra of this CTA, in the convention k_fft_reduce expects (re / 2, im / 4 applied there)
#pragma unroll
    for (int c = 0; c < 4; c++) {
        float acc[8];
        tmem_ld8(tmem + 8 * c, acc);
        const int k = tid + 1024 * c;
#pragma unroll
        for (int p = 0; p < 4; p++)
            if (J.partials[p]) J.partials[p][(size_t)cta * kBins + k] = make_float2(0.5f * acc[2 * p], acc[2 * p + 1]);
    }
    if (warp == 0) {
        float acc[8];
        tmem_ld8(tmem + 32, acc);
        if (tid == 0) {
#pragma unroll
            for (int p = 0; p < 4; p++)
                if (J.partials[p]) J.partials[p][(size_t)cta * kBins + kN / 2] = make_float2(0.5f * acc[2 * p], acc[2 * p + 1]);
        }
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
}

}  // namespace

int fft_tile_setup()
{
    return cudaFuncSetAttribute(k_fft_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, kTileSmem) == cudaSuccess &&
                   cudaFuncSetAttribute(k_fft_tiles16, cudaFuncAttributeMaxDynamicSharedMemorySize, kTileSmem) == cudaSuccess
               ? 0 : -1;
}

void launch_fft_tiles(const TileJob *d_jobs, int n_jobs, int max_cta, const float2 *d_tw, cudaStream_t st)
{
    if (n_jobs <= 0 || max_cta <= 0) return;
    static const int tile16 = getenv("TDOA_FFT_TILE16") ? atoi(getenv("TDOA_FFT_TILE16")) : 0;   // experiment switch
    if (tile16) k_fft_tiles16<<<dim3(max_cta, n_jobs), kTile16Threads, kTileSmem, st>>>(d_jobs, d_tw);
    else k_fft_tiles<<<dim3(max_cta, n_jobs), kTileThreads, kTileSmem, st>>>(d_jobs, d_tw);
}

}  // namespace tdoa
