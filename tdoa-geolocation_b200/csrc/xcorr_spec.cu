// xcorr_spec.cu -- many stations per window (BASELINE config 4: 16 stations, 120 pairs):
// every station-segment is transformed ONCE, the pairs are formed from the parked spectra.
//
// The 2 x 2 station tiles of xcorr_tile.cu transform a station again in every tile it
// appears in: 16 stations need 36 tiles = 72 transforms per segment where 16 suffice
// (15 template roles + 15 signal roles, two real signals per complex transform).  Here:
//   k_spec_fft : one CTA = one 8192-point transform (fft_tile_core.cuh) of a pair of
//                planes -- template segments zero padded after `seg` samples, signal
//                segments 8192 samples long -- unpacked into the two stations' spectra and
//                written to global memory ([segment][chunk of 32 bins][row][32]; parked in L2 / HBM)
//   k_spec_acc : one CTA = 32 frequency bins of one (window, lag chunk) for ALL its pairs, one warp
//                per 4 x 4 register tile of pairs; per segment the chunk's block of station
//                spectra arrives by cp.async and conj(T_a) S_c is added into the threads' registers;
//                after the last segment the pair spectra go straight to k_fft_finish (xcorr_fft.cu),
//                no partials, no reduce.
// Because the segment length is a parameter here, a search of 2049..4096 lags runs as ONE
// chunk of 4096-sample segments instead of two chunks of 6144-sample segments.
#include "fft_tile_core.cuh"
#include "kernels.h"
#include "xcorr_fft.h"

namespace tdoa {

using namespace fft2;

namespace {

constexpr int kRowSmem = (kBuf + kTab) * (int)sizeof(float2);
constexpr int kAccBins = kSpecBins;                          // 32 bins per CTA: a warp is one register tile
constexpr int kAccGroups = kSpecMaxTiles;                    // one warp per tile
constexpr int kAccThreads = kAccGroups * kAccBins;           // 320
constexpr int kSpecStages = 4;                               // ring of parked blocks, three segments ahead
constexpr int kStageBytes = 2 * kSpecMaxPacked * kAccBins * (int)sizeof(float2);   // 32 rows x 256 B = 8 KB
constexpr int kAccSmem = kSpecStages * kStageBytes;          // 32 KB: three CTAs per SM

// ---------------------------------------------------------------- transforms
// One CTA = one 8192-point transform of a pair of planes (Z = FFT(x0 + i x1)), then the two stations' own
// spectra, X0[k] = (Z[k] + conj Z[N-k]) / 2 and X1[k] = (Z[k] - conj Z[N-k]) / (2 i), k = 0 .. 4096, written
// to the unit's parked block.  (Round 2, first half: Z itself was parked and every accumulation CTA undid the
// packing per segment -- a quarter of that kernel's instructions; this kernel waits on memory and has the slots.)
__global__ void __launch_bounds__(kT, 2) k_spec_fft(const SpecFftJob *jobs, int n_jobs, const float2 *__restrict__ tw)
{
    extern __shared__ __align__(16) float2 sm[];
    // transform fastest: the CTAs in flight together fill ONE segment's parked block (its rows lie 512 bytes apart
    // in every chunk), so the block's lines complete in L2 before they are written back
    const SpecFftJob &J = jobs[blockIdx.x % (unsigned)n_jobs];
    const int seg = (int)(blockIdx.x / (unsigned)n_jobs);
    if (seg >= J.n_seg) return;
    const int t = threadIdx.x;
    float2 *buf = sm, *tab = sm + kBuf;
    for (int idx = t; idx < kTab; idx += kT) tab[idx] = tw[(16 * (idx & 31) * (idx >> 5)) & (kN - 1)];
    const float2 w1a = tw[2 * t], w1b = tw[2 * t + 1];
    {
        // z[m] = x0[i] sc0 + i x1[i] sc1, i = base + seg * stride + m, for m < seg_len and lo <= i < hi; sc = rank_pre
        // (xcorr_fft.h), 1 unless the two planes' powers differ widely
        const i64 first = J.base + (i64)seg * J.stride;
        const float *__restrict__ x0 = J.x0, *__restrict__ x1 = J.x1;
        const float sc0 = rank_pre(J.x0_stats, J.x1_stats), sc1 = rank_pre(J.x1_stats, J.x0_stats);
        float2 v[32];
        if (first >= J.lo && first + J.seg_len <= J.hi && (J.seg_len & 255) == 0) {
            const int rows = J.seg_len >> 8;
#pragma unroll
            for (int r = 0; r < 32; r++) v[r] = r < rows ? make_float2(x0[first + t + 256 * r], x1[first + t + 256 * r]) : make_float2(0.f, 0.f);
        } else {
#pragma unroll
            for (int r = 0; r < 32; r++) {
                const int m = t + 256 * r;
                const i64 i = first + m;
                v[r] = (m < J.seg_len && i >= J.lo && i < J.hi) ? make_float2(x0[i], x1[i]) : make_float2(0.f, 0.f);
            }
        }
        if (sc0 != 1.f || sc1 != 1.f) {
#pragma unroll
            for (int r = 0; r < 32; r++) v[r] = make_float2(__fmul_rn(v[r].x, sc0), __fmul_rn(v[r].y, sc1));
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
        spectrum_store(u0, u1, t, buf);   // Z in natural order, into the (free again) buffer
    }
    __syncthreads();
    // bins k = 2 (t + 256 w) and k + 1: 16-byte stores, a half-warp's 32 bins are one chunk's row (256 contiguous bytes)
    float2 *__restrict__ out = J.out + (size_t)seg * spec_seg_elems(J.n_rows);
    const size_t row_a = (size_t)J.row0 * kSpecBins, chunk_stride = (size_t)J.n_rows * kSpecBins;
#pragma unroll
    for (int w = 0; w < 8; w++) {
        const int k = 2 * (t + 256 * w);
        const float4 a = *reinterpret_cast<const float4 *>(buf + k);            // Z[k], Z[k + 1]
        const float2 c0 = buf[(kN - k) & (kN - 1)], c1 = buf[kN - k - 1];       // Z[N - k], Z[N - k - 1]
        float2 *o = out + (size_t)(k >> 5) * chunk_stride + row_a + (k & (kSpecBins - 1));
        *reinterpret_cast<float4 *>(o) = make_float4(0.5f * (a.x + c0.x), 0.5f * (a.y - c0.y), 0.5f * (a.z + c1.x), 0.5f * (a.w - c1.y));
        *reinterpret_cast<float4 *>(o + kSpecBins) = make_float4(0.5f * (a.y + c0.y), 0.5f * (c0.x - a.x), 0.5f * (a.w + c1.y), 0.5f * (c1.x - a.z));
    }
    if (t == 0) {   // the Nyquist bin is its own partner
        const float2 a = buf[kN / 2];
        float2 *o = out + (size_t)(kSpecChunks - 1) * chunk_stride + row_a;
        o[0] = make_float2(0.5f * (a.x + a.x), 0.5f * (a.y - a.y));
        o[kSpecBins] = make_float2(0.5f * (a.y + a.y), 0.5f * (a.x - a.x));
    }
}

// ---------------------------------------------------------------- pair accumulation
// One CTA = 32 frequency bins of one (window, lag chunk); one WARP = one 4 x 4 register tile of pairs (templates
// a0..a3 against signals c0..c3), lanes = bins.  Per segment a thread loads its 4 + 4 station values from the
// ring and adds the 16 products conj(T_a) S_c: 8 shared-memory loads and 64 FMA where the pair-by-pair kernel
// before it spent 17 instructions per pair (two PRMT, two address adds, a test and up to two loads around four
// FMA).  16 stations, all pairs: 10 tiles (the station pairs i < j in template row i, signal row j - 1 fill the
// blocks I <= J of a 4 x 4 block grid); products a tile has no pair for are computed and dropped.  The parked
// block of a segment is contiguous (xcorr_fft.h): it arrives by 16-byte cp.async, three segments ahead, and is
// read in place -- no unpacking, one barrier per segment.  Sums run segment by segment with the same two FMA
// chains per component as before: the pair spectra are bit for bit the earlier kernel's.
__global__ void __launch_bounds__(kAccThreads, 3) k_spec_acc(const SpecAccJob *jobs)
{
    extern __shared__ __align__(16) unsigned char ring[];    // [stage][row][bin] float2
    const SpecAccJob &J = jobs[blockIdx.y];
    const int chunk = blockIdx.x;
    const int k0 = chunk * kAccBins;
    const int nb = min(kAccBins, kN / 2 + 1 - k0);
    const int tid = threadIdx.x, b = tid & (kAccBins - 1), g = tid >> 5;
    const int n_rows = J.n_rows, n_seg = J.n_seg;
    const bool worker = g < J.n_tiles;
    const int gt = worker ? g : 0;
    unsigned off_t[kSpecTile], off_s[kSpecTile];
#pragma unroll
    for (int a = 0; a < kSpecTile; a++) {
        off_t[a] = (unsigned)((J.t_row[gt][a] * kAccBins + b) * sizeof(float2));
        off_s[a] = (unsigned)((J.s_row[gt][a] * kAccBins + b) * sizeof(float2));
    }
    float2 acc[kSpecTile * kSpecTile];
#pragma unroll
    for (int q = 0; q < kSpecTile * kSpecTile; q++) acc[q] = make_float2(0.f, 0.f);
    const unsigned ring_base = (unsigned)__cvta_generic_to_shared(ring);
    const int n_piece = n_rows * (kAccBins * (int)sizeof(float2) / 16);   // 16-byte pieces of a block: <= 512
    const size_t seg_stride = spec_seg_elems(n_rows);
    const float2 *__restrict__ src0 = J.spec + (size_t)chunk * n_rows * kAccBins;
    auto issue = [&](int seg) {
        if (seg < n_seg) {
            const char *src = reinterpret_cast<const char *>(src0 + (size_t)seg * seg_stride);
            const unsigned dst = ring_base + (unsigned)((seg % kSpecStages) * kStageBytes);
            for (int p = tid; p < n_piece; p += kAccThreads)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (unsigned)p), "l"(src + 16 * (size_t)p) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto lds2 = [](unsigned addr) {
        float2 v;
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
        return v;
    };
#pragma unroll
    for (int p = 0; p < kSpecStages - 1; p++) issue(p);
    for (int seg = 0; seg < n_seg; seg++) {
        asm volatile("cp.async.wait_group %0;" ::"n"(kSpecStages - 2) : "memory");   // this thread's pieces of `seg` have landed
        __syncthreads();   // everybody's have, and everybody is done with segment seg - 1, whose stage is refilled next
        issue(seg + kSpecStages - 1);
        if (worker) {
            const unsigned base = ring_base + (unsigned)((seg % kSpecStages) * kStageBytes);
            float2 tv[kSpecTile], sv[kSpecTile];
#pragma unroll
            for (int a = 0; a < kSpecTile; a++) { tv[a] = lds2(base + off_t[a]); sv[a] = lds2(base + off_s[a]); }
#pragma unroll
            for (int a = 0; a < kSpecTile; a++)
#pragma unroll
                for (int c = 0; c < kSpecTile; c++) {
                    float2 &q = acc[kSpecTile * a + c];
                    // conj(T) S
                    q.x = fmaf(tv[a].x, sv[c].x, fmaf(tv[a].y, sv[c].y, q.x));
                    q.y = fmaf(tv[a].x, sv[c].y, fmaf(-tv[a].y, sv[c].x, q.y));
                }
        }
    }
    if (worker && b < nb) {
#pragma unroll
        for (int q = 0; q < kSpecTile * kSpecTile; q++) {
            float2 *o = J.out[g][q];
            if (o) o[k0 + b] = acc[q];
        }
    }
}

}  // namespace

int spec_setup()
{
    return cudaFuncSetAttribute(k_spec_fft, cudaFuncAttributeMaxDynamicSharedMemorySize, kRowSmem) == cudaSuccess &&
                   cudaFuncSetAttribute(k_spec_acc, cudaFuncAttributeMaxDynamicSharedMemorySize, kAccSmem) == cudaSuccess
               ? 0 : -1;
}

void launch_spec_fft(const SpecFftJob *d_jobs, int n_jobs, int max_seg, const float2 *d_tw, cudaStream_t st)
{
    if (n_jobs <= 0 || max_seg <= 0) return;
    // (a 512-thread, 16-points-per-thread variant of this kernel -- 32 warps per SM instead of 16 -- measured 0.95-0.99 ms
    // against 0.94-0.98 ms on config 4: the kernel waits on the memory system, 3.2 TB/s of mostly writes, not on latency)
    k_spec_fft<<<(unsigned)max_seg * (unsigned)n_jobs, kT, kRowSmem, st>>>(d_jobs, n_jobs, d_tw);
}

void launch_spec_acc(const SpecAccJob *d_jobs, int n_jobs, cudaStream_t st)
{
    if (n_jobs <= 0) return;
    k_spec_acc<<<dim3(kSpecChunks, n_jobs), kAccThreads, kAccSmem, st>>>(d_jobs);
}

}  // namespace tdoa
