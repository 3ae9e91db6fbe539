// fft_tile_core.cuh -- second-generation 8192-point complex FFT in one CTA's shared
// memory, written against the B200's instruction budget (the transform is FP32-issue
// bound, not bandwidth bound):
//   - decimation-in-time butterflies in registers whose twiddle multiply is folded into
//     the add/subtract with FMAs: X = a + w b costs 4 FMA, Y = 2a - X costs 2 (6
//     instructions against 8 for multiply-then-add; 4 for the trivial twiddles);
//   - three Stockham passes (radix 32, 16, 16) over 256 threads, 32 points per thread;
//     rows of 32 points are padded by 2 so that the radix-32 pass writes 128-bit words
//     and every other access is a conflict-free 64-bit one, with all offsets folded
//     into the instruction (one base register per phase);
//   - pass-2 twiddles W_512^(r k) from a per-lane table, pass-3 twiddles W_8192^(r j) from
//     one seed per butterfly and a product tree with squarings.
// Everything is __host__ __device__: tests/native/fft_tile_emul.cu runs the phases one
// "thread" at a time on the CPU against a direct DFT (no GPU needed to check the maths).
#pragma once
#include <cuda_runtime.h>

namespace tdoa {
namespace fft2 {

#define TDOA_HD2 __host__ __device__ __forceinline__

constexpr int kN = 8192;                 // complex points
constexpr int kT = 256;                  // threads per transform
constexpr int kRow = 34;                 // float2 per padded row of 32 points
constexpr int kBuf = (kN / 32) * kRow;   // float2 per transform buffer (8704)
constexpr int kTab = 16 * 32;            // pass-2 twiddle table entries

TDOA_HD2 int pad2(int i) { return i + 2 * (i >> 5); }

// W_32^k = exp(-2 pi i k / 32)
__host__ __device__ constexpr float c32(int k)
{
    constexpr float c[16] = {1.0f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254524f,
                             0.70710678118654752f, 0.55557023301960218f, 0.38268343236508977f, 0.19509032201612825f,
                             0.0f, -0.19509032201612825f, -0.38268343236508977f, -0.55557023301960218f,
                             -0.70710678118654752f, -0.83146961230254524f, -0.92387953251128674f, -0.98078528040323043f};
    return c[k];
}
__host__ __device__ constexpr float s32(int k)
{
    constexpr float s[16] = {0.0f, -0.19509032201612825f, -0.38268343236508977f, -0.55557023301960218f,
                             -0.70710678118654752f, -0.83146961230254524f, -0.92387953251128674f, -0.98078528040323043f,
                             -1.0f, -0.98078528040323043f, -0.92387953251128674f, -0.83146961230254524f,
                             -0.70710678118654752f, -0.55557023301960218f, -0.38268343236508977f, -0.19509032201612825f};
    return s[k];
}

// a, b <- a + W_32^K b, a - W_32^K b
template <int K>
TDOA_HD2 void bfly(float2 &a, float2 &b)
{
    if constexpr (K == 0) {
        const float2 x = make_float2(a.x + b.x, a.y + b.y), y = make_float2(a.x - b.x, a.y - b.y);
        a = x; b = y;
    } else if constexpr (K == 8) {  // w = -i: w b = (b.y, -b.x)
        const float2 x = make_float2(a.x + b.y, a.y - b.x), y = make_float2(a.x - b.y, a.y + b.x);
        a = x; b = y;
    } else if constexpr (K == 4) {  // w = (1 - i) h: w b = h (b.x + b.y, b.y - b.x)
        constexpr float h = 0.70710678118654752f;
        const float s = b.x + b.y, d = b.y - b.x;
        const float2 x = make_float2(fmaf(h, s, a.x), fmaf(h, d, a.y)), y = make_float2(fmaf(-h, s, a.x), fmaf(-h, d, a.y));
        a = x; b = y;
    } else if constexpr (K == 12) {  // w = (-1 - i) h: w b = h (b.y - b.x, -(b.x + b.y))
        constexpr float h = 0.70710678118654752f;
        const float s = b.x + b.y, d = b.y - b.x;
        const float2 x = make_float2(fmaf(h, d, a.x), fmaf(-h, s, a.y)), y = make_float2(fmaf(-h, d, a.x), fmaf(h, s, a.y));
        a = x; b = y;
    } else {
        constexpr float c = c32(K), s = s32(K);
        const float xr = fmaf(c, b.x, fmaf(-s, b.y, a.x));
        const float xi = fmaf(c, b.y, fmaf(s, b.x, a.y));
        const float2 y = make_float2(fmaf(2.f, a.x, -xr), fmaf(2.f, a.y, -xi));
        a = make_float2(xr, xi); b = y;
    }
}

// one DIT stage of butterfly size LEN over an R-point register array
template <int R, int LEN, int B, int K>
struct DitStage {
    static TDOA_HD2 void run(float2 (&v)[R])
    {
        constexpr int i = B * LEN + K;
        bfly<K * (32 / LEN)>(v[i], v[i + LEN / 2]);
        if constexpr (K + 1 < LEN / 2) DitStage<R, LEN, B, K + 1>::run(v);
        else if constexpr (B + 1 < R / LEN) DitStage<R, LEN, B + 1, 0>::run(v);
    }
};

template <int R, int LEN>
TDOA_HD2 void dit_all(float2 (&v)[R])
{
    DitStage<R, LEN, 0, 0>::run(v);
    if constexpr (LEN < R) dit_all<R, LEN * 2>(v);
}

template <int R>
__host__ __device__ constexpr int bitrev(int i)
{
    int r = 0;
    for (int b = 1; b < R; b <<= 1) { r = (r << 1) | (i & 1); i >>= 1; }
    return r;
}

template <int R, int I>
TDOA_HD2 void scramble(const float2 (&v)[R], float2 (&o)[R])
{
    o[I] = v[bitrev<R>(I)];
    if constexpr (I + 1 < R) scramble<R, I + 1>(v, o);
}

// forward DFT of R points (R = 16 or 32), natural order in and out
template <int R>
TDOA_HD2 void dft(float2 (&v)[R])
{
    float2 o[R];
    scramble<R, 0>(v, o);
    dit_all<R, 2>(o);
#pragma unroll
    for (int i = 0; i < R; i++) v[i] = o[i];
}

TDOA_HD2 float2 cmul(float2 a, float2 b) { return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x)); }
TDOA_HD2 float2 csqr(float2 a) { return make_float2(fmaf(a.x, a.x, -a.y * a.y), 2.f * a.x * a.y); }

// v[r] *= w^r, r = 1..15
TDOA_HD2 void twiddle16(float2 (&v)[16], float2 w1)
{
    const float2 w2 = csqr(w1), w3 = cmul(w2, w1), w4 = csqr(w2);
    const float2 w5 = cmul(w4, w1), w6 = csqr(w3), w7 = cmul(w4, w3), w8 = csqr(w4);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], w3);
    v[4] = cmul(v[4], w4);
    v[5] = cmul(v[5], w5);
    v[6] = cmul(v[6], w6);
    v[7] = cmul(v[7], w7);
    v[8] = cmul(v[8], w8);
    v[9] = cmul(v[9], cmul(w8, w1));
    v[10] = cmul(v[10], cmul(w8, w2));
    v[11] = cmul(v[11], cmul(w8, w3));
    v[12] = cmul(v[12], cmul(w8, w4));
    v[13] = cmul(v[13], cmul(w8, w5));
    v[14] = cmul(v[14], cmul(w8, w6));
    v[15] = cmul(v[15], cmul(w8, w7));
}

// ---- per-thread phases of one transform (t = thread index within the transform, 0..255);
// barriers over the transform's 256 threads go between them.
//
// pass 1: radix 32.  in[t + 256 r] (already in v) -> out[32 t + r], stored as 128-bit pairs
TDOA_HD2 void pass1_store(float2 (&v)[32], int t, float2 *buf)
{
    dft<32>(v);
    float4 *row = reinterpret_cast<float4 *>(buf + kRow * t);
#pragma unroll
    for (int r = 0; r < 16; r++) row[r] = make_float4(v[2 * r].x, v[2 * r].y, v[2 * r + 1].x, v[2 * r + 1].y);
}

// passes 2 and 3: a thread owns the ADJACENT butterflies j = 2t and 2t + 1, so every
// shared-memory access moves two complex points (128 bits).  Inputs in[j + 512 r], r = 0..15.
TDOA_HD2 void pass_load(const float2 *buf, int t, float2 (&u0)[16], float2 (&u1)[16])
{
    const float4 *p = reinterpret_cast<const float4 *>(buf + pad2(2 * t));
#pragma unroll
    for (int r = 0; r < 16; r++) {
        const float4 q = p[((512 + 32) / 2) * r];
        u0[r] = make_float2(q.x, q.y);
        u1[r] = make_float2(q.z, q.w);
    }
}

// pass 2: radix 16 with twiddles W_512^(r k), k = j % 32, from tab[r * 32 + k];
// out[(j / 32) * 512 + k + 32 r]
TDOA_HD2 void pass2_twiddle(float2 (&u0)[16], float2 (&u1)[16], int t, const float2 *tab)
{
    const float4 *p = reinterpret_cast<const float4 *>(tab + ((2 * t) & 31));
#pragma unroll
    for (int r = 1; r < 16; r++) {
        const float4 w = p[16 * r];
        u0[r] = cmul(u0[r], make_float2(w.x, w.y));
        u1[r] = cmul(u1[r], make_float2(w.z, w.w));
    }
}
TDOA_HD2 void pass2_store(float2 (&u0)[16], float2 (&u1)[16], int t, float2 *buf)
{
    dft<16>(u0);
    dft<16>(u1);
    float4 *p = reinterpret_cast<float4 *>(buf + ((2 * t) >> 5) * (16 * kRow) + ((2 * t) & 31));
#pragma unroll
    for (int r = 0; r < 16; r++) p[(kRow / 2) * r] = make_float4(u0[r].x, u0[r].y, u1[r].x, u1[r].y);
}

// pass 3: radix 16 with twiddles W_8192^(r j), w1 = W_8192^j; result u[r] = X[j + 512 r]
TDOA_HD2 void pass3_compute(float2 (&u)[16], float2 w1)
{
    twiddle16(u, w1);
    dft<16>(u);
}
// spectrum in natural order: X[2t + 512 r], X[2t + 1 + 512 r]
TDOA_HD2 void spectrum_store(const float2 (&u0)[16], const float2 (&u1)[16], int t, float2 *buf)
{
    float4 *p = reinterpret_cast<float4 *>(buf) + t;
#pragma unroll
    for (int r = 0; r < 16; r++) p[256 * r] = make_float4(u0[r].x, u0[r].y, u1[r].x, u1[r].y);
}

// ---- cross-spectra of a 2 x 2 tile.  A = FFT(t0 + i t1), B = FFT(s0 + i s1) with real
// t, s.  At bin k, with a = A[k], c = A[N-k], b = B[k], d = B[N-k]:
//   2 T0 = (a.x + c.x, a.y - c.y)   2 T1 = (a.y + c.y, c.x - a.x)      (same for S from b, d)
// and acc[2 (2 ta + sb) + {0, 1}] += 4 conj(T_ta[k]) S_sb[k]  (re, im).
TDOA_HD2 void cross_accumulate(float2 a, float2 c, float2 b, float2 d, float *acc)
{
    const float t0x = a.x + c.x, t0y = a.y - c.y, t1x = a.y + c.y, t1y = c.x - a.x;
    const float s0x = b.x + d.x, s0y = b.y - d.y, s1x = b.y + d.y, s1y = d.x - b.x;
    acc[0] = fmaf(t0x, s0x, fmaf(t0y, s0y, acc[0]));
    acc[1] = fmaf(t0x, s0y, fmaf(-t0y, s0x, acc[1]));
    acc[2] = fmaf(t0x, s1x, fmaf(t0y, s1y, acc[2]));
    acc[3] = fmaf(t0x, s1y, fmaf(-t0y, s1x, acc[3]));
    acc[4] = fmaf(t1x, s0x, fmaf(t1y, s0y, acc[4]));
    acc[5] = fmaf(t1x, s0y, fmaf(-t1y, s0x, acc[5]));
    acc[6] = fmaf(t1x, s1x, fmaf(t1y, s1y, acc[6]));
    acc[7] = fmaf(t1x, s1y, fmaf(-t1y, s1x, acc[7]));
}

// Bins k < N/2 of a tile, one per register slot c = 0..7: thread t of transform g takes k = 2t + q + 512 c, whose
// X_g[k] it holds after pass 3 (u0[c] for q = 0, u1[c] for q = 1), and loads only A or B at k, A[N-k] and B[N-k].
// The two transforms' threads t split the pair {2t, 2t + 1} + 512 c between them.  Lanes 8..15 and 24..31 of a warp
// take the other parity than lanes 0..7 and 16..23, so the 16 lanes of each half warp hit 16 distinct 64-bit bank
// pairs at k and at N - k: one wavefront each, where all-even bins (a 16-byte stride) would be two-way conflicted.
TDOA_HD2 int tile_bin_parity(int g, int t) { return ((t >> 3) & 1) ^ g; }

}  // namespace fft2
}  // namespace tdoa
