// discriminate.cuh -- the FM discriminator's statement for one sample, shared by k_demod (preprocess.cu) and
// k_channel_demod (channel.cu), so that the channel filter's fused kernel gives k_demod's bits on its planes.
#pragma once
#include "common.cuh"

namespace tdoa {

// ELF 0x49d120 (no source): out[i] = atan2(Im p, Re p), p = complex64(s[i]*conj(s[i-1]))
// (f64 products, one rounding to f32); gates leave 0; out[0] = out[1].
__device__ __forceinline__ float discriminate(float2 prev, float2 cur)
{
    if (prev.x == 0.f && prev.y == 0.f) return 0.f;
    const double pr = prev.x, pi = prev.y, cr = cur.x, ci = cur.y, npi = -pi;
    const double re = __dsub_rn(__dmul_rn(pr, cr), __dmul_rn(ci, npi));
    const double im = __dadd_rn(__dmul_rn(npi, cr), __dmul_rn(ci, pr));
    const float fre = (float)re, fim = (float)im;
    if (fre == 0.f && fim == 0.f) return 0.f;
    const float m = __fadd_rn(__fmul_rn(fre, fre), __fmul_rn(fim, fim));
    if (!(m > 1e-10f)) return 0.f;
    return (float)atan2((double)fim, (double)fre);
}

}  // namespace tdoa
