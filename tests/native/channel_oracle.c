/* channel_oracle.c -- the channel filter's statement (include/tdoa_b200.h, tdoa_set_channel) restated on the CPU
 * with explicit fmaf, for tests/channel_oracle.py.  glibc's fmaf is correctly rounded, and -ffp-contract=off keeps
 * the compiler from fusing anything else.
 *
 * For every i: acc = +0 + 0j, then for k = 0 .. T-1 ascending, v = x[i + c - k] (zero outside [0, n)),
 * c = (T - 1) / 2:
 *   acc.re = fmaf(hr[k], v.re, acc.re); acc.re = fmaf(-hi[k], v.im, acc.re);
 *   acc.im = fmaf(hr[k], v.im, acc.im); acc.im = fmaf(hi[k], v.re, acc.im);
 * hi == NULL: every hi[k] is +0 (the four FMAs are still taken). */
#include <math.h>
#include <stdint.h>

typedef struct { float re, im; } c64;

__attribute__((visibility("default"))) void orc_channel(const c64 *x, int64_t n, const float *hr, const float *hi,
                                                       int32_t T, c64 *y)
{
    const int64_t c = (T - 1) / 2;
    for (int64_t i = 0; i < n; i++) {
        float ar = 0.f, ai = 0.f;
        for (int32_t k = 0; k < T; k++) {
            const int64_t q = i + c - k;
            const c64 v = (q >= 0 && q < n) ? x[q] : (c64){0.f, 0.f};
            const float h_i = hi ? hi[k] : 0.f;
            ar = fmaf(hr[k], v.re, ar);
            ar = fmaf(-h_i, v.im, ar);
            ai = fmaf(hr[k], v.im, ai);
            ai = fmaf(h_i, v.re, ai);
        }
        y[i].re = ar;
        y[i].im = ai;
    }
}
