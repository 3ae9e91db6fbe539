// Host emulation of k_fft_tiles' cross phase (csrc/xcorr_tile.cu) with the bin map of csrc/fft_tile_core.cuh:
// thread t of transform g takes the bins k = 2t + q + 512 c, q = tile_bin_parity(g, t), c = 0..7, with X_g[k] from
// its pass-3 registers and the other three operands from the spectra spectrum_store wrote.  Checks that
//   - every bin 0 .. N/2 - 1 is taken exactly once;
//   - the accumulators equal, bit for bit, those of all four operands read from shared memory;
//   - each 64-bit load (at k and at N - k) is conflict-free: the 16 lanes of each half warp read 16 distinct
//     bank pairs.
// Built and run by tests/test_fft_tile_cross.py (no GPU).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "fft_tile_core.cuh"

using namespace tdoa::fft2;

int main()
{
    srand(777);
    auto rnd = [] { return (float)rand() / RAND_MAX - 0.5f; };
    // pass-3 registers of both transforms: u[g][t][0] = X_g[2t + 512 r], u[g][t][1] = X_g[2t + 1 + 512 r]
    static float2 u[2][kT][2][16];
    std::vector<float2> Z[2] = {std::vector<float2>(kN), std::vector<float2>(kN)};
    for (int g = 0; g < 2; g++)
        for (int t = 0; t < kT; t++) {
            for (int r = 0; r < 16; r++)
                for (int h = 0; h < 2; h++) u[g][t][h][r] = make_float2(rnd(), rnd());
            spectrum_store(u[g][t][0], u[g][t][1], t, Z[g].data());
        }
    const float2 *ZA = Z[0].data(), *ZB = Z[1].data();
    std::vector<int> taken(kN / 2, 0);
    int bad_acc = 0, conflicts = 0;
    for (int g = 0; g < 2; g++)
        for (int c = 0; c < 8; c++)
            for (int w = 0; w < kT / 32; w++) {
                for (int half = 0; half < 2; half++) {   // bank pairs of one 64-bit load per half warp
                    int seen_k = 0, seen_nk = 0;
                    for (int l = 16 * half; l < 16 * half + 16; l++) {
                        const int t = 32 * w + l, k = 2 * t + tile_bin_parity(g, t) + 512 * c;
                        seen_k |= 1 << (k & 15);
                        seen_nk |= 1 << (((kN - k) & (kN - 1)) & 15);
                    }
                    conflicts += (seen_k != 0xffff) + (seen_nk != 0xffff);
                }
                for (int l = 0; l < 32; l++) {
                    const int t = 32 * w + l, q = tile_bin_parity(g, t);
                    const int k = 2 * t + q + 512 * c, nk = (kN - k) & (kN - 1);
                    taken[k]++;
                    const float2 own = u[g][t][q][c];
                    float got[8], want[8];
                    for (int i = 0; i < 8; i++) got[i] = want[i] = 0.1f * (float)i;
                    if (g == 0) cross_accumulate(own, ZA[nk], ZB[k], ZB[nk], got);
                    else cross_accumulate(ZA[k], ZA[nk], own, ZB[nk], got);
                    cross_accumulate(ZA[k], ZA[nk], ZB[k], ZB[nk], want);
                    bad_acc += memcmp(got, want, sizeof got) != 0;
                }
            }
    int bad_map = 0;
    for (int k = 0; k < kN / 2; k++) bad_map += taken[k] != 1;
    printf("bins_not_taken_once %d\naccumulators_differing %d\nconflicted_loads %d\n", bad_map, bad_acc, conflicts);
    return bad_map || bad_acc || conflicts;
}
