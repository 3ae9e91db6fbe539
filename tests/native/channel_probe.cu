// channel_probe.cu -- the two kernels of channel.cu driven directly from host arrays, for
// tests/test_gpu_channel_kernels.py (built there with channel.cu's own flags, linked with preprocess.cu for the
// plane kernels it is compared with, and loaded with ctypes).
//
// Every output array sits between two runs of kCanary canary words, and the output itself is filled with
// kUnwritten before the launch, so a stray write and a missing write both show on the host.  Return value: the
// first CUDA error of the call (0 = none).
#include "channel.cu"

#include <cstring>
#include <vector>

namespace {

constexpr int kCanary = 64;
constexpr uint32_t kCanaryWord = 0xdeadbeefu;
constexpr uint32_t kUnwritten = 0x7fc00001u;   // a NaN no filter of finite samples produces

struct Status {
    cudaError_t err = cudaSuccess;
    void operator()(cudaError_t e) { if (err == cudaSuccess && e != cudaSuccess) err = e; }
};

template <typename T>
T *alloc_guarded(Status &ok, std::vector<void *> &owned, long long n)
{
    static_assert(sizeof(T) % 4 == 0, "32-bit words");
    const size_t words = sizeof(T) / 4, total = (size_t)(n + 2 * kCanary) * words;
    std::vector<uint32_t> h(total, kUnwritten);
    for (size_t k = 0; k < (size_t)kCanary * words; k++) h[k] = h[total - 1 - k] = kCanaryWord;
    void *d = nullptr;
    ok(cudaMalloc(&d, total * 4));
    if (!d) return nullptr;
    owned.push_back(d);
    ok(cudaMemcpy(d, h.data(), total * 4, cudaMemcpyHostToDevice));
    return reinterpret_cast<T *>(d) + kCanary;
}

template <typename T>
long long read_guarded(Status &ok, const T *d, long long n, T *out)
{
    const size_t words = sizeof(T) / 4, total = (size_t)(n + 2 * kCanary) * words;
    std::vector<uint32_t> h(total, 0);
    ok(cudaMemcpy(h.data(), reinterpret_cast<const uint32_t *>(d - kCanary), total * 4, cudaMemcpyDeviceToHost));
    long long bad = 0;
    for (size_t k = 0; k < (size_t)kCanary * words; k++) bad += (h[k] != kCanaryWord) + (h[total - 1 - k] != kCanaryWord);
    if (n > 0 && out) std::memcpy(out, h.data() + (size_t)kCanary * words, (size_t)n * sizeof(T));
    return bad;
}

template <typename T>
T *dev_copy(Status &ok, std::vector<void *> &owned, const T *h, size_t count)
{
    void *d = nullptr;
    ok(cudaMalloc(&d, std::max<size_t>(count, 1) * sizeof(T)));
    if (!d) return nullptr;
    owned.push_back(d);
    if (count) ok(cudaMemcpy(d, h, count * sizeof(T), cudaMemcpyHostToDevice));
    return reinterpret_cast<T *>(d);
}

void free_all(std::vector<void *> &owned)
{
    for (void *p : owned) cudaFree(p);
    owned.clear();
}

// statistics scratch of one job: ST_COUNT doubles, partials, a zeroed counter
void stats_scratch(Status &ok, std::vector<void *> &owned, tdoa::SigJob &j, long long max_n)
{
    const size_t parts = 3 * (size_t)std::max(tdoa::stream_grid_x(max_n), tdoa::boxcar_grid_x(max_n));
    std::vector<double> zeros(tdoa::ST_COUNT, 0.0);
    j.stats = dev_copy(ok, owned, zeros.data(), zeros.size());
    std::vector<double> pz(parts, 0.0);
    j.partials = dev_copy(ok, owned, pz.data(), pz.size());
    unsigned z = 0;
    j.counter = dev_copy(ok, owned, &z, 1);
}

}  // namespace

// One launch of k_channel (demod = 0) or k_channel_demod (demod = 1) over n_jobs jobs.  Job k: the capture h_raw[k]
// (raw_bytes[k] bytes), the view of n[k] samples given by (run0_start, run0_len, run1_start)[k].  demod = 0: planes
// out_re[k] / out_im[k]; demod = 1: the discriminator plane out_re[k] and the statistics block stats[k * ST_COUNT].
// taps_im may be NULL (the real-tap kernel).  canary_bad: canary words that changed, over all outputs.
extern "C" __attribute__((visibility("default"))) int probe_channel(int n_jobs, const long long *n, const uint8_t *const *h_raw,
                                                                    const long long *raw_bytes, const long long *runs,
                                                                    const float *taps_re, const float *taps_im, int n_taps,
                                                                    int demod, float *const *out_re, float *const *out_im,
                                                                    double *stats, long long *canary_bad)
{
    Status ok;
    std::vector<void *> owned;
    std::vector<tdoa::SigJob> jobs((size_t)n_jobs);
    long long max_n = 0;
    for (int k = 0; k < n_jobs; k++) max_n = std::max(max_n, n[k]);
    std::vector<float *> d_re(n_jobs, nullptr), d_im(n_jobs, nullptr);
    for (int k = 0; k < n_jobs; k++) {
        tdoa::SigJob &j = jobs[k];
        j = tdoa::SigJob{};
        j.src.raw = dev_copy(ok, owned, h_raw[k], (size_t)raw_bytes[k]);
        j.src.run0_start = runs[3 * k]; j.src.run0_len = runs[3 * k + 1]; j.src.run1_start = runs[3 * k + 2];
        j.n = n[k];
        d_re[k] = alloc_guarded<float>(ok, owned, n[k]);
        if (!demod) d_im[k] = alloc_guarded<float>(ok, owned, n[k]);
        j.p_re = d_re[k];
        j.p_im = d_im[k];
        stats_scratch(ok, owned, j, max_n);
    }
    if (ok.err) { free_all(owned); return (int)ok.err; }
    tdoa::ChannelTaps t{};
    for (int k = 0; k < n_taps; k++) { t.re[k] = taps_re[k]; t.im[k] = taps_im ? taps_im[k] : 0.f; }
    t.n = n_taps;
    tdoa::SigJob *d_jobs = dev_copy(ok, owned, jobs.data(), jobs.size());
    if (demod) tdoa::launch_channel_demod(d_jobs, n_jobs, max_n, t, taps_im != nullptr, 0);
    else tdoa::launch_channel(d_jobs, n_jobs, max_n, t, taps_im != nullptr, 0);
    ok(cudaGetLastError());
    ok(cudaDeviceSynchronize());
    long long bad = 0;
    for (int k = 0; k < n_jobs; k++) {
        bad += read_guarded(ok, d_re[k], n[k], out_re[k]);
        if (!demod) bad += read_guarded(ok, d_im[k], n[k], out_im[k]);
        else ok(cudaMemcpy(stats + (size_t)k * tdoa::ST_COUNT, jobs[k].stats, tdoa::ST_COUNT * sizeof(double), cudaMemcpyDeviceToHost));
    }
    *canary_bad = bad;
    free_all(owned);
    return (int)ok.err;
}

// k_power, then k_demod, on the planes (re, im) of n >= 2 samples (SigSrc raw == nullptr): the discriminator plane
// and the statistics block (ST_POWER0 from k_power, the sums from k_demod)
extern "C" __attribute__((visibility("default"))) int probe_demod_planes(long long n, const float *re, const float *im, float *out,
                                                                         double *stats)
{
    Status ok;
    std::vector<void *> owned;
    tdoa::SigJob j{};
    j.src.re = dev_copy(ok, owned, re, (size_t)n);
    j.src.im = dev_copy(ok, owned, im, (size_t)n);
    j.n = n;
    float *d_out = alloc_guarded<float>(ok, owned, n);
    j.p_re = d_out;
    stats_scratch(ok, owned, j, n);
    if (ok.err) { free_all(owned); return (int)ok.err; }
    tdoa::SigJob *d_jobs = dev_copy(ok, owned, &j, 1);
    tdoa::launch_power(d_jobs, 1, n, tdoa::stream_grid_x(n), 0);
    tdoa::launch_demod(d_jobs, 1, n, tdoa::stream_grid_x(n), 0);
    ok(cudaGetLastError());
    ok(cudaDeviceSynchronize());
    read_guarded(ok, d_out, n, out);
    ok(cudaMemcpy(stats, j.stats, tdoa::ST_COUNT * sizeof(double), cudaMemcpyDeviceToHost));
    free_all(owned);
    return (int)ok.err;
}
