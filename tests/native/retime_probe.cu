// retime_probe.cu -- the two kernels of retime.cu driven directly from host arrays, for
// tests/test_gpu_retime_kernels.py (built there with retime.cu's own flags and loaded with ctypes).
//
// Every output array sits between two runs of kCanary canary words, and the output itself is filled with
// kUnwritten before the launch, so a stray write and a missing write both show on the host.  Return value: the
// first CUDA error of the call (0 = none).  Plain cudaMalloc / cudaMemcpy throughout: a pointer's alignment is
// exactly what the caller asked for.
#include "retime.cu"

#include <cstring>
#include <vector>

namespace {

constexpr int kCanary = 64;                  // elements before and after every output array
constexpr uint32_t kCanaryWord = 0xdeadbeefu;
constexpr uint32_t kUnwritten = 0xffffffffu; // a NaN pattern no gather of a finite plane produces

struct Status {
    cudaError_t err = cudaSuccess;
    void operator()(cudaError_t e) { if (err == cudaSuccess && e != cudaSuccess) err = e; }
};

// a device array of n elements of `words` 32-bit words each, canaries on both sides; returns the element pointer
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

// copies the n elements back to `out` and counts the canary words that changed
template <typename T>
long long read_guarded(Status &ok, const T *d, long long n, T *out)
{
    const size_t words = sizeof(T) / 4, total = (size_t)(n + 2 * kCanary) * words;
    std::vector<uint32_t> h(total, 0);
    ok(cudaMemcpy(h.data(), reinterpret_cast<const uint32_t *>(d - kCanary), total * 4, cudaMemcpyDeviceToHost));
    long long bad = 0;
    for (size_t k = 0; k < (size_t)kCanary * words; k++) bad += (h[k] != kCanaryWord) + (h[total - 1 - k] != kCanaryWord);
    if (n > 0) std::memcpy(out, h.data() + (size_t)kCanary * words, (size_t)n * sizeof(T));
    return bad;
}

void free_all(std::vector<void *> &owned)
{
    for (void *p : owned) cudaFree(p);
    owned.clear();
}

}  // namespace

// One launch of k_retime over n_jobs jobs.  Job k: plane h_x[k] of n[k] samples, placed x_off[k] floats past a
// cudaMalloc'd (256-byte aligned) base, re-timed by rates[station[k]] into h_y[k].  canary_bad: canary words that
// changed, over all jobs.
extern "C" __attribute__((visibility("default"))) int probe_retime(int n_jobs, const long long *n, const int *station,
                                                                   const int *x_off, const float *const *h_x,
                                                                   float *const *h_y, const double *rates, int n_rates,
                                                                   long long *canary_bad)
{
    Status ok;
    std::vector<void *> owned;
    std::vector<tdoa::RetimeJob> jobs((size_t)n_jobs);
    long long max_n = 0;
    for (int k = 0; k < n_jobs; k++) {
        void *src = nullptr;
        ok(cudaMalloc(&src, (size_t)(n[k] + x_off[k] + 1) * sizeof(float)));
        if (!src) { free_all(owned); return (int)ok.err; }
        owned.push_back(src);
        float *x = reinterpret_cast<float *>(src) + x_off[k];
        if (n[k] > 0) ok(cudaMemcpy(x, h_x[k], (size_t)n[k] * sizeof(float), cudaMemcpyHostToDevice));
        float *y = alloc_guarded<float>(ok, owned, n[k]);
        jobs[k] = tdoa::RetimeJob{x, y, n[k], station[k]};
        if (n[k] > max_n) max_n = n[k];
    }
    void *d_jobs = nullptr, *d_rates = nullptr;
    ok(cudaMalloc(&d_jobs, jobs.size() * sizeof(tdoa::RetimeJob) + 1));
    ok(cudaMalloc(&d_rates, (size_t)n_rates * sizeof(double) + 1));
    if (d_jobs) owned.push_back(d_jobs);
    if (d_rates) owned.push_back(d_rates);
    if (ok.err == cudaSuccess) {
        ok(cudaMemcpy(d_jobs, jobs.data(), jobs.size() * sizeof(tdoa::RetimeJob), cudaMemcpyHostToDevice));
        ok(cudaMemcpy(d_rates, rates, (size_t)n_rates * sizeof(double), cudaMemcpyHostToDevice));
        tdoa::launch_retime(reinterpret_cast<const tdoa::RetimeJob *>(d_jobs), n_jobs, max_n,
                            reinterpret_cast<const double *>(d_rates), 0);
        ok(cudaGetLastError());
        ok(cudaDeviceSynchronize());
        long long bad = 0;
        for (int k = 0; k < n_jobs && ok.err == cudaSuccess; k++) bad += read_guarded<float>(ok, jobs[k].y, n[k], h_y[k]);
        *canary_bad = bad;
    }
    free_all(owned);
    return (int)ok.err;
}

// One launch of k_station_rates: fit[P][kWindowFitDoubles] (P = S (S - 1) / 2 pairs) in, rate[S] and clock[S] out.
extern "C" __attribute__((visibility("default"))) int probe_station_rates(const double *fit, int S, double *rate,
                                                                          double *clock, long long *canary_bad)
{
    Status ok;
    std::vector<void *> owned;
    const size_t fit_doubles = (size_t)tdoa::kWindowFitDoubles * S * (S - 1) / 2;
    void *d_fit = nullptr;
    ok(cudaMalloc(&d_fit, fit_doubles * sizeof(double) + 1));
    if (d_fit) owned.push_back(d_fit);
    double *d_rate = alloc_guarded<double>(ok, owned, S), *d_clock = alloc_guarded<double>(ok, owned, S);
    if (ok.err == cudaSuccess) {
        ok(cudaMemcpy(d_fit, fit, fit_doubles * sizeof(double), cudaMemcpyHostToDevice));
        tdoa::launch_station_rates(reinterpret_cast<const double *>(d_fit), S, d_rate, d_clock, 0);
        ok(cudaGetLastError());
        ok(cudaDeviceSynchronize());
        long long bad = 0;
        if (ok.err == cudaSuccess) bad += read_guarded<double>(ok, d_rate, S, rate);
        if (ok.err == cudaSuccess) bad += read_guarded<double>(ok, d_clock, S, clock);
        *canary_bad = bad;
    }
    free_all(owned);
    return (int)ok.err;
}
