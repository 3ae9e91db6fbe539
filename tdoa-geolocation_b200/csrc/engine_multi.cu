// engine_multi.cu -- more than one GPU behind the C ABI (SURVEY.md 8e; processor.go:816-850 is the
// loop being sharded).
//
// The units of the path are independent: a (window, pair) correlation needs only its two
// stations' window.  Windows are dealt round-robin over the ranks of a communicator -- rank r takes
// the windows w with (cursor + w) % world == r, preprocesses each of its station-windows once and
// runs all pairs locally -- so there is no collective on the data path.  The one exchange is the
// peak records: every rank's k_peak_candidates / k_peak writes its records straight into its slot
// of the gather buffer, one ncclAllGather (in place, NVLink / NVSwitch) completes the table on every
// rank, and a permutation kernel puts it in window order.  No host round trip.
//
// Two ways to get a communicator, same code path afterwards:
//   - tdoa_config.n_devices = N: ONE process drives N GPUs (what a Go caller binding the header
//     gets).  The engine created is rank 0; it owns N - 1 peer engines on the next devices, loads
//     are forwarded to them, and a sharded tdoa_xcorr runs one host thread per device.
//   - tdoa_comm_unique_id + tdoa_comm_init: one process per GPU (torchrun, MPI): rank 0 makes the
//     id, the launcher distributes it, every rank joins.  Calls are then collective: every rank
//     makes the same tdoa_xcorr call and every rank gets the whole table.
// The cursor advances by the number of windows of each sharded call, so that back-to-back calls
// (66 REF windows, then 33 TGT windows, over 8 ranks) do not pile their remainders on rank 0.
//
// NCCL is bound at run time (dlopen of libnccl.so.2: the copy already in the process when the
// caller is PyTorch, the system's otherwise), so a single-GPU user needs no NCCL at all.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "engine_internal.h"

using namespace tdoa;

namespace tdoa {

// one process, several devices: the host threads meet here before the gather, so that a device which
// failed on the way (and will never launch its part of the collective) does not leave the others waiting
struct Rendezvous {
    std::mutex m;
    std::condition_variable cv;
    int n = 0, arrived = 0, failed = 0;
    bool arrive(bool ok)
    {
        std::unique_lock<std::mutex> lk(m);
        arrived++;
        if (!ok) failed++;
        if (arrived == n) cv.notify_all();
        else cv.wait(lk, [&] { return arrived == n; });
        return failed == 0;
    }
};

struct MultiState {
    Rendezvous *rdv = nullptr;            // set for the duration of a multi-device call
    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
    int cursor = 0;                       // rank that owns window 0 of the next sharded call
    std::vector<tdoa_engine *> peers;     // n_devices engines: [0] = the engine itself, the rest owned by it
    bool owned_by_parent = false;
};

namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
    std::string why;
};

NcclApi &nccl()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            api.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) { api.why = std::string("libnccl.so.2 not found: ") + (dlerror() ? dlerror() : ""); return; }
        auto sym = [&](const char *n) { void *p = dlsym(api.handle, n); if (!p) api.why = std::string("missing NCCL symbol ") + n; return p; };
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommInitAll && api.CommDestroy && api.AllGather && api.GetErrorString;
    });
    return api;
}

// table[w * P + p] <- gathered[(rank(w) * n_max + w / world) * P + p], rank(w) = (cursor + w) % world
__global__ void k_window_order(const PeakRec *__restrict__ gathered, PeakRec *__restrict__ table, int n_windows, int P, int world,
                               int cursor, int n_max)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_windows * P) return;
    const int w = i / P, p = i - w * P;
    const int r = (cursor + w) % world, k = w / world;
    table[i] = gathered[((size_t)r * n_max + k) * P + p];
}

// the pair loops of this rank's windows of every part (a part = one signal kind's windows), the gathers, the
// tables in window order (device), and -- out != nullptr -- their copies to the host.  Collective over the
// communicator.  All parts are correlated BEFORE the first gather, so the ranks meet once per call: with one
// gather per kind a rank that got the short end of the REF windows would wait for the others before it may
// start its TGT windows (66 + 33 windows over 8 ranks: 9 + 5 window times instead of 13).
int sharded_rank(tdoa_engine *e, const std::vector<ShardPart> &parts)
{
    MultiState &M = *e->multi;
    NcclApi &N = nccl();
    const int S = e->cfg.n_stations, P = S * (S - 1) / 2;
    const int world = M.world;
    struct Work { PeakRec *d_gather = nullptr, *d_table = nullptr, *mine = nullptr; int n_max = 0, cursor = 0; };
    std::vector<Work> work(parts.size());
    int rc = TDOA_OK;
    auto before_the_gather = [&]() -> int {
        stats_reset(e);
        cudaEventRecord(e->ev[0], e->stream);
        int cursor = M.cursor;
        for (size_t k = 0; k < parts.size(); k++) {
            const ShardPart &Q = parts[k];
            Work &W = work[k];
            W.n_max = (Q.n_windows + world - 1) / world;
            W.cursor = cursor;
            int32_t first = 0, count = 0;
            tdoa_shard_windows(Q.n_windows, M.rank, world, cursor, &first, &count);
            cursor = (cursor + Q.n_windows) % world;
            if ((rc = alloc_t(e, &W.d_gather, (size_t)world * W.n_max * P))) return rc;
            if (Q.out_is_device) W.d_table = reinterpret_cast<PeakRec *>(Q.out);
            else if ((rc = alloc_t(e, &W.d_table, (size_t)Q.n_windows * P))) return rc;
            W.mine = W.d_gather + (size_t)M.rank * W.n_max * P;
            CU(cudaMemsetAsync(W.mine, 0, (size_t)W.n_max * P * sizeof(PeakRec), e->stream));
            if (count > 0 && (rc = xcorr_core(e, Q.kind, Q.win_start + (i64)first * Q.hop, Q.len, count, Q.hop * world, W.mine, nullptr,
                                              Q.rates)))
                return rc;
        }
        return TDOA_OK;
    };
    rc = before_the_gather();
    if (M.rdv && !M.rdv->arrive(rc == TDOA_OK))
        return rc ? rc : fail(e, TDOA_E_STATE, "another device of this engine failed before the gather");
    if (rc) return rc;
    for (size_t k = 0; k < parts.size(); k++) {
        const ShardPart &Q = parts[k];
        Work &W = work[k];
        const ncclResult_t nr = N.AllGather(W.mine, W.d_gather, (size_t)W.n_max * P * sizeof(PeakRec), ncclUint8, M.comm, e->stream);
        if (nr != ncclSuccess) return fail(e, TDOA_E_CUDA, "ncclAllGather failed: %s", N.GetErrorString(nr));
        k_window_order<<<(Q.n_windows * P + 255) / 256, 256, 0, e->stream>>>(W.d_gather, W.d_table, Q.n_windows, P, world, W.cursor, W.n_max);
        count_launch(e);
    }
    cudaEventRecord(e->ev[4], e->stream);
    for (size_t k = 0; k < parts.size(); k++)
        if (parts[k].out && !parts[k].out_is_device)
            CU(cudaMemcpyAsync(parts[k].out, work[k].d_table, (size_t)parts[k].n_windows * P * sizeof(tdoa_peak), cudaMemcpyDeviceToHost,
                               e->stream));
    for (const ShardPart &Q : parts) M.cursor = (M.cursor + Q.n_windows) % world;
    rc = end_call(e, true);
    if (rc) return rc;
    e->st.launches_last = e->st.launches_total - e->launches_at_call;
    retire_lazy(e);
    spans_collect(e);
    float t = 0.f;
    cudaEventElapsedTime(&t, e->ev[0], e->ev[4]);
    e->st.ms_exact = e->ms_corr - e->st.ms_fft;
    e->st.ms_total = t;
    return TDOA_OK;
}

}  // namespace

// a communicator of one rank takes the same path (gather buffer, ncclAllGather, window order): that
// is how a one-GPU box exercises it
bool multi_wants(const tdoa_engine *e, int32_t n_windows) { return e->multi && e->multi->comm && n_windows >= 2; }

int xcorr_sharded(tdoa_engine *e, const std::vector<ShardPart> &parts)
{
    MultiState &M = *e->multi;
    if (M.peers.size() <= 1) return sharded_rank(e, parts);
    // one process, several devices: one host thread per peer (each queues on its own device and
    // joins the gather); this thread is rank 0
    const int n = (int)M.peers.size();
    // station rates (tdoa_process_windows_retimed) live on this device: each peer gets the same S doubles in its own
    std::vector<std::vector<double>> h_rates(parts.size());
    bool any_rates = false;
    for (size_t k = 0; k < parts.size(); k++) {
        if (!parts[k].rates) continue;
        h_rates[k].resize(e->cfg.n_stations);
        CU(cudaMemcpyAsync(h_rates[k].data(), parts[k].rates, h_rates[k].size() * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        any_rates = true;
    }
    if (any_rates) CU(cudaStreamSynchronize(e->stream));
    std::vector<int> rcs(n, TDOA_OK);
    std::vector<std::thread> threads;
    Rendezvous rdv;
    rdv.n = n;
    for (int r = 0; r < n; r++) M.peers[r]->multi->rdv = &rdv;
    for (int r = 1; r < n; r++)
        threads.emplace_back([&, r] {
            tdoa_engine *p = M.peers[r];
            int rc = begin_call(p);
            std::vector<ShardPart> mine = parts;   // the peer's own window lengths; its tables stay on its device
            for (size_t k = 0; k < mine.size(); k++) {
                ShardPart &Q = mine[k];
                const i64 wl = Q.len.empty() ? 0 : Q.len[0];
                Q.out = nullptr; Q.out_is_device = false;
                if (!rc) rc = window_lengths(p, Q.kind, Q.win_start, wl, Q.n_windows, Q.hop, Q.len);
                if (!rc && Q.rates) rc = upload(p, h_rates[k], &Q.rates);
            }
            if (rc) rdv.arrive(false);
            else rc = sharded_rank(p, mine);
            rcs[r] = rc;
        });
    rcs[0] = sharded_rank(e, parts);
    for (auto &t : threads) t.join();
    for (int r = 0; r < n; r++) M.peers[r]->multi->rdv = nullptr;
    cudaSetDevice(e->device);
    for (int r = 1; r < n; r++)
        if (rcs[r]) return fail(e, rcs[r], "device %d: %s", M.peers[r]->device, M.peers[r]->error.c_str());
    return rcs[0];
}

int xcorr_sharded(tdoa_engine *e, int32_t kind, int64_t win_start, const std::vector<i64> &len, int32_t n_windows, int64_t hop,
                  tdoa_peak *out, bool out_is_device)
{
    std::vector<ShardPart> parts(1);
    parts[0].kind = kind; parts[0].win_start = win_start; parts[0].len = len; parts[0].n_windows = n_windows; parts[0].hop = hop;
    parts[0].out = out; parts[0].out_is_device = out_is_device;
    return xcorr_sharded(e, parts);
}

void multi_destroy(tdoa_engine *e)
{
    if (!e->multi) return;
    MultiState *M = e->multi;
    for (size_t r = 1; r < M->peers.size(); r++) tdoa_destroy(M->peers[r]);
    if (M->comm && nccl().ok) { cudaSetDevice(e->device); nccl().CommDestroy(M->comm); }
    delete M;
    e->multi = nullptr;
}

// tdoa_create's second half for n_devices > 1: the peers and the communicator
int multi_create_peers(tdoa_engine *e, const tdoa_config *cfg)
{
    NcclApi &N = nccl();
    if (!N.ok) return fail(e, TDOA_E_NODEVICE, "n_devices = %d needs NCCL: %s", cfg->n_devices, N.why.c_str());
    const int n = cfg->n_devices;
    int n_dev = 0;
    CU(cudaGetDeviceCount(&n_dev));
    if (cfg->device + n > n_dev)
        return fail(e, TDOA_E_NODEVICE, "n_devices = %d from device %d, but the process sees %d device(s)", n, cfg->device, n_dev);
    MultiState *M = new MultiState();
    M->rank = 0; M->world = n;
    M->peers.push_back(e);
    e->multi = M;
    for (int r = 1; r < n; r++) {
        tdoa_config c = *cfg;
        c.device = cfg->device + r;
        c.n_devices = 1;
        tdoa_engine *p = nullptr;
        const int rc = tdoa_create(&p, &c);
        if (rc) return fail(e, rc, "peer engine on device %d: %s", c.device, tdoa_last_error(nullptr));
        p->multi = new MultiState();
        p->multi->rank = r; p->multi->world = n; p->multi->owned_by_parent = true;
        M->peers.push_back(p);
    }
    std::vector<ncclComm_t> comms(n);
    std::vector<int> devs(n);
    for (int r = 0; r < n; r++) devs[r] = cfg->device + r;
    const ncclResult_t nr = N.CommInitAll(comms.data(), n, devs.data());
    if (nr != ncclSuccess) return fail(e, TDOA_E_CUDA, "ncclCommInitAll failed: %s", N.GetErrorString(nr));
    for (int r = 0; r < n; r++) M->peers[r]->multi->comm = comms[r];
    CU(cudaSetDevice(e->device));
    return TDOA_OK;
}

// forward a load to the peers of a multi-device engine (every device holds every capture)
int multi_forward_load(tdoa_engine *e, int which, int32_t station, const void *p, size_t nbytes, int64_t *n_samples)
{
    if (!e->multi || e->multi->peers.size() <= 1) return TDOA_OK;
    for (size_t r = 1; r < e->multi->peers.size(); r++) {
        tdoa_engine *q = e->multi->peers[r];
        int rc = TDOA_OK;
        switch (which) {
            case 0: rc = tdoa_load_u8(q, station, static_cast<const uint8_t *>(p), nbytes); break;
            case 1: rc = tdoa_load_u8_pinned(q, station, static_cast<const uint8_t *>(p), nbytes); break;
            case 2: rc = tdoa_load_file(q, station, static_cast<const char *>(p), n_samples); break;
        }
        if (rc) { cudaSetDevice(e->device); return fail(e, rc, "device %d: %s", q->device, q->error.c_str()); }
    }
    CU(cudaSetDevice(e->device));
    return TDOA_OK;
}

}  // namespace tdoa

extern "C" {

int tdoa_shard_windows(int32_t n_windows, int32_t rank, int32_t world, int32_t cursor, int32_t *first, int32_t *count)
{
    if (n_windows < 0 || world < 1 || rank < 0 || rank >= world || cursor < 0 || !first || !count) return TDOA_E_INVALID;
    const int f = ((rank - cursor % world) % world + world) % world;   // window w belongs to rank (cursor + w) % world
    *first = f;
    *count = f < n_windows ? (n_windows - f + world - 1) / world : 0;
    return TDOA_OK;
}

int tdoa_comm_unique_id(uint8_t id[128])
{
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    if (!id) return TDOA_E_INVALID;
    NcclApi &N = nccl();
    if (!N.ok) return fail(nullptr, TDOA_E_NODEVICE, "tdoa_comm_unique_id: %s", N.why.c_str());
    ncclUniqueId u;
    const ncclResult_t nr = N.GetUniqueId(&u);
    if (nr != ncclSuccess) return fail(nullptr, TDOA_E_CUDA, "ncclGetUniqueId failed: %s", N.GetErrorString(nr));
    std::memcpy(id, &u, sizeof(u));
    return TDOA_OK;
}

int tdoa_comm_init(tdoa_engine *e, const uint8_t id[128], int32_t rank, int32_t world)
{
    if (!e) return TDOA_E_INVALID;
    int rc = begin_call(e);
    if (rc) return rc;
    if (!id || world < 1 || rank < 0 || rank >= world) return fail(e, TDOA_E_INVALID, "tdoa_comm_init: bad rank %d of %d", rank, world);
    if (e->multi) return fail(e, TDOA_E_STATE, "tdoa_comm_init: the engine already has a communicator");
    NcclApi &N = nccl();
    if (!N.ok) return fail(e, TDOA_E_NODEVICE, "tdoa_comm_init: %s", N.why.c_str());
    ncclUniqueId u;
    std::memcpy(&u, id, sizeof(u));
    ncclComm_t comm = nullptr;
    const ncclResult_t nr = N.CommInitRank(&comm, world, u, rank);
    if (nr != ncclSuccess) return fail(e, TDOA_E_CUDA, "ncclCommInitRank failed: %s", N.GetErrorString(nr));
    e->multi = new MultiState();
    e->multi->rank = rank; e->multi->world = world; e->multi->comm = comm;
    return TDOA_OK;
}

int tdoa_comm_rank(tdoa_engine *e, int32_t *rank, int32_t *world)
{
    if (!e) return TDOA_E_INVALID;
    if (rank) *rank = e->multi ? e->multi->rank : 0;
    if (world) *world = e->multi ? e->multi->world : 1;
    return TDOA_OK;
}

}  // extern "C"
