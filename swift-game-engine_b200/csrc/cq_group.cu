// cq_group.cu — the GPUs of one box behind the C ABI (include/cq.h: cq_group_*, cq_world_create_multi, cq_multi_*).
//
// The path shards by independent units (characters, sweeps, rays — SURVEY.md §8e): the mesh and its trees are
// replicated on every GPU, every GPU processes one contiguous range of the units (cq_shard_range), nothing is exchanged
// inside the algorithm.  The ONE collective a caller may want is the gather of the fixed-size result records; it goes
// through NCCL over NVLink / NVSwitch: ncclAllGather for equal shards, a group of ncclBroadcast calls for ragged ones
// (every rank's shard lands at its offset of the result without padding).
//
// Two ways to own the GPUs, both without Python:
//   * one process per GPU (how bench.py runs under torchrun): rank 0 makes a 128-byte id (cq_group_unique_id), the host
//     ships it to the other ranks by any means it has, every rank calls cq_group_create_rank on its own device;
//   * one process driving all GPUs (a Swift or C++ host such as examples/cq_multi_gpu.cpp): cq_group_create_local, then
//     cq_world_create_multi builds one replica per device and the cq_multi_* calls shard a host batch over them, one
//     worker thread per device, each running the single-GPU copy / compute pipeline of cq_api.cu on its shard.
//
// NCCL is loaded at run time (dlopen of libnccl.so.2, the soname both the system package and PyTorch's bundled copy
// carry), so libcq.so itself has no link-time dependency on it: single-GPU users never need it, and inside a PyTorch
// process the library shares the copy that is already loaded.
#include <dlfcn.h>

#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>

#include "cq_internal.h"

namespace cq {

// ---------------------------------------------------------------- NCCL, resolved at run time
typedef struct ncclComm *ncclComm_t;
typedef struct {
    char internal[128];
} ncclUniqueId;
enum { ncclSuccess = 0 };
enum { ncclChar = 0 }; // ncclInt8

struct Nccl {
    void *handle = nullptr;
    int (*GetVersion)(int *) = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
};

static Nccl &nccl() {
    static Nccl N;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            N.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (N.handle) break;
        }
        if (!N.handle) return;
        auto sym = [&](const char *s) { return dlsym(N.handle, s); };
        N.GetVersion = (int (*)(int *))sym("ncclGetVersion");
        N.GetUniqueId = (int (*)(ncclUniqueId *))sym("ncclGetUniqueId");
        N.CommInitRank = (int (*)(ncclComm_t *, int, ncclUniqueId, int))sym("ncclCommInitRank");
        N.CommInitAll = (int (*)(ncclComm_t *, int, const int *))sym("ncclCommInitAll");
        N.CommDestroy = (int (*)(ncclComm_t))sym("ncclCommDestroy");
        N.AllGather = (int (*)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t))sym("ncclAllGather");
        N.Broadcast = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))sym("ncclBroadcast");
        N.GroupStart = (int (*)())sym("ncclGroupStart");
        N.GroupEnd = (int (*)())sym("ncclGroupEnd");
        N.GetErrorString = (const char *(*)(int))sym("ncclGetErrorString");
        N.ok = N.GetUniqueId && N.CommInitRank && N.CommInitAll && N.CommDestroy && N.AllGather && N.Broadcast && N.GroupStart &&
               N.GroupEnd;
    });
    return N;
}

static int need_nccl() {
    if (nccl().ok) return CQ_OK;
    const char *why = nccl().handle ? "symbols missing" : "libnccl.so.2 could not be loaded";
    set_error("NCCL is not available: %s", why);
    return CQ_ERR_NCCL;
}

static int check_nccl(int r, const char *what) {
    if (r == ncclSuccess) return CQ_OK;
    set_error("NCCL error %d (%s) at %s", r, nccl().GetErrorString ? nccl().GetErrorString(r) : "?", what);
    return CQ_ERR_NCCL;
}
#define CQ_NCCL(x)                          \
    do {                                    \
        int _r = check_nccl((x), #x);       \
        if (_r != CQ_OK) return _r;         \
    } while (0)

// ---------------------------------------------------------------- one worker thread per device (local groups)
class Worker {
  public:
    Worker() : th_([this] { loop(); }) {}
    ~Worker() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            quit_ = true;
        }
        cv_.notify_all();
        th_.join();
    }
    void submit(std::function<int()> job) {
        std::lock_guard<std::mutex> lk(mu_);
        job_ = std::move(job);
        busy_ = true;
        cv_.notify_all();
    }
    int wait(std::string &err) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [this] { return !busy_; });
        err = err_;
        return rc_;
    }

  private:
    void loop() {
        std::unique_lock<std::mutex> lk(mu_);
        for (;;) {
            cv_.wait(lk, [this] { return quit_ || busy_; });
            if (quit_) return;
            std::function<int()> job = std::move(job_);
            lk.unlock();
            const int rc = job();
            const std::string err = rc == CQ_OK ? std::string() : std::string(cq_last_error()); // the error text is per thread
            lk.lock();
            rc_ = rc, err_ = err, busy_ = false;
            cv_.notify_all();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_;
    std::function<int()> job_;
    bool busy_ = false, quit_ = false;
    int rc_ = CQ_OK;
    std::string err_;
    std::thread th_;
};

} // namespace cq

using namespace cq;

struct cq_group {
    int nRanks = 0;
    int rank = -1;                  // process-per-GPU groups; -1 = local group (this process drives every device)
    std::vector<int> devices;       // local groups: the devices; rank groups: the one device of this rank
    std::vector<ncclComm_t> comms;  // one per entry of `devices`
    std::vector<Worker *> workers;  // local groups only
    std::vector<cudaStream_t> streams; // local groups: a stream per device for the collective calls
};

// One replica's buffers of cq_multi_move_and_slide_batch_ex with CQ_MAS_AGENTS, grown on demand.
struct MultiAgentBuffers {
    cq_character_state *states = nullptr; // the replica's shard
    cq_agent_snapshot *snap = nullptr;    // the whole crowd's snapshot
    cq_platform *platforms = nullptr;     // MAS_MAX_PLATFORMS records
    size_t capStates = 0, capSnap = 0;
};

struct cq_multi_world {
    cq_group *group = nullptr;
    std::vector<cq_world *> replicas;
    std::vector<MultiAgentBuffers> agentBufs; // one per replica
};

// every worker runs fn(i); the first failure (lowest device index) is reported in the caller's thread
static int on_every_device(cq_group *g, const std::function<int(int)> &fn) {
    const int n = (int)g->devices.size();
    for (int i = 0; i < n; i++) {
        const int dev = g->devices[i];
        g->workers[i]->submit([=] {
            if (check_cuda(cudaSetDevice(dev), "cudaSetDevice") != CQ_OK) return CQ_ERR_CUDA;
            return fn(i);
        });
    }
    int rc = CQ_OK, where = 0;
    std::string err, first;
    for (int i = 0; i < n; i++) {
        const int r = g->workers[i]->wait(err);
        if (r != CQ_OK && rc == CQ_OK) rc = r, first = err, where = g->devices[i];
    }
    if (rc != CQ_OK) set_error("device %d: %s", where, first.c_str());
    return rc;
}

extern "C" void cq_shard_range(int64_t n_units, int32_t n_ranks, int32_t rank, int64_t *lo, int64_t *hi);

template <class Fn> static int sharded(cq_multi_world *mw, int64_t n, Fn fn) { // fn(replica, lo, count)
    if (!mw || n < 0) return CQ_ERR_INVALID;
    const int ranks = (int)mw->replicas.size();
    return on_every_device(mw->group, [&](int i) {
        int64_t lo, hi;
        cq_shard_range(n, ranks, i, &lo, &hi);
        return hi > lo ? fn(mw->replicas[i], lo, (int32_t)(hi - lo)) : CQ_OK;
    });
}

// a device buffer of at least `count` records of T on the current device; a larger one frees the old (the replica's
// stream is idle between calls: every call ends with its synchronisation)
template <class T> static int grow(T *&p, size_t &cap, size_t count, const char *what) {
    if (count <= cap) return CQ_OK;
    cudaFree(p);
    p = nullptr, cap = 0;
    CQ_TRY(check_cuda(cudaMalloc((void **)&p, count * sizeof(T)), what));
    cap = count;
    return CQ_OK;
}

extern "C" {

void cq_shard_range(int64_t n_units, int32_t n_ranks, int32_t rank, int64_t *lo, int64_t *hi) {
    if (n_ranks <= 0 || rank < 0 || rank >= n_ranks || n_units < 0) {
        if (lo) *lo = 0;
        if (hi) *hi = 0;
        return;
    }
    if (lo) *lo = (int64_t)rank * n_units / n_ranks;
    if (hi) *hi = ((int64_t)rank + 1) * n_units / n_ranks;
}

int cq_group_unique_id(uint8_t id[CQ_GROUP_ID_BYTES]) {
    if (!id) return CQ_ERR_INVALID;
    CQ_TRY(need_nccl());
    ncclUniqueId u;
    CQ_NCCL(nccl().GetUniqueId(&u));
    static_assert(sizeof(u) == CQ_GROUP_ID_BYTES, "ncclUniqueId is 128 bytes");
    memcpy(id, &u, sizeof(u));
    return CQ_OK;
}

int cq_group_create_rank(int32_t n_ranks, int32_t rank, const uint8_t id[CQ_GROUP_ID_BYTES], cq_group **out) {
    if (!out || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) {
        set_error("cq_group_create_rank: invalid arguments");
        return CQ_ERR_INVALID;
    }
    *out = nullptr;
    CQ_TRY(need_nccl());
    int dev = 0;
    CQ_CUDA(cudaGetDevice(&dev));
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    ncclComm_t comm = nullptr;
    CQ_NCCL(nccl().CommInitRank(&comm, n_ranks, u, rank));
    cq_group *g = new cq_group();
    g->nRanks = n_ranks, g->rank = rank;
    g->devices = {dev};
    g->comms = {comm};
    *out = g;
    return CQ_OK;
}

int cq_group_create_local(int32_t n_gpus, const int32_t *devices, cq_group **out) {
    if (!out || n_gpus < 1) {
        set_error("cq_group_create_local: invalid arguments");
        return CQ_ERR_INVALID;
    }
    *out = nullptr;
    int visible = 0;
    CQ_CUDA(cudaGetDeviceCount(&visible));
    std::vector<int> devs(n_gpus);
    for (int i = 0; i < n_gpus; i++) {
        devs[i] = devices ? devices[i] : i;
        if (devs[i] < 0 || devs[i] >= visible) {
            set_error("cq_group_create_local: device %d of %d visible", devs[i], visible);
            return CQ_ERR_INVALID;
        }
    }
    cq_group *g = new cq_group();
    g->nRanks = n_gpus, g->rank = -1, g->devices = devs;
    g->comms.assign(n_gpus, nullptr);
    if (n_gpus > 1 || nccl().ok) { // a single-device group works without NCCL (its gather is a copy)
        int rc = need_nccl();
        if (rc == CQ_OK) rc = check_nccl(nccl().CommInitAll(g->comms.data(), n_gpus, devs.data()), "ncclCommInitAll");
        if (rc != CQ_OK && n_gpus > 1) {
            delete g;
            return rc;
        }
    }
    int prev = 0;
    cudaGetDevice(&prev);
    for (int i = 0; i < n_gpus; i++) {
        g->workers.push_back(new Worker());
        cudaStream_t st = nullptr;
        cudaSetDevice(devs[i]);
        cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
        g->streams.push_back(st);
    }
    cudaSetDevice(prev);
    *out = g;
    return CQ_OK;
}

void cq_group_destroy(cq_group *g) {
    if (!g) return;
    int prev = 0;
    cudaGetDevice(&prev);
    for (size_t i = 0; i < g->comms.size(); i++)
        if (g->comms[i]) nccl().CommDestroy(g->comms[i]);
    for (size_t i = 0; i < g->streams.size(); i++) {
        cudaSetDevice(g->devices[i]);
        if (g->streams[i]) cudaStreamDestroy(g->streams[i]);
    }
    for (Worker *w : g->workers) delete w;
    cudaSetDevice(prev);
    delete g;
}

int32_t cq_group_size(const cq_group *g) { return g ? g->nRanks : 0; }
int32_t cq_group_rank(const cq_group *g) { return g ? g->rank : -1; }
int32_t cq_group_device(const cq_group *g, int32_t i) { return g && i >= 0 && i < (int)g->devices.size() ? g->devices[i] : -1; }

// the collective itself for one communicator (called inside an NCCL group when a process owns several)
static int gather_one(cq_group *g, int idx, int rank, const void *dLocal, int64_t nUnits, size_t recBytes, void *dAll, cudaStream_t st) {
    const int n = g->nRanks;
    bool equal = nUnits % n == 0;
    if (equal) return check_nccl(nccl().AllGather(dLocal, dAll, (size_t)(nUnits / n) * recBytes, ncclChar, g->comms[idx], st), "ncclAllGather");
    for (int r = 0; r < n; r++) { // ragged: rank r's shard is broadcast straight to its offset of the result
        int64_t lo, hi;
        cq_shard_range(nUnits, n, r, &lo, &hi);
        char *dst = (char *)dAll + (size_t)lo * recBytes;
        const void *src = r == rank ? dLocal : dst; // (unused on non-root ranks)
        if (hi > lo) CQ_TRY(check_nccl(nccl().Broadcast(src, dst, (size_t)(hi - lo) * recBytes, ncclChar, r, g->comms[idx], st), "ncclBroadcast"));
    }
    return CQ_OK;
}

int cq_group_gather_records(cq_group *g, const void *d_local, int64_t n_units, size_t record_bytes, void *d_all, void *stream) {
    if (!g || g->rank < 0 || n_units < 0 || record_bytes == 0 || (n_units > 0 && (!d_local || !d_all))) {
        set_error("cq_group_gather_records: needs a process-per-GPU group (cq_group_create_rank) and device buffers");
        return CQ_ERR_INVALID;
    }
    if (n_units == 0) return CQ_OK;
    const bool ragged = n_units % g->nRanks != 0;
    if (ragged) CQ_NCCL(nccl().GroupStart());
    int rc = gather_one(g, 0, g->rank, d_local, n_units, record_bytes, d_all, (cudaStream_t)stream);
    if (ragged) {
        const int r2 = check_nccl(nccl().GroupEnd(), "ncclGroupEnd");
        if (rc == CQ_OK) rc = r2;
    }
    return rc;
}

int cq_group_gather_records_local(cq_group *g, const void *const *d_local, int64_t n_units, size_t record_bytes, void *const *d_all,
                                  void *const *streams) {
    if (!g || g->rank >= 0 || n_units < 0 || record_bytes == 0 || !d_local || !d_all) {
        set_error("cq_group_gather_records_local: needs a local group (cq_group_create_local) and one buffer pair per device");
        return CQ_ERR_INVALID;
    }
    if (n_units == 0) return CQ_OK;
    const int n = g->nRanks;
    if (n == 1) { // one device: the gather is a copy
        int prev = 0;
        cudaGetDevice(&prev);
        CQ_CUDA(cudaSetDevice(g->devices[0]));
        cudaStream_t st = streams ? (cudaStream_t)streams[0] : g->streams[0];
        if (d_all[0] != d_local[0]) CQ_CUDA(cudaMemcpyAsync(d_all[0], d_local[0], (size_t)n_units * record_bytes, cudaMemcpyDeviceToDevice, st));
        cudaSetDevice(prev);
        return CQ_OK;
    }
    CQ_TRY(need_nccl());
    CQ_NCCL(nccl().GroupStart());
    int rc = CQ_OK;
    for (int i = 0; i < n && rc == CQ_OK; i++)
        rc = gather_one(g, i, i, d_local[i], n_units, record_bytes, d_all[i], streams ? (cudaStream_t)streams[i] : g->streams[i]);
    const int r2 = check_nccl(nccl().GroupEnd(), "ncclGroupEnd");
    return rc != CQ_OK ? rc : r2;
}

int cq_group_synchronize(cq_group *g) {
    if (!g) return CQ_ERR_INVALID;
    int prev = 0;
    cudaGetDevice(&prev);
    int rc = CQ_OK;
    for (size_t i = 0; i < g->streams.size(); i++) {
        cudaSetDevice(g->devices[i]);
        const int r = check_cuda(cudaStreamSynchronize(g->streams[i]), "group stream");
        if (rc == CQ_OK) rc = r;
    }
    cudaSetDevice(prev);
    return rc;
}

// ---------------------------------------------------------------- replicated world + sharded host batches
int cq_world_create_multi(cq_group *g, const cq_mesh_part *parts, int32_t n_parts, const cq_world_options *options,
                          cq_multi_world **out) {
    if (!g || !out || g->rank >= 0) {
        set_error("cq_world_create_multi: needs a local group (cq_group_create_local)");
        return CQ_ERR_INVALID;
    }
    *out = nullptr;
    cq_multi_world *mw = new cq_multi_world();
    mw->group = g;
    mw->replicas.assign(g->devices.size(), nullptr);
    // every device builds its own replica from the caller's arrays (deterministic build: identical trees, no broadcast)
    const int rc = on_every_device(g, [&](int i) { return cq_world_create_ex(parts, n_parts, options, &mw->replicas[i]); });
    if (rc != CQ_OK) {
        const std::string keep = cq_last_error();
        cq_multi_world_destroy(mw);
        set_error("%s", keep.c_str());
        return rc;
    }
    *out = mw;
    return CQ_OK;
}

void cq_multi_world_destroy(cq_multi_world *mw) {
    if (!mw) return;
    int prev = 0;
    cudaGetDevice(&prev);
    for (size_t i = 0; i < mw->agentBufs.size(); i++) {
        MultiAgentBuffers &b = mw->agentBufs[i];
        cudaSetDevice(mw->group->devices[i]);
        cudaFree(b.states), cudaFree(b.snap), cudaFree(b.platforms);
    }
    for (cq_world *w : mw->replicas)
        if (w) cq_world_destroy(w);
    cudaSetDevice(prev);
    delete mw;
}

int32_t cq_multi_world_size(const cq_multi_world *mw) { return mw ? (int32_t)mw->replicas.size() : 0; }
cq_world *cq_multi_world_replica(cq_multi_world *mw, int32_t i) {
    return mw && i >= 0 && i < (int32_t)mw->replicas.size() ? mw->replicas[i] : nullptr;
}

int cq_multi_update_transforms(cq_multi_world *mw, const uint32_t *entity_ids, const float *models, int32_t n) {
    if (!mw) return CQ_ERR_INVALID;
    return on_every_device(mw->group, [&](int i) { return cq_world_update_transforms(mw->replicas[i], entity_ids, models, n); });
}

int cq_multi_raycast_batch(cq_multi_world *mw, const cq_ray *rays, int32_t n, cq_ray_hit *out) {
    if (n > 0 && (!rays || !out)) return CQ_ERR_INVALID;
    return sharded(mw, n, [&](cq_world *w, int64_t lo, int32_t cnt) { return cq_raycast_batch(w, rays + lo, cnt, out + lo); });
}

int cq_multi_capsule_cast_batch(cq_multi_world *mw, const cq_capsule_cast *q, int32_t n, int32_t mode, cq_cast_hit *out) {
    if (n > 0 && (!q || !out)) return CQ_ERR_INVALID;
    return sharded(mw, n, [&](cq_world *w, int64_t lo, int32_t cnt) { return cq_capsule_cast_batch(w, q + lo, cnt, mode, out + lo); });
}

int cq_multi_move_and_slide_batch(cq_multi_world *mw, cq_character_state *inout, int32_t n, const cq_controller_params *params,
                                  float dt, const float gravity[3], uint32_t flags) {
    if (n > 0 && !inout) return CQ_ERR_INVALID;
    if (flags & CQ_MAS_AGENTS) { // the batch is the crowd: agents of different shards would not see each other
        set_error("cq_multi_move_and_slide_batch: CQ_MAS_AGENTS couples the characters of a batch; use cq_multi_move_and_slide_batch_ex");
        return CQ_ERR_INVALID;
    }
    return sharded(mw, n, [&](cq_world *w, int64_t lo, int32_t cnt) {
        return cq_move_and_slide_batch(w, inout + lo, cnt, params, dt, gravity, flags);
    });
}

int cq_multi_move_and_slide_batch_ex(cq_multi_world *mw, cq_character_state *inout, int32_t n, const cq_controller_params *params,
                                     float dt, const float gravity[3], uint32_t flags, const cq_platform *platforms,
                                     int32_t n_platforms) {
    if (!mw || n < 0 || !params || !gravity || (n > 0 && !inout) || n_platforms < 0 || n_platforms > 64 ||
        (n_platforms > 0 && !platforms)) {
        set_error("cq_multi_move_and_slide_batch_ex: invalid arguments (0..64 host platforms)");
        return CQ_ERR_INVALID;
    }
    if (!(flags & CQ_MAS_AGENTS))
        return sharded(mw, n, [&](cq_world *w, int64_t lo, int32_t cnt) {
            return cq_move_and_slide_batch_ex(w, inout + lo, cnt, params, dt, gravity, flags, platforms, n_platforms);
        });
    if (n == 0) return CQ_OK;
    const int ranks = (int)mw->replicas.size();
    mw->agentBufs.resize(ranks);
    // 1. every replica uploads its shard and snapshots it into its range of a crowd-sized snapshot
    CQ_TRY(on_every_device(mw->group, [&](int i) {
        cq_world *w = mw->replicas[i];
        MultiAgentBuffers &b = mw->agentBufs[i];
        int64_t lo, hi;
        cq_shard_range(n, ranks, i, &lo, &hi);
        const int32_t cnt = (int32_t)(hi - lo);
        CQ_TRY(grow(b.states, b.capStates, (size_t)std::max(cnt, 1), "multi agents: shard"));
        CQ_TRY(grow(b.snap, b.capSnap, (size_t)n, "multi agents: snapshot"));
        if (!b.platforms) CQ_CUDA(cudaMalloc((void **)&b.platforms, 64 * sizeof(cq_platform)));
        CQ_NO_CAPTURE(w->stream, "cq_multi_move_and_slide_batch_ex");
        if (cnt == 0) return CQ_OK;
        CQ_CUDA(cudaMemcpyAsync(b.states, inout + lo, sizeof(cq_character_state) * (size_t)cnt, cudaMemcpyHostToDevice, w->stream));
        return cq_agent_snapshot_device(w, b.states, cnt, dt, gravity, flags, b.snap + lo, w->stream);
    }));
    // 2. one all-gather of the 32-byte records, in place, on the replicas' streams (ordered after the snapshots)
    std::vector<const void *> local(ranks);
    std::vector<void *> all(ranks), streams(ranks);
    for (int i = 0; i < ranks; i++) {
        int64_t lo, hi;
        cq_shard_range(n, ranks, i, &lo, &hi);
        local[i] = mw->agentBufs[i].snap + lo;
        all[i] = mw->agentBufs[i].snap;
        streams[i] = (void *)mw->replicas[i]->stream;
    }
    CQ_TRY(cq_group_gather_records_local(mw->group, local.data(), n, sizeof(cq_agent_snapshot), all.data(), streams.data()));
    // 3. every replica moves its shard against the whole snapshot and downloads it
    return on_every_device(mw->group, [&](int i) {
        cq_world *w = mw->replicas[i];
        MultiAgentBuffers &b = mw->agentBufs[i];
        int64_t lo, hi;
        cq_shard_range(n, ranks, i, &lo, &hi);
        const int32_t cnt = (int32_t)(hi - lo);
        if (n_platforms > 0)
            CQ_CUDA(cudaMemcpyAsync(b.platforms, platforms, sizeof(cq_platform) * (size_t)n_platforms, cudaMemcpyHostToDevice,
                                    w->stream));
        if (cnt > 0) {
            CQ_TRY(cq_move_and_slide_device_agents(w, b.states, cnt, b.snap, n, (int32_t)lo, params, dt, gravity, flags, b.platforms,
                                                   n_platforms, w->stream));
            CQ_CUDA(cudaMemcpyAsync(inout + lo, b.states, sizeof(cq_character_state) * (size_t)cnt, cudaMemcpyDeviceToHost, w->stream));
        }
        CQ_CUDA(cudaStreamSynchronize(w->stream));
        return check_status(w, "cq_multi_move_and_slide_batch_ex");
    });
}

} // extern "C"
