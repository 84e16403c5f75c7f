// cq_api.cu — the C ABI of include/cq.h: world lifetime, transforms/refit, batch + device query
// entry points, counters.  No CPU fallback anywhere: every path needs a usable CUDA device.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <map>

#include "cq_internal.h"

namespace cq {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return CQ_OK;
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return CQ_ERR_CUDA;
}

int ensure_scratch(ScratchBuf &b, size_t bytes) {
    if (bytes <= b.cap) return CQ_OK;
    if (b.ptr) cudaFree(b.ptr);
    b.ptr = nullptr;
    b.cap = 0;
    size_t cap = bytes + bytes / 4 + 256;
    int r = check_cuda(cudaMalloc(&b.ptr, cap), "scratch cudaMalloc");
    if (r == CQ_OK) b.cap = cap;
    return r;
}

int check_status(cq_world *w, const char *what) {
    if (!w->hStatus) return CQ_OK;
    const unsigned int v = *(volatile unsigned int *)w->hStatus;
    if (v == 0) return CQ_OK;
    *(volatile unsigned int *)w->hStatus = 0;
    set_error("%s: device status 0x%x (%s%s%s): results of the call are incomplete", what, v,
              (v & 1u) ? "traversal stack overflow " : "", (v & 2u) ? "sort look-back watchdog fired " : "",
              (v & 4u) ? "pair-pool watchdog fired" : "");
    return CQ_ERR_CUDA;
}

int *next_work_counter(cq_world *w, cudaStream_t st) {
    int *p = w->dWork + (w->workSeq++ % CQ_WORK_RING);
    if (check_cuda(cudaMemsetAsync(p, 0, sizeof(int), st), "work counter") != CQ_OK) return nullptr;
    return p;
}

int scratch_acquire(cq_world *w, ScratchBuf &b, cudaStream_t st) {
    if (!b.ev) CQ_CUDA(cudaEventCreateWithFlags(&b.ev, cudaEventDisableTiming));
    if (b.recorded && b.last != st) CQ_CUDA(cudaStreamWaitEvent(st, b.ev, 0));
    if (std::find(w->held.begin(), w->held.end(), &b) == w->held.end()) w->held.push_back(&b);
    return CQ_OK;
}

int release_held(cq_world *w, cudaStream_t st) {
    int rc = CQ_OK;
    for (ScratchBuf *b : w->held) {
        int r = check_cuda(cudaEventRecord(b->ev, st), "scratch release");
        if (r != CQ_OK) rc = r;
        b->last = st;
        b->recorded = true;
    }
    w->held.clear();
    return rc;
}

int await_trees(const cq_world *w, cudaStream_t st) {
    if (w->treesPending && st != w->treesStream) CQ_CUDA(cudaStreamWaitEvent(st, w->evTrees, 0));
    return CQ_OK;
}

// one event per stream that ever launched on the world, re-recorded by every launch on it
static int note_reader(cq_world *w, cudaStream_t st) {
    ReaderEvent *r = nullptr;
    for (ReaderEvent &e : w->readers)
        if (e.st == st) r = &e;
    if (!r) {
        ReaderEvent e;
        e.st = st;
        CQ_CUDA(cudaEventCreateWithFlags(&e.ev, cudaEventDisableTiming));
        w->readers.push_back(e);
        r = &w->readers.back();
    }
    CQ_CUDA(cudaEventRecord(r->ev, st));
    r->pending = true;
    return CQ_OK;
}

int finish_launch(cq_world *w, cudaStream_t st, const char *what) {
    const int rc = check_cuda(cudaGetLastError(), what);
    const int rr = release_held(w, st);
    const int rn = note_reader(w, st);
    return rc != CQ_OK ? rc : rr != CQ_OK ? rr : rn;
}

static void destroy_scratch(ScratchBuf &b) {
    if (b.ptr) cudaFree(b.ptr);
    if (b.ev) cudaEventDestroy(b.ev);
    b = ScratchBuf();
}

void *pool_node_scratch(cq_world *w, size_t warps, cudaStream_t st) {
    size_t bytes = warps * (size_t)2048 /* CQ_NSCAP */ * sizeof(uint2);
    if (bytes > w->nodeScratch[0].cap) {
        // grow all four regions at once (a cudaMalloc inside a timed step costs milliseconds); growing frees the
        // old blocks, so make sure no launch still uses them
        if (check_cuda(cudaDeviceSynchronize(), "node scratch sync") != CQ_OK) return nullptr;
        for (int k = 0; k < 4; k++)
            if (ensure_scratch(w->nodeScratch[k], bytes) != CQ_OK) return nullptr;
    }
    ScratchBuf &b = w->nodeScratch[w->nodeSeq++ & 3];
    if (scratch_acquire(w, b, st) != CQ_OK) return nullptr;
    return b.ptr;
}

static void make_view(cq_world *w) {
    for (int s = 0; s < 2; s++) {
        DeviceSet &S = w->set[s];
        SetView &v = w->view.set[s];
        v.tv0 = S.tv0, v.tv1 = S.tv1, v.tv2 = S.tv2;
        v.nodes = S.nodes;
        v.nodes4 = S.nodes4;
        v.hdr = S.hdr;
        v.triPart = S.triPart;
        v.triMat = S.triMat;
        v.triOffset = s == 0 ? 0 : w->set[0].nTris;
        v.refNodes = S.refNodes;
        v.refSlot = S.refSlot;
        v.refHdr = S.refHdr ? S.refHdr : S.hdr; // an empty set has no reference tree: its LBVH header says "empty" too
    }
    w->view.rank = w->order == CQ_ORDER_REFERENCE ? w->dRank : nullptr;
    w->view.encOfRank = w->dEncOfRank;
    w->view.status = nullptr;
    if (w->hStatus) cudaHostGetDevicePointer((void **)&w->view.status, w->hStatus, 0);
    w->view.materials = w->dMaterials;
    w->view.nParts = (int)w->parts.size();
    w->view.nMaterials = (int)std::max(w->hMaterials.size(), w->parts.size());
    w->view.stagedLeaves = (w->set[0].nTris + w->set[1].nTris) >= 4096 ? 1 : 0;
    w->view.refStats = w->countRef;
}

} // namespace cq

using namespace cq;

static cudaStream_t pick_stream(cq_world *w, void *stream) { return stream ? (cudaStream_t)stream : w->stream; }

// ---------------------------------------------------------------- transform updates
// Queues the refit of the rows staged in movedRows on `st`: after every launch that has read the trees since the last
// refit (any stream) and after the previous refit, then records evTrees, which every later launch on another stream waits
// for (await_trees).  The table reaches the device in one copy from a pinned slot of a ring of CQ_STAGE_SLOTS; a slot is
// reused once its copy has completed, so the caller's arrays are free when the call returns and the host blocks only when
// CQ_STAGE_SLOTS earlier updates still have their copy in flight (it then waits for the oldest).  A table larger than any
// before it grows the slot and the device table; the old buffers are retired, not freed (a free would wait for the device),
// until the next synchronous update or cq_world_destroy.
static void free_retired(cq_world *w) {
    for (void *p : w->retiredDev) cudaFree(p);
    for (void *p : w->retiredHost) cudaFreeHost(p);
    w->retiredDev.clear(), w->retiredHost.clear();
}

static int queue_refit(cq_world *w, cudaStream_t st, cudaEvent_t t0) {
    for (ReaderEvent &r : w->readers)
        if (r.pending) {
            if (r.st != st) CQ_CUDA(cudaStreamWaitEvent(st, r.ev, 0));
            r.pending = false;
        }
    CQ_TRY(await_trees(w, st));
    const size_t n0 = w->movedRows[0].size(), nRows = n0 + w->movedRows[1].size(), bytes = nRows * sizeof(MovedPart);
    StageSlot &slot = w->stage[w->stageSeq++ % CQ_STAGE_SLOTS];
    if (!slot.ev) CQ_CUDA(cudaEventCreateWithFlags(&slot.ev, cudaEventDisableTiming));
    if (slot.recorded) CQ_CUDA(cudaEventSynchronize(slot.ev));
    if (slot.cap < nRows) {
        if (slot.host) w->retiredHost.push_back(slot.host);
        slot.host = nullptr, slot.cap = 0;
        const size_t cap = nRows + nRows / 4 + 16;
        CQ_CUDA(cudaHostAlloc((void **)&slot.host, cap * sizeof(MovedPart), cudaHostAllocDefault));
        slot.cap = cap;
    }
    if (bytes > w->dTable.cap) { // the previous refit may still read the old table
        if (w->dTable.ptr) w->retiredDev.push_back(w->dTable.ptr);
        w->dTable.ptr = nullptr, w->dTable.cap = 0;
        CQ_TRY(ensure_scratch(w->dTable, bytes));
    }
    std::copy(w->movedRows[0].begin(), w->movedRows[0].end(), slot.host);
    std::copy(w->movedRows[1].begin(), w->movedRows[1].end(), slot.host + n0);
    CQ_CUDA(cudaMemcpyAsync(w->dTable.ptr, slot.host, bytes, cudaMemcpyHostToDevice, st));
    CQ_CUDA(cudaEventRecord(slot.ev, st));
    slot.recorded = true;
    if (t0) CQ_CUDA(cudaEventRecord(t0, st));
    const MovedPart *dTab = (const MovedPart *)w->dTable.ptr;
    CQ_TRY(refit_set(w, w->set[0], dTab, w->movedRows[0], st));
    CQ_TRY(refit_set(w, w->set[1], dTab + n0, w->movedRows[1], st));
    CQ_CUDA(cudaEventRecord(w->evTrees, st));
    w->treesStream = st;
    w->treesPending = true;
    return CQ_OK;
}

// Both transform-update calls: check every id before anything is queued (a failed call changes nothing), build the table
// of moved parts, queue the refit on `st`.  t0 (may be null) is recorded after the table copy, before the refit kernels.
static int update_transforms_on(cq_world *w, const uint32_t *ids, const float *models, int n, cudaStream_t st, const char *what,
                                cudaEvent_t t0) {
    for (int i = 0; i < n; i++)
        if (w->partsOfEntity.find(ids[i]) == w->partsOfEntity.end()) {
            set_error("%s: unknown entity id %u", what, ids[i]);
            return CQ_ERR_NOT_FOUND;
        }
    // every part with the id takes the model; `guard let slice = slices[e]`: parts that contributed no triangle are
    // skipped (CollisionQuery.swift:427); a part named twice keeps the last model
    for (int i = 0; i < n; i++)
        for (int p : w->partsOfEntity.find(ids[i])->second) {
            const PartInfo &pi = w->parts[p];
            if (pi.triHi <= pi.triLo) continue;
            std::vector<MovedPart> &rows = w->movedRows[pi.set];
            int32_t &row = w->movedSlot[p];
            if (row < 0) {
                row = (int32_t)rows.size();
                MovedPart r{};
                r.part = p, r.vertLo = pi.vertLo, r.triLo = pi.triLo, r.nVerts = pi.vertHi - pi.vertLo, r.nTris = pi.triHi - pi.triLo;
                rows.push_back(r);
            }
            memcpy(rows[row].model, models + 16 * (size_t)i, sizeof(float) * 16);
        }
    for (int s = 0; s < 2; s++) {
        int32_t v = 0, t = 0;
        for (MovedPart &r : w->movedRows[s]) {
            w->movedSlot[r.part] = -1;
            r.vertBase = v, r.triBase = t;
            v += r.nVerts, t += r.nTris;
        }
    }
    int rc = CQ_OK;
    if (!w->movedRows[0].empty() || !w->movedRows[1].empty()) rc = queue_refit(w, st, t0);
    else if (t0) rc = check_cuda(cudaEventRecord(t0, st), "update timing");
    w->movedRows[0].clear(), w->movedRows[1].clear();
    return rc;
}

// ---------------------------------------------------------------- host-pointer (synchronous) entry points
// Three-stage pipeline over chunks of the batch: a dedicated H2D stream streams the inputs in back to back,
// two alternating compute streams run the chunk kernels (so one chunk's tail overlaps the next chunk's
// head), a dedicated D2H stream streams the results out; events order chunk k's copy -> kernel -> copy.
// PCIe is full duplex, so the wall time approaches max(H2D, kernels, D2H) instead of their sum.
// Chunking adapts to the previous call of the same entry point: when that call was compute-bound (wall time
// >> PCIe time of its bytes) the next one uses two chunks only, because every chunk kernel pays its own tail.
// leave no copy in flight on the caller's memory when a batch call fails half-way
static int fail_batch(cq_world *w, int rc) {
    cudaStreamSynchronize(w->h2dStream);
    cudaStreamSynchronize(w->copyStream[0]);
    cudaStreamSynchronize(w->copyStream[1]);
    cudaStreamSynchronize(w->d2hStream);
    return rc;
}
#define CQ_CUDA_B(x)                                   \
    do {                                               \
        int _r = cq::check_cuda((x), #x);              \
        if (_r != CQ_OK) return fail_batch(w, _r);     \
    } while (0)

// flagsHost (may be null): one byte per unit, produced by the launch into w->aux2 at the unit's index
template <class In, class Out, class Launch>
static int run_batch(cq_world *w, const In *in, size_t inStride, Out *out, size_t outStride, int n, Launch launch,
                     bool inPlace = false, float *computeBoundHint = nullptr, bool singleChunk = false,
                     uint8_t *flagsHost = nullptr) {
    if (n <= 0) return CQ_OK;
    CQ_CUDA(cudaSetDevice(w->device));
    static const int CH = [] { // units per chunk of the copy/compute pipeline (CQ_CHUNK overrides, for tuning)
        const char *e = getenv("CQ_CHUNK");
        int v = e ? atoi(e) : 0;
        return v >= 1024 ? v : (1 << 17);
    }();
    int nChunks = (n + CH - 1) / CH;
    if (computeBoundHint && *computeBoundHint > 3.0f && nChunks > 2) nChunks = 2;
    if (nChunks > CQ_PIPE_EVENTS) nChunks = CQ_PIPE_EVENTS;
    if (singleChunk) nChunks = 1; // the units interact (agents): every one must be resident before the kernel starts
    const auto t0 = std::chrono::steady_clock::now();
    int chunk = (n + nChunks - 1) / nChunks;
    int r;
    if ((r = ensure_scratch(w->in, (size_t)n * inStride)) != CQ_OK) return r;
    if (!inPlace && (r = ensure_scratch(w->out, (size_t)n * outStride)) != CQ_OK) return r;
    if (flagsHost && (r = ensure_scratch(w->aux2, (size_t)n)) != CQ_OK) return r;
    int k = 0;
    for (int lo = 0; lo < n; lo += chunk, k++) {
        int cnt = std::min(chunk, n - lo);
        cudaStream_t cs = w->copyStream[k & 1]; // compute streams
        char *dIn = (char *)w->in.ptr + (size_t)lo * inStride;
        char *dOut = inPlace ? dIn : (char *)w->out.ptr + (size_t)lo * outStride;
        CQ_CUDA_B(cudaMemcpyAsync(dIn, (const char *)in + (size_t)lo * inStride, (size_t)cnt * inStride, cudaMemcpyHostToDevice,
                                  w->h2dStream));
        CQ_CUDA_B(cudaEventRecord(w->evIn[k], w->h2dStream));
        CQ_CUDA_B(cudaStreamWaitEvent(cs, w->evIn[k], 0));
        r = launch(dIn, dOut, cnt, lo, cs);
        if (r != CQ_OK) return fail_batch(w, r);
        CQ_CUDA_B(cudaEventRecord(w->evDone[k], cs));
        CQ_CUDA_B(cudaStreamWaitEvent(w->d2hStream, w->evDone[k], 0));
        CQ_CUDA_B(cudaMemcpyAsync((char *)out + (size_t)lo * outStride, dOut, (size_t)cnt * outStride, cudaMemcpyDeviceToHost,
                                  w->d2hStream));
        if (flagsHost)
            CQ_CUDA_B(cudaMemcpyAsync(flagsHost + lo, (const uint8_t *)w->aux2.ptr + lo, (size_t)cnt, cudaMemcpyDeviceToHost,
                                      w->d2hStream));
    }
    CQ_CUDA(cudaStreamSynchronize(w->d2hStream));
    CQ_TRY(check_status(w, "batch call"));
    if (computeBoundHint) {
        double wallMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        double pcieMs = (double)n * (double)std::max(inStride, outStride) / 50.0e6; // ~50 GB/s per direction, duplex
        *computeBoundHint = (float)(wallMs / std::max(pcieMs, 1e-3));
    }
    return CQ_OK;
}

extern "C" {

const char *cq_last_error(void) { return g_err; }
const char *cq_version(void) { return "cq-b200 0.1 (sm_100a)"; }

void *cq_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void cq_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

void cq_controller_params_default(cq_controller_params *p) { // Components.swift:380-404
    p->radius = 1.5f;
    p->half_height = 1.0f;
    p->skin_width = 0.3f;
    p->ground_snap_skin = 0.05f;
    p->snap_distance = 0.8f;
    p->fall_probe_distance = 200.0f;
    p->ground_snap_max_speed = 5.0f;
    p->ground_snap_max_toi = 0.1f;
    p->ground_snap_max_step = 0.1f;
    p->ground_sweep_max_step = 0.1f;
    p->max_slide_iterations = 4;
    p->min_ground_dot = 0.5f;
    p->collision_mask = CQ_LAYER_ALL;
}

void cq_character_state_init(cq_character_state *s, const float position[3], const float velocity[3]) {
    memset(s, 0, sizeof(*s));
    for (int k = 0; k < 3; k++) {
        s->position[k] = (double)position[k]; // PhysicsBodyComponent.init widens Float -> Double (Components.swift:566-575)
        s->velocity[k] = velocity ? (double)velocity[k] : 0.0;
    }
    s->ground_normal[1] = 1.0f;
    s->ground_distance = 3.402823466e+38f;
    s->ground_triangle_index = -1;
}

void cq_world_options_default(cq_world_options *o) {
    if (!o) return;
    memset(o, 0, sizeof(*o));
    o->order = CQ_ORDER_REFERENCE;
}

int cq_world_create(const cq_mesh_part *parts, int32_t n_parts, cq_world **out) {
    return cq_world_create_ex(parts, n_parts, nullptr, out);
}

int cq_world_create_ex(const cq_mesh_part *parts, int32_t n_parts, const cq_world_options *options, cq_world **out) {
    if (!out || n_parts < 0 || (n_parts > 0 && !parts)) {
        set_error("cq_world_create: invalid arguments");
        return CQ_ERR_INVALID;
    }
    *out = nullptr;
    cq_world_options opt;
    cq_world_options_default(&opt);
    if (options) opt = *options;
    if (opt.order != CQ_ORDER_REFERENCE && opt.order != CQ_ORDER_CANONICAL) {
        set_error("cq_world_create: unknown order %d", opt.order);
        return CQ_ERR_INVALID;
    }
    int dev = 0;
    CQ_CUDA(cudaGetDevice(&dev));
    cq_world *w = new cq_world();
    w->device = dev;
    w->order = opt.order;
    int rc = CQ_OK;
    auto fail = [&](int r) {
        cq_world_destroy(w);
        return r;
    };
    if ((rc = check_cuda(cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking), "stream")) != CQ_OK) return fail(rc);
    for (int k = 0; k < 2; k++)
        if ((rc = check_cuda(cudaStreamCreateWithFlags(&w->copyStream[k], cudaStreamNonBlocking), "stream")) != CQ_OK)
            return fail(rc);
    if ((rc = check_cuda(cudaStreamCreateWithFlags(&w->h2dStream, cudaStreamNonBlocking), "stream")) != CQ_OK) return fail(rc);
    if ((rc = check_cuda(cudaStreamCreateWithFlags(&w->d2hStream, cudaStreamNonBlocking), "stream")) != CQ_OK) return fail(rc);
    for (int k = 0; k < CQ_PIPE_EVENTS; k++) {
        if ((rc = check_cuda(cudaEventCreateWithFlags(&w->evIn[k], cudaEventDisableTiming), "event")) != CQ_OK) return fail(rc);
        if ((rc = check_cuda(cudaEventCreateWithFlags(&w->evDone[k], cudaEventDisableTiming), "event")) != CQ_OK) return fail(rc);
    }
    if ((rc = check_cuda(cudaEventCreate(&w->evA), "event")) != CQ_OK) return fail(rc);
    if ((rc = check_cuda(cudaEventCreate(&w->evB), "event")) != CQ_OK) return fail(rc);
    if ((rc = check_cuda(cudaEventCreateWithFlags(&w->evTrees, cudaEventDisableTiming), "event")) != CQ_OK) return fail(rc);

    // host-side assembly of the two sets' input arrays (partitionEntities, CollisionQuery.swift:886-900): cq_assemble.h
    SetPlan input[2];
    std::vector<PartPlacement> place;
    const PlanError bad = plan_upload(parts, n_parts, input, place);
    if (bad.code != CQ_OK) {
        if (bad.kind == 3)
            set_error("cq_world_create: more than 2^31 vertices or indices in one triangle set (at part %d)", bad.part);
        else
            set_error("cq_world_create: part %d has invalid arrays", bad.part);
        return fail(bad.code);
    }
    std::vector<float> models((size_t)n_parts * 16);
    std::vector<float4> materials(n_parts);
    // per-triangle materials (options->triangle_materials): rows appended to the table after the parts' own rows; a part
    // whose array does not have exactly one entry per triangle keeps its own material (CollisionQuery.swift:365-369)
    std::vector<int32_t> matIn[2];
    if (opt.n_triangle_materials > 0) {
        if (!opt.triangle_materials) {
            set_error("cq_world_create_ex: n_triangle_materials = %d without an array", opt.n_triangle_materials);
            return fail(CQ_ERR_INVALID);
        }
        for (int k = 0; k < opt.n_triangle_materials; k++) {
            const cq_triangle_materials &tm = opt.triangle_materials[k];
            for (int s = 0; s < 2; s++)
                for (const PartRow &row : input[s].rows) {
                    if (parts[row.part].entity_id != tm.entity_id || tm.n != row.nTris || row.nTris == 0) continue;
                    if (!tm.materials) {
                        set_error("cq_world_create_ex: triangle_materials[%d] has no array", k);
                        return fail(CQ_ERR_INVALID);
                    }
                    if (matIn[s].empty()) { // default: every input triangle points at its part's row
                        matIn[s].resize(input[s].nTris);
                        for (const PartRow &r : input[s].rows) std::fill_n(matIn[s].begin() + r.triStart, r.nTris, r.part);
                    }
                    const int32_t base = (int32_t)materials.size();
                    for (int t = 0; t < row.nTris; t++) {
                        const cq_surface_material &m = tm.materials[t];
                        materials.push_back(make_float4(m.mu_s, m.mu_k, m.flatten_ground ? 1.0f : 0.0f, 0.0f));
                        matIn[s][(size_t)row.triStart + t] = base + t;
                    }
                }
        }
    }
    w->parts.resize(n_parts);
    for (int p = 0; p < n_parts; p++) {
        const cq_mesh_part &mp = parts[p];
        PartInfo &pi = w->parts[p];
        pi.entityId = mp.entity_id;
        pi.set = place[p].set;
        pi.vertLo = place[p].vertLo, pi.vertHi = place[p].vertHi;
        pi.material = {mp.mu_s, mp.mu_k, mp.flatten_ground ? 1 : 0};
        pi.layer = mp.layer;
        memcpy(&models[(size_t)p * 16], mp.model, sizeof(float) * 16);
        materials[p] = make_float4(mp.mu_s, mp.mu_k, mp.flatten_ground ? 1.0f : 0.0f, 0.0f);
        w->partsOfEntity[mp.entity_id].push_back(p);
    }
    w->movedSlot.assign(n_parts, -1);

    if ((rc = check_cuda(cudaMalloc((void **)&w->dModels, sizeof(float) * 16 * (size_t)std::max(n_parts, 1)), "models")) != CQ_OK)
        return fail(rc);
    if ((rc = check_cuda(cudaMalloc((void **)&w->dMaterials, sizeof(float4) * std::max(materials.size(), (size_t)1)), "materials")) != CQ_OK)
        return fail(rc);
    w->hMaterials.resize(materials.size());
    for (size_t k = 0; k < materials.size(); k++) w->hMaterials[k] = {materials[k].x, materials[k].y, materials[k].z != 0.0f ? 1 : 0};
    if ((rc = check_cuda(cudaMalloc((void **)&w->dCounters, sizeof(unsigned long long) * 4), "counters")) != CQ_OK) return fail(rc);
    cudaMemsetAsync(w->dCounters, 0, sizeof(unsigned long long) * 4, w->stream);
    if ((rc = check_cuda(cudaMalloc((void **)&w->dWork, sizeof(int) * CQ_WORK_RING), "work counters")) != CQ_OK) return fail(rc);
    if ((rc = check_cuda(cudaHostAlloc((void **)&w->hStatus, sizeof(unsigned int), cudaHostAllocMapped), "status word")) != CQ_OK)
        return fail(rc);
    *w->hStatus = 0;
    cudaHostGetDevicePointer((void **)&w->view.status, w->hStatus, 0);
    if (n_parts) {
        cudaMemcpyAsync(w->dModels, models.data(), sizeof(float) * 16 * (size_t)n_parts, cudaMemcpyHostToDevice, w->stream);
        cudaMemcpyAsync(w->dMaterials, materials.data(), sizeof(float4) * materials.size(), cudaMemcpyHostToDevice, w->stream);
    }
    w->buildMs = 0.0f; // accumulated by build_set: device time of the build kernels only
    for (int s = 0; s < 2; s++) {
        std::vector<int> &partTriStart = input[s].partTriStart; // in: before the degenerate filter; out: after
        int badTri = -1;
        rc = build_set(w, w->set[s], input[s], partTriStart, &badTri, matIn[s].empty() ? nullptr : matIn[s].data());
        if (rc != CQ_OK && badTri >= 0) { // name the part and the first offending index of that triangle
            const PartRow &row = input[s].rows[part_row_of(input[s].rows.data(), (int)input[s].rows.size(), badTri, true)];
            const uint32_t *tri = parts[row.part].indices + 3 * (size_t)(badTri - row.triStart);
            uint32_t li = tri[0];
            for (int k = 2; k >= 0; k--)
                if (tri[k] >= (uint32_t)row.nVerts) li = tri[k];
            set_error("cq_world_create: part %d index %u out of range (%d vertices)", row.part, li, row.nVerts);
        }
        if (rc != CQ_OK) return fail(rc);
        for (size_t k = 0; k < input[s].partOfSet.size(); k++) {
            PartInfo &pi = w->parts[input[s].partOfSet[k]];
            pi.triLo = partTriStart[k];
            pi.triHi = partTriStart[k + 1];
        }
    }
    if ((rc = check_cuda(cudaStreamSynchronize(w->stream), "build")) != CQ_OK) return fail(rc);
    for (int s = 0; s < 2; s++)
        if (w->set[s].triMat && w->set[s].nTris > 0) { // host copy for cq_world_triangle_material
            w->hTriMat[s].resize((size_t)w->set[s].nTris);
            if ((rc = check_cuda(cudaMemcpy(w->hTriMat[s].data(), w->set[s].triMat, sizeof(int32_t) * (size_t)w->set[s].nTris,
                                            cudaMemcpyDeviceToHost), "triangle materials")) != CQ_OK)
                return fail(rc);
        }
    if (w->order == CQ_ORDER_REFERENCE && (rc = attach_ref_order(w)) != CQ_OK) return fail(rc);
    make_view(w);
    *out = w;
    return CQ_OK;
}

void cq_world_destroy(cq_world *w) {
    if (!w) return;
    cudaSetDevice(w->device);
    cudaDeviceSynchronize(); // *_device launches may still be in flight on the caller's streams
    for (int s = 0; s < 2; s++) free_set(w->set[s]);
    cudaFree(w->dModels), cudaFree(w->dMaterials), cudaFree(w->dCounters), cudaFree(w->dWork), cudaFree(w->dRank), cudaFree(w->dEncOfRank);
    if (w->hStatus) cudaFreeHost(w->hStatus);
    destroy_scratch(w->in), destroy_scratch(w->out), destroy_scratch(w->aux), destroy_scratch(w->aux2);
    for (int k = 0; k < 4; k++) destroy_scratch(w->nodeScratch[k]), destroy_scratch(w->orderScratch[k]);
    destroy_scratch(w->agentScratch);
    sep_graphs_destroy(w);
    destroy_scratch(w->sepScratch);
    destroy_scratch(w->dTable);
    free_retired(w);
    for (StageSlot &s : w->stage) {
        if (s.host) cudaFreeHost(s.host);
        if (s.ev) cudaEventDestroy(s.ev);
    }
    for (ReaderEvent &e : w->readers) cudaEventDestroy(e.ev);
    if (w->evTrees) cudaEventDestroy(w->evTrees);
    if (w->evA) cudaEventDestroy(w->evA);
    if (w->evB) cudaEventDestroy(w->evB);
    if (w->stream) cudaStreamDestroy(w->stream);
    if (w->h2dStream) cudaStreamDestroy(w->h2dStream);
    if (w->d2hStream) cudaStreamDestroy(w->d2hStream);
    for (int k = 0; k < CQ_PIPE_EVENTS; k++) {
        if (w->evIn[k]) cudaEventDestroy(w->evIn[k]);
        if (w->evDone[k]) cudaEventDestroy(w->evDone[k]);
    }
    for (int k = 0; k < 2; k++)
        if (w->copyStream[k]) cudaStreamDestroy(w->copyStream[k]);
    delete w;
}

int cq_world_get_info(const cq_world *w, cq_world_info *info) {
    if (!w || !info) return CQ_ERR_INVALID;
    info->n_static_triangles = w->set[0].nTris;
    info->n_dynamic_triangles = w->set[1].nTris;
    info->n_static_vertices = w->set[0].nVerts;
    info->n_dynamic_vertices = w->set[1].nVerts;
    info->n_static_nodes = std::max(w->set[0].nTris - 1, 0);
    info->n_dynamic_nodes = std::max(w->set[1].nTris - 1, 0);
    info->n_parts = (int)w->parts.size();
    info->device = w->device;
    info->build_ms = w->buildMs;
    info->refit_ms = w->refitMs;
    info->order = w->order;
    info->ref_order_ms = w->refBuildMs;
    info->n_ref_nodes = w->set[0].nRefInternal + w->set[0].nRefLeaves + w->set[1].nRefInternal + w->set[1].nRefLeaves;
    info->_reserved = 0;
    return CQ_OK;
}

int cq_world_update_transforms(cq_world *w, const uint32_t *entity_ids, const float *models, int32_t n) {
    if (!w || n < 0 || (n > 0 && (!entity_ids || !models))) return CQ_ERR_INVALID;
    CQ_CUDA(cudaSetDevice(w->device));
    // the documented contract of the synchronous call: everything in flight on any stream has finished first
    CQ_CUDA(cudaDeviceSynchronize());
    free_retired(w);
    CQ_TRY(update_transforms_on(w, entity_ids, models, n, w->stream, "cq_world_update_transforms", w->evA));
    cudaEventRecord(w->evB, w->stream);
    CQ_CUDA(cudaStreamSynchronize(w->stream)); // makes refit_ms readable; later launches need not wait for this refit
    w->treesPending = false;
    cudaEventElapsedTime(&w->refitMs, w->evA, w->evB);
    return CQ_OK;
}

int cq_world_update_transforms_async(cq_world *w, const uint32_t *entity_ids, const float *models, int32_t n, void *stream) {
    if (!w || n < 0 || (n > 0 && (!entity_ids || !models))) return CQ_ERR_INVALID;
    if (n == 0) return CQ_OK;
    CQ_CUDA(cudaSetDevice(w->device));
    return update_transforms_on(w, entity_ids, models, n, pick_stream(w, stream), "cq_world_update_transforms_async", nullptr);
}

int cq_world_read_soup(const cq_world *w, int32_t which, float *positions_xyz, uint32_t *indices, float *tri_aabbs,
                       uint32_t *tri_layers, int32_t *tri_parts) {
    if (!w || which < 0 || which > 1) return CQ_ERR_INVALID;
    CQ_CUDA(cudaSetDevice(w->device));
    const DeviceSet &S = w->set[which];
    CQ_TRY(await_trees(w, w->stream));
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    std::vector<float4> pos(S.nVerts);
    std::vector<uint32_t> idx((size_t)S.nTris * 3);
    if (S.nVerts) CQ_CUDA(cudaMemcpy(pos.data(), S.worldPos, sizeof(float4) * (size_t)S.nVerts, cudaMemcpyDeviceToHost));
    if (S.nTris) CQ_CUDA(cudaMemcpy(idx.data(), S.indices, sizeof(uint32_t) * 3 * (size_t)S.nTris, cudaMemcpyDeviceToHost));
    if (positions_xyz)
        for (int i = 0; i < S.nVerts; i++) {
            positions_xyz[3 * i] = pos[i].x;
            positions_xyz[3 * i + 1] = pos[i].y;
            positions_xyz[3 * i + 2] = pos[i].z;
        }
    if (indices && S.nTris) memcpy(indices, idx.data(), sizeof(uint32_t) * idx.size());
    if (tri_aabbs && S.nTris) {
        // bounds as stored on the device: leaf boxes of the sorted order, scattered back to soup order
        std::vector<float4> lo(S.nTris), hi(S.nTris);
        std::vector<uint32_t> sorted(S.nTris);
        CQ_CUDA(cudaMemcpy(lo.data(), S.boxLo + (S.nTris - 1), sizeof(float4) * (size_t)S.nTris, cudaMemcpyDeviceToHost));
        CQ_CUDA(cudaMemcpy(hi.data(), S.boxHi + (S.nTris - 1), sizeof(float4) * (size_t)S.nTris, cudaMemcpyDeviceToHost));
        CQ_CUDA(cudaMemcpy(sorted.data(), S.sortedTri, sizeof(uint32_t) * (size_t)S.nTris, cudaMemcpyDeviceToHost));
        for (int s = 0; s < S.nTris; s++) {
            float *o = tri_aabbs + 6 * (size_t)sorted[s];
            o[0] = lo[s].x, o[1] = lo[s].y, o[2] = lo[s].z, o[3] = hi[s].x, o[4] = hi[s].y, o[5] = hi[s].z;
        }
    }
    if (tri_layers && S.nTris)
        CQ_CUDA(cudaMemcpy(tri_layers, S.triLayer, sizeof(uint32_t) * (size_t)S.nTris, cudaMemcpyDeviceToHost));
    if (tri_parts && S.nTris)
        CQ_CUDA(cudaMemcpy(tri_parts, S.triPart, sizeof(int32_t) * (size_t)S.nTris, cudaMemcpyDeviceToHost));
    return CQ_OK;
}

int cq_world_triangle_material(const cq_world *w, int32_t triangle_index, cq_material *out) {
    if (!w || !out) return CQ_ERR_INVALID;
    *out = {0.8f, 0.6f, 0}; // SurfaceMaterial.default
    if (triangle_index >= 0) { // a set with per-triangle materials: the triangle's own row of the table
        const int off = w->set[0].nTris, s = triangle_index >= off ? 1 : 0, local = s ? triangle_index - off : triangle_index;
        if (!w->hTriMat[s].empty() && local < (int)w->hTriMat[s].size()) {
            const int32_t row = w->hTriMat[s][(size_t)local];
            if (row >= 0 && row < (int32_t)w->hMaterials.size()) *out = w->hMaterials[(size_t)row];
            return CQ_OK;
        }
    }
    for (const PartInfo &p : w->parts) {
        int off = p.set == 0 ? 0 : w->set[0].nTris;
        if (triangle_index >= p.triLo + off && triangle_index < p.triHi + off) {
            *out = p.material;
            return CQ_OK;
        }
    }
    return CQ_OK;
}

int cq_world_set_counting(cq_world *w, int32_t mode) {
    if (!w || mode < CQ_COUNT_OFF || mode > CQ_COUNT_PATH) return CQ_ERR_INVALID;
    w->counting = mode != CQ_COUNT_OFF ? 1 : 0;
    w->countRef = mode == CQ_COUNT_REFERENCE ? 1 : 0;
    w->view.refStats = w->countRef;
    return CQ_OK;
}

int cq_world_read_counters(cq_world *w, cq_counters *out, int32_t reset) {
    if (!w || !out) return CQ_ERR_INVALID;
    CQ_CUDA(cudaSetDevice(w->device));
    unsigned long long h[4];
    CQ_TRY(await_trees(w, w->stream));
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    CQ_CUDA(cudaMemcpy(h, w->dCounters, sizeof(h), cudaMemcpyDeviceToHost));
    CQ_TRY(check_status(w, "cq_world_read_counters"));
    out->nodes_visited = h[0];
    out->candidates = h[1];
    out->distance_evals = h[2];
    out->queries = h[3];
    out->kernel_launches = w->launches;
    if (reset) {
        CQ_CUDA(cudaMemset(w->dCounters, 0, sizeof(h)));
        w->launches = 0;
    }
    return CQ_OK;
}

// ---------------------------------------------------------------- device-pointer entry points

int cq_raycast_device_ex(cq_world *w, const cq_ray *d_rays, int32_t n, cq_ray_hit *d_out, uint8_t *d_flags, void *stream) {
    if (!w || n < 0 || (n > 0 && (!d_rays || !d_out))) return CQ_ERR_INVALID;
    return launch_raycast(w, d_rays, n, d_out, d_flags, pick_stream(w, stream));
}
int cq_raycast_device(cq_world *w, const cq_ray *d_rays, int32_t n, cq_ray_hit *d_out, void *stream) {
    return cq_raycast_device_ex(w, d_rays, n, d_out, nullptr, stream);
}
int cq_capsule_cast_device_ex(cq_world *w, const cq_capsule_cast *d_q, int32_t n, int32_t mode, cq_cast_hit *d_out,
                              uint8_t *d_flags, void *stream) {
    if (!w || n < 0 || mode < 0 || mode > 2 || (n > 0 && (!d_q || !d_out))) return CQ_ERR_INVALID;
    return launch_cast(w, d_q, n, mode, d_out, d_flags, pick_stream(w, stream));
}
int cq_capsule_cast_device(cq_world *w, const cq_capsule_cast *d_q, int32_t n, int32_t mode, cq_cast_hit *d_out, void *stream) {
    return cq_capsule_cast_device_ex(w, d_q, n, mode, d_out, nullptr, stream);
}
int cq_capsule_overlap_device_ex(cq_world *w, const cq_capsule *d_q, int32_t n, cq_overlap_hit *d_out, uint8_t *d_flags,
                                 void *stream) {
    if (!w || n < 0 || (n > 0 && (!d_q || !d_out))) return CQ_ERR_INVALID;
    return launch_overlap(w, d_q, n, d_out, d_flags, pick_stream(w, stream));
}
int cq_capsule_overlap_device(cq_world *w, const cq_capsule *d_q, int32_t n, cq_overlap_hit *d_out, void *stream) {
    return cq_capsule_overlap_device_ex(w, d_q, n, d_out, nullptr, stream);
}
int cq_capsule_overlap_all_device(cq_world *w, const cq_capsule *d_q, int32_t n, int32_t max_hits, cq_overlap_hit *d_out,
                                  int32_t *d_counts, uint8_t *d_overflow, void *stream) {
    if (!w || n < 0 || (n > 0 && (!d_q || !d_out || !d_counts))) return CQ_ERR_INVALID;
    if (max_hits < 1) max_hits = 1; // max(1, maxHits), CollisionQuery.swift:157
    if (max_hits > CQ_MAX_OVERLAP_HITS) {
        set_error("max_hits %d > %d", max_hits, CQ_MAX_OVERLAP_HITS);
        return CQ_ERR_INVALID;
    }
    return launch_overlap_all(w, d_q, n, max_hits, d_out, d_counts, d_overflow, pick_stream(w, stream));
}
int cq_move_and_slide_device_ex(cq_world *w, cq_character_state *d_inout, int32_t n, const cq_controller_params *params,
                                float dt, const float gravity[3], uint32_t flags, const cq_platform *platforms,
                                int32_t n_platforms, void *stream) {
    if (!w || n < 0 || !params || !gravity || (n > 0 && !d_inout)) return CQ_ERR_INVALID;
    return launch_move_and_slide(w, d_inout, n, *params, dt, gravity, flags, platforms, n_platforms, pick_stream(w, stream));
}
int cq_move_and_slide_device(cq_world *w, cq_character_state *d_inout, int32_t n, const cq_controller_params *params, float dt,
                             const float gravity[3], uint32_t flags, void *stream) {
    return cq_move_and_slide_device_ex(w, d_inout, n, params, dt, gravity, flags, nullptr, 0, stream);
}

int cq_raycast_batch_ex(cq_world *w, const cq_ray *rays, int32_t n, cq_ray_hit *out, uint8_t *flags) {
    if (!w || n < 0 || (n > 0 && (!rays || !out))) return CQ_ERR_INVALID;
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    return run_batch(w, rays, sizeof(cq_ray), out, sizeof(cq_ray_hit), n,
                     [&](void *di, void *dout, int cnt, int lo, cudaStream_t st) {
                         return launch_raycast(w, (const cq_ray *)di, cnt, (cq_ray_hit *)dout,
                                               flags ? (uint8_t *)w->aux2.ptr + lo : nullptr, st);
                     },
                     false, nullptr, false, flags);
}
int cq_raycast_batch(cq_world *w, const cq_ray *rays, int32_t n, cq_ray_hit *out) {
    return cq_raycast_batch_ex(w, rays, n, out, nullptr);
}

int cq_capsule_cast_batch_ex(cq_world *w, const cq_capsule_cast *q, int32_t n, int32_t mode, cq_cast_hit *out, uint8_t *flags) {
    if (!w || n < 0 || mode < 0 || mode > 2 || (n > 0 && (!q || !out))) return CQ_ERR_INVALID;
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    return run_batch(w, q, sizeof(cq_capsule_cast), out, sizeof(cq_cast_hit), n,
                     [&](void *di, void *dout, int cnt, int lo, cudaStream_t st) {
                         return launch_cast(w, (const cq_capsule_cast *)di, cnt, mode, (cq_cast_hit *)dout,
                                            flags ? (uint8_t *)w->aux2.ptr + lo : nullptr, st);
                     },
                     false, &w->hintCast, false, flags);
}
int cq_capsule_cast_batch(cq_world *w, const cq_capsule_cast *q, int32_t n, int32_t mode, cq_cast_hit *out) {
    return cq_capsule_cast_batch_ex(w, q, n, mode, out, nullptr);
}

int cq_capsule_overlap_batch_ex(cq_world *w, const cq_capsule *q, int32_t n, cq_overlap_hit *out, uint8_t *flags) {
    if (!w || n < 0 || (n > 0 && (!q || !out))) return CQ_ERR_INVALID;
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    return run_batch(w, q, sizeof(cq_capsule), out, sizeof(cq_overlap_hit), n,
                     [&](void *di, void *dout, int cnt, int lo, cudaStream_t st) {
                         return launch_overlap(w, (const cq_capsule *)di, cnt, (cq_overlap_hit *)dout,
                                               flags ? (uint8_t *)w->aux2.ptr + lo : nullptr, st);
                     },
                     false, nullptr, false, flags);
}
int cq_capsule_overlap_batch(cq_world *w, const cq_capsule *q, int32_t n, cq_overlap_hit *out) {
    return cq_capsule_overlap_batch_ex(w, q, n, out, nullptr);
}

int cq_capsule_overlap_all_batch(cq_world *w, const cq_capsule *q, int32_t n, int32_t max_hits, cq_overlap_hit *out,
                                 int32_t *counts, uint8_t *overflow) {
    if (!w || n < 0 || (n > 0 && (!q || !out || !counts))) return CQ_ERR_INVALID;
    if (max_hits < 1) max_hits = 1;
    if (max_hits > CQ_MAX_OVERLAP_HITS) {
        set_error("max_hits %d > %d", max_hits, CQ_MAX_OVERLAP_HITS);
        return CQ_ERR_INVALID;
    }
    if (n == 0) return CQ_OK;
    CQ_CUDA(cudaSetDevice(w->device));
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    cudaStream_t st = w->stream;
    int r;
    if ((r = ensure_scratch(w->in, sizeof(cq_capsule) * (size_t)n)) != CQ_OK) return r;
    if ((r = ensure_scratch(w->out, sizeof(cq_overlap_hit) * (size_t)n * max_hits)) != CQ_OK) return r;
    if ((r = ensure_scratch(w->aux, sizeof(int32_t) * (size_t)n)) != CQ_OK) return r;
    if ((r = ensure_scratch(w->aux2, (size_t)n)) != CQ_OK) return r;
    CQ_CUDA(cudaMemcpyAsync(w->in.ptr, q, sizeof(cq_capsule) * (size_t)n, cudaMemcpyHostToDevice, st));
    r = launch_overlap_all(w, (const cq_capsule *)w->in.ptr, n, max_hits, (cq_overlap_hit *)w->out.ptr, (int32_t *)w->aux.ptr,
                           (uint8_t *)w->aux2.ptr, st);
    if (r != CQ_OK) return r;
    CQ_CUDA(cudaMemcpyAsync(out, w->out.ptr, sizeof(cq_overlap_hit) * (size_t)n * max_hits, cudaMemcpyDeviceToHost, st));
    CQ_CUDA(cudaMemcpyAsync(counts, w->aux.ptr, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (overflow) CQ_CUDA(cudaMemcpyAsync(overflow, w->aux2.ptr, (size_t)n, cudaMemcpyDeviceToHost, st));
    CQ_CUDA(cudaStreamSynchronize(st));
    return CQ_OK;
}

int cq_move_and_slide_batch(cq_world *w, cq_character_state *inout, int32_t n, const cq_controller_params *params, float dt,
                            const float gravity[3], uint32_t flags) {
    return cq_move_and_slide_batch_ex(w, inout, n, params, dt, gravity, flags, nullptr, 0);
}

int cq_move_and_slide_batch_ex(cq_world *w, cq_character_state *inout, int32_t n, const cq_controller_params *params, float dt,
                               const float gravity[3], uint32_t flags, const cq_platform *platforms, int32_t n_platforms) {
    if (!w || n < 0 || !params || !gravity || (n > 0 && !inout)) return CQ_ERR_INVALID;
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    return run_batch(w, inout, sizeof(cq_character_state), inout, sizeof(cq_character_state), n,
                     [&](void *di, void *, int cnt, int, cudaStream_t st) {
                         return launch_move_and_slide(w, (cq_character_state *)di, cnt, *params, dt, gravity, flags, platforms,
                                                      n_platforms, st);
                     },
                     /*inPlace=*/true, &w->hintMas, /*singleChunk=*/(flags & CQ_MAS_AGENTS) != 0);
}

int cq_agent_separation_device(cq_world *w, cq_character_state *d_inout, int32_t n, const cq_controller_params *params,
                               const float *d_mass_weight, int32_t iterations, float separation_margin, float height_margin,
                               int32_t use_query, void *stream) {
    if (!w || n < 0 || !params || (n > 0 && !d_inout)) return CQ_ERR_INVALID;
    CQ_CUDA(cudaSetDevice(w->device));
    return launch_agent_separation(w, d_inout, n, *params, d_mass_weight, iterations, separation_margin, height_margin, use_query,
                                   pick_stream(w, stream));
}

int cq_agent_separation_batch(cq_world *w, cq_character_state *inout, int32_t n, const cq_controller_params *params,
                              const float *mass_weight, int32_t iterations, float separation_margin, float height_margin,
                              int32_t use_query) {
    if (!w || n < 0 || !params || (n > 0 && !inout)) return CQ_ERR_INVALID;
    if (n == 0) return CQ_OK;
    CQ_CUDA(cudaSetDevice(w->device));
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    int r;
    if ((r = ensure_scratch(w->in, sizeof(cq_character_state) * (size_t)n)) != CQ_OK) return r;
    if (mass_weight && (r = ensure_scratch(w->aux, sizeof(float) * (size_t)n)) != CQ_OK) return r;
    cudaStream_t st = w->stream;
    cq_character_state *d = (cq_character_state *)w->in.ptr;
    CQ_CUDA(cudaMemcpyAsync(d, inout, sizeof(cq_character_state) * (size_t)n, cudaMemcpyHostToDevice, st));
    if (mass_weight) CQ_CUDA(cudaMemcpyAsync(w->aux.ptr, mass_weight, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, st));
    r = launch_agent_separation(w, d, n, *params, mass_weight ? (const float *)w->aux.ptr : nullptr, iterations,
                                separation_margin, height_margin, use_query, st);
    if (r != CQ_OK) return r;
    CQ_CUDA(cudaMemcpyAsync(inout, d, sizeof(cq_character_state) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CQ_CUDA(cudaStreamSynchronize(st));
    return CQ_OK;
}

} // extern "C"
