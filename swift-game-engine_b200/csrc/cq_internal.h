// cq_internal.h — host-side world representation shared by the .cu translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/cq.h"
#include "cq_assemble.h"
#include "cq_world.cuh"

namespace cq {

struct PartInfo {
    uint32_t entityId;
    int set;          // 0 static, 1 dynamic
    int vertLo, vertHi; // range in the set's vertex arrays
    int triLo, triHi;   // range in the set's FILTERED triangle numbering (slice, CollisionQuery.swift:404-409)
    cq_material material;
    uint32_t layer;
};

// One TriangleMeshSet (CollisionQuery.swift:320-470) resident in HBM.
struct DeviceSet {
    void *arena = nullptr; // one allocation holds every array below
    int nVerts = 0;
    int nTrisIn = 0; // before the degenerate filter
    int nTris = 0;   // after
    // vertex arrays
    float4 *localPos = nullptr; // (x,y,z, bits(part index))
    float4 *worldPos = nullptr; // (x,y,z,0)   = simd_mul(modelMatrix, (p,1))
    // triangle arrays in soup order (the reference's numbering)
    uint32_t *indices = nullptr;  // 3 per triangle, set-global vertex ids
    uint32_t *triLayer = nullptr;
    int32_t *triPart = nullptr;
    int32_t *triMat = nullptr; // per triangle: row of the material table, only when a part of the set has per-triangle materials (own allocation)
    // sorted (Morton) order
    uint32_t *sortedTri = nullptr; // slot -> soup triangle id
    float4 *tv0 = nullptr, *tv1 = nullptr, *tv2 = nullptr;
    // LBVH
    Node *nodes = nullptr;       // nTris-1 internal nodes (>= 1 allocated)
    Node4 *nodes4 = nullptr;     // 4-wide collapse of `nodes`, indexed by the binary node each was made from
    uint8_t *depthParity = nullptr; // per internal node: depth & 1
    int32_t *parent = nullptr;   // [0,nTris-1): internal, [nTris-1, 2nTris-1): leaves
    int32_t *rangeLo = nullptr, *rangeHi = nullptr; // per internal node
    float4 *boxLo = nullptr, *boxHi = nullptr;      // 2nTris-1 subtree boxes (bottom-up scratch, kept for refit)
    int32_t *visit = nullptr;    // per internal node arrival counter
    int32_t *expect = nullptr;   // dirty-subtree refit: dirty children per internal node (zero between refits)
    uint32_t *slotOfTri = nullptr; // soup triangle id -> slot of the sorted SoA
    SetHeader *hdr = nullptr;
    // reference order (attach_ref_order): the reference's own tree, for the ray walk and its refit
    void *refArena = nullptr;
    int nRefInternal = 0, nRefLeaves = 0, refDepth = 0;
    Node *refNodes = nullptr;          // internal nodes
    uint32_t *refSlot = nullptr;       // triOrder position -> sorted slot
    int32_t *refNodeParent = nullptr;  // per internal node: (parent << 1) | which child, -1 = root
    int32_t *refLeafParent = nullptr;  // per leaf: same encoding
    int32_t *refLeafRange = nullptr;   // per leaf: (start << 2) | (count - 1)
    int32_t *refVisit = nullptr;       // per internal node arrival counter (left at zero by every fit)
    int32_t *refExpect = nullptr;      // dirty-subtree refit: dirty children per internal node
    int32_t *refLeafMark = nullptr;    // dirty-subtree refit: per leaf, claimed by one of its updated triangles
    int32_t *refLeafOfTri = nullptr;   // soup triangle id -> leaf of the reference's tree
    SetHeader *refHdr = nullptr;
};

struct ScratchBuf {
    void *ptr = nullptr;
    size_t cap = 0;
    // cross-stream reuse guard (scratch_acquire / release_held): completion of the last launch that used the block
    cudaEvent_t ev = nullptr;
    cudaStream_t last = nullptr;
    bool recorded = false;
    bool captured = false; // a stream capture recorded this block's address: on growth it is kept, not freed (take_scratch)
};

// One row of the part table a transform update stages (cq_api.cu: update_transforms_on): a moved part of one set, its
// vertex and triangle ranges, and the running totals of both over the set's earlier rows (the refit kernels find a
// thread's row by binary search over them).  The table holds the static set's rows, then the dynamic set's.
struct MovedPart {
    int32_t part;             // index into the parts array (row of dModels)
    int32_t vertLo, triLo;    // first vertex / filtered triangle of the part in its set
    int32_t nVerts, nTris;
    int32_t vertBase, triBase; // sum of nVerts / nTris over the set's earlier rows
    int32_t _pad;
    float model[16];          // the new model matrix, column-major
};

// What the refit kernels of one update do to one set.  They read these counts on the device: the host-staged path copies
// them with its table, the device path (cq_world_update_transforms_device) has k_build_moved write them, so the same
// kernels serve both.  path: which of the two refits runs (the kernels of the other one exit at once).
#define CQ_PATH_NONE 0  // no part of the set moved
#define CQ_PATH_DIRTY 1 // the dirty-subtree refit
#define CQ_PATH_FULL 2  // regather + full fit
struct RefitCounts {
    int32_t nRows;  // rows of the set in the table
    int32_t nVerts; // sum of their nVerts
    int32_t nMoved; // sum of their nTris
    int32_t path;
};
// The header in front of a table of moved parts: both sets' counts.  generation / unknown are the device path's state
// (k_resolve_ids / k_build_moved); the host-staged path leaves them zero.
struct RefitHeader {
    RefitCounts set[2];
    uint32_t generation; // of the last device-path update: its last-writer words hold (generation << 32) | input index
    int32_t unknown;     // unknown ids counted by k_resolve_ids for the update being built (reset by k_build_moved)
    int32_t _pad[14];
};
static_assert(sizeof(RefitHeader) == sizeof(MovedPart), "the header takes one row of the staged table");

// Device entity index (cq_world_update_transforms_device): the sorted unique entity ids, CSR offsets into the entries of
// their parts that have triangles, and one entry per such part.
struct EntityEntry {
    int32_t part, set, vertLo, triLo, nVerts, nTris;
};

// Host side of one staged table: pinned memory, reused once the copy that read it has completed (event).
struct StageSlot {
    MovedPart *host = nullptr;
    size_t cap = 0; // rows
    cudaEvent_t ev = nullptr;
    bool recorded = false;
};

// Completion of the last launch on `st` that read the world's trees (finish_launch); `pending` until a refit waited on it.
struct ReaderEvent {
    cudaStream_t st = nullptr;
    cudaEvent_t ev = nullptr;
    bool pending = false;
};

} // namespace cq

#define CQ_PIPE_EVENTS 64
#define CQ_STAGE_SLOTS 4 // transform updates whose table copy may be in flight at once; a fifth waits for the oldest

struct cq_world {
    int device = 0;
    int order = CQ_ORDER_REFERENCE; // tie / overflow rule of every query (include/cq.h)
    int32_t *dRank = nullptr;       // reference order: global triangle index -> visiting rank
    uint32_t *dEncOfRank = nullptr; // reference order: visiting rank -> (set << 26) | sorted slot
    unsigned int *hStatus = nullptr; // status word, mapped host memory (WorldView::status is its device alias)
    float refBuildMs = 0;           // host time of the reference-order build (download + tree + upload)
    cudaStream_t stream = nullptr;
    cudaStream_t copyStream[2] = {nullptr, nullptr}; // the two alternating compute streams of the batch pipeline
    cudaStream_t h2dStream = nullptr, d2hStream = nullptr;
    cudaEvent_t evIn[CQ_PIPE_EVENTS] = {}, evDone[CQ_PIPE_EVENTS] = {};
    cudaEvent_t evA = nullptr, evB = nullptr;
    cq::DeviceSet set[2];
    std::vector<cq::PartInfo> parts;
    float *dModels = nullptr;    // nParts * 16
    float4 *dMaterials = nullptr; // nParts
    cq::WorldView view;
    float buildMs = 0, refitMs = 0;
    int counting = 0;
    int countRef = 0; // counting mode CQ_COUNT_REFERENCE
    // material table: one row per part, then the per-triangle rows of the parts that brought their own (triangleMaterials)
    std::vector<cq_material> hMaterials;
    std::vector<int32_t> hTriMat[2]; // host copy of DeviceSet::triMat (cq_world_triangle_material)
    unsigned long long *dCounters = nullptr; // 4 x u64: nodes, cands, evals, queries
    int numSms = 0; // SMs of `device`
    std::unordered_map<const void *, int> residentBlocks; // persistent kernel -> one resident wave of its CTAs (resident_blocks)
    uint64_t launches = 0;
    cq::ScratchBuf nodeScratch[4], orderScratch[4];
    uint32_t orderSeq = 0;
    uint32_t nodeSeq = 0;
    float hintMas = 0.0f, hintCast = 0.0f; // wall/PCIe ratio of the previous host-pointer call (chunking heuristic)
    int *dWork = nullptr; // ring of dynamic-fetch counters, one per persistent-kernel launch in flight
    uint32_t workSeq = 0;
    cq::ScratchBuf in, out, aux, aux2;
    cq::ScratchBuf agentScratch; // agent snapshot + grid of the move-and-slide call in flight (CQ_MAS_AGENTS)
    cq::ScratchBuf sepScratch;   // cq_agent_separation working set
    void *sepGraphs = nullptr;   // instantiated round-loop graphs of cq_agent_separation (cq_sep.cu: SepGraphCache)
    std::vector<cq::ScratchBuf *> held; // scratch blocks acquired by the launch being enqueued (release_held)
    // transform updates (cq_api.cu: update_transforms_on)
    std::unordered_map<uint32_t, std::vector<int>> partsOfEntity; // entity id -> parts with that id, in part order
    std::vector<int32_t> movedSlot;         // per part: its row in movedRows[set] during staging, else -1
    std::vector<cq::MovedPart> movedRows[2]; // the table being staged, per set
    cq::StageSlot stage[CQ_STAGE_SLOTS];
    uint32_t stageSeq = 0;
    cq::ScratchBuf dTable; // device copy of the staged table: a RefitHeader row, then the rows (one update at a time)
    // device path (cq_world_update_transforms_device), one allocation made at creation so that the call never allocates
    void *devArena = nullptr;
    uint32_t *dEntityIds = nullptr;         // nEntities sorted unique ids
    int32_t *dEntityOff = nullptr;          // nEntities + 1 offsets into dEntries
    cq::EntityEntry *dEntries = nullptr;    // parts with triangles, grouped by entity, in part order
    unsigned long long *dLastWriter = nullptr; // per part: (generation << 32) | index of the input that claimed it last
    cq::RefitHeader *dDevHdr = nullptr;     // counts, generation and unknown-id count of the device path
    cq::MovedPart *dDevTable = nullptr;     // static set's rows at [0, devRows0), dynamic set's after
    int nEntities = 0, devRows0 = 0;
    // a device call is being recorded into a stream capture (CaptureScope, cq_api.cu): no world event is waited on,
    // recorded or created, and scratch must not grow (take_scratch refuses)
    bool capturing = false;
    std::vector<void *> graphScratch; // outgrown scratch blocks that captured graphs may still use: freed by cq_world_destroy
    std::vector<void *> retiredDev, retiredHost; // outgrown table buffers a queued update may still use (cq_api.cu: free_retired)
    // Ordering of stream-ordered refits against every other launch on the world (await_trees / note_reader):
    std::vector<cq::ReaderEvent> readers; // per stream: the last launch that read the trees
    cudaEvent_t evTrees = nullptr;        // recorded after the last kernel of the latest asynchronous refit
    cudaStream_t treesStream = nullptr;   // ... on this stream
    bool treesPending = false;            // an asynchronous refit was queued and no synchronous call has waited for it since
};

namespace cq {
inline int cdiv(int a, int b) { return (a + b - 1) / b; }
void set_error(const char *fmt, ...);
int check_cuda(cudaError_t e, const char *what);
#define CQ_CUDA(x)                                        \
    do {                                                  \
        int _r = cq::check_cuda((x), #x);                 \
        if (_r != CQ_OK) return _r;                       \
    } while (0)

#define CQ_TRY(x)                  \
    do {                           \
        int _r = (x);              \
        if (_r != CQ_OK) return _r; \
    } while (0)

int ensure_scratch(ScratchBuf &b, size_t bytes);
// CTAs of `kernel` (`threads` per CTA, `dynSmem` bytes of dynamic shared memory) that fit on the device at once: SMs x
// resident CTAs per SM (at least one per SM), cached per world.  dynSmem > 0 also raises the kernel's dynamic shared-memory
// limit to dynSmem.  0 on CUDA error.
int resident_blocks(cq_world *w, const void *kernel, int threads, size_t dynSmem);
// Chunk count of the copy/compute pipeline of a host-pointer call over n units (CQ_CHUNK sets the units per chunk): two
// chunks only when the previous call's wall / PCIe-time ratio `hint` was above `computeBoundAbove`, because every chunk
// kernel pays its own tail; at most CQ_PIPE_EVENTS; one when `singleChunk` (the units interact).
int pipeline_chunks(int n, float hint, float computeBoundAbove, bool singleChunk);
// after a synchronisation: has any kernel raised the world's status word since the last check?
int check_status(cq_world *w, const char *what);
// The world's scratch blocks (node stacks, unit order, agent grid, separation state) are shared by successive launches.
// Launches on ONE stream are ordered by the stream; a launch on ANOTHER stream must wait until the previous user of
// the block has finished.  scratch_acquire(b, st) inserts that wait and notes the block as held; the launcher calls
// release_held(w, st) once everything that touches its blocks is enqueued (records the completion events).
int scratch_acquire(cq_world *w, ScratchBuf &b, cudaStream_t st);
int release_held(cq_world *w, cudaStream_t st);
// The only code that grows the scratch a launch uses: takes ring[use] of the nRing blocks of `ring` (one block, or a ring
// of four used round-robin so that up to four launches on different streams run concurrently; a fifth waits for the
// first) for a launch on `st` and returns its address in *ptr.  A block smaller than `bytes` is refused under capture (CQ_ERR_INVALID, naming `what`;
// nothing is enqueued and the capture stays valid); uncaptured, all nRing blocks grow together after one device
// synchronisation, and a block whose address a graph recorded (ScratchBuf::captured) is moved to w->graphScratch instead
// of being freed, so replays stay valid.  Under capture the block is marked captured; then it is acquired for `st`.
int take_scratch(cq_world *w, ScratchBuf *ring, int nRing, int use, size_t bytes, cudaStream_t st, const char *what, void **ptr);
// First call of every launcher: a launch on `st` must see the trees the latest asynchronous refit writes, so `st` waits
// for that refit when it was queued on another stream.
int await_trees(const cq_world *w, cudaStream_t st);
// end of every launcher: pick up the launch error of the kernel just enqueued, release the held scratch blocks, and
// record that `st` has read the trees (the next asynchronous refit waits for it)
int finish_launch(cq_world *w, cudaStream_t st, const char *what);
#define CQ_WORK_RING 256
// zeroed work counter for the next persistent-kernel launch on `st` (nullptr on CUDA error)
int *next_work_counter(cq_world *w, cudaStream_t st);

// cq_build.cu
int build_set(cq_world *w, DeviceSet &S, const SetPlan &in /* upload plan of the set, cq_assemble.h */,
              std::vector<int> &partTriStart /* in: first input triangle of each part of the set (+ end); out: after the filter */,
              int *badTriangle /* out: smallest input triangle with an out-of-range index (CQ_ERR_INVALID), else -1 */,
              const int32_t *matIn = nullptr /* host, per INPUT triangle: row of the material table, or nullptr (row = part) */);
// Refit one set after its parts moved: dTab = the set's rows of the table on the device, counts = the set's RefitCounts
// on the device (every kernel reads its counts and path there).  rows = the same rows on the host (host-staged path):
// only the chosen path is launched, with exact grids.  rows == nullptr (device path): the host knows no counts, so both
// paths are launched with grids sized from the set's own vertex / triangle counts and the unchosen one exits at once.
// Stream-ordered on `st`; a fixed number of launches however many parts moved.
int refit_set(cq_world *w, DeviceSet &S, const MovedPart *dTab, const RefitCounts *counts, const std::vector<MovedPart> *rows,
              cudaStream_t st);
// the path the host-staged update takes for a set of which `moved` triangles moved (CQ_PATH_*)
int refit_path(const DeviceSet &S, int moved);
// Device path of cq_world_update_transforms_device: resolve the ids and build the table + counts on `st` (2 launches).
int build_moved_device(cq_world *w, const uint32_t *dIds, const float *dModels, int n, int32_t *dStatus, cudaStream_t st);
// cq_world_platforms_device: n > 0 platform records from the world-space vertices of the named entities, one launch on `st`.
int launch_platform_records(cq_world *w, const uint32_t *dIds, const float *dDeltas, int n, cq_platform *dOut, int32_t *dStatus,
                            cudaStream_t st);
// a stream capture is recording `st` (cudaStreamGetCaptureInfo)
bool stream_capturing(cudaStream_t st);
// Calls that synchronise, allocate, create events or stage host memory: CQ_ERR_INVALID while `st` is capturing (the
// capture stays valid), else CQ_OK.
int refuse_capture(cudaStream_t st, const char *what);
#define CQ_NO_CAPTURE(st, what) CQ_TRY(cq::refuse_capture((st), (what)))
// reference order: cut the reference's tree of each set on the device from its triangle boxes; ranks + tree (cq_build.cu)
int attach_ref_order(cq_world *w);
void free_set(DeviceSet &S);
// Morton-sorted processing order of n work units whose position (3 floats or 3 doubles) sits at the start of each
// `stride`-byte record.  take_unit_order takes the order's scratch for `st` (take_scratch); *scratch = nullptr when
// ordering is not worthwhile (small world / batch).  make_unit_order enqueues the keys and the sort into that scratch on
// `st` and returns the order in *order (nullptr when scratch is).
int take_unit_order(cq_world *w, int n, cudaStream_t st, uint32_t **scratch);
int make_unit_order(cq_world *w, uint32_t *scratch, const void *dUnits, size_t stride, bool positionIsDouble, int n,
                    cudaStream_t st, const uint32_t **order);
// CQ_MAS_AGENTS pre-pass of a launch that moves n characters, agents first .. first + n - 1 of a crowd of nAgents.
// take_agent_grid takes the grid's scratch for `st` (take_scratch): sort side nAgents-sized, per-character rows n-sized,
// plus room for the snapshot when the launch takes its own (ownSnapshot: the single-batch step, first = 0, nAgents = n).
// make_agent_grid enqueues on `st`: the snapshot of dStates (after the gravity rule) into that scratch when dAgents is
// nullptr, else the bounds of the snapshot dAgents; then the XZ grid and sort by cell over all nAgents, and the cell
// ranges of the n moving characters.
int take_agent_grid(cq_world *w, int nAgents, int n, bool ownSnapshot, cudaStream_t st, void **scratch);
int make_agent_grid(cq_world *w, void *scratch, const cq_character_state *dStates, const cq_agent_snapshot *dAgents, int nAgents,
                    int first, int n, float radius, float dt, const float g[3], uint32_t flags, cudaStream_t st, AgentGrid &out);
// cq_agent_snapshot_device: n > 0 snapshot records of dStates into dOut, one launch on `st`
int launch_agent_snapshot(cq_world *w, const cq_character_state *dStates, int n, float dt, const float g[3], uint32_t flags,
                          cq_agent_snapshot *dOut, cudaStream_t st);

// 32-bit key / value LSD radix sort (onesweep); `scratch` holds sort_scratch_words(n) words.  Result in (keys, vals).
size_t sort_scratch_words(int n);
int sort_pairs_u32(cq_world *w, uint32_t *keys, uint32_t *vals, uint32_t *keysTmp, uint32_t *valsTmp, int n, uint32_t *scratch,
                   size_t scratchWords, cudaStream_t st);

// cq_query.cu
// What pool_launch_setup gives one launch of a persistent pair-pool kernel.
struct PoolLaunch {
    int blocks = 0;                  // CTAs: one resident wave at most
    int ownersPerWarp = 0;           // pool_owners_per_warp
    uint2 *nodeScratch = nullptr;    // CQ_NSCAP node-stack entries per warp
    int *work = nullptr;             // the zeroed dynamic-fetch counter
    const uint32_t *order = nullptr; // unit order, nullptr = the units' own order
};
// The prologue of every pool-kernel launch of n units on `st`: await_trees; blocks = min(cdiv(n, unitsPerCta), one
// resident wave of `kernel` at `threads` threads and `smem` bytes of dynamic shared memory); owners per warp over
// blocks * threads / 32 warps.  It first takes every scratch block the launch needs (node stacks when `nodeScratch`, the
// unit order's when `units` is non-null: records of `stride` bytes, see make_unit_order), so a refused call enqueues
// nothing, and only then enqueues the work-counter memset and the unit order's keys and sort.
int pool_launch_setup(cq_world *w, const void *kernel, int threads, size_t smem, int unitsPerCta, int n, bool nodeScratch,
                      const void *units, size_t stride, bool positionIsDouble, cudaStream_t st, PoolLaunch &out);
// d_flags (may be nullptr): one CQ_HIT_* byte per query
int launch_raycast(cq_world *w, const cq_ray *d_rays, int n, cq_ray_hit *d_out, uint8_t *d_flags, cudaStream_t st);
int launch_cast(cq_world *w, const cq_capsule_cast *d_q, int n, int mode, cq_cast_hit *d_out, uint8_t *d_flags, cudaStream_t st);
int launch_overlap(cq_world *w, const cq_capsule *d_q, int n, cq_overlap_hit *d_out, uint8_t *d_flags, cudaStream_t st);
int launch_overlap_all(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                       uint8_t *d_overflow, cudaStream_t st);
// cq_mas.cu
// Kinematic platforms come either as a host array `platforms` (at most 64, copied into the kernel arguments, so a captured
// graph keeps them) or, when dPlatforms is non-null, as a device array the kernels read when they execute (any count).
// CQ_MAS_AGENTS: dAgents = nullptr makes the batch the crowd; otherwise the batch is agents first .. first + n - 1 of
// the nAgents-record snapshot dAgents.
int launch_move_and_slide(cq_world *w, cq_character_state *d_inout, int n, const cq_controller_params &p, float dt,
                          const float g[3], uint32_t flags, const cq_platform *platforms, const cq_platform *dPlatforms,
                          int nPlatforms, cudaStream_t st, const cq_agent_snapshot *dAgents = nullptr, int nAgents = 0,
                          int first = 0);
// cq_sep.cu
void sep_graphs_destroy(cq_world *w);
// Queues the whole separation on `st` without waiting for the device; the outcome goes to d_status (may be nullptr).
int launch_agent_separation(cq_world *w, cq_character_state *d_inout, int n, const cq_controller_params &p,
                            const float *d_massWeight, int iterations, float sepMargin, float heightMargin, int useQuery,
                            int32_t *d_status, cudaStream_t st);
// The synchronous calls: waits for the separation just queued on `st` and turns its outcome into an error code.
int wait_agent_separation(cq_world *w, int n, const cq_controller_params &p, float sepMargin, cudaStream_t st);
} // namespace cq
