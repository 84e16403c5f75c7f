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
    // reference order (cq_reftree.h -> attach_ref_order): the reference's own tree, for the ray walk and its refit
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
    int occ[6][4] = {}; // (raycast: [counting + 2 * reference-order walker]) // resident CTAs per SM of each persistent kernel ([counting + 2 * staged-walk variant])
    int numSms = 0;
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
    int occSep[2][2] = {};       // resident CTAs per SM of k_sep_turns / k_sep_post ([counting build])
    void *sepGraphs = nullptr;   // instantiated round-loop graphs of cq_agent_separation (cq_sep.cu: SepGraphCache)
    std::vector<cq::ScratchBuf *> held; // scratch blocks acquired by the launch being enqueued (release_held)
    // transform updates (cq_api.cu: update_transforms_on)
    std::unordered_map<uint32_t, std::vector<int>> partsOfEntity; // entity id -> parts with that id, in part order
    std::vector<int32_t> movedSlot;         // per part: its row in movedRows[set] during staging, else -1
    std::vector<cq::MovedPart> movedRows[2]; // the table being staged, per set
    cq::StageSlot stage[CQ_STAGE_SLOTS];
    uint32_t stageSeq = 0;
    cq::ScratchBuf dTable; // device copy of the staged table (read by the refit kernels of one update at a time)
    std::vector<void *> retiredDev, retiredHost; // outgrown table buffers a queued update may still use (cq_api.cu: free_retired)
    // Ordering of stream-ordered refits against every other launch on the world (await_trees / note_reader):
    std::vector<cq::ReaderEvent> readers; // per stream: the last launch that read the trees
    cudaEvent_t evTrees = nullptr;        // recorded after the last kernel of the latest asynchronous refit
    cudaStream_t treesStream = nullptr;   // ... on this stream
    bool treesPending = false;            // an asynchronous refit was queued and no synchronous call has waited for it since
};

namespace cq {
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
// after a synchronisation: has any kernel raised the world's status word since the last check?
int check_status(cq_world *w, const char *what);
// The world's scratch blocks (node stacks, unit order, agent grid, separation state) are shared by successive launches.
// Launches on ONE stream are ordered by the stream; a launch on ANOTHER stream must wait until the previous user of
// the block has finished.  scratch_acquire(b, st) inserts that wait and notes the block as held; the launcher calls
// release_held(w, st) once everything that touches its blocks is enqueued (records the completion events).
int scratch_acquire(cq_world *w, ScratchBuf &b, cudaStream_t st);
int release_held(cq_world *w, cudaStream_t st);
// First call of every launcher: a launch on `st` must see the trees the latest asynchronous refit writes, so `st` waits
// for that refit when it was queued on another stream.
int await_trees(const cq_world *w, cudaStream_t st);
// end of every launcher: pick up the launch error of the kernel just enqueued, release the held scratch blocks, and
// record that `st` has read the trees (the next asynchronous refit waits for it)
int finish_launch(cq_world *w, cudaStream_t st, const char *what);
#define CQ_WORK_RING 256
// zeroed work counter for the next persistent-kernel launch on `st` (nullptr on CUDA error)
int *next_work_counter(cq_world *w, cudaStream_t st);
// node-stack scratch for one persistent-kernel launch with `warps` warps (CQ_NSCAP uint2 entries per warp);
// four regions are used round-robin so that up to four launches on different streams run concurrently (a fifth
// waits for the first, see scratch_acquire).  nullptr on CUDA error.
void *pool_node_scratch(cq_world *w, size_t warps, cudaStream_t st);

// cq_build.cu
int build_set(cq_world *w, DeviceSet &S, const SetPlan &in /* upload plan of the set, cq_assemble.h */,
              std::vector<int> &partTriStart /* in: first input triangle of each part of the set (+ end); out: after the filter */,
              int *badTriangle /* out: smallest input triangle with an out-of-range index (CQ_ERR_INVALID), else -1 */,
              const int32_t *matIn = nullptr /* host, per INPUT triangle: row of the material table, or nullptr (row = part) */);
// Refit one set after its parts moved: dTab = the set's rows of the staged table on the device (rows = the same rows on
// the host, for the totals).  Stream-ordered on `st`; a fixed number of launches however many parts moved.
int refit_set(cq_world *w, DeviceSet &S, const MovedPart *dTab, const std::vector<MovedPart> &rows, cudaStream_t st);
// reference order: rebuild the reference's tree on the host from the set's triangle boxes, upload rank + tree (cq_reftree.h)
int attach_ref_order(cq_world *w);
void free_set(DeviceSet &S);
// Morton-sorted processing order of n work units whose position (3 floats or 3 doubles) sits at the start of each
// `stride`-byte record; nullptr when ordering is not worthwhile (small world / batch) or on error
// CQ_MAS_AGENTS pre-pass: snapshot (after the gravity rule), XZ grid, sort by cell.  Stream-ordered on `st`.
int make_agent_grid(cq_world *w, const cq_character_state *dStates, int n, float radius, float dt, const float g[3],
                    uint32_t flags, cudaStream_t st, AgentGrid &out);
const uint32_t *make_unit_order(cq_world *w, const void *dUnits, size_t stride, bool positionIsDouble, int n, cudaStream_t st);

// 32-bit key / value LSD radix sort (onesweep); `scratch` holds sort_scratch_words(n) words.  Result in (keys, vals).
size_t sort_scratch_words(int n);
int sort_pairs_u32(cq_world *w, uint32_t *keys, uint32_t *vals, uint32_t *keysTmp, uint32_t *valsTmp, int n, uint32_t *scratch,
                   size_t scratchWords, cudaStream_t st);

// cq_query.cu
// d_flags (may be nullptr): one CQ_HIT_* byte per query
int launch_raycast(cq_world *w, const cq_ray *d_rays, int n, cq_ray_hit *d_out, uint8_t *d_flags, cudaStream_t st);
int launch_cast(cq_world *w, const cq_capsule_cast *d_q, int n, int mode, cq_cast_hit *d_out, uint8_t *d_flags, cudaStream_t st);
int launch_overlap(cq_world *w, const cq_capsule *d_q, int n, cq_overlap_hit *d_out, uint8_t *d_flags, cudaStream_t st);
int launch_overlap_all(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                       uint8_t *d_overflow, cudaStream_t st);
// cq_mas.cu
int launch_move_and_slide(cq_world *w, cq_character_state *d_inout, int n, const cq_controller_params &p, float dt,
                          const float g[3], uint32_t flags, const cq_platform *platforms, int nPlatforms, cudaStream_t st);
// cq_sep.cu
void sep_graphs_destroy(cq_world *w);
int launch_agent_separation(cq_world *w, cq_character_state *d_inout, int n, const cq_controller_params &p,
                            const float *d_massWeight, int iterations, float sepMargin, float heightMargin, int useQuery,
                            cudaStream_t st);
} // namespace cq
