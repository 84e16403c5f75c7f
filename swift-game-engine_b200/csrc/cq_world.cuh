// cq_world.cuh — device-side world layout (triangle SoA, LBVH nodes, views) and small helpers shared by
// the query kernels (cq_pool.cuh, cq_query.cu, cq_mas.cu).
//
// HBM layout of one triangle set (static or dynamic, CollisionQuery.swift:710-711):
//   tv0/tv1/tv2 : float4 SoA, one entry per triangle in MORTON (leaf) order
//        tv0 = (v0.xyz, bits(layer))      tv1 = (v1.xyz, bits(triangle id in the filtered soup))
//        tv2 = (v2.xyz, bits(visiting rank)) — the global position of the triangle in the order rule of the world:
//              the reference's depth-first visiting rank (CQ_ORDER_REFERENCE) or simply its global index (canonical).
//              Exact ties go to the smaller rank; it travels with the triangle so that no query ever loads it separately.
//   nodes       : 64-byte LBVH node = the AABBs of BOTH children + their references, so one
//                 node fetch (4 x LDG.128) tests two boxes:
//        n0 = (lo0.xyz, bits(ref0))  n1 = (hi0.xyz, bits(ref1))  n2 = (lo1.xyz, -)  n3 = (hi1.xyz, -)
//        ref >= 0 : internal node index;  ref < 0 : leaf range, ~ref = (start << 2) | (count - 1),
//        1..4 consecutive triangles of the sorted SoA (subtrees with <= 4 triangles are
//        collapsed, mirroring the reference's leafTriangleLimit = 4, CollisionQuery.swift:473).
//   header      : root reference + root box, kept in device memory so a refit needs no host sync.
#pragma once
#include "cq_math.cuh"

namespace cq {

#define CQ_REF_EMPTY 0x7fffffff
#define CQ_STACK 64

struct __align__(16) Node {
    float4 n0, n1, n2, n3;
};

// 4-wide node used by the cooperative walk: the binary LBVH collapsed two levels at a time (every internal
// node at even depth absorbs its internal children), so a query descends half as many levels — and the walk
// rounds are latency bound on exactly that dependent chain of node fetches.  128 bytes:
//   q[0] = (lo0, ref0) q[1] = (hi0, ref1) q[2] = (lo1, ref2) q[3] = (hi1, ref3) q[4..7] = lo2 hi2 lo3 hi3
// ref >= 0: wide node index (= index of the binary node it was made from); ref < 0: leaf range as in Node;
// CQ_REF_EMPTY: unused child (its box is inverted, so it never overlaps anything).
struct __align__(16) Node4 {
    float4 q[8];
};

struct __align__(16) SetHeader {
    float lo[3];
    int rootRef; // CQ_REF_EMPTY when the set has no triangles
    float hi[3];
    int nTris;
};

struct SetView {
    const float4 *tv0, *tv1, *tv2;
    const Node *nodes;
    const Node4 *nodes4;
    const SetHeader *hdr;
    const int32_t *triPart; // per triangle of the set (soup numbering): index of the part (entity) it came from -> material
    const int32_t *triMat;  // per triangle: row of the material table, or nullptr = the part's own row (no per-triangle materials)
    int triOffset; // added to triangle ids of this set (dynamic set: static count, CollisionQuery.swift:782)
    // Reference order only (attach_ref_order): the reference's own median-split tree as 64-byte nodes (child 0 = left,
    // child 1 = right; a leaf reference ~((start << 2) | (count - 1)) names positions of refSlot), walked by the ray
    // kernel exactly as CollisionQuery.swift:916-978 walks it.  refSlot: triOrder position -> slot of the sorted SoA.
    const Node *refNodes;
    const uint32_t *refSlot;
    const SetHeader *refHdr;
};

struct WorldView {
    SetView set[2];
    const float4 *materials; // (muS, muK, flattenGround, -): one row per part, then the rows of per-triangle materials
    int nParts;
    int nMaterials;
    // Visiting rank of every triangle (global triangle index -> position in the reference's depth-first order, static
    // set first), or nullptr in canonical order, where the rank of a triangle is its index.  Exact ties (equal toi /
    // depth) go to the smaller rank; capsuleOverlapAll keeps the maxHits smallest ranks (CollisionQuery.swift:1272-1274).
    const int32_t *rank;
    const uint32_t *encOfRank; // reference order: visiting rank -> (set << 26) | slot of the sorted SoA (a pair-ring entry)
    // Device-visible status word in mapped host memory (zero = fine).  Bit 0: a warp's node stack would have overflowed
    // (cq_pool.cuh) — the launch's results are incomplete; the next synchronising call reports CQ_ERR_CUDA.
    unsigned int *status;
    int refStats;     // counting launches only (CQ_COUNT_REFERENCE): no bestT-based culling, `candidates` = capsuleCandidateCount
    int stagedLeaves; // which kernel variant the launchers pick: 1 = walk expands leaf ranges one triangle per lane
                      // (worlds that do not fit L1); the tiny-world variant keeps the shorter per-lane loop
};

// Snapshot of every agent of a crowd, taken before any character of the step moves (collectAgentStates,
// Systems.swift:1592-1611; one cq_agent_snapshot per agent), binned into a uniform XZ grid and sorted by cell key.  The
// launch moves characters 0..n) of its batch, which are agents first .. first + n - 1 of the crowd: the whole crowd when
// first = 0 and the grid holds n agents, one slice of it otherwise.
struct AgentGridParams { // written by k_agent_grid_params, read by the move-and-slide kernel
    float originX, originZ, invCell, cell;
    int dimX, dimZ;
    float maxSpeed; // max |velocity| over the snapshot
    float _pad;
};
struct AgentGrid {
    const float4 *pos;  // sorted by cell key; w = original index (bits)
    const float4 *vel;  // same order
    const uint32_t *keys; // sorted cell keys: iz * dimX + ix
    const AgentGridParams *params;
    const int4 *rows; // per character of the launch, 2 x int4: (start,end) in the sorted arrays of the cells ix-1..ix+1 of
                      // the rows iz-1, iz, iz+1 around its snapshot cell, then (ix, iz) -- found once, in parallel
    float4 *firstHit; // per character of the launch: (normal, toi) of the agent hit of the FIRST slide iteration, computed
                      // by a pre-pass under the assumption that depenetration does not move the character; toi -1 = none
    int n;            // agents in the grid
    int first;        // agent index of the launch's character 0
};
__device__ __forceinline__ int agent_cell(float x, float origin, float invCell, int dim) { // monotonic in x
    float c = floorf((x - origin) * invCell);
    return (int)fminf(fmaxf(c, 0.0f), (float)(dim - 1));
}

struct Counters { // per-thread work counters, flushed with atomics when COUNT
    uint32_t nodes, cands, evals, queries;
};

__device__ __forceinline__ bool box_disjoint(f3 lo, f3 hi, f3 qlo, f3 qhi) { // CollisionQuery.swift:1047-1049
    return hi.x < qlo.x || lo.x > qhi.x || hi.y < qlo.y || lo.y > qhi.y || hi.z < qlo.z || lo.z > qhi.z;
}

__device__ __forceinline__ Tri load_tri(const SetView &s, int i, uint32_t &layer, int &triId, int &rank) {
    float4 a = __ldg(s.tv0 + i), b = __ldg(s.tv1 + i), c = __ldg(s.tv2 + i);
    layer = __float_as_uint(a.w);
    triId = __float_as_int(b.w);
    rank = __float_as_int(c.w);
    return Tri{xyz(a), xyz(b), xyz(c)};
}

// row of the material table of a global triangle index (TriangleMeshSet.triangleMaterials[index], :464-469), -1 = default
__device__ __forceinline__ int world_material_row(const WorldView &W, int gid) {
    if (gid < 0) return -1;
    const int off = W.set[1].triOffset;
    const SetView &S = gid >= off ? W.set[1] : W.set[0];
    const int local = gid >= off ? gid - off : gid;
    return S.triMat ? __ldg(S.triMat + local) : __ldg(S.triPart + local);
}

#define CQ_MODE_ALL 0
#define CQ_MODE_BLOCKING 1
#define CQ_MODE_GROUND 2

// ---------------------------------------------------------------- capsule overlap
struct OverlapRec {
    float depth;
    f3 position, normal, triNormal;
    int tri, part;
};

__device__ __forceinline__ void overlap_box(f3 from, float radius, float hh, f3 &qlo, f3 &qhi) { // :1126-1133
    const f3 up = {0.0f, 1.0f, 0.0f};
    f3 a0 = from + up * hh, b0 = from - up * hh;
    f3 ext = {radius, radius, radius};
    qlo = vmin(a0, b0) - ext;
    qhi = vmax(a0, b0) + ext;
}

// contact record of one overlapping triangle — CollisionQuery.swift:1165-1190
__device__ __forceinline__ void overlap_contact(const Tri &T, float dist, f3 segPt, f3 triPt, float radius,
                                                OverlapRec &r) {
    f3 triNormal = normalize(cross(T.v1 - T.v0, T.v2 - T.v0));
    f3 n = dist < 1e-6f ? triNormal : normalize(segPt - triPt);
    f3 triN = triNormal;
    if (dot(triN, n) < 0.0f) triN = -triN;
    r.depth = radius - dist;
    r.position = triPt;
    r.normal = n;
    r.triNormal = triN;
}

// ---------------------------------------------------------------- raycast
// rayAABB — CollisionQuery.swift:1603-1631 — made conservative: the box is accepted when the slab
// interval, widened by a few ulps, is non-empty and starts before closestT.  The reference's own
// slab test is not conservative in floating point, so which grazing hits it culls depends on its
// tree; this library defines the result as the minimum-t triangle over ALL triangles (ties ->
// smallest index) and only uses the boxes to skip work (SURVEY.md §A.4-2).
__device__ __forceinline__ bool ray_box(f3 o, f3 inv, f3 lo, f3 hi, float closestT) {
    // spatial pad: a float Moller-Trumbore hit can sit a few ulps outside the triangle's box
    float ex = 2e-6f * (fabsf(o.x) + fmaxf(fabsf(lo.x), fabsf(hi.x))) + 1e-7f;
    float ey = 2e-6f * (fabsf(o.y) + fmaxf(fabsf(lo.y), fabsf(hi.y))) + 1e-7f;
    float ez = 2e-6f * (fabsf(o.z) + fmaxf(fabsf(lo.z), fabsf(hi.z))) + 1e-7f;
    float t0x = ((lo.x - ex) - o.x) * inv.x, t1x = ((hi.x + ex) - o.x) * inv.x;
    float t0y = ((lo.y - ey) - o.y) * inv.y, t1y = ((hi.y + ey) - o.y) * inv.y;
    float t0z = ((lo.z - ez) - o.z) * inv.z, t1z = ((hi.z + ez) - o.z) * inv.z;
    float tmin = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fminf(t0z, t1z));
    float tmax = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fmaxf(t0z, t1z));
    float pad = 1e-6f + 1e-6f * fmaxf(fabsf(tmin), fabsf(tmax)); // + a relative pad on the interval itself
    if (tmin - pad > tmax + pad) return false;
    if (tmax + pad < 0.0f) return false; // rayTriangle needs t >= 0
    return tmin - pad <= closestT;
}

} // namespace cq
