// cq_pool.cuh — warp-cooperative query engine: owners post queries, the warp's 32 lanes share the
// (query, candidate-triangle) work items.
//
// Measured facts that shape this file (B200, ncu; profiles/):
//  * thread-per-query with nested loops runs 2.0 of 32 lanes (v1);
//  * a flat per-lane state machine fixes the nesting but not the WORKLOAD skew: distance evaluations per
//    character-step are median 29-37 / p99 ~1000 (hulls) and median 29 / p99 ~36,000 (render mesh) — a
//    character that touches geometry sweeps tens of "creeping" candidates for up to L/minAdvance trips
//    each, exactly as the reference does (CollisionQuery.swift:1295-1356).  One lane per character then
//    leaves most of the warp idle.
// So the unit of scheduling here is one (query, candidate) PAIR, not a query and not a character:
//  * each lane is the OWNER of one work unit (a character / a batch query): it runs the unit's serial
//    logic, walks the LBVH for the unit's current query and pushes every candidate triangle into a
//    per-warp ring in shared memory;
//  * every lane is also an EXECUTOR: it takes any pair from the ring, runs its conservative
//    advancement one distance evaluation per trip of the main loop, and commits the contact to the
//    owner's record.  The best accepted toi of the query is shared, so the exact-safe prune
//    `lastSafeT > bestT` (SURVEY.md §A.4-3) works across lanes;
//  * a query completes when its walk is finished and its pending-pair counter is back to zero.
// The main loop is: [front end, only when the ring is dry and enough lanes idle: owner logic -> cooperative walk /
// push] -> job pickup (ballot ranked; query kernels drop candidates that cannot matter) -> ONE distance
// evaluation on every lane that holds a pair -> commit per owner (warp reductions / grouped rounds, pool_commit)
// -> warp-uniform exit test.
// Results are deterministic: a cast's answer is the accepted pair with the smallest (toi, visiting rank), an
// order-free reduction, whatever the order in which the lanes finish.
#pragma once
#include "../../include/cq.h"
#include "cq_world.cuh"

namespace cq {

enum { PH_NONE = 0, PH_ADV = 1, PH_BIS = 2, PH_FIN = 3, PH_OVL = 4 };
#define CQ_KIND_OVERLAP 3 /* query mode: two-deepest overlap (move-and-slide depenetration) */
#define CQ_QCAP 256       /* pair-ring entries per warp */
#ifndef CQ_WALK_FILL /* walk rounds run until the pair ring holds this many pairs.  Swept on one box after the slim pair state
                        (profiles/r2_ab_same_box.txt, call 20; 96 everywhere before): the move-and-slide kernels gain 0.3-0.8% with a
                        fuller ring (a round always leaves room for 128 more, so 160 means "up to 128"), the query kernels
                        2.8% on C2 with a shorter one (fresher bestT for the culling of the next walk rounds; C4 unchanged) */
#define CQ_WALK_FILL (LOOKAHEAD ? 64 : 160)
#endif
#define CQ_NSCAP 2048     /* node-stack entries per warp (global memory; 32 concurrent walks) */
// Stack budget.  A walk round with 32 poppers grows the stack by at most 32 x (4 - 1) = 96 entries; posting roots adds at
// most 32 owners x 2 sets = 64.  Above CQ_NS_WIDE only ONE lane pops per round (depth-first), which grows the stack by
// at most 3 per level below the popped entry: CQ_NS_DFS_RESERVE covers 48 four-wide levels (a binary LBVH over 2^26
// triangles with 30-bit keys + index tie-breaks is at most 56 levels = 28 wide ones).  Owners post new queries only
// below CQ_NS_POST.  Should a lone popper still not find room, the walk round drops the children and raises the world's
// status word (one warp-uniform test per round, nothing per push).
#define CQ_NS_DFS_RESERVE 144
#define CQ_NS_WIDE (CQ_NSCAP - CQ_NS_DFS_RESERVE - 96)
#define CQ_NS_POST (CQ_NS_WIDE - 64)

struct QShared { // one per owner lane, shared memory: what executors need + the query's result
    float from[3], radius, hh;
    // sweeps only.  An overlap query of the move-and-slide kernel reuses these ten words (ovl_words): the eight smallest
    // visiting ranks seen, the number of overlapping triangles, and the rank limit of a second pass (reference order).
    float dir[3], delta[3], L, minNormalY, minAdvance;
    int maxIter;
    int mode; // low byte: CQ_MODE_* / CQ_KIND_OVERLAP; CQ_QF_* flags above it
    float qlo[3], qhi[3]; // the query's (swept) AABB: node / triangle boxes are tested against it
    uint32_t mask;
    // result.  cast: rT/rTri/rPart + contact.  overlap: two deepest, d0=rT t0=rTri n0=rN | d1=rPos[0] t1=rPart n1=rTriN
    float rT;
    int rTri, rPart;
    int rRank, rRank1; // visiting rank of rTri (and, overlap queries, of the second deepest rPart): exact ties go to the smaller
    float rPos[3], rN[3], rTriN[3];
    int pending; // stack entries + pairs pushed for this query and not yet consumed; 0 = query complete
};

#define CQ_QF_TIE 0x100 /* another accepted candidate had exactly the best key: the answer depended on the order rule */
__device__ __forceinline__ int *ovl_words(QShared &s) { return reinterpret_cast<int *>(s.dir); }
// ovl_words: [0..7] the eight smallest ranks seen so far (unsorted), [8] overlapping triangles counted (-1 = second pass: nothing
// is counted or kept), [9] the largest of the eight kept ranks (valid once eight are kept)
enum { OVL_TOTAL = 8, OVL_MAXRANK = 9 };

struct QResult { // what owner logic reads back
    float bestT;
    int bestTri, bestPart;
    f3 bestPos, bestN, bestTriN;
};

struct Job { // executor-side pair state (registers)
    // Everything here stays live across the distance function, whose own working set fills the register file: values
    // that are only needed between evaluations (|delta|, minAdvance, maxIter) are re-read from the owner's QShared, and
    // the phases share slots — round 2's terrain capture showed 11% of the stall samples on reloads of spilled pair state
    // that the node / triangle traffic had evicted from L1 (profiles/r2_by_region_midround.txt).
    int phase;
    uint32_t enc; // ring entry (owner | set | slot): lets an owner reload a winning triangle later
    float radius, hh;
    Tri T;
    int gid, rank;      // global triangle index; visiting rank (tv2.w)
    float t, lastSafeT; // PH_ADV: conservative advancement.  PH_BIS / PH_FIN: refineTOI's hi (in t) and lo (in lastSafeT)
    int it;             // PH_ADV: iterations done.  PH_BIS: bisection steps done
    __device__ __forceinline__ int owner() const { return (int)(enc >> 27); }
};

struct Commit { // a finished pair's contribution, applied in the serialized commit step
    int kind; // 0 none, 1 cast contact, 2 overlap
    float key;
    f3 pos, n, triN;
};

struct WarpPool { // per-warp handles
    QShared *qs;             // [32]                shared
    uint32_t *ring;          // [CQ_QCAP] pairs     shared
    volatile uint32_t *head; // pairs consumed      shared
    volatile uint32_t *tail; // pairs produced      shared
    volatile uint32_t *ntop; // node-stack height   shared
    volatile uint32_t *fePasses; // front-end passes of this launch (watchdog)   shared
    uint2 *nstack;           // [CQ_NSCAP] (owner<<2 | set<<1 | isLeaf, ref)   global (L2 resident)
    uint32_t *stage;         // [CQ_STAGE] triangles of the leaf ranges popped in this walk round   shared
    const int32_t *rank;     // visiting rank per global triangle index (reference order) or nullptr (rank = index)
    unsigned int *status;    // the world's status word (mapped host memory)
};

__device__ __forceinline__ int pool_rank(const int32_t *rank, int gid) { return rank ? __ldg(rank + gid) : gid; }
#define CQ_STAGE 128 /* 32 leaf ranges x <= 4 triangles */
#define CQ_POOL_WORDS (CQ_QCAP + 4 + CQ_STAGE) /* shared words per warp besides QShared */

__device__ __forceinline__ void pool_bind(WarpPool &wp, QShared *qsAll, uint32_t *words, uint2 *nodeScratch, int warp,
                                          int warpsPerBlock, const int32_t *rank, unsigned int *status) {
    wp.qs = qsAll + warp * 32;
    wp.ring = words + warp * CQ_POOL_WORDS;
    wp.head = wp.ring + CQ_QCAP;
    wp.tail = wp.ring + CQ_QCAP + 1;
    wp.ntop = wp.ring + CQ_QCAP + 2;
    wp.fePasses = wp.ring + CQ_QCAP + 3;
    wp.stage = wp.ring + CQ_QCAP + 4;
    wp.nstack = nodeScratch + ((size_t)blockIdx.x * warpsPerBlock + warp) * CQ_NSCAP;
    wp.rank = rank;
    wp.status = status;
}

__device__ __forceinline__ void pool_read_result(const QShared &s, QResult &r) {
    r.bestT = s.rT;
    r.bestTri = s.rTri;
    r.bestPart = s.rPart;
    r.bestPos = mk3(s.rPos[0], s.rPos[1], s.rPos[2]);
    r.bestN = mk3(s.rN[0], s.rN[1], s.rN[2]);
    r.bestTriN = mk3(s.rTriN[0], s.rTriN[1], s.rTriN[2]);
}

__device__ __forceinline__ void store3s(float *o, f3 v) {
    o[0] = v.x;
    o[1] = v.y;
    o[2] = v.z;
}

// push the roots of both triangle sets (static first, CollisionQuery.swift:990-1008) onto the warp's node stack
__device__ __forceinline__ void pool_push_roots(const WorldView &W, const WarpPool &wp, int lane, QShared &s, f3 qlo, f3 qhi,
                                                Counters &ctr, bool count) {
    int pushed = 0;
#pragma unroll 1
    for (int set = 0; set < 2; set++) {
        SetHeader h = *(set ? W.set[1].hdr : W.set[0].hdr);
        if (h.rootRef == CQ_REF_EMPTY) continue;
        if (count) {
            ctr.queries++;
            ctr.nodes++;
        }
        if (box_disjoint(mk3(h.lo[0], h.lo[1], h.lo[2]), mk3(h.hi[0], h.hi[1], h.hi[2]), qlo, qhi)) continue;
        bool leaf = h.rootRef < 0;
        uint32_t pos = atomicAdd((uint32_t *)wp.ntop, 1u); // (room for 64 roots is what CQ_NS_POST keeps free)
        wp.nstack[pos] = make_uint2(((uint32_t)lane << 2) | ((uint32_t)set << 1) | (leaf ? 1u : 0u),
                                    (uint32_t)(leaf ? ~h.rootRef : h.rootRef));
        pushed++;
    }
    s.pending = pushed;
}

// capsuleCastCombined prologue — CollisionQuery.swift:980-1043
template <bool COUNT>
__device__ __forceinline__ void pool_post_cast(const WorldView &W, const WarpPool &wp, int lane, QShared &s, f3 from, f3 delta,
                                               float radius, float hh, uint32_t mask, int mode, float minNormalY,
                                               Counters &ctr) {
    s.rTri = -1;
    s.rPart = -1;
    s.pending = 0;
    s.mode = mode;
    float L = len(delta);
    if (L < 1e-6f) return; // nil without any traversal (:988)
    f3 dir = delta / L;
    float minAdvance = smax(radius * 0.02f, 1e-4f); // :1295
    store3s(s.from, from);
    store3s(s.dir, dir);
    store3s(s.delta, delta);
    s.L = L;
    s.radius = radius;
    s.hh = hh;
    s.minNormalY = minNormalY;
    s.minAdvance = minAdvance;
    s.maxIter = min(256, (int)ceilf(L / minAdvance) + 1); // :1296
    s.rT = L;                                             // bestT starts at |delta| (:1038)
    const f3 up = {0.0f, 1.0f, 0.0f};
    f3 a0 = from + up * hh, b0 = from - up * hh;
    f3 a1 = a0 + delta, b1 = b0 + delta;
    f3 ext = {radius, radius, radius};
    f3 qlo = vmin(vmin(a0, b0), vmin(a1, b1)) - ext;
    f3 qhi = vmax(vmax(a0, b0), vmax(a1, b1)) + ext;
    store3s(s.qlo, qlo);
    store3s(s.qhi, qhi);
    s.mask = mask;
    pool_push_roots(W, wp, lane, s, qlo, qhi, ctr, COUNT);
}

// capsuleOverlapAll prologue — CollisionQuery.swift:1209-1216 (two deepest kept, Systems.swift:764-767)
template <bool COUNT>
__device__ __forceinline__ void pool_post_overlap(const WorldView &W, const WarpPool &wp, int lane, QShared &s, f3 from,
                                                  float radius, float hh, uint32_t mask, Counters &ctr) {
    s.mode = CQ_KIND_OVERLAP;
    store3s(s.from, from);
    s.radius = radius;
    s.hh = hh;
    ovl_words(s)[OVL_TOTAL] = 0;
    s.rT = 0.0f, s.rTri = -1, store3s(s.rN, mk3(0, 0, 0));         // deepest
    s.rPos[0] = 0.0f, s.rPart = -1, store3s(s.rTriN, mk3(0, 0, 0)); // second deepest
    f3 qlo, qhi;
    overlap_box(from, radius, hh, qlo, qhi);
    store3s(s.qlo, qlo);
    store3s(s.qhi, qhi);
    s.mask = mask;
    pool_push_roots(W, wp, lane, s, qlo, qhi, ctr, COUNT);
}

// Cooperative LBVH walk: all 32 lanes pop one stack entry each (any owner's), test it against that owner's
// query box, and push what survives — internal children / leaf ranges back on the stack, candidate triangles
// (layer mask + triangle AABB passed, CollisionQuery.swift:1057-1065) into the pair ring.  One round of the walk
// for the whole warp costs what one step of a single lane's walk used to cost.
// Sweep with a hit on record (LOOKAHEAD kernels): only contacts at or before bestT can still matter, and the capsule moves at
// unit speed, so the walk may use the box of the capsule swept over [0, bestT] (plus the float margin of the look-ahead
// prune) instead of the whole sweep's box.  Returns false when the query is not such a sweep (the caller keeps qlo/qhi).
__device__ __forceinline__ bool sweep_reach(const QShared &s, float &bestT, float &margin) {
    if ((s.mode & 0xff) == CQ_KIND_OVERLAP || *(volatile const int *)&s.rTri < 0) return false;
    bestT = *(volatile const float *)&s.rT;
    margin = 1e-3f + (fabsf(s.from[0]) + fabsf(s.from[1]) + fabsf(s.from[2]) + s.L) * 8e-6f;
    return true;
}
__device__ __forceinline__ void sweep_reach_box(const QShared &s, float bestT, float margin, f3 &qlo, f3 &qhi) {
    const f3 a = mk3(s.from[0], s.from[1], s.from[2]);
    const f3 b = a + mk3(s.dir[0], s.dir[1], s.dir[2]) * (bestT + margin);
    const f3 ext = mk3(s.radius + margin, s.radius + s.hh + margin, s.radius + margin);
    qlo = vmax(qlo, vmin(a, b) - ext); // (never wider than the whole sweep's box)
    qhi = vmin(qhi, vmax(a, b) + ext);
}
// The triangle-level form: (a) best toi 0 with a tie on record and this triangle visited later than the best — it could
// only tie behind it; (b) the capsule's axis at t = 0 is farther from the triangle's box than radius + bestT + margin.
__device__ __forceinline__ bool sweep_cannot_matter(const QShared &s, float bestT, float margin, f3 tlo, f3 thi, int rank) {
    if (bestT == 0.0f && (*(volatile const int *)&s.mode & CQ_QF_TIE) != 0 && rank > *(volatile const int *)&s.rRank) return true;
    const float dx = smax(smax(tlo.x - s.from[0], s.from[0] - thi.x), 0.0f);
    const float dz = smax(smax(tlo.z - s.from[2], s.from[2] - thi.z), 0.0f);
    const float dy = smax(smax(tlo.y - (s.from[1] + s.hh), (s.from[1] - s.hh) - thi.y), 0.0f);
    const float reach = s.radius + bestT + margin;
    return dx * dx + dy * dy + dz * dz > reach * reach * 1.0001f;
}

template <bool COUNT, bool STAGED, bool LOOKAHEAD>
__device__ __forceinline__ void pool_walk_round(const WorldView &W, const WarpPool &wp, int lane, Counters &ctr) {
    const uint32_t top = *wp.ntop;
    const uint32_t poppers = top > (uint32_t)CQ_NS_WIDE ? 1u : 32u; // nearly full: depth-first with one lane
    // warp-uniform overflow guard: a lone popper replaces its entry by at most four.  Should even that not fit, the
    // children are dropped and the world's status word is raised (the call then fails with CQ_ERR_CUDA).
    const bool full = top + 3u > (uint32_t)CQ_NSCAP;
    if (full && lane == 0) atomicOr(wp.status, 1u);
    const uint32_t k = min(top, poppers);
    uint2 e = make_uint2(0u, 0u);
    const bool have = (uint32_t)lane < k;
    if (have) e = wp.nstack[top - 1u - (uint32_t)lane];
    __syncwarp();
    if (lane == 0) *wp.ntop = top - k;
    __syncwarp();
    const bool isLeaf = have && (e.x & 1u) != 0u;
    if (have && !isLeaf) { // 4-wide internal node: test up to four children
        const int owner = e.x >> 2, set = (e.x >> 1) & 1;
        QShared &s = wp.qs[owner];
        f3 qlo = mk3(s.qlo[0], s.qlo[1], s.qlo[2]), qhi = mk3(s.qhi[0], s.qhi[1], s.qhi[2]);
        if (LOOKAHEAD && !(COUNT && W.refStats)) {
            float bestT, margin;
            if (sweep_reach(s, bestT, margin)) sweep_reach_box(s, bestT, margin, qlo, qhi);
        }
        int net = -1; // this entry is consumed
        const Node4 *n = (set ? W.set[1].nodes4 : W.set[0].nodes4) + e.y;
        float4 q0 = __ldg(&n->q[0]), q1 = __ldg(&n->q[1]), q2 = __ldg(&n->q[2]), q3 = __ldg(&n->q[3]);
        float4 q4 = __ldg(&n->q[4]), q5 = __ldg(&n->q[5]), q6 = __ldg(&n->q[6]), q7 = __ldg(&n->q[7]);
        const int r0 = __float_as_int(q0.w), r1 = __float_as_int(q1.w), r2 = __float_as_int(q2.w), r3 = __float_as_int(q3.w);
        // empty children have inverted boxes: they fail the overlap test by themselves
        bool h0 = !box_disjoint(xyz(q0), xyz(q1), qlo, qhi), h1 = !box_disjoint(xyz(q2), xyz(q3), qlo, qhi);
        bool h2 = !box_disjoint(xyz(q4), xyz(q5), qlo, qhi), h3 = !box_disjoint(xyz(q6), xyz(q7), qlo, qhi);
        if (COUNT) ctr.nodes += 2 + (r2 != CQ_REF_EMPTY) + (r3 != CQ_REF_EMPTY);
        int cnt = full ? 0 : (h0 ? 1 : 0) + (h1 ? 1 : 0) + (h2 ? 1 : 0) + (h3 ? 1 : 0);
        if (cnt) {
            uint32_t pos = atomicAdd((uint32_t *)wp.ntop, (uint32_t)cnt);
            const uint32_t tag = e.x & ~1u;
            if (h0) wp.nstack[pos++] = make_uint2(tag | (r0 < 0 ? 1u : 0u), (uint32_t)(r0 < 0 ? ~r0 : r0));
            if (h1) wp.nstack[pos++] = make_uint2(tag | (r1 < 0 ? 1u : 0u), (uint32_t)(r1 < 0 ? ~r1 : r1));
            if (h2) wp.nstack[pos++] = make_uint2(tag | (r2 < 0 ? 1u : 0u), (uint32_t)(r2 < 0 ? ~r2 : r2));
            if (h3) wp.nstack[pos] = make_uint2(tag | (r3 < 0 ? 1u : 0u), (uint32_t)(r3 < 0 ? ~r3 : r3));
            net += cnt;
        }
        if (net) atomicAdd(&s.pending, net);
    }
    // Leaf ranges (1..4 consecutive triangles of the sorted SoA).  Big worlds: expanded to ONE TRIANGLE PER LANE through
    // a staging list, so that the triangle fetches of the whole round are in flight together instead of a few lanes
    // looping over their ranges while the others wait (C4: +18%, terrain move-and-slide: +10%).
    if (!STAGED) { // tiny worlds (everything L1 resident): the plain per-lane loop has less overhead and less code
        if (isLeaf) {
            const int owner = e.x >> 2, set = (e.x >> 1) & 1;
            QShared &s = wp.qs[owner];
            const f3 qlo = mk3(s.qlo[0], s.qlo[1], s.qlo[2]), qhi = mk3(s.qhi[0], s.qhi[1], s.qhi[2]);
            const int start = (int)(e.y >> 2), count = (int)(e.y & 3u) + 1;
            const uint32_t mask = s.mask;
            const float4 *p0 = set ? W.set[1].tv0 : W.set[0].tv0;
            const float4 *p1 = set ? W.set[1].tv1 : W.set[0].tv1;
            const float4 *p2 = set ? W.set[1].tv2 : W.set[0].tv2;
            int net = -1;
#pragma unroll 1
            for (int i = 0; i < count; i++) {
                const int slot = start + i;
                float4 a = __ldg(p0 + slot), b = __ldg(p1 + slot), c = __ldg(p2 + slot);
                if ((__float_as_uint(a.w) & mask) == 0u) continue; // layer mask, CollisionQuery.swift:1057
                f3 v0 = xyz(a), v1 = xyz(b), v2 = xyz(c);
                f3 tlo = vmin(v0, vmin(v1, v2)), thi = vmax(v0, vmax(v1, v2));
                if (box_disjoint(tlo, thi, qlo, qhi)) continue; // :1060-1065
                if (COUNT) ctr.cands++;
                uint32_t pos = atomicAdd((uint32_t *)wp.tail, 1u);
                wp.ring[pos % CQ_QCAP] = ((uint32_t)owner << 27) | ((uint32_t)set << 26) | (uint32_t)slot;
                net++;
            }
            if (net) atomicAdd(&s.pending, net);
        }
        __syncwarp();
        return;
    }
    const uint32_t leafMask = __ballot_sync(0xffffffffu, isLeaf);
    const int total = __popc(leafMask) * 4; // four staging slots per leaf range, unused ones marked empty
    if (total) {
        if (isLeaf) {
            const uint32_t owner = e.x >> 2, set = (e.x >> 1) & 1u;
            const uint32_t item = (owner << 27) | (set << 26) | (e.y >> 2);
            const uint32_t count = (e.y & 3u) + 1u;
            uint32_t *slot4 = wp.stage + 4 * __popc(leafMask & ((1u << lane) - 1u));
#pragma unroll
            for (uint32_t i = 0; i < 4; i++) slot4[i] = i < count ? item + i : 0xffffffffu;
            atomicAdd(&wp.qs[owner].pending, -1); // this entry is consumed
        }
        __syncwarp();
        for (int t = lane; t < total; t += 32) {
            const uint32_t item = wp.stage[t];
            if (item == 0xffffffffu) continue;
            const int owner = item >> 27, set = (item >> 26) & 1, slot = item & 0x3ffffffu;
            QShared &s = wp.qs[owner];
            const float4 *p0 = set ? W.set[1].tv0 : W.set[0].tv0;
            const float4 *p1 = set ? W.set[1].tv1 : W.set[0].tv1;
            const float4 *p2 = set ? W.set[1].tv2 : W.set[0].tv2;
            float4 a = __ldg(p0 + slot), b = __ldg(p1 + slot), c = __ldg(p2 + slot);
            if ((__float_as_uint(a.w) & s.mask) == 0u) continue; // layer mask, CollisionQuery.swift:1057
            const f3 qlo = mk3(s.qlo[0], s.qlo[1], s.qlo[2]), qhi = mk3(s.qhi[0], s.qhi[1], s.qhi[2]);
            f3 v0 = xyz(a), v1 = xyz(b), v2 = xyz(c);
            f3 tlo = vmin(v0, vmin(v1, v2)), thi = vmax(v0, vmax(v1, v2));
            if (box_disjoint(tlo, thi, qlo, qhi)) continue; // :1060-1065
            if (LOOKAHEAD && !(COUNT && W.refStats)) {
                float bestT, margin;
                if (sweep_reach(s, bestT, margin) && sweep_cannot_matter(s, bestT, margin, tlo, thi, __float_as_int(c.w))) continue;
            }
            if (COUNT) ctr.cands++;
            uint32_t pos = atomicAdd((uint32_t *)wp.tail, 1u);
            wp.ring[pos % CQ_QCAP] = item;
            atomicAdd(&s.pending, 1);
        }
    }
    __syncwarp();
}

// job pickup: idle lanes take ring entries, ranked by ballot.
// LOOKAHEAD kernels drop a sweep candidate right here, before its first distance evaluation, when it cannot matter
// (both exact-safe, same argument as the look-ahead prune of pool_eval):
//  (a) the owner's best toi is 0 with a tie already on record and this triangle is visited later than the best: every toi
//      is >= 0, so it could only tie behind it;
//  (b) the distance from the capsule's axis at t = 0 to the triangle's BOX exceeds radius + bestT + margin: the capsule
//      moves at unit speed, so no contact exists at or before bestT.
// A lane that dropped its candidate takes another one (up to four pickups per trip), so that drops do not leave lanes idle
// through the evaluation.  C2 (profiles/r2_ab_same_box.txt, call 11).
// OVLDROP (the staged-walk move-and-slide kernel and the query kernels): an overlap candidate is dropped when the kernel's
// bookkeeping says it cannot matter (OverlapTop2::cannot_matter: reference order, eight overlaps on record, this triangle
// visited after all of them; OverlapTopK::cannot_matter: the same once the overflow of capsuleOverlapAll is established).
template <bool COUNT, bool LOOKAHEAD, bool OVLDROP, class OvlCommit>
__device__ __forceinline__ void pool_take_jobs(const WorldView &W, const WarpPool &wp, Job &job, int lane, const OvlCommit &ovl) {
#pragma unroll 1
    for (int rep = 0; rep < (LOOKAHEAD ? 4 : 1); rep++) { // (an overlap drop is rare: its lane simply idles one trip)
        uint32_t idle = __ballot_sync(0xffffffffu, job.phase == PH_NONE);
        uint32_t h = *wp.head, avail = *wp.tail - h;
        bool dropped = false;
        if (job.phase == PH_NONE) {
            uint32_t rank = __popc(idle & ((1u << lane) - 1u));
            if (rank < avail) {
                uint32_t e = wp.ring[(h + rank) % CQ_QCAP];
                int owner = e >> 27, set = (e >> 26) & 1, slot = e & 0x3ffffffu;
                QShared &s = wp.qs[owner];
                job.enc = e;
                job.radius = s.radius;
                job.hh = s.hh;
                const float4 *p0 = set ? W.set[1].tv0 : W.set[0].tv0;
                const float4 *p1 = set ? W.set[1].tv1 : W.set[0].tv1;
                const float4 *p2 = set ? W.set[1].tv2 : W.set[0].tv2;
                float4 a = __ldg(p0 + slot), b = __ldg(p1 + slot), c = __ldg(p2 + slot);
                job.T.v0 = xyz(a), job.T.v1 = xyz(b), job.T.v2 = xyz(c);
                job.gid = __float_as_int(b.w) + (set ? W.set[1].triOffset : 0);
                job.rank = __float_as_int(c.w);
                job.t = 0.0f;
                job.lastSafeT = 0.0f;
                job.it = 0;
                const int mode = s.mode;
                job.phase = (mode & 0xff) == CQ_KIND_OVERLAP ? PH_OVL : PH_ADV;
                if (LOOKAHEAD && job.phase == PH_ADV && !(COUNT && W.refStats)) {
                    float bestT, margin;
                    if (sweep_reach(s, bestT, margin))
                        dropped = sweep_cannot_matter(s, bestT, margin, vmin(job.T.v0, vmin(job.T.v1, job.T.v2)),
                                                      vmax(job.T.v0, vmax(job.T.v1, job.T.v2)), job.rank);
                }
                if (OVLDROP && job.phase == PH_OVL && !(COUNT && W.refStats)) dropped = ovl.cannot_matter(s, job.rank, e);
                if ((LOOKAHEAD || OVLDROP) && dropped) {
                    job.phase = PH_NONE;
                    atomicSub(&s.pending, 1);
                }
            }
        }
        __syncwarp();
        if (lane == 0) *wp.head = h + min((uint32_t)__popc(idle), avail);
        if (!LOOKAHEAD) break;
        __syncwarp();
        if (!__any_sync(0xffffffffu, dropped) || (uint32_t)__popc(idle) >= avail) break; // nobody freed a lane / ring is empty
    }
}

// one distance evaluation + the pair's state transition.  `retired` = the pair is finished (with or
// without a contribution in `cm`).
// LOOKAHEAD: the look-ahead prune below.  Measured on one box (profiles/r2_ab_same_box.txt): the batched sweep kernel gains
// where candidates are many (C2: distance evaluations per sweep 5352 -> 4108, 32.8 -> 28.1 ms) and loses 1% on C4; the
// move-and-slide kernel LOSES 3-5% on the hulls and terrain scenes (few candidates per query, the extra compares and the
// longer loop body cost more than the 1.5% of evaluations they save), so only the query kernels instantiate it.
// Bisection steps a bound decides (exact-safe, DESIGN.md §5.1 "Decided bisection steps"): the capsule only translates
// along a unit direction, so the distance is 1-Lipschitz in t up to the float error `margin`; once this trip's evaluation
// at tc returned dist, a refineTOI midpoint m with |m - tc| + margin < |dist - radius| would evaluate to the same side
// of the radius and is applied without evaluating it.  The midpoints are the same floats 0.5f * (lo + hi), so lo and hi
// end bit-identical.  No prediction for capsules of radius <= 5 mm (a missed piercing of a nearly vertical triangle can
// read up to 4.6 mm) or half height > 16 radii (near-parallel edge error), nor in reference-stats counting launches.
// Only the plain-walk kernels (worlds below 4096 triangles) instantiate it: measured on one box (profiles/r3_ab_same_box.txt)
// the hulls step gains 13.5% (evaluations per character-step 27.9 -> 17.5), but the staged-walk kernels lose more to the
// longer loop than they save (terrain +4.4%, C4 +2.6% for 6% / 2.5% fewer evaluations; render and C2 gain 3%).
__device__ __forceinline__ float bisect_margin(const QShared &s, float radius, float hh) {
    const volatile float *f = s.from; // (re-read: the copies loaded for the centre would stay live across the distance function)
    const float scale = fabsf(f[0]) + fabsf(f[1]) + fabsf(f[2]) + s.L + hh + radius;
    return radius > 5e-3f && hh <= 16.0f * radius ? scale * 1.9073486e-6f /* 16 * 2^-23 */ : INFINITY;
}

template <bool COUNT, bool LOOKAHEAD>
__device__ __forceinline__ void pool_eval(Job &job, const WarpPool &wp, Commit &cm, bool &retired, Counters &ctr, bool predict) {
    const int ph = job.phase;
    const QShared &s = wp.qs[job.owner()];
    float &hi = job.t, &lo = job.lastSafeT; // (slots shared between the phases, see Job)
    float tc = ph == PH_ADV ? job.t : (ph == PH_BIS ? 0.5f * (lo + hi) : hi);
    f3 center = mk3(s.from[0], s.from[1], s.from[2]);
    if (ph != PH_OVL) center = center + mk3(s.dir[0], s.dir[1], s.dir[2]) * tc;
    f3 sp, tp;
    if (COUNT) ctr.evals++;
    float dist = segment_triangle_distance<true>(center, job.hh, job.T, sp, tp);
    const float bestT = *(volatile const float *)&s.rT; // shared across the query's pairs
    // A contact whose toi is bounded below by `tLow` cannot win when tLow > bestT.  LOOKAHEAD kernels also retire the pair
    // when it can at best TIE (tLow == bestT) behind an earlier-visited best whose tie is already on record: neither the
    // answer nor its CQ_HIT_TIE flag can change.  (A capsule that starts a sweep inside the mesh meets dozens of toi == 0
    // contacts, two evaluations each: C2.)
    auto hopeless = [&](float tLow) {
        if (tLow > bestT) return true;
        if (!LOOKAHEAD || tLow != bestT) return false;
        return (*(volatile const int *)&s.mode & CQ_QF_TIE) != 0 && job.rank > *(volatile const int *)&s.rRank;
    };
    if (ph == PH_ADV) { // sweepCapsuleTriangle loop body, CollisionQuery.swift:1303-1356
        if (dist <= job.radius + 1e-5f) {
            const float L = s.L;
            float c0 = smax(0.0f, smin(job.lastSafeT, L)); // refineTOI prologue, :1371-1377
            float c1 = smax(0.0f, smin(job.t, L));
            lo = smin(c0, c1);
            hi = smax(c0, c1);
            const bool fin = hi - lo < 1e-5f;
            job.it = 0; // (now the bisection counter)
            if (hopeless(fin ? hi : lo)) retired = true;
            else job.phase = fin ? PH_FIN : PH_BIS;
        } else {
            job.lastSafeT = job.t;
            const float minAdvance = s.minAdvance, L = s.L;
            float advance = smax(dist - job.radius, minAdvance);
            job.t += advance <= 0.0f ? minAdvance : advance;
            job.it++;
            // next trip: `for _ in 0..<maxIter { if t > maxDistance return nil ...`; prune: toi >= lastSafeT > bestT
            if (job.it >= s.maxIter || job.t > L || job.lastSafeT > bestT) retired = true;
            // Look-ahead prune (exact-safe): this was a true conservative-advancement step (advance = dist - r, not the
            // minAdvance floor) and it lands beyond bestT by more than `margin`.  The capsule moves at unit speed, so
            // the distance at any t <= bestT is at least dist - (t - lastSafeT) > r + margin: if the NEXT evaluation
            // reports contact, every bisection point of refineTOI at or before bestT still evaluates to "no contact"
            // (margin covers the float error of positions and distances), the refined toi ends beyond bestT and the
            // hit is rejected by `toi < bestT` (:1084); contacts found later have lastSafeT > bestT anyway.
            // margin: float error of positions and distances at this query's scale (1 mm + 8e-6 of the coordinates' size)
            else if (LOOKAHEAD && dist - job.radius >= minAdvance &&
                     job.t > bestT + (1e-3f + (fabsf(s.from[0]) + fabsf(s.from[1]) + fabsf(s.from[2]) + L) * 8e-6f))
                retired = true;
        }
    } else if (ph == PH_BIS) { // refineTOI bisection, :1379-1392 (threshold is radius, not radius+eps)
        if (dist <= job.radius) hi = tc;
        else lo = tc;
        job.it++;
    }
    if (job.phase == PH_BIS && !retired) { // (also right after the PH_ADV -> PH_BIS transition)
        const float margin = bisect_margin(s, job.radius, job.hh), gap = fabsf(dist - job.radius);
#pragma unroll 1
        for (; predict && job.it < 10; job.it++) { // decided steps (a NaN dist never decides)
            const float mid = 0.5f * (lo + hi);
            if (!(fabsf(mid - tc) + margin < gap)) break;
            if (dist <= job.radius) hi = mid;
            else lo = mid;
        }
        if (job.it == 10) {
            if (hopeless(hi)) retired = true;
            else job.phase = PH_FIN;
        } else if (lo > bestT) {
            retired = true;
        }
    }
    // PH_FIN evaluates at hi: when that is this trip's point (the last bisection step evaluated had contact, or the
    // hi - lo < 1e-5 entry with hi = t), the centre, and so dist / sp / tp, are bit-identical: finish in this trip.
    if (job.phase == PH_FIN && !retired && (ph == PH_FIN || (predict && __float_as_uint(hi) == __float_as_uint(tc)))) {
        // contact at tHit = hi, :1325-1346; acceptance filters of :1087-1097
        retired = true;
        f3 triNormal = normalize(cross(job.T.v1 - job.T.v0, job.T.v2 - job.T.v0));
        f3 n;
        if (dist < 1e-6f) n = dot(triNormal, mk3(s.dir[0], s.dir[1], s.dir[2])) > 0.0f ? -triNormal : triNormal;
        else n = normalize(sp - tp);
        f3 triN = triNormal;
        if (dot(triN, n) < 0.0f) triN = -triN;
        bool ok = true;
        const int mode = s.mode & 0xff;
        if (mode == CQ_MODE_BLOCKING) {
            f3 delta = mk3(s.delta[0], s.delta[1], s.delta[2]);
            ok = !(dot(delta, n) >= 0.0f) && !(dot(delta, triN) >= 0.0f);
        } else if (mode == CQ_MODE_GROUND) {
            ok = !(triN.y < s.minNormalY);
        }
        if (ok) {
            cm.kind = 1;
            cm.key = tc;
            cm.pos = tp;
            cm.n = n;
            cm.triN = triN;
        }
    } else if (ph == PH_OVL) { // capsuleOverlapBVHAll leaf body, :1248-1271
        retired = true;
        if (dist < job.radius) {
            f3 triNormal = normalize(cross(job.T.v1 - job.T.v0, job.T.v2 - job.T.v0));
            cm.kind = 2;
            cm.key = job.radius - dist; // depth
            cm.n = dist < 1e-6f ? triNormal : normalize(sp - tp);
        }
    }
}

// (the commit step itself is pool_commit below)
// default overlap commit: the two deepest overlaps kept in the owner's QShared (move-and-slide depenetration)
// Reference order (byRank): the reference's depenetration takes the first maxHits = 8 overlaps in visiting order, sorts
// them by depth (stably) and uses one or two (Systems.swift:751-767).  The first pass keeps the two deepest of ALL
// overlapping triangles (ties: smaller rank), counts them and remembers the eight smallest ranks; only when more than
// eight triangles overlap does the owner run a second pass over exactly those eight (pool_post_first_hits).
// Out of line on purpose: overlap commits are rare in the scenes the kernel is tuned on (a character that starts a step
// inside geometry) while the commit step sits in the steady-state loop whose code size decides the small-scene throughput
// (DESIGN.md §5.1) — inlined, this bookkeeping made the loop 4 KB longer and the hulls step 12% slower.
static __device__ __noinline__ void overlap_top2_commit(QShared &s, float depth, int gid, int rk, f3 n, bool byRank) {
    if (byRank) {
        int *ov = ovl_words(s);
        const int total = ov[OVL_TOTAL];
        if (total >= 0) { // first pass: count, and keep the eight smallest ranks seen (unsorted list + its maximum)
            if (total < CQ_MAX_OVERLAP_HITS) {
                ov[total] = rk;
                if (total == CQ_MAX_OVERLAP_HITS - 1) {
                    int mx = ov[0];
#pragma unroll 1
                    for (int k = 1; k < CQ_MAX_OVERLAP_HITS; k++) mx = max(mx, ov[k]);
                    ov[OVL_MAXRANK] = mx;
                }
            } else if (rk < ov[OVL_MAXRANK]) { // replaces the largest kept rank
                const int out = ov[OVL_MAXRANK];
                int mx = rk;
#pragma unroll 1
                for (int k = 0; k < CQ_MAX_OVERLAP_HITS; k++) {
                    int v = ov[k];
                    if (v == out) ov[k] = v = rk;
                    mx = max(mx, v);
                }
                ov[OVL_MAXRANK] = mx;
            }
            ov[OVL_TOTAL] = total + 1;
        }
    }
    float d0 = s.rT, d1 = s.rPos[0];
    int t0 = s.rTri, t1 = s.rPart;
    bool before0 = t0 < 0 || depth > d0 || (depth == d0 && rk < s.rRank);
    bool before1 = t1 < 0 || depth > d1 || (depth == d1 && rk < s.rRank1);
    if (before0) {
        s.rPos[0] = d0, s.rPart = t0, s.rRank1 = s.rRank;
        store3s(s.rTriN, mk3(s.rN[0], s.rN[1], s.rN[2]));
        s.rT = depth, s.rTri = gid, s.rRank = rk;
        store3s(s.rN, n);
    } else if (before1) {
        s.rPos[0] = depth, s.rPart = gid, s.rRank1 = rk;
        store3s(s.rTriN, n);
    }
}
struct OverlapTop2 {
    bool byRank;
    // Reference order, eight overlaps on record: a triangle the reference visits after all eight cannot be among the first
    // eight, whether it overlaps or not.  (The count then stays short of the true total, but not below eight, and whenever
    // it is exactly eight the two deepest seen are the two deepest of exactly those eight.)
    __device__ __forceinline__ bool cannot_matter(QShared &s, int rk, uint32_t) const {
        if (!byRank) return false;
        const volatile int *ov = ovl_words(s);
        return ov[OVL_TOTAL] >= CQ_MAX_OVERLAP_HITS && rk > ov[OVL_MAXRANK];
    }
    __device__ __forceinline__ void operator()(QShared &s, float depth, int gid, int rk, uint32_t, f3 n) const {
        overlap_top2_commit(s, depth, gid, rk, n, byRank);
    }
};

// second depenetration pass in reference order: the owner's query becomes the (<= 8) triangles the reference visited
// first, posted straight into the pair ring (no walk); the top-2 bookkeeping starts over
static __device__ __noinline__ void pool_post_first_hits(const uint32_t *__restrict__ encOfRank, uint32_t *ring, volatile uint32_t *tail,
                                                         int lane, QShared &s) {
    int *ov = ovl_words(s);
    const uint32_t pos = atomicAdd((uint32_t *)tail, (uint32_t)CQ_MAX_OVERLAP_HITS);
#pragma unroll 1
    for (int k = 0; k < CQ_MAX_OVERLAP_HITS; k++) ring[(pos + k) % CQ_QCAP] = ((uint32_t)lane << 27) | __ldg(encOfRank + ov[k]);
    ov[OVL_TOTAL] = -1; // second pass
    s.rT = 0.0f, s.rTri = -1, store3s(s.rN, mk3(0, 0, 0));
    s.rPos[0] = 0.0f, s.rPart = -1, store3s(s.rTriN, mk3(0, 0, 0));
    s.pending = CQ_MAX_OVERLAP_HITS;
}

// Commit step: the lanes that finished a pair this trip hand their contribution to the owner's record; pending counters drop.
// Contributions to DIFFERENT owners touch different records and commute; contributions to the same owner are order-free
// reductions (smallest (toi, rank); deepest two / smallest ranks; counts).  So the lanes are grouped by owner (one MATCH) and
// round r serves the r-th finishing lane of every owner at once: the serialized rounds are the largest group, not the
// number of finishing lanes.
// REDUCE (the query kernels): sweep hits (:1084,1098 + the order rule — the accepted candidate with the smallest (toi, rank)
// wins) are settled among the finishing lanes of an owner with two warp reductions, so that ONE lane per owner touches the
// record and no rounds are needed for sweeps.  Lane-at-a-time rounds cost the C2 kernel 8.3 rounds per trip: a capsule that
// starts inside the mesh collects dozens of toi == 0 hits, all exact ties that each took a round to compare ranks
// (profiles/r2_by_region_midround.txt).  A contribution already behind the owner's best is dropped before anything else.
// Measured on one box (profiles/r2_ab_same_box.txt, calls 9-10): C2 28.1 -> 16.7 ms (with the tie-aware prune of pool_eval);
// in the move-and-slide kernel the reductions gain 3.6% on the render mesh and 1.2% on the terrain but cost the hulls step
// 4% (0.7 KB more code in the steady-state loop), so only its staged-walk variant (worlds of >= 4096 triangles) uses them;
// owner-grouped rounds alone gained the hulls step 2% over lane-at-a-time rounds.
template <bool REDUCE, class OvlCommit>
__device__ __forceinline__ void pool_commit(const WarpPool &wp, Job &job, const Commit &cm, bool retired, int lane,
                                            OvlCommit ovl) {
    const uint32_t retMask = __ballot_sync(0xffffffffu, retired);
    if (retMask == 0u) return; // (warp-uniform) nothing finished this trip
    bool cast = retired && cm.kind == 1;
    if (cast) cast = !(cm.key > *(volatile const float *)&wp.qs[job.owner()].rT);
    const uint32_t below = (1u << lane) - 1u;
    const uint32_t sameOwner = retired ? __match_any_sync(retMask, job.owner()) : 0u; // the finishing lanes of my owner
    bool mine = retired && cm.kind == 2;
    if (REDUCE) {
        const uint32_t castMask = __ballot_sync(0xffffffffu, cast);
        if (cast) {
            const uint32_t grp = sameOwner & castMask;
            const uint32_t kb = __float_as_uint(cm.key + 0.0f); // toi >= 0: the bit pattern orders like the value
            const bool atMin = kb == __reduce_min_sync(grp, kb);
            const uint32_t rmin = __reduce_min_sync(grp, atMin ? (uint32_t)job.rank : 0xffffffffu);
            const bool tiedInGroup = __popc(__ballot_sync(grp, atMin)) > 1;
            if (atMin && (uint32_t)job.rank == rmin) {
                QShared &s = wp.qs[job.owner()];
                const float bestT = s.rT;
                const bool better = cm.key < bestT;
                const bool tie = s.rTri >= 0 && cm.key == bestT; // exactly equal toi: the reference keeps the first it visited
                const bool tieWin = tie && job.rank < s.rRank;
                int mode = s.mode;
                if (better) mode &= ~CQ_QF_TIE;
                if (tie || ((better || tieWin) && tiedInGroup)) mode |= CQ_QF_TIE;
                s.mode = mode;
                if (better || tieWin) {
                    s.rT = cm.key;
                    s.rTri = job.gid;
                    s.rRank = job.rank;
                    store3s(s.rPos, cm.pos);
                    store3s(s.rN, cm.n);
                    store3s(s.rTriN, cm.triN);
                }
            }
        }
    } else {
        mine = mine || cast;
    }
    // Overlaps: the bookkeeping is the kernel's (two deepest + first-visited list, or top-K) and is order-free, but a
    // read-modify-write of the owner's record, hence the rounds.
    const uint32_t todo = __ballot_sync(0xffffffffu, mine);
    const int myRound = __popc(sameOwner & todo & below); // my place among my owner's lanes
#pragma unroll 1
    for (int round = 0; __any_sync(0xffffffffu, mine && myRound >= round); round++) {
        if (mine && myRound == round) {
            QShared &s = wp.qs[job.owner()];
            if (!REDUCE && cm.kind == 1) {
                float bestT = s.rT;
                int bestTri = s.rTri;
                bool better = cm.key < bestT;
                bool tie = bestTri >= 0 && cm.key == bestT;
                bool tieWin = tie && job.rank < s.rRank;
                if (tie) s.mode |= CQ_QF_TIE;
                if (better) s.mode &= ~CQ_QF_TIE;
                if (better || tieWin) {
                    s.rT = cm.key;
                    s.rTri = job.gid;
                    s.rRank = job.rank;
                    store3s(s.rPos, cm.pos);
                    store3s(s.rN, cm.n);
                    store3s(s.rTriN, cm.triN);
                }
            } else {
                ovl(s, cm.key, job.gid, job.rank, job.enc, cm.n);
            }
        }
        __syncwarp();
    }
    if (retired) {
        if ((sameOwner & below) == 0u) atomicSub(&wp.qs[job.owner()].pending, __popc(sameOwner)); // one lane per owner
        job.phase = PH_NONE;
    }
    __syncwarp();
}

// The warp's main loop.  `advance(mine, ctr)` is the owner-role callback: it is invoked when the lane's
// current query is complete (pending == 0), consumes the result from `mine`, runs the unit's serial logic and
// posts the next query (pool_post_*) — or returns false when the lane has no more work units.
// `ownersPerWarp` (1..32): how many lanes of each warp take the owner role.  Small batches of heavy units
// use fewer owners per warp so that every owner still processes several units (dynamic fetch then balances
// the warps against each other) while all 32 lanes keep executing pairs.
template <bool COUNT, bool STAGED, int FE_IDLE, bool LOOKAHEAD, class Advance, class OvlCommit>
__device__ __forceinline__ void pool_run(const WorldView &W, const WarpPool &wp, int lane, int ownersPerWarp, Counters &ctr,
                                         Advance advance, OvlCommit ovl) {
    QShared &mine = wp.qs[lane];
    mine.pending = 0;
    mine.rTri = -1;
    if (lane == 0) {
        *wp.head = 0;
        *wp.tail = 0;
        *wp.ntop = 0;
        *wp.fePasses = 0;
    }
    Job job;
    job.phase = PH_NONE;
    bool alive = lane < ownersPerWarp;
    __syncwarp();
    for (;;) { // (exits through the vote at the bottom, or through the watchdog on the front-end passes)
        // The front end (owners' unit logic + walk rounds) runs only when the pair ring has run dry AND at least FE_IDLE
        // lanes have nothing to execute: the divergent unit logic then runs for many owners at once, and — what matters
        // most on small scenes — its ~40 KB of code passes through the instruction caches far less often, evicting the
        // ~20 KB distance loop less often (measured, 1 M characters: hulls 374 -> 416 M/s with FE_IDLE 8, 426 M/s with
        // 16; terrain +4%; C4 +1.6% with 8 but -2% with 16; the candidate-heavy render mesh loses 3% either way).
        const uint32_t idleNow = (uint32_t)__popc(__ballot_sync(0xffffffffu, job.phase == PH_NONE));
        if (*wp.tail == *wp.head && idleNow >= (uint32_t)FE_IDLE) {
            // Watchdog.  Every pair retires within maxIter + 12 trips and the ring only drains between front-end passes, so a
            // loop that does not end must keep coming through here; counted in shared memory (a counter in a register would
            // be one more value kept alive across the distance function, i.e. one more spill).
            const uint32_t passes = *wp.fePasses;
            if (passes > (1u << 24)) {
                if (lane == 0) atomicOr(wp.status, 4u);
                break;
            }
            __syncwarp();
            if (lane == 0) *wp.fePasses = passes + 1u;
            // The owners' logic runs only when enough owners are ready (or nothing at all is left to execute), so that the
            // divergent front end serves many owners per pass.  Measured on one box (profiles/r2_ab_same_box.txt, call 7):
            // with 24 of 32 the render-mesh step (heavy queries, owners rarely ready together) gains 23% (21.98 -> 17.88 ms),
            // the terrain step is unchanged, the hulls step loses 0.8% — hence only the staged-walk variant (worlds of
            // >= 4096 triangles) of the move-and-slide kernel waits; the plain query kernels own few units per warp.
            const bool ready = alive && *(volatile int *)&mine.pending == 0 && *wp.ntop <= (uint32_t)CQ_NS_POST;
            bool go = ready;
            if (FE_IDLE >= 16 && STAGED) { // (compile-time)
                const uint32_t nReady = (uint32_t)__popc(__ballot_sync(0xffffffffu, ready));
                go = ready && (nReady >= 24u || (idleNow == 32u && *wp.ntop == 0u));
            }
            if (go) alive = advance(mine, ctr);
            __syncwarp();
            // cooperative walk: rounds until the ring holds ~3 trips of work (or the stack is empty)
            while (*wp.ntop != 0u && *wp.tail - *wp.head < (uint32_t)CQ_WALK_FILL && *wp.tail - *wp.head + 128u <= (uint32_t)CQ_QCAP)
                pool_walk_round<COUNT, STAGED, LOOKAHEAD>(W, wp, lane, ctr);
        }
        // executor: idle lanes take pairs; every lane holding a pair does ONE distance evaluation
        pool_take_jobs<COUNT, LOOKAHEAD, (STAGED && FE_IDLE >= 16) || LOOKAHEAD>(W, wp, job, lane, ovl);
        Commit cm;
        cm.kind = 0;
        bool retired = false;
        if (job.phase != PH_NONE) pool_eval<COUNT, LOOKAHEAD>(job, wp, cm, retired, ctr, !STAGED && !(COUNT && W.refStats));
        pool_commit<LOOKAHEAD || (STAGED && FE_IDLE >= 16)>(wp, job, cm, retired, lane, ovl);
        if (__all_sync(0xffffffffu, !alive && job.phase == PH_NONE) && *wp.ntop == 0u && *wp.tail == *wp.head) break;
    }
}

// host side: owners per warp for a batch of n units on `warps` resident warps (aim: >= 4 units per owner)
static inline int pool_owners_per_warp(long long n, long long warps) {
    if (n >= warps * 32) return 32;      // at least one unit per lane: every lane owns
    long long o = n / (warps * 4);       // otherwise aim at >= 4 units per owner
    return (int)(o < 4 ? 4 : (o > 32 ? 32 : o));
}

__device__ __forceinline__ void pool_flush_counters(const Counters &c, unsigned long long *g, bool count) {
    if (!count) return;
    uint32_t v[4] = {c.nodes, c.cands, c.evals, c.queries};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        unsigned long long s = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(g + k, s);
    }
}

} // namespace cq
