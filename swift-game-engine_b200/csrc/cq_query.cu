// cq_query.cu — batched query kernels: raycast, capsule cast (3 modes), capsule overlap (deepest),
// capsule overlap-all (max_hits hits).  One thread per query; the BVH walk and the narrow phase live in
// cq_world.cuh / cq_math.cuh.  Replaces the per-call CPU entry points of CollisionQuery.swift:85-159.
#include "cq_pool.cuh"
#include "cq_internal.h"

namespace cq {

#define Q_THREADS 128

__device__ __forceinline__ void store3(float *o, f3 v) {
    o[0] = v.x;
    o[1] = v.y;
    o[2] = v.z;
}
__device__ __forceinline__ f3 load3(const float *p) { return {p[0], p[1], p[2]}; }

// ---------------------------------------------------------------- raycast (CollisionQuery.swift:768-785, 916-978)
// rayAABB (:1603-1631) with the same operations: the slab test of the reference's own walk
__device__ __forceinline__ bool ref_ray_aabb(f3 o, f3 inv, f3 lo, f3 hi, float &tminOut) {
    float tmin = (lo.x - o.x) * inv.x, tmax = (hi.x - o.x) * inv.x;
    if (tmin > tmax) {
        float t = tmin;
        tmin = tmax, tmax = t;
    }
    float tymin = (lo.y - o.y) * inv.y, tymax = (hi.y - o.y) * inv.y;
    if (tymin > tymax) {
        float t = tymin;
        tymin = tymax, tymax = t;
    }
    if (tmin > tymax || tymin > tmax) return false;
    tmin = tymin >= tmin ? tymin : tmin; // Swift max(x, y) = y >= x ? y : x ; min(x, y) = y < x ? y : x
    tmax = tymax < tmax ? tymax : tmax;
    float tzmin = (lo.z - o.z) * inv.z, tzmax = (hi.z - o.z) * inv.z;
    if (tzmin > tzmax) {
        float t = tzmin;
        tzmin = tzmax, tzmax = t;
    }
    if (tmin > tzmax || tzmin > tmax) return false;
    tminOut = tzmin >= tmin ? tzmin : tmin;
    return true;
}

// One kernel, both order rules (REF):
//   canonical  the triangle with the smallest t over ALL triangles (ties -> smallest index); boxes only skip work and the
//              box test is conservative (see ray_box).
//   reference  the reference's walk itself (CollisionQuery.swift:916-978) over the reference's own tree (cut on the device
//              by attach_ref_order): per set, closestT starts at maxDistance; pop a node, cull it when rayAABB
//              (ref_ray_aabb) misses or starts beyond closestT, test a leaf's triangles in triOrder with strict
//              `t < closestT`, push left then right.  The slab test of a child is evaluated when its parent is visited (a
//              miss never depends on closestT) and its tmin travels with the stack entry, so the `tmin > closestT` test
//              happens at pop time with the value closestT has THEN — the same nodes are culled as in the reference,
//              including the grazing hits its non-conservative slab test loses.  Static and dynamic sets are walked
//              independently and merged with `<=` (:902-907).
// Phase voting.  ncu on the earlier one-step-per-trip kernels (profiles/r2_c5_raycast_v12_summary.txt): 7.2 of 32 lanes
// active per warp instruction, 65% of the stall samples long-scoreboard.  A ray of C5 takes ~8 node steps, ~1.4 triangle
// steps and one finish + fetch; with one step of whatever kind per trip every trip pays for all three bodies while each
// is populated by a third of the lanes or fewer.  Here the three bodies are PHASES of the warp:
//   refill    finished lanes write their hit and fetch the next ray — only when at least RAY_REFILL_MIN lanes are idle
//             (or nobody has anything else to do), so the long, latency-heavy body runs for many lanes at once;
//   nodes     lanes with a non-empty stack pop / test / push, and the phase REPEATS while at least RAY_NODE_MIN lanes
//             still want a node step: the dependent node fetches of most of the warp are in flight together;
//   triangles lanes holding a leaf range test their next triangle, repeated while RAY_TRI_MIN lanes have one.
// Every phase runs at least once per round when any lane wants it, so progress never depends on the thresholds.
#ifndef RAY_REFILL_MIN
#define RAY_REFILL_MIN 8
#endif
#ifndef RAY_NODE_MIN /* measured on C5, one box: reference order 12 -> 3.18 ms, 16 -> 3.00, 20 -> 2.94, 24 -> 3.00; canonical order */
#define RAY_NODE_MIN (REF ? 20 : 12) /* 12 -> 2.01 ms, 16 -> 2.01, 20 -> 2.05 (the reference's binary tree takes more node steps per ray) */
#endif
#ifndef RAY_TRI_MIN
#define RAY_TRI_MIN 8
#endif
#ifndef RAY_SMEM_STACK
#define RAY_SMEM_STACK (REF ? 20 : 24) /* entries per lane in shared memory (the rest of CQ_STACK in local memory) */
#endif
template <bool COUNT, bool REF>
__global__ void __launch_bounds__(Q_THREADS) k_raycast_phased(WorldView W, const cq_ray *__restrict__ rays, int n,
                                                              cq_ray_hit *__restrict__ out, uint8_t *__restrict__ flagsOut,
                                                              int *workCounter, const uint32_t *__restrict__ order,
                                                              unsigned long long *gctr) {
    Counters ctr = {0, 0, 0, 0};
    // Traversal stack: the first RAY_SMEM_STACK entries of every lane live in shared memory ([entry][thread]: a warp's
    // accesses fall into 32 different banks whatever the lanes' depths), deeper entries in local memory.  With the whole
    // stack in local memory the two loads of a pop were the kernel's top long-scoreboard stall (15% of the samples of
    // profiles/r2_ray_c5_ref_summary.txt's capture): rays and triangles stream through L1 and keep evicting it.
    int sp = 0;
    __shared__ int sRef[RAY_SMEM_STACK][Q_THREADS];
    __shared__ float sT[REF ? RAY_SMEM_STACK : 1][Q_THREADS];
    int deepRef[CQ_STACK - RAY_SMEM_STACK];
    float deepT[REF ? CQ_STACK - RAY_SMEM_STACK : 1];
    const int tid = threadIdx.x;
    auto push = [&](int ref, float t) {
        if (sp < RAY_SMEM_STACK) {
            sRef[sp][tid] = ref;
            if (REF) sT[sp][tid] = t;
        } else {
            deepRef[sp - RAY_SMEM_STACK] = ref;
            if (REF) deepT[sp - RAY_SMEM_STACK] = t;
        }
        sp++;
    };
    auto pop = [&](int &ref, float &t) {
        --sp;
        if (sp < RAY_SMEM_STACK) {
            ref = sRef[sp][tid];
            if (REF) t = sT[sp][tid];
        } else {
            ref = deepRef[sp - RAY_SMEM_STACK];
            if (REF) t = deepT[sp - RAY_SMEM_STACK];
        }
    };
    int set = 2, leafPos = 0, leafEnd = 0, cur = -1;
    int bestTri = -1, setTri = -1;
    float closestT = 0.0f, bestT = 0.0f, maxDist = 0.0f;
    f3 o = {0, 0, 0}, d = {0, 0, 0}, inv = {0, 0, 0}, bestN = {0, 0, 0}, setN = {0, 0, 0};
    uint32_t mask = 0, tie = 0, setTie = 0;
    bool alive = true;
    const int lane = threadIdx.x & 31;
    while (true) {
        // ---------------- refill / set transitions: lanes whose stack and leaf range are empty
        const bool idle = alive && sp == 0 && leafPos >= leafEnd;
        const uint32_t idleMask = __ballot_sync(0xffffffffu, idle);
        const uint32_t busyMask = __ballot_sync(0xffffffffu, alive && !idle);
        if (idleMask != 0u && (__popc(idleMask) >= RAY_REFILL_MIN || busyMask == 0u)) {
            if (idle) {
                if (REF) { // the set just walked: merge its hit (static wins `<=`, :902-907)
                    if (setTri >= 0 && (bestTri < 0 || !(bestT <= closestT))) bestT = closestT, bestTri = setTri, bestN = setN, tie = setTie;
                    setTri = -1, setTie = 0;
                }
                // one atomic per warp: the lanes that need a new ray take consecutive positions of the processing order
                const bool finished = set >= 2; // (also true on a lane's first trip)
                const uint32_t takers = __ballot_sync(idleMask, finished);
                if (finished) {
                    if (cur >= 0) { // write the finished ray
                        cq_ray_hit hres;
                        const float tHit = REF ? bestT : closestT;
                        if (bestTri >= 0) {
                            hres.distance = tHit;
                            store3(hres.position, o + d * tHit); // :962
                            store3(hres.normal, bestN);
                            hres.triangle_index = bestTri;
                        } else {
                            hres.distance = 0.0f;
                            store3(hres.position, mk3(0, 0, 0));
                            store3(hres.normal, mk3(0, 0, 0));
                            hres.triangle_index = -1;
                        }
                        out[cur] = hres;
                        if (flagsOut) flagsOut[cur] = (uint8_t)tie;
                    }
                    int base = 0;
                    const int leader = __ffs(takers) - 1;
                    if (lane == leader) base = atomicAdd(workCounter, __popc(takers));
                    base = __shfl_sync(takers, base, leader);
                    cur = base + __popc(takers & ((1u << lane) - 1u));
                    if (cur >= n) {
                        cur = -1;
                        alive = false;
                    } else {
                        if (order) cur = (int)order[cur];
                        cq_ray r = rays[cur];
                        o = load3(r.origin), d = load3(r.direction);
                        maxDist = r.max_distance;
                        closestT = maxDist;
                        mask = r.mask;
                        bestTri = -1, setTri = -1, tie = 0, setTie = 0;
                        inv = mk3(d.x != 0.0f ? 1.0f / d.x : FLT_MAX, d.y != 0.0f ? 1.0f / d.y : FLT_MAX,
                                  d.z != 0.0f ? 1.0f / d.z : FLT_MAX); // :1606-1608
                        set = 0;
                    }
                }
                // Roots.  Reference order walks one set at a time (closestT starts over at maxDistance, :921): push the next
                // set's root and stop.  Canonical order pushes both roots at once, the dynamic one first so that the static
                // set is popped first.
                while (alive && set < 2 && (!REF || sp == 0)) {
                    const int s1 = REF ? set : 1 - set;
                    const SetHeader h = *(REF ? (s1 ? W.set[1].refHdr : W.set[0].refHdr) : (s1 ? W.set[1].hdr : W.set[0].hdr));
                    if (REF) closestT = maxDist;
                    set++;
                    if (h.rootRef == CQ_REF_EMPTY) continue;
                    if (COUNT) {
                        ctr.queries++;
                        ctr.nodes++;
                    }
                    const f3 lo = mk3(h.lo[0], h.lo[1], h.lo[2]), hi = mk3(h.hi[0], h.hi[1], h.hi[2]);
                    const int tagged = h.rootRef < 0 ? ~((~h.rootRef) | (s1 << 30)) : (h.rootRef | (s1 << 30)); // bit 30 = set
                    if (REF) {
                        float tmin;
                        if (ref_ray_aabb(o, inv, lo, hi, tmin)) push(tagged, tmin);
                    } else if (ray_box(o, inv, lo, hi, closestT)) {
                        push(tagged, 0.0f);
                    }
                }
            }
        }
        if (__all_sync(0xffffffffu, !alive)) break;
        // ---------------- node phase
        while (true) {
            const bool wantN = alive && sp > 0 && leafPos >= leafEnd;
            const uint32_t nMask = __ballot_sync(0xffffffffu, wantN);
            if (nMask == 0u) break;
            if (wantN) {
                int ref;
                float tNear = 0.0f;
                pop(ref, tNear);
                bool visit = true;
                if (REF) visit = !(tNear > closestT); // :933, with the closestT of NOW
                if (visit) {
                    if (ref < 0) {
                        int enc = ~ref;
                        const int s1 = (enc >> 30) & 1;
                        enc &= 0x3fffffff;
                        leafPos = (enc >> 2) | (s1 << 30);
                        leafEnd = leafPos + (enc & 3) + 1;
                    } else {
                        const int s1 = (ref >> 30) & 1;
                        const Node *nd = (REF ? W.set[s1].refNodes : W.set[s1].nodes) + (ref & 0x3fffffff);
                        const float4 n0 = __ldg(&nd->n0), n1 = __ldg(&nd->n1), n2 = __ldg(&nd->n2), n3 = __ldg(&nd->n3);
                        if (COUNT) ctr.nodes += 2;
                        int r0 = __float_as_int(n0.w), r1 = __float_as_int(n1.w);
                        r0 = r0 < 0 ? ~((~r0) | (s1 << 30)) : (r0 | (s1 << 30));
                        r1 = r1 < 0 ? ~((~r1) | (s1 << 30)) : (r1 | (s1 << 30));
                        if (REF) {
                            float t0, t1;
                            const bool h0 = ref_ray_aabb(o, inv, xyz(n0), xyz(n1), t0); // left
                            const bool h1 = ref_ray_aabb(o, inv, xyz(n2), xyz(n3), t1); // right
                            if (h0) push(r0, t0); // push left, then right: right is popped first (:965-966)
                            if (h1) push(r1, t1);
                        } else {
                            const bool h0 = ray_box(o, inv, xyz(n0), xyz(n1), closestT);
                            const bool h1 = ray_box(o, inv, xyz(n2), xyz(n3), closestT);
                            if (h1) push(r1, 0.0f);
                            if (h0) push(r0, 0.0f);
                        }
                    }
                }
            }
            if (__popc(nMask) < RAY_NODE_MIN) break;
        }
        // ---------------- triangle phase
        while (true) {
            const bool wantT = alive && leafPos < leafEnd;
            const uint32_t tMask = __ballot_sync(0xffffffffu, wantT);
            if (tMask == 0u) break;
            if (wantT) {
                const int s1 = (leafPos >> 30) & 1, pos = leafPos & 0x3fffffff;
                leafPos++;
                const SetView &S = W.set[s1];
                const int slot = REF ? (int)__ldg(S.refSlot + pos) : pos; // reference order: ascending triOrder positions (:938-940)
                uint32_t layer;
                int triId, part;
                Tri T = load_tri(S, slot, layer, triId, part);
                if ((layer & mask) != 0u) {
                    if (COUNT) ctr.cands++;
                    float t;
                    if (ray_triangle(o, d, T, t)) {
                        const int gid = triId + S.triOffset;
                        if (REF) {
                            if (t < closestT) { // strict: the first visited keeps an exact tie (:944)
                                closestT = t;
                                setTri = gid;
                                setTie = 0;
                                f3 nrm = normalize(cross(T.v1 - T.v0, T.v2 - T.v0));
                                setN = dot(nrm, d) > 0.0f ? -nrm : nrm;
                            } else if (t == closestT && setTri >= 0) {
                                setTie = CQ_HIT_TIE;
                            }
                        } else {
                            if (bestTri >= 0 && t == closestT) tie = CQ_HIT_TIE;
                            if (t < closestT) tie = 0;
                            if (t < closestT || (bestTri >= 0 && t == closestT && gid < bestTri)) {
                                closestT = t;
                                bestTri = gid;
                                f3 nrm = normalize(cross(T.v1 - T.v0, T.v2 - T.v0)); // :960-961
                                bestN = dot(nrm, d) > 0.0f ? -nrm : nrm;
                            }
                        }
                    }
                }
            }
            if (__popc(tMask) < RAY_TRI_MIN) break;
        }
    }
    pool_flush_counters(ctr, gctr, COUNT);
}

// ---------------------------------------------------------------- capsule cast (CollisionQuery.swift:787-828, 980-1117)
// Warp-cooperative pool engine (cq_pool.cuh): every lane owns one sweep at a time (fetched dynamically),
// walks the LBVH for it and pushes its candidate triangles into the warp's ring; all 32 lanes execute
// the (sweep, triangle) pairs, one distance evaluation per trip.
#define CAST_WARPS (Q_THREADS / 32)
#ifndef CAST_MIN_BLOCKS
#define CAST_MIN_BLOCKS 5 /* 96 registers: +9% on C4 against 4 CTAs/SM (107 registers); 6 CTAs/SM (80) gains nothing */
#endif
template <bool COUNT, bool STAGED>
__global__ void __launch_bounds__(Q_THREADS, CAST_MIN_BLOCKS) k_capsule_cast(WorldView W, const cq_capsule_cast *__restrict__ qs, int n,
                                                               int mode, cq_cast_hit *__restrict__ out,
                                                               uint8_t *__restrict__ flagsOut, int ownersPerWarp,
                                                               uint2 *nodeScratch, int *workCounter,
                                                               const uint32_t *__restrict__ order,
                                                               unsigned long long *gctr) {
    __shared__ QShared qsAll[Q_THREADS];
    __shared__ uint32_t words[CQ_POOL_WORDS * CAST_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpPool wp;
    pool_bind(wp, qsAll, words, nodeScratch, warp, CAST_WARPS, W.rank, W.status);
    Counters ctr = {0, 0, 0, 0};
    int cur = -1;
    pool_run<COUNT, STAGED, 8, true>(W, wp, lane, ownersPerWarp, ctr, [&](QShared &mine, Counters &ct) {
        if (cur >= 0) { // write the finished hit
            cq_cast_hit h;
            if (mine.rTri >= 0) {
                h.toi = mine.rT;
                store3(h.position, mk3(mine.rPos[0], mine.rPos[1], mine.rPos[2]));
                store3(h.normal, mk3(mine.rN[0], mine.rN[1], mine.rN[2]));
                store3(h.triangle_normal, mk3(mine.rTriN[0], mine.rTriN[1], mine.rTriN[2]));
                h.triangle_index = mine.rTri;
            } else {
                h.toi = 0.0f;
                store3(h.position, mk3(0, 0, 0));
                store3(h.normal, mk3(0, 0, 0));
                store3(h.triangle_normal, mk3(0, 0, 0));
                h.triangle_index = -1;
            }
            out[cur] = h;
            if (flagsOut) flagsOut[cur] = (mine.mode & CQ_QF_TIE) ? CQ_HIT_TIE : 0;
        }
        cur = atomicAdd(workCounter, 1); // dynamic fetch of the next sweep
        if (cur >= n) {
            cur = -1;
            return false;
        }
        if (order) cur = (int)order[cur]; // Morton-coherent processing order (big worlds)
        cq_capsule_cast c = qs[cur];
        pool_post_cast<COUNT>(W, wp, lane, mine, load3(c.from), load3(c.delta), c.radius, c.half_height, c.mask, mode,
                              c.min_normal_y, ct);
        return true;
    }, OverlapTop2{W.rank != nullptr});
    pool_flush_counters(ctr, gctr, COUNT);
}

__device__ __forceinline__ void write_overlap(cq_overlap_hit &h, const OverlapRec &r) {
    h.depth = r.depth;
    store3(h.position, r.position);
    store3(h.normal, r.normal);
    store3(h.triangle_normal, r.triNormal);
    h.triangle_index = r.tri;
}
__device__ __forceinline__ void write_overlap_nil(cq_overlap_hit &h) {
    h.depth = 0.0f;
    store3(h.position, mk3(0, 0, 0));
    store3(h.normal, mk3(0, 0, 0));
    store3(h.triangle_normal, mk3(0, 0, 0));
    h.triangle_index = -1;
}

// ---------------------------------------------------------------- capsule overlap / overlap-all
// (CollisionQuery.swift:830-882, 1119-1283) on the pair pool: one distance evaluation per (capsule, triangle)
// pair, shared by the warp.  The owner keeps its winners as (depth, rank, triangle, ring entry) in shared memory —
// inserted in the serialized commit step — and, when its query completes, re-evaluates those <= 8 winners to emit the
// full contact records (same arithmetic, so the records are bit-identical to what the pair's executor saw).
//   capsuleOverlap    = the deepest one; exactly equal depths go to the smaller visiting rank (strict `>`, :1172)
//   capsuleOverlapAll, reference order = the maxHits triangles the reference visits FIRST (:1272-1274), in that order
//                     (its callers sort by depth themselves, Systems.swift:759);
//                     canonical order = the maxHits deepest, deepest first.  Both agree as sets whenever at most
//                     maxHits triangles overlap; `overflow` flags the queries where more do.
struct OvlTop {
    float depth[CQ_MAX_OVERLAP_HITS];
    int rank[CQ_MAX_OVERLAP_HITS];
    int gid[CQ_MAX_OVERLAP_HITS];
    uint32_t enc[CQ_MAX_OVERLAP_HITS];
    int count, total, cap, tie;
};

struct OverlapTopK {
    OvlTop *tops; // the warp's 32 records
    bool byRank; // keep the smallest ranks (overlap-all in reference order) instead of the deepest
    // capsuleOverlapAll in reference order keeps the maxHits overlaps visited first (:1272-1274).  Once MORE than maxHits
    // overlaps are on record the count (= maxHits) and the overflow flag are settled, and a triangle visited after all the
    // kept ones cannot enter the list whether it overlaps or not: it is not evaluated.
    __device__ __forceinline__ bool cannot_matter(QShared &, int rk, uint32_t enc) const {
        if (!byRank) return false;
        const OvlTop &t = tops[enc >> 27];
        return t.total > t.cap && rk > t.rank[t.cap - 1];
    }
    __device__ __forceinline__ void operator()(QShared &, float depth, int gid, int rk, uint32_t enc, f3) const {
        OvlTop &t = tops[enc >> 27];
        t.total++;
        int pos = t.count;
        if (byRank) {
            while (pos > 0 && t.rank[pos - 1] > rk) pos--;
        } else {
            if (t.count > 0 && t.depth[0] == depth) t.tie = 1; // exactly as deep as the deepest so far
            while (pos > 0 && (t.depth[pos - 1] < depth || (t.depth[pos - 1] == depth && t.rank[pos - 1] > rk))) pos--;
            if (pos == 0 && t.count > 0 && t.depth[0] != depth) t.tie = 0; // a strictly deeper one: the old tie is moot
        }
        if (pos >= t.cap) return;
        int last = t.count < t.cap ? t.count : t.cap - 1;
        for (int k = last; k > pos; k--) {
            t.depth[k] = t.depth[k - 1];
            t.rank[k] = t.rank[k - 1];
            t.gid[k] = t.gid[k - 1];
            t.enc[k] = t.enc[k - 1];
        }
        t.depth[pos] = depth;
        t.rank[pos] = rk;
        t.gid[pos] = gid;
        t.enc[pos] = enc;
        if (t.count < t.cap) t.count++;
    }
};

// contact record of a winning triangle — CollisionQuery.swift:1165-1190 (re-evaluated by the owner)
__device__ __forceinline__ void overlap_record(const WorldView &W, uint32_t enc, int gid, f3 from, float radius, float hh,
                                               cq_overlap_hit &h) {
    int set = (enc >> 26) & 1, slot = enc & 0x3ffffffu;
    const SetView &S = W.set[set];
    uint32_t layer;
    int triId, part;
    Tri T = load_tri(S, slot, layer, triId, part);
    f3 sp, tp;
    float dist = segment_triangle_distance<true>(from, hh, T, sp, tp);
    OverlapRec r;
    overlap_contact(T, dist, sp, tp, radius, r);
    r.tri = gid;
    write_overlap(h, r);
}

template <bool COUNT, bool ALL, bool STAGED>
__global__ void __launch_bounds__(Q_THREADS, 4) k_capsule_overlap_pool(WorldView W, const cq_capsule *__restrict__ qs, int n,
                                                                       int maxHits, cq_overlap_hit *__restrict__ out,
                                                                       int32_t *__restrict__ counts,
                                                                       uint8_t *__restrict__ overflow, int ownersPerWarp,
                                                                       uint2 *nodeScratch, int *workCounter,
                                                                       unsigned long long *gctr) {
    __shared__ QShared qsAll[Q_THREADS];
    __shared__ OvlTop tops[Q_THREADS];
    __shared__ uint32_t words[CQ_POOL_WORDS * CAST_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpPool wp;
    pool_bind(wp, qsAll, words, nodeScratch, warp, CAST_WARPS, W.rank, W.status);
    OvlTop &top = tops[threadIdx.x];
    Counters ctr = {0, 0, 0, 0};
    int cur = -1;
    f3 curFrom = {0, 0, 0};
    float curR = 0.0f, curHH = 0.0f;
    pool_run<COUNT, STAGED, 8, true>(W, wp, lane, ownersPerWarp, ctr, [&](QShared &mine, Counters &ct) {
        if (cur >= 0) { // emit the finished query
            const int stride = ALL ? maxHits : 1;
            for (int k = 0; k < stride; k++) {
                cq_overlap_hit h;
                if (k < top.count) {
                    if (COUNT) ct.evals++;
                    overlap_record(W, top.enc[k], top.gid[k], curFrom, curR, curHH, h);
                } else {
                    write_overlap_nil(h);
                }
                out[(size_t)cur * stride + k] = h;
            }
            if (ALL) {
                counts[cur] = top.count;
                if (overflow) overflow[cur] = top.total > maxHits ? 1 : 0;
            } else if (overflow) { // capsuleOverlap: the flags byte
                overflow[cur] = top.tie ? CQ_HIT_TIE : 0;
            }
        }
        cur = atomicAdd(workCounter, 1);
        if (cur >= n) {
            cur = -1;
            return false;
        }
        cq_capsule c = qs[cur];
        curFrom = load3(c.from), curR = c.radius, curHH = c.half_height;
        top.count = 0, top.total = 0, top.cap = ALL ? maxHits : 1, top.tie = 0;
        pool_post_overlap<COUNT>(W, wp, lane, mine, curFrom, curR, curHH, c.mask, ct);
        return true;
    }, OverlapTopK{tops + warp * 32, ALL && W.rank != nullptr});
    pool_flush_counters(ctr, gctr, COUNT);
}

// ---------------------------------------------------------------- capsule overlap-all, wide path (max_hits > CQ_OVL_WIDE_ABOVE)
// OvlTop keeps 8 winners per owner in shared memory and the owner emits them serially; neither scales to a large maxHits.
// The wide path keeps each query's winners in its own output slots and emits them in two more launches:
//   k_capsule_overlap_wide  the pair pool; an owner's kept list is a binary heap in global memory, one OvlEntry at the head
//                           of each of the query's cq_overlap_hit slots, with the WORST kept entry at the root, so that a
//                           commit costs O(log maxHits).  Per owner, shared memory holds only OvlHead.  At completion the
//                           owner writes counts / overflow and nothing else;
//   k_overlap_wide_sort     one thread per query: heapsort of the kept entries in place (best first);
//   k_overlap_wide_emit     one thread per slot: entry k -> full record k (the arithmetic of overlap_record), nil past count.
// Both orders keep the same entries as OverlapTopK: the smallest visiting ranks (reference order), or the deepest with
// exact ties to the smaller rank (canonical order); ranks are unique, so the kept set and its sorted order are too.
#ifndef CQ_OVL_WIDE_ABOVE
#define CQ_OVL_WIDE_ABOVE CQ_MAX_OVERLAP_HITS /* max_hits above this runs the wide path (0: every call, for A/B builds) */
#endif

struct OvlEntry { // 16 B at the head of a 44 B output slot until the emit pass overwrites it
    float depth;
    int rank, gid;
    uint32_t enc;
};
struct OvlHead { // per owner: the heap's size, overlaps committed, the query, and the root (worst kept) entry's key
    int count, total, cur, worstRank;
    float worstDepth;
};

// a sits nearer the root than b: larger rank (reference order), or shallower with exact ties to the larger rank
__device__ __forceinline__ bool ovl_worse(bool byRank, float da, int ra, float db, int rb) {
    return byRank ? ra > rb : (da < db || (da == db && ra > rb));
}
__device__ __forceinline__ OvlEntry *ovl_slot(cq_overlap_hit *out, size_t base, unsigned i) {
    return reinterpret_cast<OvlEntry *>(out + base + i);
}
__device__ __forceinline__ void ovl_put(cq_overlap_hit *out, size_t base, unsigned i, const OvlEntry &e) {
    OvlEntry *p = ovl_slot(out, base, i); // (4-byte aligned only: four word stores)
    p->depth = e.depth, p->rank = e.rank, p->gid = e.gid, p->enc = e.enc;
}
__device__ __forceinline__ OvlEntry ovl_get(const cq_overlap_hit *out, size_t base, unsigned i) {
    const OvlEntry *p = ovl_slot(const_cast<cq_overlap_hit *>(out), base, i);
    return OvlEntry{p->depth, p->rank, p->gid, p->enc};
}
// sift e down from the root of the heap out[base .. base + n); returns the new root
__device__ __forceinline__ OvlEntry ovl_sift_down(cq_overlap_hit *out, size_t base, unsigned n, const OvlEntry &e, bool byRank) {
    unsigned i = 0;
    OvlEntry root = e;
#pragma unroll 1
    for (;;) {
        const unsigned l = 2u * i + 1u; // (i < n / 2 < 2^30: no wrap)
        if (l >= n) break;
        unsigned c = l;
        OvlEntry C = ovl_get(out, base, l);
        if (l + 1u < n) {
            const OvlEntry R = ovl_get(out, base, l + 1u);
            if (ovl_worse(byRank, R.depth, R.rank, C.depth, C.rank)) c = l + 1u, C = R;
        }
        if (!ovl_worse(byRank, C.depth, C.rank, e.depth, e.rank)) break;
        ovl_put(out, base, i, C);
        if (i == 0) root = C;
        i = c;
    }
    ovl_put(out, base, i, e);
    return root;
}

// Commit of one overlap, run by the executor lane in the owner's pool_commit round.  Out of line for the same reason as
// overlap_top2_commit: it sits in the steady-state loop.
static __device__ __noinline__ void overlap_heap_commit(OvlHead &h, cq_overlap_hit *out, int cap, bool byRank, float depth, int gid,
                                                        int rk, uint32_t enc) {
    h.total++;
    const OvlEntry e{depth, rk, gid, enc};
    const size_t base = (size_t)h.cur * cap;
    if (h.count < cap) { // not full: sift up
        unsigned i = (unsigned)h.count;
#pragma unroll 1
        while (i > 0) {
            const unsigned p = (i - 1u) >> 1;
            const OvlEntry P = ovl_get(out, base, p);
            if (!ovl_worse(byRank, e.depth, e.rank, P.depth, P.rank)) break;
            ovl_put(out, base, i, P);
            i = p;
        }
        ovl_put(out, base, i, e);
        h.count++;
        if (i == 0) h.worstDepth = depth, h.worstRank = rk;
    } else if (ovl_worse(byRank, h.worstDepth, h.worstRank, depth, rk)) { // full: replaces the worst kept entry
        const OvlEntry root = ovl_sift_down(out, base, (unsigned)cap, e, byRank);
        h.worstDepth = root.depth, h.worstRank = root.rank;
    }
}

struct OverlapHeapK {
    OvlHead *heads; // the warp's 32 owners
    cq_overlap_hit *out;
    int cap;
    bool byRank;
    // OverlapTopK::cannot_matter: more than maxHits overlaps on record and this triangle visited after every kept one
    __device__ __forceinline__ bool cannot_matter(QShared &, int rk, uint32_t enc) const {
        if (!byRank) return false;
        const OvlHead &h = heads[enc >> 27];
        return h.total > cap && rk > h.worstRank;
    }
    __device__ __forceinline__ void operator()(QShared &, float depth, int gid, int rk, uint32_t enc, f3) const {
        overlap_heap_commit(heads[enc >> 27], out, cap, byRank, depth, gid, rk, enc);
    }
};

template <bool COUNT, bool STAGED>
__global__ void __launch_bounds__(Q_THREADS, 4) k_capsule_overlap_wide(WorldView W, const cq_capsule *__restrict__ qs, int n,
                                                                       int maxHits, cq_overlap_hit *out, int32_t *__restrict__ counts,
                                                                       uint8_t *__restrict__ overflow, int ownersPerWarp,
                                                                       uint2 *nodeScratch, int *workCounter,
                                                                       unsigned long long *gctr) {
    __shared__ QShared qsAll[Q_THREADS];
    __shared__ OvlHead heads[Q_THREADS];
    __shared__ uint32_t words[CQ_POOL_WORDS * CAST_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpPool wp;
    pool_bind(wp, qsAll, words, nodeScratch, warp, CAST_WARPS, W.rank, W.status);
    OvlHead &head = heads[threadIdx.x];
    Counters ctr = {0, 0, 0, 0};
    int cur = -1;
    pool_run<COUNT, STAGED, 8, true>(W, wp, lane, ownersPerWarp, ctr, [&](QShared &mine, Counters &ct) {
        if (cur >= 0) { // the records are the emit pass's
            counts[cur] = head.count;
            if (overflow) overflow[cur] = head.total > maxHits ? 1 : 0;
        }
        cur = atomicAdd(workCounter, 1);
        if (cur >= n) {
            cur = -1;
            return false;
        }
        cq_capsule c = qs[cur];
        head.count = 0, head.total = 0, head.cur = cur, head.worstRank = 0, head.worstDepth = 0.0f;
        pool_post_overlap<COUNT>(W, wp, lane, mine, load3(c.from), c.radius, c.half_height, c.mask, ct);
        return true;
    }, OverlapHeapK{heads + warp * 32, out, maxHits, W.rank != nullptr});
    pool_flush_counters(ctr, gctr, COUNT);
}

// heapsort in place: the worst entry goes to the end first, so the slots end best first — ascending rank (reference
// order), deepest first with ties to the smaller rank (canonical order)
__global__ void __launch_bounds__(Q_THREADS) k_overlap_wide_sort(int n, int maxHits, bool byRank, cq_overlap_hit *out,
                                                                 const int32_t *__restrict__ counts) {
    for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < (size_t)n; q += (size_t)gridDim.x * blockDim.x) {
        const size_t base = q * maxHits;
#pragma unroll 1
        for (unsigned end = (unsigned)counts[q]; end > 1u; end--) {
            const OvlEntry root = ovl_get(out, base, 0), last = ovl_get(out, base, end - 1u);
            ovl_sift_down(out, base, end - 1u, last, byRank);
            ovl_put(out, base, end - 1u, root);
        }
    }
}

// slot i = query i / maxHits, entry i % maxHits: reads its entry and writes its record from the same thread
template <bool COUNT>
__global__ void __launch_bounds__(Q_THREADS) k_overlap_wide_emit(WorldView W, const cq_capsule *__restrict__ qs, int n,
                                                                 int maxHits, cq_overlap_hit *out,
                                                                 const int32_t *__restrict__ counts, unsigned long long *gctr) {
    Counters ctr = {0, 0, 0, 0};
    const size_t slots = (size_t)n * maxHits;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < slots; i += (size_t)gridDim.x * blockDim.x) {
        const size_t q = i / (size_t)maxHits;
        const int k = (int)(i - q * (size_t)maxHits);
        cq_overlap_hit h;
        if (k < counts[q]) {
            const OvlEntry e = ovl_get(out, i, 0);
            const cq_capsule c = qs[q];
            if (COUNT) ctr.evals++;
            overlap_record(W, e.enc, e.gid, load3(c.from), c.radius, c.half_height, h);
        } else {
            write_overlap_nil(h);
        }
        out[i] = h;
    }
    pool_flush_counters(ctr, gctr, COUNT);
}

// ---------------------------------------------------------------- launchers
int pool_launch_setup(cq_world *w, const void *kernel, int threads, size_t smem, int unitsPerCta, int n, bool nodeScratch,
                      const void *units, size_t stride, bool positionIsDouble, cudaStream_t st, PoolLaunch &out) {
    CQ_TRY(await_trees(w, st));
    const int resident = resident_blocks(w, kernel, threads, smem);
    if (!resident) return CQ_ERR_CUDA;
    const int warps = threads / 32;
    out.blocks = std::min(cdiv(n, unitsPerCta), resident); // one resident wave of persistent lanes
    out.ownersPerWarp = pool_owners_per_warp(n, (long long)out.blocks * warps);
    const size_t nodeBytes = (size_t)out.blocks * warps * CQ_NSCAP * sizeof(uint2);
    void *ns = nullptr;
    uint32_t *orderScratch = nullptr;
    if (nodeScratch) CQ_TRY(take_scratch(w, w->nodeScratch, 4, w->nodeSeq++ & 3, nodeBytes, st, "node scratch", &ns));
    if (units) CQ_TRY(take_unit_order(w, n, st, &orderScratch));
    out.nodeScratch = (uint2 *)ns;
    out.work = next_work_counter(w, st);
    if (!out.work) return CQ_ERR_CUDA;
    return make_unit_order(w, orderScratch, units, stride, positionIsDouble, n, st, &out.order);
}

int launch_raycast(cq_world *w, const cq_ray *d_rays, int n, cq_ray_hit *d_out, uint8_t *d_flags, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    const bool ref = w->order == CQ_ORDER_REFERENCE; // the reference's own walk over the reference's own tree
    const int ci = (w->counting ? 1 : 0) + (ref ? 2 : 0);
    using Kernel = void (*)(WorldView, const cq_ray *, int, cq_ray_hit *, uint8_t *, int *, const uint32_t *, unsigned long long *);
    static const Kernel kernels[4] = {k_raycast_phased<false, false>, k_raycast_phased<true, false>, k_raycast_phased<false, true>,
                                      k_raycast_phased<true, true>};
    const Kernel kernel = kernels[ci];
    PoolLaunch L;
    CQ_TRY(pool_launch_setup(w, (const void *)kernel, Q_THREADS, 0, Q_THREADS, n, false, d_rays, sizeof(cq_ray), false, st, L));
    kernel<<<L.blocks, Q_THREADS, 0, st>>>(w->view, d_rays, n, d_out, d_flags, L.work, L.order, w->dCounters);
    w->launches++;
    return finish_launch(w, st, ref ? "k_raycast_ref" : "k_raycast");
}

int launch_cast(cq_world *w, const cq_capsule_cast *d_q, int n, int mode, cq_cast_hit *d_out, uint8_t *d_flags, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    const int ci = (w->counting ? 1 : 0) + 2 * (w->view.stagedLeaves ? 1 : 0);
    using Kernel = void (*)(WorldView, const cq_capsule_cast *, int, int, cq_cast_hit *, uint8_t *, int, uint2 *, int *,
                            const uint32_t *, unsigned long long *);
    static const Kernel kernels[4] = {k_capsule_cast<false, false>, k_capsule_cast<true, false>, k_capsule_cast<false, true>,
                                      k_capsule_cast<true, true>};
    const Kernel kernel = kernels[ci];
    PoolLaunch L;
    CQ_TRY(pool_launch_setup(w, (const void *)kernel, Q_THREADS, 0, 4, n, true, d_q, sizeof(cq_capsule_cast), false, st, L));
    kernel<<<L.blocks, Q_THREADS, 0, st>>>(w->view, d_q, n, mode, d_out, d_flags, L.ownersPerWarp, L.nodeScratch, L.work, L.order,
                                           w->dCounters);
    w->launches++;
    return finish_launch(w, st, "k_capsule_cast");
}

template <bool ALL>
static int launch_overlap_pool(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                               uint8_t *d_overflow, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    const int ci = (w->counting ? 1 : 0) + 2 * (w->view.stagedLeaves ? 1 : 0);
    using Kernel = void (*)(WorldView, const cq_capsule *, int, int, cq_overlap_hit *, int32_t *, uint8_t *, int, uint2 *, int *,
                            unsigned long long *);
    static const Kernel kernels[4] = {k_capsule_overlap_pool<false, ALL, false>, k_capsule_overlap_pool<true, ALL, false>,
                                      k_capsule_overlap_pool<false, ALL, true>, k_capsule_overlap_pool<true, ALL, true>};
    const Kernel kernel = kernels[ci];
    PoolLaunch L;
    CQ_TRY(pool_launch_setup(w, (const void *)kernel, Q_THREADS, 0, 4, n, true, nullptr, 0, false, st, L));
    kernel<<<L.blocks, Q_THREADS, 0, st>>>(w->view, d_q, n, maxHits, d_out, d_counts, d_overflow, L.ownersPerWarp, L.nodeScratch,
                                           L.work, w->dCounters);
    w->launches++;
    return finish_launch(w, st, "k_capsule_overlap_pool");
}

int launch_overlap(cq_world *w, const cq_capsule *d_q, int n, cq_overlap_hit *d_out, uint8_t *d_flags, cudaStream_t st) {
    return launch_overlap_pool<false>(w, d_q, n, 1, d_out, nullptr, d_flags, st);
}

// the wide path: the pool kernel, the sort and the emit pass, always three launches
static int launch_overlap_wide(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                               uint8_t *d_overflow, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    const int ci = (w->counting ? 1 : 0) + 2 * (w->view.stagedLeaves ? 1 : 0);
    using Kernel = void (*)(WorldView, const cq_capsule *, int, int, cq_overlap_hit *, int32_t *, uint8_t *, int, uint2 *, int *,
                            unsigned long long *);
    static const Kernel kernels[4] = {k_capsule_overlap_wide<false, false>, k_capsule_overlap_wide<true, false>,
                                      k_capsule_overlap_wide<false, true>, k_capsule_overlap_wide<true, true>};
    const Kernel kernel = kernels[ci];
    PoolLaunch L;
    CQ_TRY(pool_launch_setup(w, (const void *)kernel, Q_THREADS, 0, 4, n, true, nullptr, 0, false, st, L));
    kernel<<<L.blocks, Q_THREADS, 0, st>>>(w->view, d_q, n, maxHits, d_out, d_counts, d_overflow, L.ownersPerWarp, L.nodeScratch,
                                           L.work, w->dCounters);
    // grid-stride passes: a few waves of 128-thread blocks whatever n and maxHits
    const long long wave = (long long)w->numSms * 16;
    const int sortBlocks = (int)std::min<long long>(cdiv(n, Q_THREADS), wave);
    k_overlap_wide_sort<<<sortBlocks, Q_THREADS, 0, st>>>(n, maxHits, w->view.rank != nullptr, d_out, d_counts);
    const long long slots = (long long)n * maxHits;
    const int emitBlocks = (int)std::min<long long>((slots + Q_THREADS - 1) / Q_THREADS, wave);
    if (w->counting) k_overlap_wide_emit<true><<<emitBlocks, Q_THREADS, 0, st>>>(w->view, d_q, n, maxHits, d_out, d_counts, w->dCounters);
    else k_overlap_wide_emit<false><<<emitBlocks, Q_THREADS, 0, st>>>(w->view, d_q, n, maxHits, d_out, d_counts, w->dCounters);
    w->launches += 3; // the number cq.h documents
    return finish_launch(w, st, "k_capsule_overlap_wide");
}

int launch_overlap_all(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                       uint8_t *d_overflow, cudaStream_t st) {
    if (maxHits > CQ_OVL_WIDE_ABOVE) return launch_overlap_wide(w, d_q, n, maxHits, d_out, d_counts, d_overflow, st);
    return launch_overlap_pool<true>(w, d_q, n, maxHits, d_out, d_counts, d_overflow, st);
}

} // namespace cq
