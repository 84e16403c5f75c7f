// cq_query.cu — batched query kernels: raycast, capsule cast (3 modes), capsule overlap (deepest),
// capsule overlap-all (8 deepest).  One thread per query; the BVH walk and the narrow phase live in
// cq_world.cuh / cq_math.cuh.  Replaces the per-call CPU entry points of CollisionQuery.swift:85-159.
#include "cq_pool.cuh"
#include "cq_internal.h"

namespace cq {

#define Q_THREADS 128

template <bool COUNT> __device__ __forceinline__ void flush_counters(const Counters &c, unsigned long long *g) {
    if (!COUNT) return;
    // warp-reduce, one atomic per warp per counter
    uint32_t v[4] = {c.nodes, c.cands, c.evals, c.queries};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        unsigned long long s = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(g + k, s);
    }
}

__device__ __forceinline__ void store3(float *o, f3 v) {
    o[0] = v.x;
    o[1] = v.y;
    o[2] = v.z;
}
__device__ __forceinline__ f3 load3(const float *p) { return {p[0], p[1], p[2]}; }

// ---------------------------------------------------------------- raycast (CollisionQuery.swift:768-785, 916-978)
// Flat per-lane state machine over persistent lanes: every trip of the loop each lane performs exactly ONE step
// of its ray — a node step (fetch a 64-byte node, test both child boxes, push/descend) or a triangle step
// (Moller-Trumbore on the next triangle of the current leaf range) — and a lane whose ray is finished writes the
// hit and fetches the next ray in the same trip.  The nested while-while version ran 3.5 of 32 lanes (ncu).
// Result = the triangle with the smallest t over ALL triangles (ties -> smallest index); boxes only skip work and
// the box test is conservative (see ray_box).
template <bool COUNT>
__global__ void __launch_bounds__(Q_THREADS) k_raycast(WorldView W, const cq_ray *__restrict__ rays, int n,
                                                       cq_ray_hit *__restrict__ out, uint8_t *__restrict__ flagsOut,
                                                       int *workCounter, const uint32_t *__restrict__ order,
                                                       unsigned long long *gctr) {
    Counters ctr = {0, 0, 0, 0};
    uint32_t tie = 0;
    int stack[CQ_STACK];
    int sp = 0, set = 2, leafPos = 0, leafEnd = 0, cur = -1;
    int bestTri = -1;
    float closestT = 0.0f;
    f3 o = {0, 0, 0}, d = {0, 0, 0}, inv = {0, 0, 0}, bestN = {0, 0, 0};
    uint32_t mask = 0;
    bool alive = true;
    while (true) {
        if (alive && leafPos >= leafEnd && sp == 0) {
            if (set < 2) { // next triangle set of this ray (static, then dynamic), or finish the ray
                const SetHeader h = *(set ? W.set[1].hdr : W.set[0].hdr);
                if (h.rootRef != CQ_REF_EMPTY) {
                    if (COUNT) {
                        ctr.queries++;
                        ctr.nodes++;
                    }
                    if (ray_box(o, inv, mk3(h.lo[0], h.lo[1], h.lo[2]), mk3(h.hi[0], h.hi[1], h.hi[2]), closestT))
                        stack[sp++] = h.rootRef < 0 ? ~((~h.rootRef) | (set << 30)) : (h.rootRef | (set << 30)); // bit 30 = set
                }
                set++;
            } else {
                if (cur >= 0) {
                    cq_ray_hit hres;
                    if (bestTri >= 0) {
                        hres.distance = closestT;
                        store3(hres.position, o + d * closestT); // :962
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
                cur = atomicAdd(workCounter, 1);
                if (cur >= n) {
                    cur = -1;
                    alive = false;
                } else {
                    if (order) cur = (int)order[cur];
                    cq_ray r = rays[cur];
                    o = load3(r.origin), d = load3(r.direction);
                    closestT = r.max_distance;
                    mask = r.mask;
                    bestTri = -1, tie = 0;
                    // CollisionQuery.swift:1606-1608: 1/d, or greatestFiniteMagnitude when d == 0
                    inv = mk3(d.x != 0.0f ? 1.0f / d.x : FLT_MAX, d.y != 0.0f ? 1.0f / d.y : FLT_MAX,
                              d.z != 0.0f ? 1.0f / d.z : FLT_MAX);
                    set = 0;
                }
            }
        } else if (alive && leafPos < leafEnd) { // triangle step
            const int s1 = (leafPos >> 30) & 1, slot = leafPos & 0x3fffffff;
            leafPos++;
            const SetView &S = W.set[s1];
            uint32_t layer;
            int triId, part;
            Tri T = load_tri(S, slot, layer, triId, part);
            if ((layer & mask) != 0u) {
                if (COUNT) ctr.cands++;
                float t;
                if (ray_triangle(o, d, T, t)) {
                    int gid = triId + S.triOffset;
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
        } else if (alive) { // node step
            int ref = stack[--sp];
            if (ref < 0) {
                int enc = ~ref;
                const int s1 = (enc >> 30) & 1;
                enc &= 0x3fffffff;
                leafPos = (enc >> 2) | (s1 << 30);
                leafEnd = leafPos + (enc & 3) + 1;
            } else {
                const int s1 = (ref >> 30) & 1;
                const Node *nd = W.set[s1].nodes + (ref & 0x3fffffff);
                float4 n0 = __ldg(&nd->n0), n1 = __ldg(&nd->n1), n2 = __ldg(&nd->n2), n3 = __ldg(&nd->n3);
                if (COUNT) ctr.nodes += 2;
                bool h0 = ray_box(o, inv, xyz(n0), xyz(n1), closestT);
                bool h1 = ray_box(o, inv, xyz(n2), xyz(n3), closestT);
                int r0 = __float_as_int(n0.w), r1 = __float_as_int(n1.w);
                // tag the set into bit 30 (internal refs are < 2^26; leaf encodings are stored complemented)
                r0 = r0 < 0 ? ~((~r0) | (s1 << 30)) : (r0 | (s1 << 30));
                r1 = r1 < 0 ? ~((~r1) | (s1 << 30)) : (r1 | (s1 << 30));
                if (h1) stack[sp++] = r1;
                if (h0) stack[sp++] = r0;
            }
        }
        if (__all_sync(0xffffffffu, !alive)) break;
    }
    flush_counters<COUNT>(ctr, gctr);
}

// ---------------------------------------------------------------- raycast in REFERENCE order
// The reference's walk itself (CollisionQuery.swift:916-978) over the reference's own tree (cq_reftree.h, uploaded by
// attach_ref_order): per set, closestT starts at maxDistance; pop a node, cull it when rayAABB (:1603-1631, restated
// below with the same operations) misses or starts beyond closestT, test a leaf's triangles in triOrder with strict
// `t < closestT`, push left then right.  The slab test of a child is evaluated when its parent is visited (a miss
// never depends on closestT) and its tmin travels with the stack entry, so the `tmin > closestT` test happens at pop
// time with the value closestT has THEN — the same nodes are culled as in the reference, including the grazing hits its
// non-conservative slab test loses.  Static and dynamic sets are walked independently and merged with `<=` (:902-907).
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

template <bool COUNT>
__global__ void __launch_bounds__(Q_THREADS) k_raycast_ref(WorldView W, const cq_ray *__restrict__ rays, int n,
                                                           cq_ray_hit *__restrict__ out, uint8_t *__restrict__ flagsOut,
                                                           int *workCounter, const uint32_t *__restrict__ order,
                                                           unsigned long long *gctr) {
    Counters ctr = {0, 0, 0, 0};
    int stackRef[CQ_STACK];
    float stackT[CQ_STACK];
    int sp = 0, set = 2, leafPos = 0, leafEnd = 0, cur = -1;
    int bestTri = -1, setTri = -1;
    float closestT = 0.0f, bestT = 0.0f, maxDist = 0.0f;
    f3 o = {0, 0, 0}, d = {0, 0, 0}, inv = {0, 0, 0}, bestN = {0, 0, 0}, setN = {0, 0, 0};
    uint32_t mask = 0, tie = 0, setTie = 0;
    bool alive = true;
    while (true) {
        if (alive && leafPos >= leafEnd && sp == 0) {
            // a set's walk is over: merge its hit (static wins `<=`, :902-907), then the next set or the next ray
            if (setTri >= 0 && (bestTri < 0 || !(bestT <= closestT))) bestT = closestT, bestTri = setTri, bestN = setN, tie = setTie;
            setTri = -1, setTie = 0;
            if (set < 2) {
                const SetHeader h = *(set ? W.set[1].refHdr : W.set[0].refHdr);
                closestT = maxDist;
                if (h.rootRef != CQ_REF_EMPTY) {
                    if (COUNT) {
                        ctr.queries++;
                        ctr.nodes++;
                    }
                    float tmin;
                    if (ref_ray_aabb(o, inv, mk3(h.lo[0], h.lo[1], h.lo[2]), mk3(h.hi[0], h.hi[1], h.hi[2]), tmin)) {
                        stackRef[sp] = h.rootRef < 0 ? ~((~h.rootRef) | (set << 30)) : (h.rootRef | (set << 30));
                        stackT[sp++] = tmin;
                    }
                }
                set++;
            } else {
                if (cur >= 0) {
                    cq_ray_hit hres;
                    if (bestTri >= 0) {
                        hres.distance = bestT;
                        store3(hres.position, o + d * bestT); // :962
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
                cur = atomicAdd(workCounter, 1);
                if (cur >= n) {
                    cur = -1;
                    alive = false;
                } else {
                    if (order) cur = (int)order[cur];
                    cq_ray r = rays[cur];
                    o = load3(r.origin), d = load3(r.direction);
                    maxDist = r.max_distance;
                    mask = r.mask;
                    bestTri = -1, setTri = -1, tie = 0;
                    inv = mk3(d.x != 0.0f ? 1.0f / d.x : FLT_MAX, d.y != 0.0f ? 1.0f / d.y : FLT_MAX,
                              d.z != 0.0f ? 1.0f / d.z : FLT_MAX); // :1606-1608
                    set = 0;
                }
            }
        } else if (alive && leafPos < leafEnd) { // triangle step, ascending triOrder positions (:938-940)
            const int s1 = (leafPos >> 30) & 1, pos = leafPos & 0x3fffffff;
            leafPos++;
            const SetView &S = W.set[s1];
            const int slot = (int)__ldg(S.refSlot + pos);
            uint32_t layer;
            int triId, part;
            Tri T = load_tri(S, slot, layer, triId, part);
            if ((layer & mask) != 0u) {
                if (COUNT) ctr.cands++;
                float t;
                if (ray_triangle(o, d, T, t)) {
                    if (t < closestT) { // strict: the first visited keeps an exact tie (:944)
                        closestT = t;
                        setTri = triId + S.triOffset;
                        setTie = 0;
                        f3 nrm = normalize(cross(T.v1 - T.v0, T.v2 - T.v0));
                        setN = dot(nrm, d) > 0.0f ? -nrm : nrm;
                    } else if (t == closestT && setTri >= 0) {
                        setTie = CQ_HIT_TIE;
                    }
                }
            }
        } else if (alive) { // node step
            --sp;
            const int ref = stackRef[sp];
            const float tminNode = stackT[sp];
            if (!(tminNode > closestT)) { // :933, with the closestT of NOW
                if (ref < 0) {
                    int enc = ~ref;
                    const int s1 = (enc >> 30) & 1;
                    enc &= 0x3fffffff;
                    leafPos = (enc >> 2) | (s1 << 30);
                    leafEnd = leafPos + (enc & 3) + 1;
                } else {
                    const int s1 = (ref >> 30) & 1;
                    const Node *nd = W.set[s1].refNodes + (ref & 0x3fffffff);
                    float4 n0 = __ldg(&nd->n0), n1 = __ldg(&nd->n1), n2 = __ldg(&nd->n2), n3 = __ldg(&nd->n3);
                    if (COUNT) ctr.nodes += 2;
                    float t0, t1;
                    const bool h0 = ref_ray_aabb(o, inv, xyz(n0), xyz(n1), t0); // left
                    const bool h1 = ref_ray_aabb(o, inv, xyz(n2), xyz(n3), t1); // right
                    int r0 = __float_as_int(n0.w), r1 = __float_as_int(n1.w);
                    r0 = r0 < 0 ? ~((~r0) | (s1 << 30)) : (r0 | (s1 << 30));
                    r1 = r1 < 0 ? ~((~r1) | (s1 << 30)) : (r1 | (s1 << 30));
                    if (h0) stackRef[sp] = r0, stackT[sp++] = t0; // push left, then right: the right child is popped first (:965-966)
                    if (h1) stackRef[sp] = r1, stackT[sp++] = t1;
                }
            }
        }
        if (__all_sync(0xffffffffu, !alive)) break;
    }
    flush_counters<COUNT>(ctr, gctr);
}

// ---------------------------------------------------------------- raycast, phase-voted (both order rules)
// ncu on the one-step-per-trip kernels above (profiles/r2_c5_raycast_v12_summary.txt): 7.2 of 32 lanes active per warp
// instruction, 65% of the stall samples long-scoreboard.  A ray of C5 takes ~8 node steps, ~1.4 triangle steps and one
// finish + fetch; with one step of whatever kind per trip every trip pays for all three bodies while each is populated
// by a third of the lanes or fewer.  Here the three bodies are PHASES of the warp:
//   refill    finished lanes write their hit and fetch the next ray — only when at least RAY_REFILL_MIN lanes are idle
//             (or nobody has anything else to do), so the long, latency-heavy body runs for many lanes at once;
//   nodes     lanes with a non-empty stack pop / test / push, and the phase REPEATS while at least RAY_NODE_MIN lanes
//             still want a node step: the dependent node fetches of most of the warp are in flight together;
//   triangles lanes holding a leaf range test their next triangle, repeated while RAY_TRI_MIN lanes have one.
// Every phase runs at least once per round when any lane wants it, so progress never depends on the thresholds.
// The per-ray logic is exactly that of k_raycast (canonical: nearest over all triangles, conservative padded slabs,
// ties to the smaller index) and k_raycast_ref (the reference's walk over the reference's tree, its own slab test,
// tmin re-tested at pop time, sets walked independently and merged with `<=`).
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
    flush_counters<COUNT>(ctr, gctr);
}

// ---------------------------------------------------------------- capsule cast (CollisionQuery.swift:787-828, 980-1117)
// Warp-cooperative pool engine (cq_pool.cuh): every lane owns one sweep at a time (fetched dynamically),
// walks the LBVH for it and pushes its candidate triangles into the warp's ring; all 32 lanes execute
// the (sweep, triangle) pairs, one distance evaluation per trip.
#define CAST_WARPS (Q_THREADS / 32)
#ifndef CQ_UNIT_BATCH
#define CQ_UNIT_BATCH 1 /* > 1: sweeps claimed per atomic by k_capsule_cast, with an L2 prefetch of their records (round-2 A/B) */
#endif
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
#if CQ_UNIT_BATCH > 1
    int batchNext = 0, batchEnd = 0; // [batchNext, batchEnd): positions in the processing order this owner has claimed
#endif
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
#if CQ_UNIT_BATCH > 1
        // claim CQ_UNIT_BATCH sweeps per atomic and start their query records towards L2 right away: the chain
        // atomic -> order[] -> query record is three dependent long-latency accesses, paid once per sweep on a single lane
        // (C4: 8% of the kernel's stall samples sit in this fetch + posting, 64-78% of them long-scoreboard waits)
        if (batchNext == batchEnd) {
            batchNext = atomicAdd(workCounter, CQ_UNIT_BATCH);
            batchEnd = min(batchNext + CQ_UNIT_BATCH, n);
            if (batchNext >= n) {
                batchNext = batchEnd = 0;
                cur = -1;
                return false;
            }
            for (int k = batchNext + 1; k < batchEnd; k++) {
                const int id = order ? (int)order[k] : k;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(qs + id));
            }
        }
        cur = batchNext++;
#else
        cur = atomicAdd(workCounter, 1); // dynamic fetch of the next sweep
        if (cur >= n) {
            cur = -1;
            return false;
        }
#endif
        if (order) cur = (int)order[cur]; // Morton-coherent processing order (big worlds)
        cq_capsule_cast c = qs[cur];
        pool_post_cast<COUNT>(W, wp, lane, mine, load3(c.from), load3(c.delta), c.radius, c.half_height, c.mask, mode,
                              c.min_normal_y, ct);
        return true;
    }, OverlapTop2{W.rank != nullptr});
    flush_counters<COUNT>(ctr, gctr);
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
    flush_counters<COUNT>(ctr, gctr);
}

// ---------------------------------------------------------------- launchers
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

#undef CQ_OCC_SLOT
#define CQ_OCC_SLOT 1
int launch_raycast(cq_world *w, const cq_ray *d_rays, int n, cq_ray_hit *d_out, uint8_t *d_flags, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    CQ_TRY(await_trees(w, st));
    int *blocksPerSm = w->occ[CQ_OCC_SLOT]; int &numSms = w->numSms;
    const bool ref = w->order == CQ_ORDER_REFERENCE; // the reference's own walk over the reference's own tree
    const int ci = (w->counting ? 1 : 0) + (ref ? 2 : 0);
    using Kernel = void (*)(WorldView, const cq_ray *, int, cq_ray_hit *, uint8_t *, int *, const uint32_t *, unsigned long long *);
    static const bool stepwise = getenv("CQ_RAY_STEPWISE") != nullptr; // the older one-step-per-trip kernels (A/B)
    static const Kernel phased[4] = {k_raycast_phased<false, false>, k_raycast_phased<true, false>, k_raycast_phased<false, true>,
                                     k_raycast_phased<true, true>};
    static const Kernel kernels_old[4] = {k_raycast<false>, k_raycast<true>, k_raycast_ref<false>, k_raycast_ref<true>};
    const Kernel *kernels = stepwise ? kernels_old : phased;
    const Kernel kernel = kernels[ci];
    if (!blocksPerSm[ci]) {
        cudaDeviceProp prop;
        CQ_CUDA(cudaGetDeviceProperties(&prop, w->device));
        numSms = prop.multiProcessorCount;
        int b = 0;
        CQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel, Q_THREADS, 0));
        blocksPerSm[ci] = b > 0 ? b : 1;
    }
    int blocks = std::min(cdiv(n, Q_THREADS), numSms * blocksPerSm[ci]); // one resident wave of persistent lanes
    int *work = next_work_counter(w, st);
    if (!work) return CQ_ERR_CUDA;
    const uint32_t *order = make_unit_order(w, d_rays, sizeof(cq_ray), false, n, st);
    kernel<<<blocks, Q_THREADS, 0, st>>>(w->view, d_rays, n, d_out, d_flags, work, order, w->dCounters);
    w->launches++;
    return finish_launch(w, st, ref ? "k_raycast_ref" : "k_raycast");
}

#undef CQ_OCC_SLOT
#define CQ_OCC_SLOT 2
int launch_cast(cq_world *w, const cq_capsule_cast *d_q, int n, int mode, cq_cast_hit *d_out, uint8_t *d_flags, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    CQ_TRY(await_trees(w, st));
    int *blocksPerSm = w->occ[CQ_OCC_SLOT]; int &numSms = w->numSms;
    const int ci = (w->counting ? 1 : 0) + 2 * (w->view.stagedLeaves ? 1 : 0);
    using Kernel = void (*)(WorldView, const cq_capsule_cast *, int, int, cq_cast_hit *, uint8_t *, int, uint2 *, int *,
                            const uint32_t *, unsigned long long *);
    static const Kernel kernels[4] = {k_capsule_cast<false, false>, k_capsule_cast<true, false>, k_capsule_cast<false, true>,
                                      k_capsule_cast<true, true>};
    const Kernel kernel = kernels[ci];
    if (!blocksPerSm[ci]) {
        cudaDeviceProp prop;
        CQ_CUDA(cudaGetDeviceProperties(&prop, w->device));
        numSms = prop.multiProcessorCount;
        int b = 0;
        CQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel, Q_THREADS, 0));
        blocksPerSm[ci] = b > 0 ? b : 1;
    }
    int blocks = std::min(cdiv(n, 4), numSms * blocksPerSm[ci]); // one resident wave of persistent lanes
    const int opw = pool_owners_per_warp(n, (long long)blocks * CAST_WARPS);
    int *work = next_work_counter(w, st);
    if (!work) return CQ_ERR_CUDA;
    uint2 *ns = (uint2 *)pool_node_scratch(w, (size_t)blocks * CAST_WARPS, st);
    if (!ns) return CQ_ERR_CUDA;
    const uint32_t *order = make_unit_order(w, d_q, sizeof(cq_capsule_cast), false, n, st);
    kernel<<<blocks, Q_THREADS, 0, st>>>(w->view, d_q, n, mode, d_out, d_flags, opw, ns, work, order, w->dCounters);
    w->launches++;
    return finish_launch(w, st, "k_capsule_cast");
}

#undef CQ_OCC_SLOT
#define CQ_OCC_SLOT (3 + (ALL ? 1 : 0))
template <bool ALL>
static int launch_overlap_pool(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                               uint8_t *d_overflow, cudaStream_t st) {
    if (n <= 0) return CQ_OK;
    CQ_TRY(await_trees(w, st));
    int &numSms = w->numSms;
    const int ci = (w->counting ? 1 : 0) + 2 * (w->view.stagedLeaves ? 1 : 0);
    int &blocksPerSm = w->occ[CQ_OCC_SLOT][ci];
    using Kernel = void (*)(WorldView, const cq_capsule *, int, int, cq_overlap_hit *, int32_t *, uint8_t *, int, uint2 *, int *,
                            unsigned long long *);
    static const Kernel kernels[4] = {k_capsule_overlap_pool<false, ALL, false>, k_capsule_overlap_pool<true, ALL, false>,
                                      k_capsule_overlap_pool<false, ALL, true>, k_capsule_overlap_pool<true, ALL, true>};
    const Kernel kernel = kernels[ci];
    if (!blocksPerSm) {
        cudaDeviceProp prop;
        CQ_CUDA(cudaGetDeviceProperties(&prop, w->device));
        numSms = prop.multiProcessorCount;
        int b = 0;
        CQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel, Q_THREADS, 0));
        blocksPerSm = b > 0 ? b : 1;
    }
    int blocks = std::min(cdiv(n, 4), numSms * blocksPerSm);
    const int opw = pool_owners_per_warp(n, (long long)blocks * CAST_WARPS);
    int *work = next_work_counter(w, st);
    if (!work) return CQ_ERR_CUDA;
    uint2 *ns = (uint2 *)pool_node_scratch(w, (size_t)blocks * CAST_WARPS, st);
    if (!ns) return CQ_ERR_CUDA;
    kernel<<<blocks, Q_THREADS, 0, st>>>(w->view, d_q, n, maxHits, d_out, d_counts, d_overflow, opw, ns, work, w->dCounters);
    w->launches++;
    return finish_launch(w, st, "k_capsule_overlap_pool");
}

int launch_overlap(cq_world *w, const cq_capsule *d_q, int n, cq_overlap_hit *d_out, uint8_t *d_flags, cudaStream_t st) {
    return launch_overlap_pool<false>(w, d_q, n, 1, d_out, nullptr, d_flags, st);
}

int launch_overlap_all(cq_world *w, const cq_capsule *d_q, int n, int maxHits, cq_overlap_hit *d_out, int32_t *d_counts,
                       uint8_t *d_overflow, cudaStream_t st) {
    return launch_overlap_pool<true>(w, d_q, n, maxHits, d_out, d_counts, d_overflow, st);
}

} // namespace cq
