// cq_mas.cu — in-kernel move-and-slide: one fixed step of the reference's
// KinematicMoveStopSystem.fixedUpdate per-entity body (Game/Systems.swift:1842-1901) for a batch of
// independent characters:
//   gravity (SYS:603) -> cache decay (SYS:1105) -> VelocityGate (SYS:1037) -> pre-sweep depenetration
//   (SYS:734,1635) -> <= maxSlideIterations blocking casts + SlideResolver plane clipping (SYS:1229,1658)
//   -> GroundProbe snap/fall/offset casts (SYS:826) -> GroundSnap (SYS:945) -> SlopeFriction (SYS:965)
//   -> writeBack (SYS:1802).
//
// Execution model (cq_pool.cuh): persistent warps; each lane OWNS one character at a time and is a resumable state
// machine.  Its controller working set lives in shared memory (CharCtx), the 168-byte record stays in HBM/L2.  The
// owner posts one collision query at a time into the warp's pool (QShared slot + roots on the warp's node stack); the
// LBVH walk and the (query, triangle) distance evaluations are shared by all 32 lanes of the warp; when the query's
// pending counter returns to zero the owner's logic (`mas_advance`) consumes the result, clips against the contact
// plane, and posts the next query — without leaving the kernel.
// Double precision exactly where the reference uses Double (velocity; SYS:792,882,958,1045,1368).
#include "cq_pool.cuh"
#include <cstring>

#include "cq_internal.h"

namespace cq {

#define MAS_THREADS 128
#ifndef MAS_MIN_BLOCKS
#define MAS_MIN_BLOCKS 5
#endif
#define MAS_WARPS (MAS_THREADS / 32)
#define MAS_SMEM_BYTES \
    (sizeof(CharCtx) * MAS_THREADS + sizeof(QShared) * MAS_THREADS + sizeof(uint32_t) * CQ_POOL_WORDS * MAS_WARPS)

#define MAS_MAX_PLATFORMS 64

struct MasArgs {
    cq_controller_params p;
    float dt;
    float gx, gy, gz;
    uint32_t flags;
    int nPlatforms;
    cq_platform platforms[MAS_MAX_PLATFORMS]; // kinematic platforms travel in the kernel arguments (2.3 KB at most)...
    const cq_platform *dPlatforms;            // ... or, when non-null, in device memory read at execution (any count)
    AgentGrid agents;                         // CQ_MAS_AGENTS: snapshot + grid of this launch
};

// PlatformCarry.computeDelta (SYS:644-732): carry by the platform stood on, push by a platform moving into the side
__device__ __noinline__ f3 platform_carry_delta(f3 position, const cq_controller_params &c, const cq_platform *platforms,
                                                int nPlatforms) {
    float capsuleHalf = c.half_height + c.radius;
    float baseY = position.y - capsuleHalf;
    f3 capMin = {position.x - c.radius, position.y - capsuleHalf, position.z - c.radius};
    f3 capMax = {position.x + c.radius, position.y + capsuleHalf, position.z + c.radius};
    float sideTol = smax(c.skin_width, c.ground_snap_skin);
    f3 bestCarry = {0, 0, 0}, pushDelta = {0, 0, 0};
    for (int k = 0; k < nPlatforms; k++) {
        const cq_platform &pl = platforms[k];
        f3 pDelta = {pl.delta[0], pl.delta[1], pl.delta[2]};
        if (len2(pDelta) < 1e-8f) continue;
        f3 amin = {pl.aabb_min[0], pl.aabb_min[1], pl.aabb_min[2]}, amax = {pl.aabb_max[0], pl.aabb_max[1], pl.aabb_max[2]};
        f3 emin = amin - mk3(sideTol, sideTol, sideTol), emax = amax + mk3(sideTol, sideTol, sideTol);
        bool overlap = capMin.x <= emax.x && capMax.x >= emin.x && capMin.y <= emax.y && capMax.y >= emin.y &&
                       capMin.z <= emax.z && capMax.z >= emin.z;
        if (!overlap) continue;
        bool withinXZ = position.x >= amin.x - c.radius && position.x <= amax.x + c.radius &&
                        position.z >= amin.z - c.radius && position.z <= amax.z + c.radius;
        float topY = amax.y;
        float topTol = c.snap_distance + smax(c.skin_width, c.ground_snap_skin) + 0.05f;
        bool onTop = withinXZ && baseY >= topY - topTol && baseY <= topY + topTol;
        if (onTop) {
            if (len2(pDelta) > len2(bestCarry)) bestCarry = pDelta;
        } else {
            float yMin = amin.y - capsuleHalf, yMax = amax.y + capsuleHalf;
            if (position.y >= yMin && position.y <= yMax) {
                bool outsideX = position.x < amin.x - c.radius || position.x > amax.x + c.radius;
                bool outsideZ = position.z < amin.z - c.radius || position.z > amax.z + c.radius;
                if (!outsideX && !outsideZ) continue;
                float cx = smax(amin.x, smin(position.x, amax.x));
                float cz = smax(amin.z, smin(position.z, amax.z));
                float dx = position.x - cx, dz = position.z - cz;
                float sideDistSq = dx * dx + dz * dz;
                float sidePushTol = c.radius + sideTol;
                if (sideDistSq <= sidePushTol * sidePushTol) {
                    float dirLen = sqrtf(smax(sideDistSq, 0.0f));
                    if (dirLen > 1e-5f) {
                        f3 dir = {dx / dirLen, 0.0f, dz / dirLen};
                        float moveToward = dot(mk3(pDelta.x, 0.0f, pDelta.z), dir);
                        if (moveToward > 0.0f) pushDelta = pushDelta + mk3(pDelta.x, 0.0f, pDelta.z);
                    }
                }
            }
        }
    }
    if (len2(bestCarry) > 1e-8f) return bestCarry;
    if (len2(pushDelta) > 1e-8f) return pushDelta;
    return mk3(0, 0, 0);
}

// AgentSweepSolver.bestHit (SYS:1053-1091) over the grid cells the sweep can reach instead of every agent.  Exact:
// an agent outside the reach box cannot produce a hit, and ties keep the smallest index, which is what the
// reference's strict `<` over its index-ordered loop keeps.  selfIndex: the character's index in the launch (agent G.first + selfIndex).
__device__ __noinline__ bool agent_best_hit(const AgentGrid &G, f3 position, f3 remaining, float remainingLen, float baseMoveLen,
                                            float dt, int selfIndex, float radius, float halfHeight, AgentHit &best) {
    const AgentGridParams gp = *G.params;
    const float timeScale = baseMoveLen > 1e-6f ? smin(remainingLen / baseMoveLen, 1.0f) : 1.0f;
    const float segmentDt = dt * timeScale;
    // XZ reach: both radii + own motion + the fastest agent's motion over the segment, padded against rounding
    const float reach = (2.0f * radius + remainingLen + gp.maxSpeed * fabsf(segmentDt)) * 1.001f + 1e-3f;
    const int ix0 = agent_cell(position.x - reach, gp.originX, gp.invCell, gp.dimX);
    const int ix1 = agent_cell(position.x + reach, gp.originX, gp.invCell, gp.dimX);
    const int iz0 = agent_cell(position.z - reach, gp.originZ, gp.invCell, gp.dimZ);
    const int iz1 = agent_cell(position.z + reach, gp.originZ, gp.invCell, gp.dimZ);
    bool have = false;
    // fast path: the reach stays inside the 3x3 cells around the agent's snapshot cell (the cell size is chosen so
    // that it does unless a platform or a depenetration push moved it far): ranges were found in the pre-pass
    const int4 r0 = __ldg(G.rows + 2 * (size_t)selfIndex), r1 = __ldg(G.rows + 2 * (size_t)selfIndex + 1);
    const bool precomputed = ix0 >= r1.z - 1 && ix1 <= r1.z + 1 && iz0 >= r1.w - 1 && iz1 <= r1.w + 1;
    const int rowLo = precomputed ? r1.w - 1 : iz0, rowHi = precomputed ? r1.w + 1 : iz1;
    for (int iz = rowLo; iz <= rowHi; iz++) {
        int j, end;
        if (precomputed) {
            const int k = iz - (r1.w - 1);
            j = k == 0 ? r0.x : (k == 1 ? r0.z : r1.x);
            end = k == 0 ? r0.y : (k == 1 ? r0.w : r1.y);
        } else {
            const uint32_t keyLo = (uint32_t)iz * (uint32_t)gp.dimX + (uint32_t)ix0, keyHi = keyLo + (uint32_t)(ix1 - ix0);
            int lo = 0, hi = G.n; // lower_bound(keyLo): a row of cells is one contiguous key range
            while (lo < hi) {
                int mid = (lo + hi) >> 1;
                if (__ldg(G.keys + mid) < keyLo) lo = mid + 1;
                else hi = mid;
            }
            j = lo;
            for (end = lo; end < G.n && __ldg(G.keys + end) <= keyHi;) end++;
        }
        for (; j < end; j++) {
            const float4 op = __ldg(G.pos + j);
            const int other = __float_as_int(op.w);
            if (other - G.first == selfIndex) continue;
            // cheap exact reject: farther apart in XZ than the reach -> the sweep cannot hit
            const float dx = op.x - position.x, dz = op.z - position.z;
            if (dx * dx + dz * dz > reach * reach) continue;
            const float4 ov = __ldg(G.vel + j);
            const f3 otherDelta = mk3(ov.x, ov.y, ov.z) * segmentDt;
            AgentHit hit;
            if (capsule_pair_sweep(position, remaining, radius, halfHeight, other, mk3(op.x, op.y, op.z), otherDelta, radius,
                                   halfHeight, hit)) {
                if (!have || hit.toi < best.toi || (hit.toi == best.toi && hit.other < best.other)) {
                    best = hit;
                    have = true;
                }
            }
        }
    }
    return have;
}

// What a character brings into its fixed step: GravitySystem (SYS:603-619), positionF, applyPlatformDelta
// (SYS:1618-1633), VelocityGate (SYS:1037-1051).  Shared by the kernel's load stage and the agent pre-pass so that
// both derive bit-identical sweep inputs.
__device__ __forceinline__ void mas_entry_motion(const cq_character_state &S, const MasArgs &A, f3 &pos, f3 &rem, d3 &vel) {
    const bool wasGrounded = S.grounded != 0, wasGroundedNear = S.grounded_near != 0;
    vel = d3{S.velocity[0], S.velocity[1], S.velocity[2]};
    if (A.flags & CQ_MAS_APPLY_GRAVITY) {
        if (!(wasGrounded && wasGroundedNear)) vel = vel + to_d3(mk3(A.gx, A.gy, A.gz)) * (double)A.dt;
    }
    pos = mk3((float)S.position[0], (float)S.position[1], (float)S.position[2]);
    if (A.nPlatforms > 0) {
        f3 platformDelta = platform_carry_delta(pos, A.p, A.dPlatforms ? A.dPlatforms : A.platforms, A.nPlatforms);
        if (len2(platformDelta) > 1e-8f) pos = pos + platformDelta;
    }
    if (wasGrounded && wasGroundedNear && vel.y < 0.0) vel.y = 0.0;
    d3 remD = vel * (double)A.dt;
    if (wasGrounded && wasGroundedNear && remD.y < 0.0) remD.y = 0.0;
    rem = to_f3(remD);
}

// Agent pre-pass: the agent hit of every character's FIRST slide iteration, one thread per character at full
// occupancy.  Valid whenever depenetration leaves the character alone (the kernel checks); later iterations and
// pushed characters run agent_best_hit inside the kernel.
__global__ void k_agent_first_hit(const cq_character_state *__restrict__ states, int n, const __grid_constant__ MasArgs A) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f3 pos, rem;
    d3 vel;
    mas_entry_motion(states[i], A, pos, rem, vel);
    const float slideLen = len(rem);
    float4 out = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
    if (!(slideLen < 1e-6f)) {
        const float baseMoveLen = len(to_f3(vel) * A.dt);
        AgentHit hit;
        if (agent_best_hit(A.agents, pos, rem, slideLen, baseMoveLen, A.dt, i, A.p.radius, A.p.half_height, hit))
            out = make_float4(hit.normal.x, hit.normal.y, hit.normal.z, hit.toi);
    }
    A.agents.firstHit[i] = out;
}

enum { W_NONE = 0, W_DEPEN, W_SLIDE, W_SNAP, W_FALL, W_OFFSET };
enum { NX_LOAD = 0, NX_DEPEN, NX_SLIDE, NX_SNAP, NX_FALL, NX_GATE, NX_OFFSET, NX_FINISH, NX_POST };
#ifndef CQ_MAS_FE_IDLE
#define CQ_MAS_FE_IDLE 16 /* idle lanes that open the front end (cq_pool.cuh: pool_run); >= 16 also selects the readiness rule */
#endif
enum {
    F_WAS_G = 1, F_WAS_GN = 2, F_HAVE_LAST = 4, F_HAVE_CENTER = 8, F_GROUNDED = 16, F_GROUNDED_NEAR = 32,
    F_CAN_SNAP = 64, F_NEAR_GROUND = 128, F_PROBE_HIT = 256, F_DID_RESOLVE = 512
};

struct CharCtx { // per-lane controller working set, shared memory (the 168-byte record itself stays in HBM/L2:
                 // it is touched only by the owner's logic, a few times per step, and keeping it out of shared
                 // memory lets 5-6 CTAs share an SM instead of 4)
    cq_character_state *st;
    float pos[3], rem[3], lastN[3];
    float slideLen;
    float cNormal[3], cTriNormal[3];
    float cToi, cPosY;
    int cTri, cPart;
    float gDistance;
    float nSum[3];
    float combineTol; // slide phase (agents): baseMoveLen
    float dSum[3];
    float dWeight;
    int wait, slideIt, offsetIt, depenIt;
    uint32_t flags;
    int charIndex;
    int _pad;
};

__device__ __forceinline__ f3 ld3(const float *p) { return {p[0], p[1], p[2]}; }
__device__ __forceinline__ void st3(float *o, f3 v) {
    o[0] = v.x;
    o[1] = v.y;
    o[2] = v.z;
}
__device__ __forceinline__ d3 ldv(const cq_character_state &s) { return {s.velocity[0], s.velocity[1], s.velocity[2]}; }
__device__ __forceinline__ void stv(cq_character_state &s, d3 v) {
    s.velocity[0] = v.x;
    s.velocity[1] = v.y;
    s.velocity[2] = v.z;
}

// ---- ContactManifoldCache / DefaultContactCachePolicy (SYS:1102-1205)
__device__ __forceinline__ bool manifold_normal_for(const cq_character_state &c, int tri, f3 &out) {
    int cnt = c.manifold_count;
    for (int i = 0; i < cnt; i++)
        if (c.manifold_triangles[i] == tri) {
            out = ld3(c.manifold_normals[i]);
            return true;
        }
    return false;
}

__device__ __noinline__ void manifold_update(cq_character_state &c, int tri, f3 normal) {
    f3 n = normal;
    if (len2(n) < 1e-8f) return;
    c.manifold_frames = 8;
    int cnt = c.manifold_count;
    for (int i = 0; i < cnt; i++) {
        if (c.manifold_triangles[i] == tri) {
            f3 cached = ld3(c.manifold_normals[i]);
            if (dot(cached, n) < 0.0f) n = -n;
            const float blend = 0.25f;
            f3 combined = normalize(cached * (1.0f - blend) + n * blend);
            st3(c.manifold_normals[i], combined);
            st3(c.side_contact_normal, combined);
            return;
        }
    }
    if (cnt >= CQ_MANIFOLD_MAX) cnt -= 1; // removeLast
    for (int i = cnt; i > 0; i--) {      // insert at 0
        c.manifold_triangles[i] = c.manifold_triangles[i - 1];
        st3(c.manifold_normals[i], ld3(c.manifold_normals[i - 1]));
    }
    f3 nn = normalize(n);
    c.manifold_triangles[0] = tri;
    st3(c.manifold_normals[0], nn);
    c.manifold_count = cnt + 1;
    st3(c.side_contact_normal, nn);
}

__device__ __forceinline__ void cache_record(cq_character_state &c, int tri, f3 normal, bool isSide) {
    manifold_update(c, tri, normal);
    if (isSide) {
        st3(c.side_contact_normal, normalize(normal));
        c.side_contact_frames = 3;
    }
}

// SlideResolver.resolveHit, kinematicMove options, static hit (SYS:1229-1375).  Returns shouldBreak.
// `isStatic` false selects the .agentHit case: no skin, never ground-like, no cached side normal.
__device__ __forceinline__ bool slide_resolve(CharCtx &c, const cq_controller_params &P, f3 hitN, f3 hitTriN, float hitToi,
                                              bool haveCachedSide, f3 cachedSide, int sideFrames, bool isStatic) {
    const bool wasGrounded = c.flags & F_WAS_G, wasGroundedNear = c.flags & F_WAS_GN;
    f3 position = ld3(c.pos), remaining = ld3(c.rem);
    const float slideLen = c.slideLen;
    f3 slideNormal = hitN;
    bool groundLike = isStatic && hitTriN.y >= P.min_ground_dot;
    float contactSkin = !isStatic ? 0.0f : (groundLike ? P.ground_snap_skin : P.skin_width); // SYS:1255-1271
    bool shouldBreak = false;
    if (isStatic && slideNormal.y < P.min_ground_dot && sideFrames > 0) { // SYS:1273-1292
        if (haveCachedSide) {
            f3 cn = cachedSide;
            if (dot(cn, slideNormal) < 0.0f) cn = -cn;
            slideNormal = cn;
        } else {
            f3 cached = ld3(c.st->side_contact_normal);
            float cl = len2(cached);
            if (cl > 1e-6f) {
                f3 cn = cached / sqrtf(cl);
                float dc = dot(cn, slideNormal);
                if (fabsf(dc) > 0.5f) slideNormal = dc >= 0.0f ? cn : -cn;
            }
        }
    }
    bool resolved = false;
    if (slideNormal.y < P.min_ground_dot) { // SYS:1294-1309
        if (groundLike) slideNormal = hitTriN;
        if (slideNormal.y < P.min_ground_dot) {
            slideNormal.y = 0.0f;
            float nl = len(slideNormal);
            if (nl > 1e-5f) {
                slideNormal = slideNormal / nl;
            } else {
                position = position + remaining;
                remaining = mk3(0, 0, 0);
                shouldBreak = true;
                resolved = true;
            }
        }
    }
    if (!resolved) {
        float into = dot(remaining, slideNormal);
        float intoEps = 1e-4f * slideLen;
        float effectiveSkin = (hitToi <= contactSkin && into < -intoEps) ? smin(contactSkin, hitToi * 0.5f) : contactSkin;
        float sticky = contactSkin * 0.1f;
        if (hitToi <= sticky && into < -intoEps) { // SYS:1320
            remaining = remaining - slideNormal * into;
            shouldBreak = false;
        } else if (into >= -intoEps) { // SYS:1324
            if (wasGroundedNear && isStatic && !groundLike && remaining.y < 0.0f) remaining.y = 0.0f;
            position = position + remaining;
            remaining = mk3(0, 0, 0);
            shouldBreak = true;
        } else if ((hitToi <= effectiveSkin && fabsf(into) <= intoEps) || into >= 0.0f) {
            position = position + remaining;
            remaining = mk3(0, 0, 0);
            shouldBreak = true;
        } else {
            float moveDist = smax(hitToi - effectiveSkin, 0.0f); // SYS:1343
            if (slideNormal.y >= P.min_ground_dot && remaining.y < 0.0f && moveDist > P.ground_sweep_max_step)
                moveDist = P.ground_sweep_max_step;
            f3 dir = remaining / slideLen;
            position = position + dir * moveDist;
            f3 leftover = remaining - dir * moveDist;
            leftover = leftover - slideNormal * dot(leftover, slideNormal);
            if (wasGrounded && wasGroundedNear && leftover.y < 0.0f) leftover.y = 0.0f;
            float residual = dot(leftover, slideNormal);
            if (fabsf(residual) < 1e-5f) leftover = leftover - slideNormal * residual;
            if (len2(leftover) < 1e-8f) {
                remaining = mk3(0, 0, 0);
                shouldBreak = true;
            } else {
                remaining = leftover;
                d3 vel = ldv(*c.st);
                d3 sn = to_d3(slideNormal);
                double vInto = dot(vel, sn); // SYS:1367-1372
                if (vInto < 0.0) stv(*c.st, vel - sn * vInto);
                shouldBreak = false;
            }
        }
    }
    st3(c.pos, position);
    st3(c.rem, remaining);
    return shouldBreak;
}

// GroundProbe tail + GroundSnap + SlopeFriction + writeBack (SYS:923-1021, 1787-1821)
__device__ __forceinline__ void mas_finish(CharCtx &c, const WorldView &W, const MasArgs &A, cq_character_state *out,
                                           bool count, uint32_t evalsNow) {
    const cq_controller_params &P = A.p;
    cq_character_state &S = *c.st;
    const f3 gravity = {A.gx, A.gy, A.gz};
    const bool wasGroundedNear = c.flags & F_WAS_GN;
    const bool grounded = c.flags & F_GROUNDED;
    f3 position = ld3(c.pos);
    d3 vel = ldv(S);
    f3 centerTriNormal = ld3(c.cTriNormal), centerNormal = ld3(c.cNormal);
    f3 gNormal = {0, 1, 0};
    float matMuS = 0.8f, matMuK = 0.6f;
    bool matFlatten = false;
    if (grounded) {
        f3 normalSum = ld3(c.nSum);
        float nl = len(normalSum);
        gNormal = nl > 1e-6f ? normalSum / nl : centerTriNormal;
        if (wasGroundedNear) {
            f3 prevNormal = ld3(S.ground_normal);
            if (dot(prevNormal, gNormal) > 0.9f) {
                const float blend = 0.2f;
                gNormal = normalize(prevNormal * (1.0f - blend) + gNormal * blend);
            }
        }
        if (c.cPart >= 0 && c.cPart < W.nMaterials) { // (cPart: row of the material table)
            float4 m = __ldg(W.materials + c.cPart);
            matMuS = m.x, matMuK = m.y, matFlatten = m.z != 0.0f;
        }
        if (matFlatten) gNormal = mk3(0, 1, 0);
    }
    if ((c.flags & F_CAN_SNAP) && (c.flags & F_PROBE_HIT)) { // GroundSnap.apply (SYS:945-963)
        float moveDist = smax(c.cToi - P.ground_snap_skin, 0.0f);
        if ((c.flags & F_NEAR_GROUND) && moveDist > P.ground_snap_max_step) moveDist = P.ground_snap_max_step;
        position = position + mk3(0.0f, -1.0f, 0.0f) * moveDist;
        d3 cn = to_d3(centerNormal);
        double vIntoSnap = dot(vel, cn);
        if (vIntoSnap < 0.0) vel = vel - cn * vIntoSnap;
    }
    int transitionFrames = S.ground_transition_frames;
    bool sliding = S.ground_sliding != 0;
    if (grounded) { // SYS:1787-1792
        float normalUpDelta = gNormal.y - S.ground_normal[1];
        if (c.cTri != S.ground_triangle_index && normalUpDelta > 0.02f) transitionFrames = 3;
    }
    if (!grounded) { // SlopeFriction.apply (SYS:965-1021)
        sliding = false;
    } else {
        f3 normal = normalize(gNormal);
        if (normal.y > 0.98f) {
            transitionFrames = 0;
            sliding = false;
        } else if (transitionFrames > 0) {
            transitionFrames -= 1;
            sliding = false;
        } else {
            float gN = dot(gravity, normal);
            f3 gTan = gravity - normal * gN;
            float gTanLen = len(gTan);
            if (gTanLen > 0.5f) {
                float gNMag = fabsf(gN);
                f3 gTanDir = gTan / gTanLen;
                d3 gTanDirD = to_d3(gTanDir), normalD = to_d3(normal);
                float stickLimit = matMuS * gNMag;
                bool enterSlide = gTanLen > stickLimit * 1.05f;
                bool exitSlide = gTanLen < stickLimit * 0.9f;
                if (sliding) {
                    if (exitSlide) sliding = false;
                } else if (enterSlide) {
                    sliding = true;
                }
                if (!sliding && gTanLen <= stickLimit) {
                    d3 vTan = vel - normalD * dot(vel, normalD);
                    double downhill = dot(vTan, gTanDirD);
                    if (downhill > 0.0) vel = vel - gTanDirD * downhill;
                } else {
                    float slideAccelMag = smax(gTanLen - matMuK * gNMag, 0.0f);
                    if (slideAccelMag > 0.0f) vel = vel + gTanDirD * (double)slideAccelMag * (double)A.dt;
                }
            }
        }
    }
    // writeBack (SYS:1802-1821)
    S.position[0] = (double)position.x;
    S.position[1] = (double)position.y;
    S.position[2] = (double)position.z;
    stv(S, vel);
    S.grounded = grounded ? 1 : 0;
    S.grounded_near = (c.flags & F_GROUNDED_NEAR) ? 1 : 0;
    S.ground_sliding = sliding ? 1 : 0;
    S.ground_transition_frames = transitionFrames;
    st3(S.ground_normal, grounded ? gNormal : mk3(0, 1, 0));
    S.ground_distance = c.gDistance;
    if (grounded) S.ground_triangle_index = c.cTri;
    if (count) { // counting build only: distance evaluations spent on this character -> _pad[1..4] (debug)
        uint32_t e = evalsNow - (uint32_t)c._pad;
        S._pad[1] = e & 255u, S._pad[2] = (e >> 8) & 255u, S._pad[3] = (e >> 16) & 255u, S._pad[4] = (e >> 24) & 255u;
    }
    (void)out; // the record was updated in place
}

// Stage L of the move-and-slide kernel: consume the finished query, run the controller logic up to the
// next query, post it.  Returns false when the lane has no more characters.
template <bool COUNT, bool AGENTS>
__device__ __forceinline__ bool mas_advance(CharCtx &c, const QResult &q, QShared &s, const WarpPool &wp, int lane,
                                            const WorldView &W, const MasArgs &A, cq_character_state *states, int n,
                                            int *workCounter, const uint32_t *order, Counters &ctr) {
    const cq_controller_params &P = A.p;
    const f3 down = {0.0f, -1.0f, 0.0f};
    int next = NX_LOAD;
    f3 postFrom = {0.0f, 0.0f, 0.0f}, postDelta = {0.0f, 0.0f, 0.0f};
    int postMode = CQ_MODE_ALL, postWait = W_NONE;
    float postMinY = 0.0f;
    // ---------------- consume
    switch (c.wait) {
    case W_DEPEN: { // DepenetrationResolver.resolve loop body after the overlap query (SYS:756-799)
        if (W.rank) { // more than maxHits triangles overlap: the reference only ever saw the first eight it visited (CQ:1272-1274)
            const int *ov = ovl_words(s);
            if (ov[OVL_TOTAL] > CQ_MAX_OVERLAP_HITS) { // (-1 after the second pass)
                pool_post_first_hits(W.encOfRank, wp.ring, wp.tail, lane, s);
                return true; // still waiting in W_DEPEN, now for the eight pairs
            }
        }
        next = NX_SLIDE;
        float d0 = q.bestT, d1 = q.bestPos.x;
        int t0 = q.bestTri, t1 = q.bestPart;
        f3 n0 = q.bestN, n1 = q.bestTriN;
        if (t0 >= 0) {
            bool sideContact = n0.y < P.min_ground_dot;
            int useCount = sideContact ? 1 : (t1 >= 0 ? 2 : 1);
            float maxDepth = d0;
            f3 frameNormal = {0, 0, 0};
            for (int k = 0; k < useCount; k++) {
                float hd = k == 0 ? d0 : d1;
                int ht = k == 0 ? t0 : t1;
                f3 hn = k == 0 ? n0 : n1;
                maxDepth = smax(maxDepth, hd);
                f3 nn = hn;
                f3 cached;
                if (manifold_normal_for(*c.st, ht, cached)) nn = cached; // SYS:770-776
                frameNormal = frameNormal + nn * hd;
                cache_record(*c.st, ht, nn, hn.y < P.min_ground_dot);
            }
            float fl = len(frameNormal);
            f3 depenNormal = fl > 1e-6f ? frameNormal / fl : frameNormal;
            const float slop = smax(P.skin_width * 0.5f, 0.001f);
            float push = sideContact ? smax(maxDepth, 0.0f) : smax(maxDepth + slop, 0.0f);
            if (sideContact) push = smin(push, P.skin_width);
            if (!(push <= 1e-6f)) {
                st3(c.pos, ld3(c.pos) + depenNormal * push);
                d3 vel = ldv(*c.st);
                d3 dn = to_d3(depenNormal);
                double vInto = dot(vel, dn);
                if (vInto < 0.0) stv(*c.st, vel - dn * vInto);
                c.flags |= F_DID_RESOLVE;
                st3(c.dSum, ld3(c.dSum) + depenNormal * maxDepth);
                c.dWeight += maxDepth;
                if (++c.depenIt < 4) next = NX_DEPEN;
            }
        }
        if (next == NX_SLIDE && (c.flags & F_DID_RESOLVE)) { // SYS:800-807, 1651-1654
            f3 normalSum = ld3(c.dSum);
            f3 depenN = c.dWeight > 1e-6f ? normalize(normalSum / c.dWeight) : normalize(normalSum);
            f3 remaining = ld3(c.rem);
            float into = dot(remaining, depenN);
            if (into < 0.0f) st3(c.rem, remaining - depenN * into);
        }
        break;
    }
    case W_SLIDE: { // resolveKinematicSweep loop body after the blocking cast (SYS:1683-1763)
        c.slideIt++;
        const bool haveHit = q.bestTri >= 0;
        f3 hitN = q.bestN;
        f3 hitTriN = q.bestTriN;
        float hitToi = q.bestT;
        const int tri = q.bestTri;
        bool haveCachedSide = false;
        f3 cachedSide = {0, 0, 0};
        const int sideFrames = c.st->side_contact_frames;
        if (haveHit && hitN.y < P.min_ground_dot && sideFrames > 0) { // SYS:1683-1694
            f3 cached;
            if (manifold_normal_for(*c.st, tri, cached)) {
                if (dot(cached, hitN) < 0.0f) cached = -cached;
                hitN = cached;
            }
        }
        bool useAgent = false;
        if (AGENTS) { // AgentSweepSolver.bestHit + HitSelector.selectBestHit (SYS:1695-1705, 1378-1399)
            AgentHit aHit;
            bool haveAgent;
            if (c.slideIt == 1 && !(c.flags & F_DID_RESOLVE)) { // untouched since load: the pre-pass had the same inputs
                const float4 m = __ldg(A.agents.firstHit + c.charIndex);
                haveAgent = m.w != -1.0f;
                aHit.toi = m.w, aHit.normal = mk3(m.x, m.y, m.z), aHit.other = -1;
            } else {
                haveAgent = agent_best_hit(A.agents, ld3(c.pos), ld3(c.rem), c.slideLen, c.combineTol, A.dt, c.charIndex,
                                           P.radius, P.half_height, aHit);
            }
            if (haveAgent) {
                useAgent = true;
                if (haveHit) {
                    float staticSkin = hitN.y >= P.min_ground_dot ? P.ground_snap_skin : P.skin_width;
                    float staticStop = smax(hitToi - staticSkin, 0.0f), agentStop = smax(aHit.toi, 0.0f);
                    useAgent = !(staticStop <= agentStop);
                }
                if (useAgent) hitN = aHit.normal, hitTriN = mk3(0, 0, 0), hitToi = aHit.toi;
            }
        }
        if (!haveHit && !useAgent) {
            st3(c.pos, ld3(c.pos) + ld3(c.rem));
            st3(c.rem, mk3(0, 0, 0));
            next = NX_SNAP;
            break;
        }
        const bool sideCache = !useAgent && hitN.y < P.min_ground_dot;
        if (sideCache && sideFrames > 0) haveCachedSide = manifold_normal_for(*c.st, tri, cachedSide);
        bool shouldBreak = slide_resolve(c, P, hitN, hitTriN, hitToi, haveCachedSide, cachedSide, sideFrames, !useAgent);
        if (sideCache) cache_record(*c.st, tri, hitN, true); // SYS:1738-1743
        if (c.flags & F_HAVE_LAST) {                                       // SYS:1744-1754
            f3 last = ld3(c.lastN);
            float dn = dot(last, hitN);
            if (fabsf(dn) < 0.98f) {
                f3 axis = cross(last, hitN);
                float al = len(axis);
                if (al > 1e-5f) {
                    f3 an = axis / al;
                    st3(c.rem, an * dot(ld3(c.rem), an));
                }
            }
        }
        st3(c.lastN, hitN);
        c.flags |= F_HAVE_LAST;
        next = shouldBreak ? NX_SNAP : NX_SLIDE;
        break;
    }
    case W_SNAP: // centre ground cast (SYS:844-853)
        if (q.bestTri >= 0) {
            c.flags |= F_HAVE_CENTER;
            c.cToi = q.bestT;
            c.cPosY = q.bestPos.y;
            st3(c.cNormal, q.bestN);
            st3(c.cTriNormal, q.bestTriN);
            c.cTri = q.bestTri;
            c.cPart = world_material_row(W, q.bestTri);
        }
        // Dead-query elimination (exact): the fall probe only feeds state.distance (SYS:864), and that field is
        // overwritten by centerHit.toi as soon as the guard `centerHit.toi <= snapDistance` passes (SYS:868-880).
        // Queries have no other side effect, so the 200 m probe is issued only when the guard will fail.
        next = ((c.flags & F_HAVE_CENTER) && c.cToi <= P.snap_distance) ? NX_GATE : NX_FALL;
        break;
    case W_FALL: // fall probe (SYS:855-866)
        if (q.bestTri >= 0) c.gDistance = q.bestT;
        next = NX_GATE;
        break;
    case W_OFFSET: // slope sample casts (SYS:906-921)
        if (q.bestTri >= 0 && q.bestT <= c.cToi + c.combineTol) {
            if (dot(q.bestTriN, ld3(c.cTriNormal)) > 0.98f) st3(c.nSum, ld3(c.nSum) + q.bestTriN);
        }
        next = ++c.offsetIt == 4 ? NX_FINISH : NX_OFFSET;
        break;
    default:
        next = NX_LOAD;
        break;
    }
    // ---------------- post
    while (true) {
        if (next == NX_LOAD) {
            c.charIndex = atomicAdd(workCounter, 1); // dynamic fetch: lanes never wait on a slow neighbour's character
            if (c.charIndex >= n) {
                c.wait = W_NONE;
                return false;
            }
            if (order) c.charIndex = (int)order[c.charIndex]; // Morton-coherent processing order (big worlds)
            c.st = states + c.charIndex;
            cq_character_state &S = *c.st;
            const bool wasGrounded = S.grounded != 0, wasGroundedNear = S.grounded_near != 0;
            c.flags = (wasGrounded ? F_WAS_G : 0) | (wasGroundedNear ? F_WAS_GN : 0);
            f3 position, remaining;
            d3 vel;
            mas_entry_motion(S, A, position, remaining, vel); // gravity, positionF, platform carry, VelocityGate
            st3(c.pos, position);
            { // decay (SYS:1105-1116)
                int scf = S.side_contact_frames;
                if (scf > 0) S.side_contact_frames = scf - 1;
                int mf = S.manifold_frames;
                if (mf > 0) {
                    mf -= 1;
                    S.manifold_frames = mf;
                    if (mf == 0) {
                        S.manifold_count = 0;
                        st3(S.side_contact_normal, mk3(0, 0, 0));
                    }
                }
            }
            stv(S, vel);
            st3(c.rem, remaining);
            c.depenIt = 0, c.slideIt = 0, c.offsetIt = 0;
            c._pad = (int)ctr.evals;
            st3(c.dSum, mk3(0, 0, 0));
            c.dWeight = 0.0f;
            c.gDistance = FLT_MAX;
            c.cTri = -1, c.cPart = -1;
            c.cToi = 0.0f, c.cPosY = 0.0f;
            st3(c.cNormal, mk3(0, 0, 0));
            st3(c.cTriNormal, mk3(0, 0, 0));
            st3(c.nSum, mk3(0, 0, 0));
            next = NX_DEPEN;
        }
        if (next == NX_DEPEN) {
            pool_post_overlap<COUNT>(W, wp, lane, s, ld3(c.pos), P.radius, P.half_height, P.collision_mask, ctr);
            c.wait = W_DEPEN;
            return true;
        }
        if (next == NX_SLIDE) {
            f3 remaining = ld3(c.rem);
            c.slideLen = len(remaining);
            // baseMoveLen = |linearVelocityF * dt| at sweep entry (SYS:1671-1672); parked in combineTol, which the
            // ground probe only starts using after the slide loop
            if (AGENTS && c.slideIt == 0) c.combineTol = len(to_f3(ldv(*c.st)) * A.dt);
            if (c.slideIt >= P.max_slide_iterations || c.slideLen < 1e-6f) { // SYS:1674-1676
                next = NX_SNAP;
            } else {
                postFrom = ld3(c.pos), postDelta = remaining, postMode = CQ_MODE_BLOCKING, postMinY = 0.0f, postWait = W_SLIDE;
                next = NX_POST;
            }
        }
        if (next == NX_SNAP) {
            if (!(P.snap_distance > 0.0f)) { // SYS:845
                next = NX_FALL;
            } else {
                postFrom = ld3(c.pos), postDelta = down * P.snap_distance, postMode = CQ_MODE_GROUND, postMinY = P.min_ground_dot;
                postWait = W_SNAP;
                next = NX_POST;
            }
        }
        if (next == NX_FALL) {
            if (!(P.fall_probe_distance > 0.0f)) { // SYS:855
                next = NX_GATE;
            } else {
                postFrom = ld3(c.pos), postDelta = down * P.fall_probe_distance, postMode = CQ_MODE_GROUND;
                postMinY = P.min_ground_dot, postWait = W_FALL;
                next = NX_POST;
            }
        }
        if (next == NX_GATE) { // validity gates after the centre + fall casts (SYS:868-925)
            next = NX_FINISH;
            if ((c.flags & F_HAVE_CENTER) && c.cToi <= P.snap_distance) {
                const bool wasGroundedNear = c.flags & F_WAS_GN;
                c.flags |= F_PROBE_HIT;
                f3 position = ld3(c.pos);
                float baseCenterY = position.y - P.half_height;
                float bottomY = baseCenterY - P.radius;
                float groundTol = smax(P.skin_width, P.ground_snap_skin);
                bool validGroundPoint = c.cPosY <= bottomY + groundTol;
                float groundNearThreshold = smax(P.ground_snap_skin, P.skin_width);
                bool nearGround = c.cToi <= groundNearThreshold;
                if (nearGround) c.flags |= F_NEAR_GROUND | F_GROUNDED_NEAR;
                c.gDistance = c.cToi;
                d3 vel = ldv(*c.st);
                bool groundGateVel = vel.y <= 0.0;
                double vInto = dot(vel, to_d3(ld3(c.cNormal)));
                bool groundGateSpeed = vInto >= -(double)P.ground_snap_max_speed;
                bool groundGateToi = c.cToi <= P.ground_snap_max_toi;
                bool canSnap = validGroundPoint && groundGateVel && (nearGround || groundGateSpeed || groundGateToi);
                if (wasGroundedNear && c.cToi <= P.snap_distance) canSnap = validGroundPoint;
                if (canSnap) c.flags |= F_CAN_SNAP;
                if (validGroundPoint && (nearGround || canSnap)) {
                    c.flags |= F_GROUNDED;
                    f3 ctn = ld3(c.cTriNormal);
                    st3(c.nSum, ctn);
                    if (ctn.y < 0.98f && (wasGroundedNear || nearGround)) { // SYS:897
                        c.combineTol = smax(smax(P.ground_snap_skin, P.skin_width), 0.05f);
                        c.offsetIt = 0;
                        next = NX_OFFSET;
                    }
                }
            }
        }
        if (next == NX_OFFSET) { // SYS:898-914
            float offset = P.radius * 0.6f;
            int oi = c.offsetIt;
            float ox = oi == 0 ? offset : (oi == 1 ? -offset : 0.0f);
            float oz = oi == 2 ? offset : (oi == 3 ? -offset : 0.0f);
            postFrom = ld3(c.pos) + mk3(ox, 0.0f, oz), postDelta = down * P.snap_distance, postMode = CQ_MODE_GROUND;
            postMinY = P.min_ground_dot, postWait = W_OFFSET;
            next = NX_POST;
        }
        // the one place a sweep is posted from: pool_post_cast is ~150 instructions per inlined copy, and one site instead of
        // four keeps 7 KB of code out of the front end (DESIGN.md §5.1)
        if (next == NX_POST) {
            pool_post_cast<COUNT>(W, wp, lane, s, postFrom, postDelta, P.radius, P.half_height, P.collision_mask, postMode, postMinY,
                                  ctr);
            c.wait = postWait;
            return true;
        }
        if (next == NX_FINISH) {
            mas_finish(c, W, A, states + c.charIndex, COUNT, ctr.evals);
            next = NX_LOAD;
        }
    }
}

template <bool COUNT, bool AGENTS, bool STAGED>
__global__ void __launch_bounds__(MAS_THREADS, MAS_MIN_BLOCKS) k_move_and_slide(WorldView W, cq_character_state *__restrict__ states,
                                                                                int n, const __grid_constant__ MasArgs A,
                                                                                int ownersPerWarp,
                                                                                uint2 *nodeScratch, int *workCounter,
                                                                                const uint32_t *__restrict__ order,
                                                                                unsigned long long *gctr) {
    extern __shared__ __align__(16) unsigned char masSmem[]; // MAS_SMEM_BYTES, dynamic
    CharCtx *ctxs = reinterpret_cast<CharCtx *>(masSmem);
    QShared *qsAll = reinterpret_cast<QShared *>(masSmem + sizeof(CharCtx) * MAS_THREADS);
    uint32_t *words = reinterpret_cast<uint32_t *>(masSmem + (sizeof(CharCtx) + sizeof(QShared)) * MAS_THREADS);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpPool wp;
    pool_bind(wp, qsAll, words, nodeScratch, warp, MAS_WARPS, W.rank, W.status);
    CharCtx &c = ctxs[threadIdx.x];
    c.charIndex = -1;
    c.wait = W_NONE;
    c.flags = 0;
    Counters ctr = {0, 0, 0, 0};
    pool_run<COUNT, STAGED, CQ_MAS_FE_IDLE, false>(W, wp, lane, ownersPerWarp, ctr, [&](QShared &mine, Counters &ct) {
        QResult r;
        pool_read_result(mine, r);
        return mas_advance<COUNT, AGENTS>(c, r, mine, wp, lane, W, A, states, n, workCounter, order, ct);
    }, OverlapTop2{W.rank != nullptr});
    pool_flush_counters(ctr, gctr, COUNT);
}

int launch_move_and_slide(cq_world *w, cq_character_state *d_inout, int n, const cq_controller_params &p, float dt,
                          const float g[3], uint32_t flags, const cq_platform *platforms, const cq_platform *dPlatforms,
                          int nPlatforms, cudaStream_t st, const cq_agent_snapshot *dAgents, int nAgents, int first) {
    if (n <= 0) return CQ_OK;
    if (!dPlatforms && (nPlatforms < 0 || nPlatforms > MAS_MAX_PLATFORMS || (nPlatforms > 0 && !platforms))) {
        set_error("cq_move_and_slide: 0..%d platforms supported, got %d", MAS_MAX_PLATFORMS, nPlatforms);
        return CQ_ERR_INVALID;
    }
    MasArgs A;
    memset(&A, 0, sizeof(A));
    A.p = p;
    A.dt = dt;
    A.gx = g[0], A.gy = g[1], A.gz = g[2];
    A.flags = flags;
    A.nPlatforms = nPlatforms;
    A.dPlatforms = dPlatforms;
    if (!dPlatforms)
        for (int k = 0; k < nPlatforms; k++) A.platforms[k] = platforms[k];
    const bool agents = (flags & CQ_MAS_AGENTS) != 0;
    const int staged = w->view.stagedLeaves ? 1 : 0;
    const int ci = (w->counting ? 1 : 0) + 2 * staged;
    using Kernel = void (*)(WorldView, cq_character_state *, int, const MasArgs, int, uint2 *, int *, const uint32_t *,
                            unsigned long long *);
    static const Kernel kernels[2][4] = {{k_move_and_slide<false, false, false>, k_move_and_slide<true, false, false>,
                                          k_move_and_slide<false, false, true>, k_move_and_slide<true, false, true>},
                                         {k_move_and_slide<false, true, false>, k_move_and_slide<true, true, false>,
                                          k_move_and_slide<false, true, true>, k_move_and_slide<true, true, true>}};
    const Kernel kernel = kernels[agents ? 1 : 0][ci];
    void *agentScratch = nullptr;
    if (!dAgents) nAgents = n, first = 0;
    if (agents) CQ_TRY(take_agent_grid(w, nAgents, n, dAgents == nullptr, st, &agentScratch));
    // persistent lanes: one resident wave of CTAs, lanes stride over characters; small batches still fill the machine
    // (>= 4 units per CTA)
    PoolLaunch L;
    CQ_TRY(pool_launch_setup(w, (const void *)kernel, MAS_THREADS, MAS_SMEM_BYTES, 4, n, true, d_inout, sizeof(cq_character_state),
                             true, st, L));
    if (agents) {
        CQ_TRY(make_agent_grid(w, agentScratch, d_inout, dAgents, nAgents, first, n, p.radius, dt, g, flags, st, A.agents));
        k_agent_first_hit<<<(n + 255) / 256, 256, 0, st>>>(d_inout, n, A);
        w->launches++;
    }
    kernel<<<L.blocks, MAS_THREADS, MAS_SMEM_BYTES, st>>>(w->view, d_inout, n, A, L.ownersPerWarp, L.nodeScratch, L.work, L.order,
                                                          w->dCounters);
    w->launches++;
    return finish_launch(w, st, "k_move_and_slide");
}

} // namespace cq
