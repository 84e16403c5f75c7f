// cq_sep.cu — AgentSeparationSystem.fixedUpdate (Game/Systems.swift:1906-2210) for a batch of characters, with the
// reference's SEQUENTIAL semantics reproduced exactly on the GPU.
//
// The reference resolves overlapping agent pairs in one Gauss-Seidel sweep in entity order: agent i ("turn i") reads
// itself once, then visits the agents j > i registered in the 3x3 grid cells around its current cell, and every
// correction it applies moves the inputs of later pairs.  Two turns commute exactly when they touch disjoint agents.
// Turn h touches h and agents whose REBUILD cell is within 1 of h's CURRENT cell; as long as h has drifted at most R
// cells since the grid was rebuilt (checked at the start of every turn), two turns can only share an agent when their
// rebuild cells are within D = 2(R+1) of each other.  So:
//   * k_sep_count_blockers: blockers(h) = #{h' < h within D cells}; agents without blockers are ready;
//   * rounds: k_sep_turns runs every ready turn (they are pairwise independent, and everything they depend on is
//     finished), k_sep_release decrements the counters of the higher-indexed agents within D cells of each finished
//     one and queues those that reach zero.  The schedule is a topological order of the conflict DAG, hence the result
//     is bit-identical to the sequential loop.  With random entity order the DAG is O(log n) deep.
//   * if any agent drifted more than R cells the sweep is repeated from a saved copy with a larger R.  Every sweep queues
//     its four attempts (R = 1, 3, 7, 15) up front and the device decides which of them run (k_sep_attempt_begin /
//     k_sep_attempt_end), so a call never waits for the device and can be captured in a CUDA graph.
// The world casts inside a turn (SYS:1994-2033) and the per-agent slide + ground snap afterwards (SYS:2043-2117) run on
// the warp-cooperative pair pool (cq_pool.cuh), like every other capsule query of the library.
#include "cq_pool.cuh"
#include <cstdlib>
#include <cstring>
#include <vector>

#include "cq_internal.h"

namespace cq {

#define SEP_THREADS 128
#define SEP_WARPS (SEP_THREADS / 32)

struct SepGridParams {
    int minX, minZ, dimX, dimZ;
    int err; // 1 = the crowd spans more cells than a 32-bit key can number
    int _pad[3];
};

// What the device decided so far in one call (one per call, in the scratch block; zeroed when the call starts).
struct SepState {
    int status; // CQ_SEP_STATUS_*: set once; every later attempt and the post-process then skip
    int done;   // the current sweep had an attempt without drift
    int skip;   // the current attempt does not run (the sweep is done, or the call failed)
    int rounds; // rounds run by every attempt of the call (the synchronous calls count their launches)
    int stalledAt; // turns processed when the schedule stalled (the synchronous calls' error message)
};

struct SepArgs {
    cq_controller_params p;
    float sepMargin, heightMargin, cellSize;
    int useQuery, R, n;
    float4 *pos; // current agents[].position, w = invWeight
    float4 *vel; // current agents[].velocity
    const int2 *cell0;      // rebuild cell of every agent (relative coordinates)
    const uint32_t *keys;   // sorted cell keys
    const uint32_t *sidx;   // agent indices in (cell, index) order = the reference's per-cell lists
    const int4 *rows;       // per agent, 2 x int4: [start, end) of the rows cz-1, cz, cz+1 (cells cx-1..cx+1) around its
                            // REBUILD cell in the sorted arrays — valid for the turn when the agent has not left that cell
    const SepGridParams *gp;
    const int *queue;       // ready turns of this round
    const int *qcount;
    int *flags;             // [0] drift violation, [1] processed turns
};

__device__ __forceinline__ int sep_lower_bound(const uint32_t *keys, int n, uint32_t key) {
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ int sep_upper_bound(const uint32_t *keys, int n, uint32_t key, int lo) {
    int hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (keys[mid] <= key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// collection loop of fixedUpdate (SYS:2151-2176): positionF, linearVelocityF, invWeight = 1 / massWeight
__global__ void k_sep_collect(const cq_character_state *__restrict__ states, const float *__restrict__ massWeight, int n,
                              float4 *pos, float4 *vel, float4 *orig) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const cq_character_state &S = states[i];
    float mw = massWeight ? massWeight[i] : 1.0f;
    float invWeight = mw > 0.0f ? 1.0f / mw : 0.0f;
    float4 p = make_float4((float)S.position[0], (float)S.position[1], (float)S.position[2], invWeight);
    pos[i] = p;
    orig[i] = p;
    vel[i] = make_float4((float)S.velocity[0], (float)S.velocity[1], (float)S.velocity[2], 0.0f);
}

// AgentSeparationGrid.cellCoord (SYS:1939-1943): Int(floor(pos / cellSize)) per axis
__device__ __forceinline__ int sep_cell(float v, float cellSize) {
    float c = floorf(v / cellSize);
    return (int)fminf(fmaxf(c, -1.0e9f), 1.0e9f);
}

__global__ void k_sep_cells(const float4 *__restrict__ pos, int n, float cellSize, int2 *cellRaw, int *bounds) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int v[4] = {INT_MAX, INT_MAX, INT_MIN, INT_MIN};
    if (i < n) {
        float4 p = pos[i];
        int ix = sep_cell(p.x, cellSize), iz = sep_cell(p.z, cellSize);
        cellRaw[i] = make_int2(ix, iz);
        v[0] = ix, v[1] = iz, v[2] = ix, v[3] = iz;
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        int x = v[k];
        for (int o = 16; o > 0; o >>= 1) {
            int y = __shfl_xor_sync(0xffffffffu, x, o);
            x = k < 2 ? min(x, y) : max(x, y);
        }
        if ((threadIdx.x & 31) == 0) {
            if (k < 2) atomicMin(bounds + k, x);
            else atomicMax(bounds + k, x);
        }
    }
}

__global__ void k_sep_bounds_init(int *bounds, int *flags) {
    if (threadIdx.x < 4) bounds[threadIdx.x] = threadIdx.x < 2 ? INT_MAX : INT_MIN;
    if (threadIdx.x < 8) flags[threadIdx.x] = 0;
}

__global__ void k_sep_grid_params(const int *bounds, SepGridParams *gp) {
    long long dx = (long long)bounds[2] - bounds[0] + 1, dz = (long long)bounds[3] - bounds[1] + 1;
    gp->minX = bounds[0], gp->minZ = bounds[1];
    gp->err = (dx <= 0 || dz <= 0 || dx * dz > 0x7fffffffll) ? 1 : 0;
    gp->dimX = gp->err ? 1 : (int)dx;
    gp->dimZ = gp->err ? 1 : (int)dz;
}

__global__ void k_sep_keys(const int2 *__restrict__ cellRaw, int n, const SepGridParams *__restrict__ gp, uint32_t *keys,
                           uint32_t *vals, int2 *cell0) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int2 c = cellRaw[i];
    int cx = c.x - gp->minX, cz = c.y - gp->minZ;
    if (gp->err) cx = 0, cz = 0;
    cell0[i] = make_int2(cx, cz);
    keys[i] = (uint32_t)cz * (uint32_t)gp->dimX + (uint32_t)cx;
    vals[i] = (uint32_t)i;
}

// the three sorted-array ranges of an agent's 3x3 neighbourhood (a row of cells is one contiguous key range, and
// (key, index) order inside it = the reference's dx-then-list order), found once per sweep at full occupancy
__device__ __forceinline__ void sep_row_range(const uint32_t *keys, int n, int dimX, int dimZ, int cx, int z, int &k0, int &k1) {
    k0 = k1 = 0;
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, dimX - 1);
    if (z < 0 || z >= dimZ || x0 > x1) return; // no agent was registered there: `cells[neighbor]` is nil
    const uint32_t keyLo = (uint32_t)z * (uint32_t)dimX + (uint32_t)x0, keyHi = keyLo + (uint32_t)(x1 - x0);
    k0 = sep_lower_bound(keys, n, keyLo);
    k1 = sep_upper_bound(keys, n, keyHi, k0);
}

__global__ void k_sep_rows(const uint32_t *__restrict__ keys, const int2 *__restrict__ cell0,
                           const SepGridParams *__restrict__ gp, int n, int4 *rows) {
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n) return;
    const int2 c = cell0[h];
    int se[6];
    for (int r = 0; r < 3; r++) sep_row_range(keys, n, gp->dimX, gp->dimZ, c.x, c.y + r - 1, se[2 * r], se[2 * r + 1]);
    rows[2 * (size_t)h] = make_int4(se[0], se[1], se[2], se[3]);
    rows[2 * (size_t)h + 1] = make_int4(se[4], se[5], 0, 0);
}

// blockers(h) = lower-indexed agents whose rebuild cell is within D cells (Chebyshev) of h's
__global__ void k_sep_count_blockers(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ sidx,
                                     const int2 *__restrict__ cell0, const SepGridParams *__restrict__ gp, int n, int D,
                                     int *cnt, int *queue, int *qcount, const SepState *S) {
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n || S->skip) return;
    const int dimX = gp->dimX, dimZ = gp->dimZ;
    const int2 c = cell0[h];
    const int x0 = max(c.x - D, 0), x1 = min(c.x + D, dimX - 1);
    int count = 0;
    for (int z = max(c.y - D, 0); z <= min(c.y + D, dimZ - 1); z++) {
        const uint32_t keyLo = (uint32_t)z * (uint32_t)dimX + (uint32_t)x0, keyHi = keyLo + (uint32_t)(x1 - x0);
        for (int k = sep_lower_bound(keys, n, keyLo); k < n && keys[k] <= keyHi; k++)
            if ((int)sidx[k] < h) count++;
    }
    cnt[h] = count;
    if (count == 0) queue[atomicAdd(qcount, 1)] = h;
}

// one thread per (finished turn, row of its D-neighbourhood): release the higher-indexed agents in reach
__global__ void k_sep_release(const int *__restrict__ queue, const int *__restrict__ qcount, const uint32_t *__restrict__ keys,
                              const uint32_t *__restrict__ sidx, const int2 *__restrict__ cell0,
                              const SepGridParams *__restrict__ gp, int n, int D, int *cnt, int *nextQueue, int *nextCount) {
    const int rows = 2 * D + 1;
    const long long total = (long long)*qcount * rows;
    const int dimX = gp->dimX, dimZ = gp->dimZ;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int h = queue[t / rows];
        const int2 c = cell0[h];
        const int z = c.y - D + (int)(t % rows);
        if (z < 0 || z >= dimZ) continue;
        const int x0 = max(c.x - D, 0), x1 = min(c.x + D, dimX - 1);
        const uint32_t keyLo = (uint32_t)z * (uint32_t)dimX + (uint32_t)x0, keyHi = keyLo + (uint32_t)(x1 - x0);
        for (int k = sep_lower_bound(keys, n, keyLo); k < n && keys[k] <= keyHi; k++) {
            const int j = (int)sidx[k];
            if (j > h && atomicSub(cnt + j, 1) == 1) nextQueue[atomicAdd(nextCount, 1)] = j;
        }
    }
}

// The end of a round, inside the CUDA-graph WHILE node that runs the rounds of an attempt on the device (sep_add_attempt
// below): the consumed queue becomes the next round's output.  The body of the loop holds two rounds (the queues swap
// roles); its last node decides whether the body runs again: turns remain, no agent drifted out of the safety radius,
// and the pass retired at least one turn.
// flags: [0] drift violation, [1] processed turns, [2] processed at the end of the previous pass, [3] stalled, [4] rounds
__global__ void k_sep_round_end_dev(int *qcount, int *flags, int *work, int n, int last, cudaGraphConditionalHandle loop) {
    flags[1] += *qcount;
    flags[4] += 1;
    *qcount = 0;
    *work = 0;
    if (last) {
        const int processed = flags[1];
        int go = processed < n && !flags[0];
        if (go && processed == flags[2]) flags[3] = 1, go = 0;
        flags[2] = processed;
        cudaGraphSetConditional(loop, go ? 1u : 0u);
    }
}

// The head of one attempt (safety radius R) of a sweep.  It is queued whatever happened before it, and skips the attempt
// when the sweep is already done or the call failed (a crowd too wide for the grid is caught here, before any round runs
// on the 1x1 fallback grid); otherwise it resets the attempt's counters.  Either way it sets the loop condition of the
// attempt's rounds, whose WHILE node tests it before the first pass.
__global__ void k_sep_attempt_begin(const SepGridParams *gp, int *flags, int *qcount, SepState *S, int first,
                                    cudaGraphConditionalHandle loop) {
    if (first) S->done = 0;
    if (!S->status && gp->err) S->status = CQ_SEP_STATUS_GRID;
    const int skip = S->done || S->status;
    S->skip = skip;
    if (!skip) {
        for (int k = 0; k < 8; k++) flags[k] = 0;
        qcount[0] = qcount[1] = qcount[2] = 0; // both queue counters + the work counter
    }
    cudaGraphSetConditional(loop, skip ? 0u : 1u);
}

// The outcome of an attempt that ran (flags as k_sep_round_end_dev left them): an agent drifted more than R cells, so
// the sweep's inputs are restored for the next attempt (after the last one the call fails); the schedule stalled; or the
// sweep is done.  Grid-stride over the agents for the restore.
__global__ void k_sep_attempt_end(const int *flags, SepState *S, int last, float4 *pos, float4 *vel,
                                  const float4 *__restrict__ posSave, const float4 *__restrict__ velSave, int n) {
    if (S->skip) return;
    const bool drift = flags[0] != 0;
    if (drift)
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            pos[i] = posSave[i];
            vel[i] = velSave[i];
        }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        S->rounds += flags[4];
        if (drift) {
            if (last) S->status = CQ_SEP_STATUS_DRIFT;
        } else if (flags[3]) {
            S->status = CQ_SEP_STATUS_STALLED;
            S->stalledAt = flags[1];
        } else {
            S->done = 1;
        }
    }
}

__global__ void k_sep_status(const SepState *S, int32_t *out) {
    if (out) *out = S->status;
}

// ---------------------------------------------------------------- turns (AgentSeparationResolver.resolve, SYS:1946-2041)
enum { SW_NONE = 0, SW_CASTA, SW_CASTB };

struct SepCtx { // per-lane turn state, shared memory
    int agent, wait;
    float aPos[3], aVel[3]; // `let a = agents[i]`: the copy taken at the start of the turn
    float aInvW;
    float cPos[3], cVel[3]; // agents[i] as the turn's own corrections accumulate
    int cx, cz;             // current cell (relative coordinates)
    int cellIt, k0, k1;     // which of the 3 rows of cells, cursor / end in the sorted arrays
    int rowSE[6];           // the rows' ranges when the agent still sits in its rebuild cell, else rowSE[0] = -1
    int j;                  // the pair in flight
    float nx, nz, penetration;
    float moveA[3], moveB[3], bPos[3];
    int blockedA;
};

__device__ __forceinline__ f3 sld3(const float *p) { return {p[0], p[1], p[2]}; }
__device__ __forceinline__ void sst3(float *o, f3 v) {
    o[0] = v.x;
    o[1] = v.y;
    o[2] = v.z;
}

// position the cursor on row number c.cellIt of the 3x3 block (dz outer, dx inner: SYS:1955-1956)
__device__ __forceinline__ void sep_open_cell(SepCtx &c, const SepArgs &A) {
    if (c.rowSE[0] >= 0) {
        c.k0 = c.rowSE[2 * c.cellIt], c.k1 = c.rowSE[2 * c.cellIt + 1];
        return;
    }
    sep_row_range(A.keys, A.n, A.gp->dimX, A.gp->dimZ, c.cx, c.cz + c.cellIt - 1, c.k0, c.k1);
}

__device__ __forceinline__ void sep_apply_pair(SepCtx &c, const SepArgs &A) { // SYS:2035-2036
    sst3(c.cPos, sld3(c.cPos) + sld3(c.moveA));
    f3 b = sld3(c.bPos) + sld3(c.moveB);
    float4 old = A.pos[c.j];
    A.pos[c.j] = make_float4(b.x, b.y, b.z, old.w);
}

// the blocked / unblocked decision after both casts (SYS:2022-2033); returns false when the pair is skipped
__device__ __forceinline__ bool sep_decide_blocked(SepCtx &c, bool blockedB) {
    const bool blockedA = c.blockedA != 0;
    if (blockedA && !blockedB) {
        sst3(c.moveA, mk3(0, 0, 0));
        sst3(c.moveB, mk3(-c.nx * c.penetration, 0.0f, -c.nz * c.penetration));
    } else if (blockedB && !blockedA) {
        sst3(c.moveB, mk3(0, 0, 0));
        sst3(c.moveA, mk3(c.nx * c.penetration, 0.0f, c.nz * c.penetration));
    } else if (blockedA && blockedB) {
        return false;
    }
    return true;
}

template <bool COUNT>
__device__ __forceinline__ bool sep_advance(SepCtx &c, const QResult &q, QShared &s, const WarpPool &wp, int lane,
                                            const WorldView &W, const SepArgs &A, int *workCounter, Counters &ctr) {
    const cq_controller_params &P = A.p;
    const float eps = 1e-6f;
    int stage = 0; // 0 scan, 1 decide cast B, 2 apply
    bool blockedB = false;
    if (c.wait == SW_CASTA) {
        c.blockedA = (q.bestTri >= 0 && q.bestT <= P.skin_width && q.bestN.y < P.min_ground_dot) ? 1 : 0;
        stage = 1;
    } else if (c.wait == SW_CASTB) {
        blockedB = q.bestTri >= 0 && q.bestT <= P.skin_width && q.bestN.y < P.min_ground_dot;
        stage = 2;
    }
    c.wait = SW_NONE;
    while (true) {
        if (stage == 1) { // cast for B (SYS:2009-2021)
            if (len(sld3(c.moveB)) > eps) {
                pool_post_cast<COUNT>(W, wp, lane, s, sld3(c.bPos), sld3(c.moveB), P.radius, P.half_height, P.collision_mask,
                                      CQ_MODE_BLOCKING, 0.0f, ctr);
                c.wait = SW_CASTB;
                return true;
            }
            blockedB = false;
            stage = 2;
        }
        if (stage == 2) {
            if (sep_decide_blocked(c, blockedB)) sep_apply_pair(c, A);
            c.k0++;
            stage = 0;
        }
        // ---- scan
        if (c.agent < 0) {
            int t = atomicAdd(workCounter, 1);
            if (t >= *A.qcount) return false;
            const int h = A.queue[t];
            c.agent = h;
            const float4 p = A.pos[h], v = A.vel[h];
            sst3(c.aPos, mk3(p.x, p.y, p.z));
            sst3(c.aVel, mk3(v.x, v.y, v.z));
            c.aInvW = p.w;
            sst3(c.cPos, mk3(p.x, p.y, p.z));
            sst3(c.cVel, mk3(v.x, v.y, v.z));
            c.cx = sep_cell(p.x, A.cellSize) - A.gp->minX; // `grid.cellCoord(for: a.position)` at the start of the turn
            c.cz = sep_cell(p.z, A.cellSize) - A.gp->minZ;
            const int2 c0 = A.cell0[h];
            if (abs(c.cx - c0.x) > A.R || abs(c.cz - c0.y) > A.R) atomicExch(A.flags, 1); // drifted too far: schedule unsafe
            c.rowSE[0] = -1;
            if (c.cx == c0.x && c.cz == c0.y) { // still in the rebuild cell: the pre-pass already found the ranges
                const int4 r0 = A.rows[2 * (size_t)h], r1 = A.rows[2 * (size_t)h + 1];
                c.rowSE[0] = r0.x, c.rowSE[1] = r0.y, c.rowSE[2] = r0.z, c.rowSE[3] = r0.w, c.rowSE[4] = r1.x, c.rowSE[5] = r1.y;
            }
            c.cellIt = 0;
            sep_open_cell(c, A);
        }
        bool posted = false;
        while (true) {
            if (c.k0 >= c.k1) {
                if (++c.cellIt == 3) break;
                sep_open_cell(c, A);
                continue;
            }
            const int j = (int)A.sidx[c.k0];
            if (!(j > c.agent)) { // `for j in list where j > i`
                c.k0++;
                continue;
            }
            const float4 bp = A.pos[j];
            const f3 aPos = sld3(c.aPos);
            const float hh = P.half_height;
            const float aMin = aPos.y - hh, aMax = aPos.y + hh, bMin = bp.y - hh, bMax = bp.y + hh;
            const float dx = aPos.x - bp.x, dz = aPos.z - bp.z;
            const float distSq = dx * dx + dz * dz;
            const float skinAllowance = smin(P.skin_width, P.skin_width);
            const float margin = smin(A.sepMargin, skinAllowance);
            const float minDist = P.radius + P.radius + margin;
            const bool heightSeparated = aMax < bMin - A.heightMargin || aMin > bMax + A.heightMargin;
            if (heightSeparated || distSq >= minDist * minDist) {
                c.k0++;
                continue;
            }
            const float dist = sqrtf(smax(distSq, 1e-8f));
            const float nx = dx / dist, nz = dz / dist;
            const float penetration = minDist - dist;
            const float aW = c.aInvW, bW = bp.w;
            const float wSum = aW + bW;
            if (wSum <= 0.0f) {
                c.k0++;
                continue;
            }
            const float corr = penetration / wSum;
            const f3 moveA = {nx * corr * aW, 0.0f, nz * corr * aW};
            const f3 moveB = {-nx * corr * bW, 0.0f, -nz * corr * bW};
            const float4 bv = A.vel[j];
            const f3 aVel = sld3(c.aVel);
            const f3 relV = aVel - mk3(bv.x, bv.y, bv.z);
            const float vn = relV.x * nx + relV.z * nz;
            if (vn < 0.0f) { // SYS:1985-1993
                const float impulse = -vn;
                const float scaleA = aW / wSum, scaleB = bW / wSum;
                c.cVel[0] += nx * impulse * scaleA;
                c.cVel[2] += nz * impulse * scaleA;
                A.vel[j] = make_float4(bv.x - nx * impulse * scaleB, bv.y, bv.z - nz * impulse * scaleB, bv.w);
            }
            c.j = j;
            c.nx = nx, c.nz = nz, c.penetration = penetration;
            sst3(c.moveA, moveA);
            sst3(c.moveB, moveB);
            sst3(c.bPos, mk3(bp.x, bp.y, bp.z));
            c.blockedA = 0;
            if (A.useQuery) {
                if (len(moveA) > eps) { // SYS:1997-2008
                    pool_post_cast<COUNT>(W, wp, lane, s, sld3(c.cPos), moveA, P.radius, P.half_height, P.collision_mask,
                                          CQ_MODE_BLOCKING, 0.0f, ctr);
                    c.wait = SW_CASTA;
                    return true;
                }
                stage = 1;
            } else {
                stage = 2;
                blockedB = false;
            }
            posted = true;
            break;
        }
        if (posted) continue; // run stage 1 / 2 for the pair just found
        // ---- end of the turn: publish agents[i]
        A.pos[c.agent] = make_float4(c.cPos[0], c.cPos[1], c.cPos[2], c.aInvW);
        const float4 v0 = A.vel[c.agent];
        A.vel[c.agent] = make_float4(c.cVel[0], c.cVel[1], c.cVel[2], v0.w);
        c.agent = -1;
    }
}

#define SEP_SMEM_BYTES(CTX) ((sizeof(CTX) + sizeof(QShared)) * SEP_THREADS + sizeof(uint32_t) * CQ_POOL_WORDS * SEP_WARPS)

template <bool COUNT>
__global__ void __launch_bounds__(SEP_THREADS, 4) k_sep_turns(WorldView W, const __grid_constant__ SepArgs A, uint2 *nodeScratch,
                                                              int *workCounter, unsigned long long *gctr) {
    extern __shared__ __align__(16) unsigned char sepSmem[];
    SepCtx *ctxs = reinterpret_cast<SepCtx *>(sepSmem);
    QShared *qsAll = reinterpret_cast<QShared *>(sepSmem + sizeof(SepCtx) * SEP_THREADS);
    uint32_t *words = reinterpret_cast<uint32_t *>(sepSmem + (sizeof(SepCtx) + sizeof(QShared)) * SEP_THREADS);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpPool wp;
    pool_bind(wp, qsAll, words, nodeScratch, warp, SEP_WARPS, W.rank, W.status);
    SepCtx &c = ctxs[threadIdx.x];
    c.agent = -1;
    c.wait = SW_NONE;
    Counters ctr = {0, 0, 0, 0};
    pool_run<COUNT, true, 8, false>(W, wp, lane, 32, ctr, [&](QShared &mine, Counters &ct) {
        QResult r;
        pool_read_result(mine, r);
        return sep_advance<COUNT>(c, r, mine, wp, lane, W, A, workCounter, ct);
    }, OverlapTop2{W.rank != nullptr});
    pool_flush_counters(ctr, gctr, COUNT);
}

// ---------------------------------------------------------------- post-process (SYS:2043-2117) + write-back (:2196-2208)
enum { PW_NONE = 0, PW_SLIDE, PW_SNAP };

struct PostCtx {
    int agent, wait, it, moved;
    float pos[3], rem[3];
    float segLen;
};

// SlideResolver.resolveHit with SlideOptions.agentSeparation, static hit, wasGrounded = wasGroundedNear = false, no
// cached side normal (SYS:1229-1375 with :1218-1221)
__device__ __forceinline__ bool sep_slide_resolve(const cq_controller_params &P, const cq_character_state &S, f3 &position,
                                                  f3 &remaining, float segLen, f3 hitN, f3 hitTriN, float hitToi) {
    if (fabsf(remaining.y) < 1e-5f && hitN.y >= P.min_ground_dot) { // allowHorizontalGroundPass (:1240-1247)
        position = position + remaining;
        remaining = mk3(0, 0, 0);
        return true;
    }
    const float contactSkin = P.skin_width; // useGroundSnapSkinForStatic = false
    f3 slideNormal = hitN;
    (void)hitTriN; // allowTriangleNormalGroundLike = false: the triangle normal is never substituted
    if (slideNormal.y < P.min_ground_dot && S.side_contact_frames > 0) { // :1273-1292, cachedSideNormal == nil
        f3 cached = {S.side_contact_normal[0], S.side_contact_normal[1], S.side_contact_normal[2]};
        float cl = len2(cached);
        if (cl > 1e-6f) {
            f3 cn = cached / sqrtf(cl);
            float dc = dot(cn, slideNormal);
            if (fabsf(dc) > 0.5f) slideNormal = dc >= 0.0f ? cn : -cn;
        }
    }
    if (slideNormal.y < P.min_ground_dot) { // :1294-1309
        slideNormal.y = 0.0f;
        float nl = len(slideNormal);
        if (nl > 1e-5f) {
            slideNormal = slideNormal / nl;
        } else {
            position = position + remaining;
            remaining = mk3(0, 0, 0);
            return true;
        }
    }
    const float into = dot(remaining, slideNormal);
    const float intoEps = 1e-4f * segLen;
    const float effectiveSkin = (hitToi <= contactSkin && into < -intoEps) ? smin(contactSkin, hitToi * 0.5f) : contactSkin;
    const float sticky = contactSkin * 0.1f;
    if (hitToi <= sticky && into < -intoEps) {
        remaining = remaining - slideNormal * into;
        return false;
    }
    if (into >= -intoEps || (hitToi <= effectiveSkin && fabsf(into) <= intoEps) || into >= 0.0f) {
        position = position + remaining;
        remaining = mk3(0, 0, 0);
        return true;
    }
    float moveDist = smax(hitToi - effectiveSkin, 0.0f);
    if (slideNormal.y >= P.min_ground_dot && remaining.y < 0.0f && moveDist > P.ground_sweep_max_step)
        moveDist = P.ground_sweep_max_step;
    const f3 dir = remaining / segLen;
    position = position + dir * moveDist;
    f3 leftover = remaining - dir * moveDist;
    leftover = leftover - slideNormal * dot(leftover, slideNormal);
    const float residual = dot(leftover, slideNormal);
    if (fabsf(residual) < 1e-5f) leftover = leftover - slideNormal * residual;
    if (len2(leftover) < 1e-8f) {
        remaining = mk3(0, 0, 0);
        return true;
    }
    remaining = leftover; // adjustVelocity = false
    return false;
}

struct PostArgs {
    cq_controller_params p;
    int useQuery, n;
    const float4 *pos, *vel, *orig;
    cq_character_state *states;
    const int *status; // SepState::status: a failed call writes no record
};

template <bool COUNT>
__device__ __forceinline__ bool post_advance(PostCtx &c, const QResult &q, QShared &s, const WarpPool &wp, int lane,
                                             const WorldView &W, const PostArgs &A, int *workCounter, Counters &ctr) {
    const cq_controller_params &P = A.p;
    const f3 down = {0.0f, -1.0f, 0.0f};
    enum { N_LOAD, N_SLIDE, N_SNAP, N_FINISH };
    int next = N_LOAD;
    if (c.wait == PW_SLIDE) { // SYS:2061-2084
        f3 position = sld3(c.pos), remaining = sld3(c.rem);
        if (q.bestTri >= 0) {
            bool done = sep_slide_resolve(P, A.states[c.agent], position, remaining, c.segLen, q.bestN, q.bestTriN, q.bestT);
            next = done ? N_SNAP : N_SLIDE;
        } else {
            position = position + remaining;
            remaining = mk3(0, 0, 0);
            next = N_SNAP;
        }
        sst3(c.pos, position);
        sst3(c.rem, remaining);
        c.it++;
    } else if (c.wait == PW_SNAP) { // SYS:2091-2112
        cq_character_state &S = A.states[c.agent];
        if (q.bestTri >= 0 && q.bestT <= P.snap_distance) {
            float rawMove = smax(q.bestT - P.ground_snap_skin, 0.0f);
            float moveDist = smin(rawMove, P.ground_snap_max_step);
            sst3(c.pos, sld3(c.pos) + down * moveDist);
            S.grounded = 1;
            S.grounded_near = q.bestT <= smax(P.ground_snap_skin, P.skin_width) ? 1 : 0;
            bool flatten = false;
            const int row = world_material_row(W, q.bestTri);
            if (row >= 0 && row < W.nMaterials) flatten = __ldg(W.materials + row).z != 0.0f;
            f3 gn = flatten ? mk3(0, 1, 0) : q.bestTriN;
            S.ground_normal[0] = gn.x, S.ground_normal[1] = gn.y, S.ground_normal[2] = gn.z;
            S.ground_triangle_index = q.bestTri;
        }
        next = N_FINISH;
    }
    c.wait = PW_NONE;
    while (true) {
        if (next == N_LOAD) {
            int t = atomicAdd(workCounter, 1);
            if (t >= A.n) return false;
            c.agent = t;
            const float4 p = A.pos[t], o = A.orig[t];
            f3 position = {p.x, p.y, p.z}, start = {o.x, o.y, o.z};
            c.moved = 0;
            c.it = 0;
            sst3(c.rem, mk3(0, 0, 0));
            next = N_FINISH;
            if (A.useQuery) {
                f3 delta = position - start;
                if (len(delta) > 1e-6f) {
                    c.moved = 1;
                    sst3(c.rem, delta);
                    position = start;
                    next = N_SLIDE;
                } else {
                    next = N_SNAP;
                }
            }
            sst3(c.pos, position);
        }
        if (next == N_SLIDE) {
            f3 remaining = sld3(c.rem);
            c.segLen = len(remaining);
            if (c.it >= 2 || c.segLen < 1e-6f) {
                next = N_SNAP;
            } else {
                pool_post_cast<COUNT>(W, wp, lane, s, sld3(c.pos), remaining, P.radius, P.half_height, P.collision_mask,
                                      CQ_MODE_BLOCKING, 0.0f, ctr);
                c.wait = PW_SLIDE;
                return true;
            }
        }
        if (next == N_SNAP) {
            next = N_FINISH;
            if (c.moved && A.states[c.agent].velocity[1] <= 0.0 && P.snap_distance > 0.0f) {
                pool_post_cast<COUNT>(W, wp, lane, s, sld3(c.pos), down * P.snap_distance, P.radius, P.half_height,
                                      P.collision_mask, CQ_MODE_GROUND, P.min_ground_dot, ctr);
                c.wait = PW_SNAP;
                return true;
            }
        }
        if (next == N_FINISH) { // body.position = d3(position); body.linearVelocity = d3(agents[idx].velocity)
            cq_character_state &S = A.states[c.agent];
            const float4 v = A.vel[c.agent];
            S.position[0] = (double)c.pos[0], S.position[1] = (double)c.pos[1], S.position[2] = (double)c.pos[2];
            S.velocity[0] = (double)v.x, S.velocity[1] = (double)v.y, S.velocity[2] = (double)v.z;
            next = N_LOAD;
        }
    }
}

template <bool COUNT>
__global__ void __launch_bounds__(SEP_THREADS, 4) k_sep_post(WorldView W, const __grid_constant__ PostArgs A, uint2 *nodeScratch,
                                                             int *workCounter, unsigned long long *gctr) {
    if (*A.status) return;
    extern __shared__ __align__(16) unsigned char sepSmem[];
    PostCtx *ctxs = reinterpret_cast<PostCtx *>(sepSmem);
    QShared *qsAll = reinterpret_cast<QShared *>(sepSmem + sizeof(PostCtx) * SEP_THREADS);
    uint32_t *words = reinterpret_cast<uint32_t *>(sepSmem + (sizeof(PostCtx) + sizeof(QShared)) * SEP_THREADS);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpPool wp;
    pool_bind(wp, qsAll, words, nodeScratch, warp, SEP_WARPS, W.rank, W.status);
    PostCtx &c = ctxs[threadIdx.x];
    c.agent = -1;
    c.wait = PW_NONE;
    Counters ctr = {0, 0, 0, 0};
    pool_run<COUNT, true, 8, false>(W, wp, lane, 32, ctr, [&](QShared &mine, Counters &ct) {
        QResult r;
        pool_read_result(mine, r);
        return post_advance<COUNT>(c, r, mine, wp, lane, W, A, workCounter, ct);
    }, OverlapTop2{W.rank != nullptr});
    pool_flush_counters(ctr, gctr, COUNT);
}

// ---------------------------------------------------------------- host driver
// One attempt of a sweep as graph nodes: begin -> count blockers -> WHILE{2 x (turns -> release -> round end)} -> end.
// k_sep_round_end_dev sets the loop condition, so the host neither launches rounds nor reads progress back while the
// schedule runs, and k_sep_attempt_begin / k_sep_attempt_end decide on the device whether the attempt runs and what its
// outcome is.  Uncaptured, each attempt is its own instantiated graph, kept per world and keyed by every launch
// parameter (R, and the node-scratch block, which rotates over four buffers: a few entries per crowd size).  Under a
// stream capture the same nodes are added to the capture graph itself (sep_attempt).
struct SepGraph {
    std::vector<unsigned char> key;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    uint64_t used = 0;
};
struct SepGraphCache {
    std::vector<SepGraph> items;
    uint64_t tick = 0;
};

void sep_graphs_destroy(cq_world *w) {
    SepGraphCache *c = (SepGraphCache *)w->sepGraphs;
    if (!c) return;
    for (SepGraph &g : c->items) {
        if (g.exec) cudaGraphExecDestroy(g.exec);
        if (g.graph) cudaGraphDestroy(g.graph);
    }
    delete c;
    w->sepGraphs = nullptr;
}

struct SepAttempt {
    const void *turnKernel;
    int turnBlocks, releaseBlocks;
    size_t turnSmem;
    WorldView view;
    SepArgs A; // queue / qcount are filled per half
    uint2 *ns;
    int *work;
    unsigned long long *counters;
    int *queue[2], *qcount;
    const uint32_t *keys, *vals;
    const int2 *cell0;
    const SepGridParams *gp;
    int n, D, first, last;
    int *cnt, *flags;
    SepState *state;
    float4 *pos, *vel;
    const float4 *posSave, *velSave;
};

static int add_kernel(cudaGraph_t g, cudaGraphNode_t *node, const cudaGraphNode_t *deps, size_t nDeps, const void *func,
                      int blocks, int threads, size_t smem, void **args) {
    cudaKernelNodeParams kp = {};
    kp.func = (void *)func;
    kp.gridDim = dim3(blocks), kp.blockDim = dim3(threads);
    kp.sharedMemBytes = (unsigned)smem;
    kp.kernelParams = args;
    CQ_CUDA(cudaGraphAddKernelNode(node, g, deps, nDeps, &kp));
    return CQ_OK;
}

// adds the attempt's nodes to `g` after `deps`; *end = its last node
static int sep_add_attempt(cudaGraph_t g, const cudaGraphNode_t *deps, size_t nDeps, SepAttempt &L, cudaGraphNode_t *end) {
    cudaGraphConditionalHandle loop;
    CQ_CUDA(cudaGraphConditionalHandleCreate(&loop, g, 0, cudaGraphCondAssignDefault));
    cudaGraphNode_t node;
    void *beginArgs[] = {(void *)&L.gp, (void *)&L.flags, (void *)&L.qcount, (void *)&L.state, (void *)&L.first, (void *)&loop};
    CQ_TRY(add_kernel(g, &node, deps, nDeps, (const void *)k_sep_attempt_begin, 1, 1, 0, beginArgs));
    void *countArgs[] = {(void *)&L.keys, (void *)&L.vals, (void *)&L.cell0, (void *)&L.gp, (void *)&L.n, (void *)&L.D,
                         (void *)&L.cnt, (void *)&L.queue[0], (void *)&L.qcount, (void *)&L.state};
    CQ_TRY(add_kernel(g, &node, &node, 1, (const void *)k_sep_count_blockers, cdiv(L.n, 256), 256, 0, countArgs));
    cudaGraphNodeParams cp = {cudaGraphNodeTypeConditional};
    cp.conditional.handle = loop;
    cp.conditional.type = cudaGraphCondTypeWhile;
    cp.conditional.size = 1;
    CQ_CUDA(cudaGraphAddNode(&node, g, &node, 1, &cp));
    const cudaGraphNode_t whileNode = node;
    cudaGraph_t body = cp.conditional.phGraph_out[0];
    cudaGraphNode_t prev = nullptr;
    for (int half = 0; half < 2; half++) {
        int *q = L.queue[half], *qn = L.queue[half ^ 1];
        int *qc = L.qcount + half, *qcn = L.qcount + (half ^ 1);
        SepArgs A = L.A;
        A.queue = q, A.qcount = qc;
        void *turnArgs[] = {(void *)&L.view, (void *)&A, (void *)&L.ns, (void *)&L.work, (void *)&L.counters};
        CQ_TRY(add_kernel(body, &node, prev ? &prev : nullptr, prev ? 1 : 0, L.turnKernel, L.turnBlocks, SEP_THREADS,
                          L.turnSmem, turnArgs));
        prev = node;
        void *relArgs[] = {(void *)&q, (void *)&qc, (void *)&L.keys, (void *)&L.vals, (void *)&L.cell0, (void *)&L.gp,
                           (void *)&L.n, (void *)&L.D, (void *)&L.cnt, (void *)&qn, (void *)&qcn};
        CQ_TRY(add_kernel(body, &node, &prev, 1, (const void *)k_sep_release, L.releaseBlocks, 256, 0, relArgs));
        prev = node;
        int last = half;
        void *endArgs[] = {(void *)&qc, (void *)&L.flags, (void *)&L.work, (void *)&L.n, (void *)&last, (void *)&loop};
        CQ_TRY(add_kernel(body, &node, &prev, 1, (const void *)k_sep_round_end_dev, 1, 1, 0, endArgs));
        prev = node;
    }
    void *endArgs[] = {(void *)&L.flags, (void *)&L.state, (void *)&L.last, (void *)&L.pos, (void *)&L.vel,
                       (void *)&L.posSave, (void *)&L.velSave, (void *)&L.n};
    return add_kernel(g, end, &whileNode, 1, (const void *)k_sep_attempt_end, L.releaseBlocks, 256, 0, endArgs);
}

// Queues one attempt on `st`: into the capture graph while `st` is captured (cudaStreamGetCaptureInfo gives the graph and
// the current dependencies, cudaStreamUpdateCaptureDependencies makes later work wait for the attempt's last node), else
// as a launch of its cached instantiated graph.  3 kernel launches are counted; the rounds are not known here.
static int sep_attempt(cq_world *w, SepAttempt &L, cudaStream_t st) {
    w->launches += 3;
    if (w->capturing) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        cudaGraph_t g = nullptr;
        const cudaGraphNode_t *d = nullptr;
        size_t nd = 0;
        CQ_CUDA(cudaStreamGetCaptureInfo(st, &cs, nullptr, &g, &d, &nd));
        const std::vector<cudaGraphNode_t> deps(d, d + nd);
        cudaGraphNode_t end;
        CQ_TRY(sep_add_attempt(g, deps.data(), deps.size(), L, &end));
        CQ_CUDA(cudaStreamUpdateCaptureDependencies(st, &end, 1, cudaStreamSetCaptureDependencies));
        return CQ_OK;
    }
    if (!w->sepGraphs) w->sepGraphs = new SepGraphCache();
    SepGraphCache &cache = *(SepGraphCache *)w->sepGraphs;
    L.A.queue = nullptr, L.A.qcount = nullptr;
    std::vector<unsigned char> key(sizeof(L));
    memcpy(key.data(), &L, sizeof(L)); // (L is memset before it is filled: padding compares equal)
    for (SepGraph &g : cache.items)
        if (g.key == key) {
            g.used = ++cache.tick;
            CQ_CUDA(cudaGraphLaunch(g.exec, st));
            return CQ_OK;
        }
    if (cache.items.size() >= 32) { // evict the least recently used
        size_t lru = 0;
        for (size_t i = 1; i < cache.items.size(); i++)
            if (cache.items[i].used < cache.items[lru].used) lru = i;
        cudaGraphExecDestroy(cache.items[lru].exec);
        cudaGraphDestroy(cache.items[lru].graph);
        cache.items.erase(cache.items.begin() + lru);
    }
    SepGraph g;
    g.key = key;
    CQ_CUDA(cudaGraphCreate(&g.graph, 0));
    cudaGraphNode_t end;
    int rc = sep_add_attempt(g.graph, nullptr, 0, L, &end);
    if (rc == CQ_OK) rc = check_cuda(cudaGraphInstantiate(&g.exec, g.graph, 0), "sep graph instantiate");
    if (rc != CQ_OK) {
        cudaGraphDestroy(g.graph);
        return rc;
    }
    g.used = ++cache.tick;
    cache.items.push_back(g);
    CQ_CUDA(cudaGraphLaunch(g.exec, st));
    return CQ_OK;
}

static float sep_cell_size(const cq_controller_params &p, float sepMargin) {
    return std::max(p.radius * 2 + sepMargin, 0.001f); // SYS:2180 (every agent has the controller radius)
}

// Where the scratch block of a call for n agents keeps its small words: bounds[4] flags[8] qcount[2] work[1], the grid
// parameters at +16, the SepState at +24.
static int *sep_small(void *scratch, int n) {
    return (int *)((uint32_t *)((char *)scratch + (size_t)n * (7 * 16 + 2 * 8 + 3 * 4 + 4 * 4)) + sort_scratch_words(n));
}

int launch_agent_separation(cq_world *w, cq_character_state *d_inout, int n, const cq_controller_params &p,
                            const float *d_massWeight, int iterations, float sepMargin, float heightMargin, int useQuery,
                            int32_t *d_status, cudaStream_t st) {
    if (n <= 1) return CQ_OK; // `guard agents.count > 1` (SYS:2178)
    CQ_TRY(await_trees(w, st));
    iterations = std::max(1, iterations);
    const size_t sortWords = sort_scratch_words(n);
    // float4 x5 (pos vel orig posSave velSave), int4 x2 (rows), int2 x2 (cellRaw cell0), int x3 (cnt queueA queueB),
    // u32 x4 (sort), scratch
    const size_t bytes = (size_t)n * (7 * 16 + 2 * 8 + 3 * 4 + 4 * 4) + sortWords * 4 + 256;
    void *sepScratch = nullptr;
    CQ_TRY(take_scratch(w, &w->sepScratch, 1, 0, bytes, st, "agent separation scratch", &sepScratch));
    float4 *pos = (float4 *)sepScratch, *vel = pos + n, *orig = vel + n, *posSave = orig + n, *velSave = posSave + n;
    int4 *rows = (int4 *)(velSave + n);
    int2 *cellRaw = (int2 *)(rows + 2 * (size_t)n), *cell0 = cellRaw + n;
    int *cnt = (int *)(cell0 + n), *queueA = cnt + n, *queueB = queueA + n;
    uint32_t *keys = (uint32_t *)(queueB + n), *vals = keys + n, *keysTmp = vals + n, *valsTmp = keysTmp + n;
    uint32_t *scratch = valsTmp + n;
    int *small = sep_small(sepScratch, n);
    int *bounds = small, *flags = small + 4, *qcount = small + 12, *work = small + 14;
    SepGridParams *gp = (SepGridParams *)(small + 16);
    SepState *state = (SepState *)(small + 24);

    const int ci = w->counting ? 1 : 0;
    const void *turnKernel = ci ? (const void *)k_sep_turns<true> : (const void *)k_sep_turns<false>;
    const void *postKernel = ci ? (const void *)k_sep_post<true> : (const void *)k_sep_post<false>;
    const size_t turnSmem = SEP_SMEM_BYTES(SepCtx), postSmem = SEP_SMEM_BYTES(PostCtx);
    const int turnBlocksMax = resident_blocks(w, turnKernel, SEP_THREADS, turnSmem);
    const int postBlocksMax = resident_blocks(w, postKernel, SEP_THREADS, postSmem);
    if (!turnBlocksMax || !postBlocksMax) return CQ_ERR_CUDA;
    const int turnBlocks = std::min(cdiv(n, 4), turnBlocksMax), postBlocks = std::min(cdiv(n, 4), postBlocksMax);
    const size_t nodeBytes = (size_t)std::max(turnBlocks, postBlocks) * SEP_WARPS * CQ_NSCAP * sizeof(uint2);
    void *nodeScratch = nullptr;
    CQ_TRY(take_scratch(w, w->nodeScratch, 4, w->nodeSeq++ & 3, nodeBytes, st, "node scratch", &nodeScratch));
    uint2 *ns = (uint2 *)nodeScratch;

    const float cellSize = sep_cell_size(p, sepMargin);
    CQ_CUDA(cudaMemsetAsync(state, 0, sizeof(SepState), st));
    k_sep_collect<<<cdiv(n, 256), 256, 0, st>>>(d_inout, d_massWeight, n, pos, vel, orig);
    w->launches++;

    SepAttempt L;
    memset(&L, 0, sizeof(L));
    L.A.p = p;
    L.A.sepMargin = sepMargin, L.A.heightMargin = heightMargin, L.A.cellSize = cellSize;
    L.A.useQuery = useQuery, L.A.n = n;
    L.A.pos = pos, L.A.vel = vel, L.A.cell0 = cell0, L.A.keys = keys, L.A.sidx = vals, L.A.rows = rows, L.A.gp = gp;
    L.A.flags = flags;
    L.turnKernel = turnKernel, L.turnBlocks = turnBlocks, L.releaseBlocks = std::min(cdiv(n, 64), 148 * 8);
    L.turnSmem = turnSmem, L.view = w->view, L.ns = ns, L.work = work, L.counters = w->dCounters;
    L.queue[0] = queueA, L.queue[1] = queueB, L.qcount = qcount;
    L.keys = keys, L.vals = vals, L.cell0 = cell0, L.gp = gp, L.n = n, L.cnt = cnt, L.flags = flags, L.state = state;
    L.pos = pos, L.vel = vel, L.posSave = posSave, L.velSave = velSave;
    for (int it = 0; it < iterations; it++) {
        // grid.rebuild(agents) (SYS:1931-1937): cells of the CURRENT positions; a stable sort keeps each cell's list in
        // ascending agent index = the reference's append order
        k_sep_bounds_init<<<1, 32, 0, st>>>(bounds, flags);
        k_sep_cells<<<cdiv(n, 256), 256, 0, st>>>(pos, n, cellSize, cellRaw, bounds);
        k_sep_grid_params<<<1, 1, 0, st>>>(bounds, gp);
        k_sep_keys<<<cdiv(n, 256), 256, 0, st>>>(cellRaw, n, gp, keys, vals, cell0);
        w->launches += 4;
        CQ_TRY(sort_pairs_u32(w, keys, vals, keysTmp, valsTmp, n, scratch, sortWords, st));
        k_sep_rows<<<cdiv(n, 256), 256, 0, st>>>(keys, cell0, gp, n, rows);
        w->launches++;
        CQ_CUDA(cudaMemcpyAsync(posSave, pos, sizeof(float4) * n, cudaMemcpyDeviceToDevice, st));
        CQ_CUDA(cudaMemcpyAsync(velSave, vel, sizeof(float4) * n, cudaMemcpyDeviceToDevice, st));
        for (int R = 1; R <= 15; R = 2 * R + 1) { // a sweep whose agents drift more than R cells is rerun with a wider R
            L.A.R = R, L.D = 2 * (R + 1);
            L.first = R == 1, L.last = R == 15;
            CQ_TRY(sep_attempt(w, L, st));
        }
    }

    PostArgs PA;
    memset(&PA, 0, sizeof(PA));
    PA.p = p;
    PA.useQuery = useQuery, PA.n = n;
    PA.pos = pos, PA.vel = vel, PA.orig = orig, PA.states = d_inout, PA.status = &state->status;
    CQ_CUDA(cudaMemsetAsync(work, 0, sizeof(int), st));
    void *args[] = {(void *)&w->view, (void *)&PA, (void *)&ns, (void *)&work, (void *)&w->dCounters};
    CQ_CUDA(cudaLaunchKernel(postKernel, dim3(postBlocks), dim3(SEP_THREADS), args, postSmem, st));
    k_sep_status<<<1, 1, 0, st>>>(state, d_status);
    w->launches += 2;
    return finish_launch(w, st, "agent separation");
}

int wait_agent_separation(cq_world *w, int n, const cq_controller_params &p, float sepMargin, cudaStream_t st) {
    if (n <= 1) return CQ_OK;
    const int *small = sep_small(w->sepScratch.ptr, n);
    SepState S;
    CQ_CUDA(cudaMemcpyAsync(&S, small + 24, sizeof(S), cudaMemcpyDeviceToHost, st));
    CQ_CUDA(cudaStreamSynchronize(st));
    w->launches += 3 * (uint64_t)S.rounds;
    switch (S.status) {
    case CQ_SEP_STATUS_OK: return CQ_OK;
    case CQ_SEP_STATUS_GRID:
        set_error("cq_agent_separation: the crowd spans more than 2^31 grid cells of %.3f m", sep_cell_size(p, sepMargin));
        return CQ_ERR_INVALID;
    case CQ_SEP_STATUS_DRIFT:
        set_error("cq_agent_separation: agents drifted more than 15 cells within one sweep");
        return CQ_ERR_INVALID;
    default:
        set_error("cq_agent_separation: the turn schedule stalled at %d of %d agents", S.stalledAt, n);
        return CQ_ERR_CUDA;
    }
}

} // namespace cq
