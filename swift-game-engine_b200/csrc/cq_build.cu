// cq_build.cu — mesh upload + LBVH build/refit on the device (sm_100a).
//
// Replaces, B200-first, what the reference does on one CPU thread:
//   TriangleMeshSet.rebuild           CollisionQuery.swift:331-417  -> k_transform, k_filter_flags, k_compact
//   StaticTriMesh.BVH.build (top-down median split, :577-670) -> LBVH: k_centroid_bounds, k_morton,
//        radix sort (rs_*), k_karras (Karras 2012 radix tree), k_fit (bottom-up boxes)
//   TriangleMeshSet.updateTransforms  :419-462 + BVH.refit :528-575 -> k_update_parts + dirty-subtree refit or k_fit
// The tree differs from the reference's (allowed: capsule candidate sets are tree-independent,
// SURVEY.md §A.4); triangle NUMBERING and world-space vertices are bit-identical to the reference's.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "cq_internal.h"
#include "cq_reftree.h"

namespace cq {

// ---------------------------------------------------------------- small helpers
__device__ __forceinline__ int float_to_ordered(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

// simd_mul(modelMatrix, (p,1)) = ((c0*x + c1*y) + c2*z) + c3*1   (CollisionQuery.swift:349-351)
__device__ __forceinline__ float4 transform_point(const float *m, float4 p) {
    float x = ((m[0] * p.x + m[4] * p.y) + m[8] * p.z) + m[12] * 1.0f;
    float y = ((m[1] * p.x + m[5] * p.y) + m[9] * p.z) + m[13] * 1.0f;
    float z = ((m[2] * p.x + m[6] * p.y) + m[10] * p.z) + m[14] * 1.0f;
    return make_float4(x, y, z, 0.0f);
}

__global__ void k_transform(const float4 *__restrict__ local, float4 *__restrict__ world, const float *__restrict__ models,
                            int lo, int hi) {
    int i = lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    float4 p = local[i];
    world[i] = transform_point(models + 16 * __float_as_int(p.w), p);
}

// ---- mesh upload, device half (cq_assemble.h): the raw arrays of the parts -> the set's input arrays
// packed xyz -> float4 (x, y, z, bits(part index)): one vertex per thread, the 12-byte reads of a warp are contiguous
__global__ void k_expand_verts(const float *__restrict__ raw, int nVerts, const PartRow *__restrict__ rows, int nRows,
                               float4 *__restrict__ local) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nVerts) return;
    const int r = part_row_of(rows, nRows, i, false);
    local[i] = make_float4(raw[3 * (size_t)i], raw[3 * (size_t)i + 1], raw[3 * (size_t)i + 2], __int_as_float(rows[r].part));
}

// part-local indices -> set-global vertex ids (in place), layer and part word per triangle (CollisionQuery.swift:376-400);
// an index outside its part's vertex range is clamped (so that nothing downstream reads out of bounds) and reported
// through errTri = the smallest offending input triangle
__global__ void k_expand_tris(uint32_t *__restrict__ idx, int nTrisIn, const PartRow *__restrict__ rows, int nRows,
                              uint32_t *__restrict__ layer, int32_t *__restrict__ part, int *__restrict__ errTri) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nTrisIn) return;
    const PartRow row = rows[part_row_of(rows, nRows, t, true)];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        uint32_t li = idx[3 * (size_t)t + k];
        if (li >= (uint32_t)row.nVerts) bad = true, li = 0;
        idx[3 * (size_t)t + k] = (uint32_t)row.vertLo + li;
    }
    layer[t] = row.layer;
    part[t] = row.part;
    if (bad) atomicMin(errTri, t);
}

// keep flag: |cross(e1,e2)|^2 > 1e-10 in WORLD space (CollisionQuery.swift:383-389)
__global__ void k_filter_flags(const float4 *__restrict__ world, const uint32_t *__restrict__ idxIn, int nTrisIn,
                               uint32_t *__restrict__ flags) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nTrisIn) return;
    f3 p0 = xyz(world[idxIn[3 * t]]), p1 = xyz(world[idxIn[3 * t + 1]]), p2 = xyz(world[idxIn[3 * t + 2]]);
    f3 e1 = p1 - p0, e2 = p2 - p0;
    flags[t] = len2(cross(e1, e2)) <= 1e-10f ? 0u : 1u;
}

// ---------------------------------------------------------------- exclusive scan (u32), 3 kernels
#define SCAN_THREADS 256
#define SCAN_ITEMS 8
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *smemWarp /*[32]*/, uint32_t &total) {
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) smemWarp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < (blockDim.x >> 5) ? smemWarp[lane] : 0u;
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t n = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += n;
        }
        smemWarp[lane] = winc - w; // exclusive warp base
        if (lane == 31) smemWarp[32] = winc;
    }
    __syncthreads();
    total = smemWarp[32];
    uint32_t r = smemWarp[warp] + inc - v;
    __syncthreads();
    return r;
}

__global__ void k_scan_tile_sums(const uint32_t *__restrict__ in, int n, uint32_t *__restrict__ tileSums) {
    __shared__ uint32_t sw[33];
    int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
        if (base + k < n) s += in[base + k];
    uint32_t total;
    block_exclusive_scan(s, sw, total);
    if (threadIdx.x == 0) tileSums[blockIdx.x] = total;
}

// single-block in-place exclusive scan of `n` entries (n up to a few million; L2 resident)
__global__ void k_scan_single_block(uint32_t *__restrict__ data, int n, uint32_t *__restrict__ totalOut) {
    __shared__ uint32_t sw[33];
    int per = (n + blockDim.x - 1) / blockDim.x;
    int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
    uint32_t s = 0;
    for (int i = lo; i < hi; i++) s += data[i];
    uint32_t total;
    uint32_t run = block_exclusive_scan(s, sw, total);
    for (int i = lo; i < hi; i++) {
        uint32_t v = data[i];
        data[i] = run;
        run += v;
    }
    if (threadIdx.x == 0 && totalOut) *totalOut = total;
}

__global__ void k_scan_apply(const uint32_t *__restrict__ in, int n, const uint32_t *__restrict__ tileBase,
                             uint32_t *__restrict__ out) {
    __shared__ uint32_t sw[33];
    int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = base + k < n ? in[base + k] : 0u;
        s += v[k];
    }
    uint32_t total;
    uint32_t run = block_exclusive_scan(s, sw, total) + tileBase[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < n) out[base + k] = run;
        run += v[k];
    }
}

__global__ void k_compact(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ offs, int nTrisIn,
                          const uint32_t *__restrict__ idxIn, const uint32_t *__restrict__ layerIn,
                          const int32_t *__restrict__ partIn, uint32_t *__restrict__ idxOut,
                          uint32_t *__restrict__ layerOut, int32_t *__restrict__ partOut) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nTrisIn || !flags[t]) return;
    uint32_t o = offs[t];
    idxOut[3 * o] = idxIn[3 * t];
    idxOut[3 * o + 1] = idxIn[3 * t + 1];
    idxOut[3 * o + 2] = idxIn[3 * t + 2];
    layerOut[o] = layerIn[t];
    partOut[o] = partIn[t];
}

__global__ void k_compact_i32(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ offs, int nTrisIn,
                              const int32_t *__restrict__ in, int32_t *__restrict__ out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nTrisIn && flags[t]) out[offs[t]] = in[t];
}

__global__ void k_gather_u32(const uint32_t *__restrict__ src, const int32_t *__restrict__ pos, int n,
                             uint32_t *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[pos[i]];
}

// ---------------------------------------------------------------- Morton codes
// bounds[0..2] = ordered-int min of triangle-AABB centroids, [3..5] = max
__global__ void k_init_bounds(int *bounds) {
    if (threadIdx.x < 3) bounds[threadIdx.x] = 0x7fffffff;
    else if (threadIdx.x < 6) bounds[threadIdx.x] = (int)0x80000000;
}

__device__ __forceinline__ f3 tri_centroid(const float4 *__restrict__ world, const uint32_t *__restrict__ idx, int t) {
    f3 p0 = xyz(world[idx[3 * t]]), p1 = xyz(world[idx[3 * t + 1]]), p2 = xyz(world[idx[3 * t + 2]]);
    f3 lo = vmin(p0, vmin(p1, p2)), hi = vmax(p0, vmax(p1, p2));
    return (lo + hi) * 0.5f; // BVH.centroid, CollisionQuery.swift:700
}

__global__ void k_centroid_bounds(const float4 *__restrict__ world, const uint32_t *__restrict__ idx, int nTris,
                                  int *__restrict__ bounds) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    f3 lo = {FLT_MAX, FLT_MAX, FLT_MAX}, hi = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    if (t < nTris) lo = hi = tri_centroid(world, idx, t);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo.x = fminf(lo.x, __shfl_xor_sync(0xffffffffu, lo.x, o));
        lo.y = fminf(lo.y, __shfl_xor_sync(0xffffffffu, lo.y, o));
        lo.z = fminf(lo.z, __shfl_xor_sync(0xffffffffu, lo.z, o));
        hi.x = fmaxf(hi.x, __shfl_xor_sync(0xffffffffu, hi.x, o));
        hi.y = fmaxf(hi.y, __shfl_xor_sync(0xffffffffu, hi.y, o));
        hi.z = fmaxf(hi.z, __shfl_xor_sync(0xffffffffu, hi.z, o));
    }
    // block-level reduction, then six atomics per CTA (one per warp made this kernel atomic-bound)
    __shared__ float red[6][8];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        red[0][warp] = lo.x, red[1][warp] = lo.y, red[2][warp] = lo.z;
        red[3][warp] = hi.x, red[4][warp] = hi.y, red[5][warp] = hi.z;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float v = red[threadIdx.x][0];
        int nw = blockDim.x >> 5;
        for (int k = 1; k < nw; k++) v = threadIdx.x < 3 ? fminf(v, red[threadIdx.x][k]) : fmaxf(v, red[threadIdx.x][k]);
        if (threadIdx.x < 3) atomicMin(bounds + threadIdx.x, float_to_ordered(v));
        else atomicMax(bounds + threadIdx.x, float_to_ordered(v));
    }
}

// 30-bit Morton code with the bits handed out longest-cell-axis first: every bit halves the currently longest side of
// the cell, so cells stay as cubic as the bounds allow.  For a cubic bound this IS the classic x,y,z interleave; for a
// flat world (a 4.5 km x 50 m x 4.5 km terrain) the classic code spends 10 bits on the 50 m and resolves only 4.4 m in
// the plane, so ~10 terrain triangles share a code and the leaves built from them overlap; this one resolves ~0.5 m.
__device__ __forceinline__ uint32_t morton30_adaptive(f3 p, f3 lo, f3 ext) {
    float ux = ext.x > 0.0f ? fminf(fmaxf((p.x - lo.x) / ext.x, 0.0f), 0.99999994f) : 0.0f;
    float uy = ext.y > 0.0f ? fminf(fmaxf((p.y - lo.y) / ext.y, 0.0f), 0.99999994f) : 0.0f;
    float uz = ext.z > 0.0f ? fminf(fmaxf((p.z - lo.z) / ext.z, 0.0f), 0.99999994f) : 0.0f;
    float cx = ext.x, cy = ext.y, cz = ext.z;
    uint32_t key = 0;
#pragma unroll 1
    for (int b = 0; b < 30; b++) {
        const int axis = (cx >= cy && cx >= cz) ? 0 : (cy >= cz ? 1 : 2); // ties: x, y, z — the classic order
        float u = axis == 0 ? ux : (axis == 1 ? uy : uz);
        u *= 2.0f;
        const uint32_t bit = u >= 1.0f ? 1u : 0u;
        u -= (float)bit;
        key = (key << 1) | bit;
        if (axis == 0) ux = u, cx *= 0.5f;
        else if (axis == 1) uy = u, cy *= 0.5f;
        else uz = u, cz *= 0.5f;
    }
    return key;
}

__global__ void k_morton(const float4 *__restrict__ world, const uint32_t *__restrict__ idx, int nTris,
                         const int *__restrict__ bounds, uint32_t *__restrict__ keys, uint32_t *__restrict__ vals) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nTris) return;
    f3 lo = {ordered_to_float(bounds[0]), ordered_to_float(bounds[1]), ordered_to_float(bounds[2])};
    f3 hi = {ordered_to_float(bounds[3]), ordered_to_float(bounds[4]), ordered_to_float(bounds[5])};
    f3 c = tri_centroid(world, idx, t);
    keys[t] = morton30_adaptive(c, lo, hi - lo);
    vals[t] = (uint32_t)t;
}

// ---------------------------------------------------------------- LSD radix sort, 8-bit digits, key/value u32
// Per pass: tile histograms -> single-block scan (digit-major) -> stable scatter with warp
// match/ballot ranking.  4 passes cover the 30-bit Morton key (+2 always-zero bits).
#define RS_THREADS 256
#define RS_ITEMS 16
#define RS_TILE (RS_THREADS * RS_ITEMS)
#define RS_WARPS (RS_THREADS / 32)

__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const uint32_t *__restrict__ keys, int n, int shift,
                                                        uint32_t *__restrict__ hist, int nBlocks) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    int base = blockIdx.x * RS_TILE;
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        int i = base + r * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[threadIdx.x * nBlocks + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const uint32_t *__restrict__ keysIn,
                                                           const uint32_t *__restrict__ valsIn,
                                                           uint32_t *__restrict__ keysOut,
                                                           uint32_t *__restrict__ valsOut, int n, int shift,
                                                           const uint32_t *__restrict__ histScanned, int nBlocks) {
    __shared__ uint32_t wh[RS_WARPS][256];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < RS_WARPS * 256; i += RS_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();
    int base = blockIdx.x * RS_TILE + warp * (32 * RS_ITEMS);
    uint32_t key[RS_ITEMS], val[RS_ITEMS], off[RS_ITEMS];
    const uint32_t ltMask = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        int i = base + r * 32 + lane;
        bool valid = i < n;
        key[r] = valid ? keysIn[i] : 0u;
        val[r] = valid ? valsIn[i] : 0u;
        uint32_t digit = valid ? ((key[r] >> shift) & 255u) : (256u + lane);
        uint32_t peers = __match_any_sync(0xffffffffu, digit);
        int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (valid && lane == leader) {
            old = wh[warp][digit];
            wh[warp][digit] = old + __popc(peers);
        }
        old = __shfl_sync(0xffffffffu, old, leader);
        off[r] = old + __popc(peers & ltMask);
        __syncwarp();
    }
    __syncthreads();
    { // digit d = threadIdx.x: exclusive prefix over warps + global base of (digit, block)
        uint32_t run = histScanned[threadIdx.x * nBlocks + blockIdx.x];
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) {
            uint32_t c = wh[w][threadIdx.x];
            wh[w][threadIdx.x] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        int i = base + r * 32 + lane;
        if (i < n) {
            uint32_t digit = (key[r] >> shift) & 255u;
            uint32_t o = wh[warp][digit] + off[r];
            keysOut[o] = key[r];
            valsOut[o] = val[r];
        }
    }
}

// ---------------------------------------------------------------- onesweep (Adinets & Merrill 2022)
// One upfront histogram kernel counts all four digits of every key; then each of the four passes is ONE
// kernel: tiles are handed out in launch order by an atomic ticket, every tile publishes its per-digit
// counts in a status word (aggregate / inclusive flag in the two top bits) and resolves its exclusive
// prefix by decoupled look-back over the preceding tiles, then scatters with the same stable
// warp-match ranking as the classic path.  3 key reads + 4 key/value read-write sweeps in total instead
// of 4 x (2 reads + 1 read-write) and 13 launches instead of 12 + scans of per-tile histograms.
#define OS_FLAG_AGG 0x40000000u
#define OS_FLAG_INC 0x80000000u
#define OS_MASK 0x3fffffffu

__global__ void __launch_bounds__(RS_THREADS) k_os_histogram(const uint32_t *__restrict__ keys, int n,
                                                             uint32_t *__restrict__ hist /* [4][256] */) {
    __shared__ uint32_t h[4][256];
    for (int i = threadIdx.x; i < 1024; i += RS_THREADS) (&h[0][0])[i] = 0;
    __syncthreads();
    for (int i = blockIdx.x * RS_THREADS + threadIdx.x; i < n; i += gridDim.x * RS_THREADS) {
        uint32_t k = keys[i];
        atomicAdd(&h[0][k & 255u], 1u);
        atomicAdd(&h[1][(k >> 8) & 255u], 1u);
        atomicAdd(&h[2][(k >> 16) & 255u], 1u);
        atomicAdd(&h[3][(k >> 24) & 255u], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 1024; i += RS_THREADS) {
        uint32_t v = (&h[0][0])[i];
        if (v) atomicAdd(hist + i, v);
    }
}

__global__ void k_os_scan(uint32_t *__restrict__ hist /* [4][256] -> exclusive per pass */) {
    __shared__ uint32_t sw[33];
    for (int p = 0; p < 4; p++) {
        uint32_t v = hist[p * 256 + threadIdx.x];
        uint32_t total;
        uint32_t ex = block_exclusive_scan(v, sw, total);
        hist[p * 256 + threadIdx.x] = ex;
    }
}

__global__ void __launch_bounds__(RS_THREADS) k_os_pass(const uint32_t *__restrict__ keysIn,
                                                        const uint32_t *__restrict__ valsIn,
                                                        uint32_t *__restrict__ keysOut, uint32_t *__restrict__ valsOut,
                                                        int n, int shift, const uint32_t *__restrict__ digitBase /* [256] */,
                                                        volatile uint32_t *status /* [nTiles][256] */, uint32_t *ticket,
                                                        int *errorFlag, unsigned int *worldStatus) {
    __shared__ uint32_t wh[RS_WARPS][256];
    __shared__ uint32_t sTile;
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) sTile = atomicAdd(ticket, 1u); // tiles are claimed in launch order: look-back never waits on a
    for (int i = threadIdx.x; i < RS_WARPS * 256; i += RS_THREADS) (&wh[0][0])[i] = 0; // tile whose CTA has not started
    __syncthreads();
    const int tile = (int)sTile;
    int base = tile * RS_TILE + warp * (32 * RS_ITEMS);
    uint32_t key[RS_ITEMS], val[RS_ITEMS], off[RS_ITEMS];
    const uint32_t ltMask = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        int i = base + r * 32 + lane;
        bool valid = i < n;
        key[r] = valid ? keysIn[i] : 0u;
        val[r] = valid ? valsIn[i] : 0u;
        uint32_t digit = valid ? ((key[r] >> shift) & 255u) : (256u + lane);
        uint32_t peers = __match_any_sync(0xffffffffu, digit);
        int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (valid && lane == leader) {
            old = wh[warp][digit];
            wh[warp][digit] = old + __popc(peers);
        }
        old = __shfl_sync(0xffffffffu, old, leader);
        off[r] = old + __popc(peers & ltMask);
        __syncwarp();
    }
    __syncthreads();
    { // thread d owns digit d: tile count -> publish -> look back -> exclusive prefix -> per-warp bases
        const int d = threadIdx.x;
        uint32_t cnt = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) cnt += wh[w][d];
        volatile uint32_t *mine = status + (size_t)tile * 256 + d;
        *mine = cnt | (tile == 0 ? OS_FLAG_INC : OS_FLAG_AGG);
        uint32_t prefix = 0;
        for (int t = tile - 1; t >= 0; t--) {
            volatile uint32_t *p = status + (size_t)t * 256 + d;
            uint32_t s = *p;
            uint32_t spins = 0;
            while ((s & (OS_FLAG_AGG | OS_FLAG_INC)) == 0u) {
                if (++spins > (1u << 26)) { // watchdog: never hang the device
                    *errorFlag = 1;
                    if (worldStatus) atomicOr(worldStatus, 2u); // asynchronous callers: reported at the next synchronising call
                    break;
                }
                s = *p;
            }
            prefix += s & OS_MASK;
            if (s & OS_FLAG_INC) break;
        }
        if (tile > 0) *mine = ((prefix + cnt) & OS_MASK) | OS_FLAG_INC;
        uint32_t run = digitBase[d] + prefix;
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) {
            uint32_t c = wh[w][d];
            wh[w][d] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        int i = base + r * 32 + lane;
        if (i < n) {
            uint32_t digit = (key[r] >> shift) & 255u;
            uint32_t o = wh[warp][digit] + off[r];
            keysOut[o] = key[r];
            valsOut[o] = val[r];
        }
    }
}

// NB: k_rs_hist walks the tile thread-strided while k_rs_scatter walks it warp-chunked; both count the
// same multiset per tile, which is all the histogram needs.

// ---------------------------------------------------------------- gather into the sorted float4 SoA
__global__ void k_gather_sorted(const uint32_t *__restrict__ sortedTri, int nTris, const float4 *__restrict__ world,
                                const uint32_t *__restrict__ idx, const uint32_t *__restrict__ layer,
                                const int32_t *__restrict__ rank /* global index -> visiting rank, or null */, int triOffset,
                                float4 *__restrict__ tv0, float4 *__restrict__ tv1, float4 *__restrict__ tv2) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nTris) return;
    uint32_t t = sortedTri[s];
    float4 a = world[idx[3 * t]], b = world[idx[3 * t + 1]], c = world[idx[3 * t + 2]];
    a.w = __uint_as_float(layer[t]);
    b.w = __int_as_float((int)t);
    c.w = __int_as_float(rank ? rank[triOffset + (int)t] : triOffset + (int)t); // canonical order: rank = global index
    tv0[s] = a;
    tv1[s] = b;
    tv2[s] = c;
}

// ---------------------------------------------------------------- Karras 2012 radix tree
__device__ __forceinline__ int delta_fn(const uint32_t *__restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    uint32_t a = keys[i], b = keys[j];
    if (a == b) return 32 + __clz((uint32_t)i ^ (uint32_t)j); // duplicate keys: fall back to the index
    return __clz(a ^ b);
}

__device__ __forceinline__ int leaf_ref(int start, int count) { return ~((start << 2) | (count - 1)); }

__global__ void k_karras(const uint32_t *__restrict__ keys, int n, Node *__restrict__ nodes, int32_t *__restrict__ parent,
                         int32_t *__restrict__ rangeLo, int32_t *__restrict__ rangeHi) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = (delta_fn(keys, n, i, i + 1) - delta_fn(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta_fn(keys, n, i, i - d);
    int lmax = 2;
    while (delta_fn(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t > 0; t >>= 1)
        if (delta_fn(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta_fn(keys, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (delta_fn(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int first = min(i, j), last = max(i, j);
    rangeLo[i] = first;
    rangeHi[i] = last;
    // children: [first, gamma] and [gamma+1, last]
    int leftIsLeaf = first == gamma, rightIsLeaf = last == gamma + 1;
    int leftBox = leftIsLeaf ? (n - 1) + gamma : gamma;             // index into boxLo/boxHi/parent
    int rightBox = rightIsLeaf ? (n - 1) + gamma + 1 : gamma + 1;
    parent[leftBox] = i;
    parent[rightBox] = i;
    if (i == 0) parent[0] = -1;
    int lc = gamma - first + 1, rc = last - gamma;
    int ref0 = lc <= 4 ? leaf_ref(first, lc) : gamma;
    int ref1 = rc <= 4 ? leaf_ref(gamma + 1, rc) : gamma + 1;
    nodes[i].n0.w = __int_as_float(ref0);
    nodes[i].n1.w = __int_as_float(ref1);
    // box slots of the children, stashed until k_fit overwrites n2.w/n3.w are unused afterwards
    nodes[i].n2.w = __int_as_float(leftBox);
    nodes[i].n3.w = __int_as_float(rightBox);
}

// bottom-up boxes: one thread per leaf slot climbs while it is the second to arrive
__global__ void k_fit(int n, const float4 *__restrict__ tv0, const float4 *__restrict__ tv1,
                      const float4 *__restrict__ tv2, Node *__restrict__ nodes, const int32_t *__restrict__ parent,
                      float4 *__restrict__ boxLo, float4 *__restrict__ boxHi, int32_t *__restrict__ visit) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    f3 a = xyz(tv0[s]), b = xyz(tv1[s]), c = xyz(tv2[s]);
    f3 lo = vmin(a, vmin(b, c)), hi = vmax(a, vmax(b, c));
    int me = (n - 1) + s;
    boxLo[me] = make_float4(lo.x, lo.y, lo.z, 0.0f);
    boxHi[me] = make_float4(hi.x, hi.y, hi.z, 0.0f);
    if (n == 1) return;
    __threadfence();
    int p = parent[me];
    while (p >= 0) {
        if (atomicAdd(&visit[p], 1) == 0) return; // first arrival: the sibling subtree is not done yet
        __threadfence();
        Node nd = nodes[p];
        int lb = __float_as_int(nd.n2.w), rb = __float_as_int(nd.n3.w);
        // volatile-ish reads: boxes were published before the sibling's atomicAdd
        float4 l0 = __ldcg(boxLo + lb), h0 = __ldcg(boxHi + lb), l1 = __ldcg(boxLo + rb), h1 = __ldcg(boxHi + rb);
        nd.n0 = make_float4(l0.x, l0.y, l0.z, nd.n0.w);
        nd.n1 = make_float4(h0.x, h0.y, h0.z, nd.n1.w);
        nd.n2 = make_float4(l1.x, l1.y, l1.z, nd.n2.w);
        nd.n3 = make_float4(h1.x, h1.y, h1.z, nd.n3.w);
        nodes[p] = nd;
        boxLo[p] = make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), 0.0f);
        boxHi[p] = make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), 0.0f);
        __threadfence();
        p = parent[p];
    }
}

// depth parity of every internal node (root = depth 0): only even-depth nodes become 4-wide nodes
__global__ void k_depth_parity(int nInternal, const int32_t *__restrict__ parent, uint8_t *__restrict__ parity) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nInternal) return;
    int d = 0;
    for (int p = parent[i]; p >= 0; p = parent[p]) d++;
    parity[i] = (uint8_t)(d & 1);
}

// collapse: wide node i = binary node i (even depth) with its internal children replaced by THEIR children
__device__ __forceinline__ void collapse4_node(int i, const Node *nodes, Node4 *nodes4);
__global__ void k_collapse4(int nInternal, const Node *__restrict__ nodes, const uint8_t *__restrict__ parity,
                            Node4 *__restrict__ nodes4) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nInternal || parity[i]) return;
    collapse4_node(i, nodes, nodes4);
}
__device__ __forceinline__ void collapse4_node(int i, const Node *nodes, Node4 *nodes4) {
    Node nb = nodes[i];
    float4 lo[4], hi[4];
    int ref[4];
    int cnt = 0;
#pragma unroll
    for (int c = 0; c < 2; c++) {
        float4 clo = c == 0 ? nb.n0 : nb.n2, chi = c == 0 ? nb.n1 : nb.n3;
        int r = __float_as_int(c == 0 ? nb.n0.w : nb.n1.w);
        if (r < 0) {
            lo[cnt] = clo, hi[cnt] = chi, ref[cnt] = r;
            cnt++;
        } else {
            Node nc = nodes[r];
            lo[cnt] = nc.n0, hi[cnt] = nc.n1, ref[cnt] = __float_as_int(nc.n0.w);
            cnt++;
            lo[cnt] = nc.n2, hi[cnt] = nc.n3, ref[cnt] = __float_as_int(nc.n1.w);
            cnt++;
        }
    }
    Node4 w;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        bool used = k < cnt;
        float4 l = used ? lo[k] : make_float4(FLT_MAX, FLT_MAX, FLT_MAX, 0.0f);
        float4 h = used ? hi[k] : make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, 0.0f);
        int r = used ? ref[k] : CQ_REF_EMPTY;
        if (k < 2) {
            w.q[2 * k] = make_float4(l.x, l.y, l.z, __int_as_float(r));
            w.q[2 * k + 1] = make_float4(h.x, h.y, h.z, 0.0f);
        } else {
            w.q[2 * k] = make_float4(l.x, l.y, l.z, 0.0f);
            w.q[2 * k + 1] = make_float4(h.x, h.y, h.z, 0.0f);
        }
    }
    // refs: q[0].w = ref0, q[1].w = ref1, q[2].w = ref2, q[3].w = ref3
    w.q[0].w = __int_as_float(cnt > 0 ? ref[0] : CQ_REF_EMPTY);
    w.q[1].w = __int_as_float(cnt > 1 ? ref[1] : CQ_REF_EMPTY);
    w.q[2].w = __int_as_float(cnt > 2 ? ref[2] : CQ_REF_EMPTY);
    w.q[3].w = __int_as_float(cnt > 3 ? ref[3] : CQ_REF_EMPTY);
    nodes4[i] = w;
}

__global__ void k_header(int n, const float4 *__restrict__ boxLo, const float4 *__restrict__ boxHi, SetHeader *hdr) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    SetHeader h;
    h.nTris = n;
    if (n == 0) {
        h.rootRef = CQ_REF_EMPTY;
        h.lo[0] = h.lo[1] = h.lo[2] = FLT_MAX;
        h.hi[0] = h.hi[1] = h.hi[2] = -FLT_MAX;
    } else {
        int rootBox = n == 1 ? 0 : 0; // n==1: leaf slot 0 lives at index (n-1)+0 = 0 as well
        h.rootRef = n <= 4 ? leaf_ref(0, n) : 0;
        float4 lo = boxLo[rootBox], hi = boxHi[rootBox];
        h.lo[0] = lo.x, h.lo[1] = lo.y, h.lo[2] = lo.z;
        h.hi[0] = hi.x, h.hi[1] = hi.y, h.hi[2] = hi.z;
    }
    *hdr = h;
}

// ---------------------------------------------------------------- transform update + dirty-subtree refit
// (TriangleMeshSet.updateTransforms :419-462, BVH.refit :528-575)
// A transform update stages a table of the moved parts (MovedPart, cq_internal.h); every kernel below runs over that
// table in ONE launch per set, whatever the number of parts: a thread finds its row by binary search over the rows'
// running totals.  k_update_parts writes the parts' model rows and re-transforms their vertices.
// The reference then recomputes the leaves of the updated triangles and only their ancestors, deepest first.  Here, when
// fewer than a quarter of a set's triangles moved, three launches per tree:
//   mark  — one thread per moved triangle rewrites its slot of the sorted SoA and its leaf box, and MARKS its ancestors:
//           `expect[p]` counts the dirty children of p (1 or 2); the thread that finds p already marked stops, so every
//           dirty edge is counted once;
//   climb — the last of a node's expected arrivals recomputes it from its children's boxes (the clean child's box is
//           still valid), re-collapses the 4-wide node when the depth is even, and goes on.  `expect` is final once the
//           mark launch has ended and nothing in the climb writes it, so an arrival can never see a counter a sibling
//           arrival has already reset;
//   clear — resets `visit` / `expect` along the same paths for the next refit.
// Same min / max arithmetic as the full fit, so the boxes are identical; cost O(updated triangles x depth).
__global__ void k_invert_sorted(const uint32_t *__restrict__ sortedTri, int n, uint32_t *__restrict__ slotOfTri) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) slotOfTri[sortedTri[s]] = (uint32_t)s;
}

// the row of the table that holds unit i (a vertex when tris == false, else a triangle): the last row whose base <= i
__device__ __forceinline__ const MovedPart &moved_row(const MovedPart *__restrict__ tab, int nRows, int i, bool tris) {
    int lo = 0, hi = nRows - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((tris ? tab[mid].triBase : tab[mid].vertBase) <= i) lo = mid;
        else hi = mid - 1;
    }
    return tab[lo];
}
__device__ __forceinline__ int moved_triangle(const MovedPart *__restrict__ tab, int nRows, int i) {
    const MovedPart &r = moved_row(tab, nRows, i, true);
    return r.triLo + (i - r.triBase);
}

// one thread per vertex of the moved parts; the arithmetic of k_transform, so the positions are bit-identical
__global__ void k_update_parts(const MovedPart *__restrict__ tab, int nRows, int nVerts, const float4 *__restrict__ local,
                               float4 *__restrict__ world, float *__restrict__ models) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nVerts) return;
    const MovedPart &r = moved_row(tab, nRows, i, false);
    const int k = i - r.vertBase;
    if (k == 0)
        for (int c = 0; c < 16; c++) models[16 * r.part + c] = r.model[c];
    const int v = r.vertLo + k;
    world[v] = transform_point(r.model, local[v]);
}

__global__ void k_refit_mark(const MovedPart *__restrict__ tab, int nRows, int nMoved, const uint32_t *__restrict__ slotOfTri,
                             int n, const float4 *__restrict__ world, const uint32_t *__restrict__ idx, float4 *tv0, float4 *tv1,
                             float4 *tv2, const int32_t *__restrict__ parent, float4 *boxLo, float4 *boxHi, int32_t *expect) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMoved) return;
    const int t = moved_triangle(tab, nRows, i);
    const int slot = (int)slotOfTri[t];
    const float4 a = world[idx[3 * t]], b = world[idx[3 * t + 1]], c = world[idx[3 * t + 2]];
    float4 o0 = tv0[slot], o1 = tv1[slot], o2 = tv2[slot]; // the w words (layer, triangle id, rank) stay
    o0.x = a.x, o0.y = a.y, o0.z = a.z, o1.x = b.x, o1.y = b.y, o1.z = b.z, o2.x = c.x, o2.y = c.y, o2.z = c.z;
    tv0[slot] = o0, tv1[slot] = o1, tv2[slot] = o2;
    const f3 lo = vmin(xyz(a), vmin(xyz(b), xyz(c))), hi = vmax(xyz(a), vmax(xyz(b), xyz(c)));
    int node = (n - 1) + slot;
    boxLo[node] = make_float4(lo.x, lo.y, lo.z, 0.0f);
    boxHi[node] = make_float4(hi.x, hi.y, hi.z, 0.0f);
    if (n == 1) return;
    for (int p = parent[node]; p >= 0; p = parent[p])
        if (atomicAdd(&expect[p], 1) != 0) break; // p was already marked through its other child
}

__global__ void k_refit_climb(const MovedPart *__restrict__ tab, int nRows, int nMoved, const uint32_t *__restrict__ slotOfTri,
                              int n, Node *nodes, const int32_t *__restrict__ parent, float4 *boxLo, float4 *boxHi, int32_t *visit,
                              const int32_t *__restrict__ expect, const uint8_t *__restrict__ parity, Node4 *nodes4) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMoved || n == 1) return;
    int p = parent[(n - 1) + (int)slotOfTri[moved_triangle(tab, nRows, i)]];
    while (p >= 0) {
        if (atomicAdd(&visit[p], 1) + 1 < expect[p]) return; // a dirty sibling subtree is not done yet
        __threadfence();
        Node nd = nodes[p];
        const int lb = __float_as_int(nd.n2.w), rb = __float_as_int(nd.n3.w);
        const float4 l0 = __ldcg(boxLo + lb), h0 = __ldcg(boxHi + lb), l1 = __ldcg(boxLo + rb), h1 = __ldcg(boxHi + rb);
        nd.n0 = make_float4(l0.x, l0.y, l0.z, nd.n0.w);
        nd.n1 = make_float4(h0.x, h0.y, h0.z, nd.n1.w);
        nd.n2 = make_float4(l1.x, l1.y, l1.z, nd.n2.w);
        nd.n3 = make_float4(h1.x, h1.y, h1.z, nd.n3.w);
        nodes[p] = nd;
        boxLo[p] = make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), 0.0f);
        boxHi[p] = make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), 0.0f);
        __threadfence();
        // 4-wide nodes: an even-depth node absorbs its internal (odd-depth) children, which are final by now
        if (!parity[p]) collapse4_node(p, nodes, nodes4);
        __threadfence();
        p = parent[p];
    }
}

// Every marked node lies on the path of a moved triangle, so walking those paths clears them all.  A thread stops at the
// first node another thread has cleared: that thread goes on above it.
__global__ void k_refit_clear(const MovedPart *__restrict__ tab, int nRows, int nMoved, const uint32_t *__restrict__ slotOfTri,
                              int n, const int32_t *__restrict__ parent, int32_t *visit, int32_t *expect) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMoved || n == 1) return;
    for (int p = parent[(n - 1) + (int)slotOfTri[moved_triangle(tab, nRows, i)]]; p >= 0; p = parent[p]) {
        visit[p] = 0;
        if (atomicExch(&expect[p], 0) == 0) break;
    }
}

// the same three steps on the reference's tree (reference order): leaves hold <= 4 triangles; a leaf is refitted by the
// moved triangle that claims it first in the mark launch (leafMark = its triangle id + 1), which also climbs for it
__device__ __forceinline__ void ref_store_child_box(Node *nd, int which, f3 lo, f3 hi);
__global__ void k_ref_refit_mark(const MovedPart *__restrict__ tab, int nRows, int nMoved, const int32_t *__restrict__ leafOfTri,
                                 const int32_t *__restrict__ leafRange, const int32_t *__restrict__ leafParent,
                                 const int32_t *__restrict__ nodeParent, const uint32_t *__restrict__ refSlot,
                                 const float4 *__restrict__ tv0, const float4 *__restrict__ tv1, const float4 *__restrict__ tv2,
                                 Node *nodes, int32_t *leafMark, int32_t *expect, SetHeader *hdr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMoved) return;
    const int t = moved_triangle(tab, nRows, i);
    const int l = leafOfTri[t];
    if (atomicCAS(&leafMark[l], 0, t + 1) != 0) return; // another triangle of the same leaf got here first
    const int range = leafRange[l], start = range >> 2, count = (range & 3) + 1;
    f3 lo = {0, 0, 0}, hi = {0, 0, 0};
    for (int k = 0; k < count; k++) {
        const uint32_t slot = refSlot[start + k];
        const f3 a = xyz(tv0[slot]), b = xyz(tv1[slot]), c = xyz(tv2[slot]);
        const f3 tlo = vmin(a, vmin(b, c)), thi = vmax(a, vmax(b, c));
        lo = k ? vmin(lo, tlo) : tlo;
        hi = k ? vmax(hi, thi) : thi;
    }
    int pw = leafParent[l];
    if (pw < 0) {
        hdr->lo[0] = lo.x, hdr->lo[1] = lo.y, hdr->lo[2] = lo.z;
        hdr->hi[0] = hi.x, hdr->hi[1] = hi.y, hdr->hi[2] = hi.z;
        return;
    }
    ref_store_child_box(nodes + (pw >> 1), pw & 1, lo, hi);
    for (; pw >= 0; pw = nodeParent[pw >> 1])
        if (atomicAdd(&expect[pw >> 1], 1) != 0) break;
}

__global__ void k_ref_refit_climb(const MovedPart *__restrict__ tab, int nRows, int nMoved, const int32_t *__restrict__ leafOfTri,
                                  const int32_t *__restrict__ leafParent, const int32_t *__restrict__ nodeParent, Node *nodes,
                                  const int32_t *__restrict__ leafMark, int32_t *visit, const int32_t *__restrict__ expect,
                                  SetHeader *hdr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMoved) return;
    const int t = moved_triangle(tab, nRows, i);
    const int l = leafOfTri[t];
    if (leafMark[l] != t + 1) return; // one climber per marked leaf: the triangle that claimed it
    int pw = leafParent[l];
    while (pw >= 0) {
        const int p = pw >> 1;
        if (atomicAdd(&visit[p], 1) + 1 < expect[p]) return;
        __threadfence();
        const float4 *q = reinterpret_cast<const float4 *>(nodes + p);
        const float4 l0 = __ldcg(q), h0 = __ldcg(q + 1), l1 = __ldcg(q + 2), h1 = __ldcg(q + 3);
        const f3 lo = vmin(xyz(l0), xyz(l1)), hi = vmax(xyz(h0), xyz(h1));
        pw = nodeParent[p];
        if (pw < 0) {
            hdr->lo[0] = lo.x, hdr->lo[1] = lo.y, hdr->lo[2] = lo.z;
            hdr->hi[0] = hi.x, hdr->hi[1] = hi.y, hdr->hi[2] = hi.z;
            return;
        }
        ref_store_child_box(nodes + (pw >> 1), pw & 1, lo, hi);
        __threadfence();
    }
}

__global__ void k_ref_refit_clear(const MovedPart *__restrict__ tab, int nRows, int nMoved, const int32_t *__restrict__ leafOfTri,
                                  const int32_t *__restrict__ leafParent, const int32_t *__restrict__ nodeParent, int32_t *leafMark,
                                  int32_t *visit, int32_t *expect) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nMoved) return;
    const int l = leafOfTri[moved_triangle(tab, nRows, i)];
    leafMark[l] = 0;
    for (int pw = leafParent[l]; pw >= 0; pw = nodeParent[pw >> 1]) {
        visit[pw >> 1] = 0;
        if (atomicExch(&expect[pw >> 1], 0) == 0) break;
    }
}

// ---------------------------------------------------------------- host orchestration
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// One cudaMalloc per triangle set (+ one for build temporaries): GB-scale cudaMalloc/cudaFree calls cost
// tens to hundreds of milliseconds each on this driver, far more than the build kernels themselves.
struct Arena {
    char *base = nullptr;
    size_t off = 0, cap = 0;
    template <class T> T *take(size_t count) {
        if (count == 0) count = 1;
        off = (off + 255) & ~(size_t)255;
        T *p = reinterpret_cast<T *>(base + off);
        off += count * sizeof(T);
        return p;
    }
};

void free_set(DeviceSet &S) {
    cudaFree(S.triMat);
    cudaFree(S.arena);
    cudaFree(S.refArena);
    S = DeviceSet();
}

static int exclusive_scan_u32(cq_world *w, const uint32_t *in, int n, uint32_t *out, uint32_t *tileSums /* cdiv(n,TILE)+1 */,
                              uint32_t *dTotal) {
    cudaStream_t st = w->stream;
    int tiles = cdiv(n, SCAN_TILE);
    k_scan_tile_sums<<<tiles, SCAN_THREADS, 0, st>>>(in, n, tileSums);
    k_scan_single_block<<<1, 1024, 0, st>>>(tileSums, tiles, dTotal);
    k_scan_apply<<<tiles, SCAN_THREADS, 0, st>>>(in, n, tileSums, out);
    w->launches += 3;
    return check_cuda(cudaGetLastError(), "scan");
}

static int radix_sort_pairs_classic(cq_world *w, uint32_t *keys, uint32_t *vals, uint32_t *keysTmp, uint32_t *valsTmp,
                                    int n, uint32_t *hist /* 256 * nBlocks */) {
    cudaStream_t st = w->stream;
    int nBlocks = cdiv(n, RS_TILE);
    uint32_t *kin = keys, *vin = vals, *kout = keysTmp, *vout = valsTmp;
    for (int pass = 0; pass < 4; pass++) {
        int shift = pass * 8;
        k_rs_hist<<<nBlocks, RS_THREADS, 0, st>>>(kin, n, shift, hist, nBlocks);
        k_scan_single_block<<<1, 1024, 0, st>>>(hist, 256 * nBlocks, nullptr);
        k_rs_scatter<<<nBlocks, RS_THREADS, 0, st>>>(kin, vin, kout, vout, n, shift, hist, nBlocks);
        w->launches += 3;
        std::swap(kin, kout);
        std::swap(vin, vout);
    }
    // 4 passes: result is back in (keys, vals)
    return check_cuda(cudaGetLastError(), "radix sort");
}

// onesweep: status = [4][nTiles][256] u32 + [4] tickets + [4][256] digit histograms + error flag, in `scratch`
static int radix_sort_pairs_onesweep(cq_world *w, uint32_t *keys, uint32_t *vals, uint32_t *keysTmp, uint32_t *valsTmp,
                                     int n, uint32_t *scratch, size_t scratchWords, cudaStream_t st = nullptr,
                                     bool checkError = true) {
    if (!st) st = w->stream;
    int nTiles = cdiv(n, RS_TILE);
    size_t statusWords = (size_t)4 * nTiles * 256;
    if (statusWords + 4 + 1024 + 1 > scratchWords) {
        set_error("onesweep scratch too small");
        return CQ_ERR_INVALID;
    }
    uint32_t *status = scratch, *tickets = scratch + statusWords, *hist = tickets + 4;
    int *err = (int *)(hist + 1024);
    CQ_CUDA(cudaMemsetAsync(scratch, 0, sizeof(uint32_t) * (statusWords + 4 + 1024 + 1), st));
    int hb = std::min(nTiles, 148 * 8);
    k_os_histogram<<<hb, RS_THREADS, 0, st>>>(keys, n, hist);
    k_os_scan<<<1, 256, 0, st>>>(hist);
    w->launches += 2;
    uint32_t *kin = keys, *vin = vals, *kout = keysTmp, *vout = valsTmp;
    for (int pass = 0; pass < 4; pass++) {
        k_os_pass<<<nTiles, RS_THREADS, 0, st>>>(kin, vin, kout, vout, n, pass * 8, hist + pass * 256,
                                                 status + (size_t)pass * nTiles * 256, tickets + pass, err, w->view.status);
        w->launches++;
        std::swap(kin, kout);
        std::swap(vin, vout);
    }
    if (!checkError) return check_cuda(cudaGetLastError(), "onesweep"); // asynchronous use: no host round trip
    int hostErr = 0;
    CQ_CUDA(cudaMemcpyAsync(&hostErr, err, sizeof(int), cudaMemcpyDeviceToHost, st));
    CQ_CUDA(cudaStreamSynchronize(st));
    if (hostErr) {
        set_error("onesweep look-back watchdog fired");
        return CQ_ERR_CUDA;
    }
    return check_cuda(cudaGetLastError(), "onesweep");
}

static bool use_classic_sort() {
    const char *e = getenv("CQ_SORT");
    return e && !strcmp(e, "classic");
}

static int build_tree(cq_world *w, DeviceSet &S, const uint32_t *sortedKeys /* may be null on refit */, cudaStream_t st) {
    int n = S.nTris;
    if (n > 0) {
        const int triOffset = &S == &w->set[1] ? w->set[0].nTris : 0;
        k_gather_sorted<<<cdiv(n, 256), 256, 0, st>>>(S.sortedTri, n, S.worldPos, S.indices, S.triLayer,
                                                      w->order == CQ_ORDER_REFERENCE ? w->dRank : nullptr, triOffset, S.tv0, S.tv1,
                                                      S.tv2);
        w->launches++;
        if (n > 1) {
            if (sortedKeys) {
                k_karras<<<cdiv(n - 1, 256), 256, 0, st>>>(sortedKeys, n, S.nodes, S.parent, S.rangeLo, S.rangeHi);
                w->launches++;
            }
            CQ_CUDA(cudaMemsetAsync(S.visit, 0, sizeof(int32_t) * (size_t)(n - 1), st));
        }
        k_fit<<<cdiv(n, 256), 256, 0, st>>>(n, S.tv0, S.tv1, S.tv2, S.nodes, S.parent, S.boxLo, S.boxHi, S.visit);
        w->launches++;
        if (n > 1) CQ_CUDA(cudaMemsetAsync(S.visit, 0, sizeof(int32_t) * (size_t)(n - 1), st)); // clean for a dirty-subtree refit
        if (n > 1) {
            if (sortedKeys) { // topology is new: depth parities
                k_depth_parity<<<cdiv(n - 1, 256), 256, 0, st>>>(n - 1, S.parent, S.depthParity);
                w->launches++;
            }
            k_collapse4<<<cdiv(n - 1, 256), 256, 0, st>>>(n - 1, S.nodes, S.depthParity, S.nodes4);
            w->launches++;
        }
    }
    k_header<<<1, 32, 0, st>>>(n, S.boxLo, S.boxHi, S.hdr);
    w->launches++;
    return check_cuda(cudaGetLastError(), "build_tree");
}

template <class Fn> static size_t arena_layout(Fn fn) { // run the carving once without memory to learn the size
    Arena a;
    fn(a);
    return a.off + 256;
}

int build_set(cq_world *w, DeviceSet &S, const SetPlan &in,
              std::vector<int> &partTriStartIn /* in: first input triangle of each part of this set (+ end), out: filtered */,
              int *badTriangle /* out: smallest input triangle with an index outside its part's vertices, or -1 */,
              const int32_t *matIn /* host, per input triangle: row of the material table, or nullptr */) {
    cudaStream_t st = w->stream;
    *badTriangle = -1;
    S.nVerts = (int)in.nVerts;
    S.nTrisIn = (int)in.nTris;
    const int nIn = S.nTrisIn;
    const int nCap = std::max(nIn, 1); // nTris (after the filter) <= nIn: size everything by the upper bound
    // ---- persistent arrays
    auto carve = [&](Arena &a) {
        S.localPos = a.take<float4>(S.nVerts);
        S.worldPos = a.take<float4>(S.nVerts);
        S.hdr = a.take<SetHeader>(1);
        S.indices = a.take<uint32_t>((size_t)nCap * 3);
        S.triLayer = a.take<uint32_t>(nCap);
        S.triPart = a.take<int32_t>(nCap);
        S.sortedTri = a.take<uint32_t>(nCap);
        S.tv0 = a.take<float4>(nCap);
        S.tv1 = a.take<float4>(nCap);
        S.tv2 = a.take<float4>(nCap);
        S.nodes = a.take<Node>(nCap);
        S.nodes4 = a.take<Node4>(nCap);
        S.depthParity = a.take<uint8_t>(nCap);
        S.parent = a.take<int32_t>((size_t)2 * nCap);
        S.rangeLo = a.take<int32_t>(nCap);
        S.rangeHi = a.take<int32_t>(nCap);
        S.boxLo = a.take<float4>((size_t)2 * nCap);
        S.boxHi = a.take<float4>((size_t)2 * nCap);
        S.visit = a.take<int32_t>(nCap);
        S.expect = a.take<int32_t>(nCap);
        S.slotOfTri = a.take<uint32_t>(nCap);
    };
    Arena arena;
    arena.cap = arena_layout(carve);
    CQ_CUDA(cudaMalloc((void **)&arena.base, arena.cap));
    S.arena = arena.base;
    carve(arena);
    // ---- temporaries
    uint32_t *dIdxIn, *dLayerIn, *dFlags, *dOffs, *dTileSums, *dTotal, *dKeys, *dKeysTmp, *dValsTmp, *dHist, *dGatherOut;
    int32_t *dPartIn, *dGatherPos;
    int *dBounds, *dErrTri;
    float *dRawPos;
    PartRow *dRows;
    const int nRows = (int)in.rows.size();
    const int np = (int)partTriStartIn.size();
    const size_t histWords = (size_t)4 * 256 * cdiv(nCap, RS_TILE) + 4 + 1024 + 1; // classic: 256*tiles; onesweep: 4x + extras
    auto carveTmp = [&](Arena &a) {
        dIdxIn = a.take<uint32_t>((size_t)nCap * 3);
        dLayerIn = a.take<uint32_t>(nCap);
        dPartIn = a.take<int32_t>(nCap);
        dFlags = a.take<uint32_t>(nCap);
        dOffs = a.take<uint32_t>((size_t)nCap + 1);
        dTileSums = a.take<uint32_t>((size_t)cdiv(nCap, SCAN_TILE) + 1);
        dTotal = a.take<uint32_t>(1);
        dKeys = a.take<uint32_t>(nCap);
        dKeysTmp = a.take<uint32_t>(nCap);
        dValsTmp = a.take<uint32_t>(nCap);
        dHist = a.take<uint32_t>(histWords);
        dBounds = a.take<int>(8);
        dGatherPos = a.take<int32_t>(std::max(np, 1));
        dGatherOut = a.take<uint32_t>(std::max(np, 1));
        dRawPos = a.take<float>((size_t)3 * S.nVerts);
        dRows = a.take<PartRow>(nRows);
        dErrTri = a.take<int>(1);
    };
    Arena tmp;
    tmp.cap = arena_layout(carveTmp);
    CQ_CUDA(cudaMalloc((void **)&tmp.base, tmp.cap));
    carveTmp(tmp);
    struct TmpGuard { // the temporaries go away on every path out of this function
        char *p;
        ~TmpGuard() { cudaFree(p); }
    } tmpGuard{tmp.base};
    auto done = [&](int rc) { return rc; };
    // ---- upload: the raw arrays as the plan says (large parts from the caller's memory, small ones staged), then expand
    for (const UploadCopy &c : in.copies) {
        if (c.kind == 0) {
            const float *src = c.src ? (const float *)c.src : in.stagedPos.data() + 3 * c.stagedOffset;
            CQ_CUDA(cudaMemcpyAsync(dRawPos + 3 * c.dstUnit, src, sizeof(float) * 3 * c.nUnits, cudaMemcpyHostToDevice, st));
        } else {
            const uint32_t *src = c.src ? (const uint32_t *)c.src : in.stagedIdx.data() + 3 * c.stagedOffset;
            CQ_CUDA(cudaMemcpyAsync(dIdxIn + 3 * c.dstUnit, src, sizeof(uint32_t) * 3 * c.nUnits, cudaMemcpyHostToDevice, st));
        }
    }
    if (nRows) CQ_CUDA(cudaMemcpyAsync(dRows, in.rows.data(), sizeof(PartRow) * (size_t)nRows, cudaMemcpyHostToDevice, st));
    if (nIn && np) CQ_CUDA(cudaMemcpyAsync(dGatherPos, partTriStartIn.data(), sizeof(int32_t) * np, cudaMemcpyHostToDevice, st));
    if (S.nVerts) {
        k_expand_verts<<<cdiv(S.nVerts, 256), 256, 0, st>>>(dRawPos, S.nVerts, dRows, nRows, S.localPos);
        w->launches++;
    }
    if (nIn) {
        int errTri = INT32_MAX;
        CQ_CUDA(cudaMemcpyAsync(dErrTri, &errTri, sizeof(int), cudaMemcpyHostToDevice, st));
        k_expand_tris<<<cdiv(nIn, 256), 256, 0, st>>>(dIdxIn, nIn, dRows, nRows, dLayerIn, dPartIn, dErrTri);
        w->launches++;
        CQ_CUDA(cudaMemcpyAsync(&errTri, dErrTri, sizeof(int), cudaMemcpyDeviceToHost, st));
        CQ_CUDA(cudaStreamSynchronize(st));
        if (errTri != INT32_MAX) {
            *badTriangle = errTri;
            return done(CQ_ERR_INVALID);
        }
    }
    // ---- kernels (timed: build_ms is device time of the build kernels, uploads and allocations excluded)
    cudaEvent_t e0, e1;
    CQ_CUDA(cudaEventCreate(&e0));
    CQ_CUDA(cudaEventCreate(&e1));
    cudaEventRecord(e0, st);
    uint32_t total = 0;
    if (S.nVerts) {
        k_transform<<<cdiv(S.nVerts, 256), 256, 0, st>>>(S.localPos, S.worldPos, w->dModels, 0, S.nVerts);
        w->launches++;
    }
    if (nIn) {
        k_filter_flags<<<cdiv(nIn, 256), 256, 0, st>>>(S.worldPos, dIdxIn, nIn, dFlags);
        w->launches++;
        int r = exclusive_scan_u32(w, dFlags, nIn, dOffs, dTileSums, dTotal);
        if (r != CQ_OK) {
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            return done(r);
        }
        CQ_CUDA(cudaMemcpyAsync(dOffs + nIn, dTotal, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st)); // dOffs[nIn] = total
        if (np) {
            k_gather_u32<<<cdiv(np, 256), 256, 0, st>>>(dOffs, dGatherPos, np, dGatherOut);
            w->launches++;
        }
        std::vector<uint32_t> outv(std::max(np, 1));
        CQ_CUDA(cudaMemcpyAsync(&total, dTotal, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (np) CQ_CUDA(cudaMemcpyAsync(outv.data(), dGatherOut, sizeof(uint32_t) * np, cudaMemcpyDeviceToHost, st));
        CQ_CUDA(cudaStreamSynchronize(st)); // the filtered triangle count sizes the remaining launches
        for (int i = 0; i < np; i++) partTriStartIn[i] = (int)outv[i];
    } else {
        for (auto &v : partTriStartIn) v = 0;
    }
    if (total > (1u << 26)) { // ring entries and leaf references carry 26-bit triangle slots (cq_pool.cuh, cq_query.cu)
        set_error("cq_world_create: %u triangles in one set after the degenerate filter; the limit is 2^26 = 67,108,864", total);
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        return done(CQ_ERR_INVALID);
    }
    S.nTris = (int)total;
    const int n = S.nTris;
    int rc = CQ_OK;
    if (n > 0) {
        k_compact<<<cdiv(nIn, 256), 256, 0, st>>>(dFlags, dOffs, nIn, dIdxIn, dLayerIn, dPartIn, S.indices, S.triLayer, S.triPart);
        if (matIn) { // per-triangle materials: the rows travel through the same compaction (triSource[triLocal], :363-396)
            int32_t *dMatIn = nullptr;
            CQ_CUDA(cudaMalloc((void **)&dMatIn, sizeof(int32_t) * (size_t)nIn));
            int r = check_cuda(cudaMalloc((void **)&S.triMat, sizeof(int32_t) * (size_t)n), "triangle materials");
            if (r == CQ_OK) r = check_cuda(cudaMemcpyAsync(dMatIn, matIn, sizeof(int32_t) * (size_t)nIn, cudaMemcpyHostToDevice, st), "triangle materials");
            if (r == CQ_OK) {
                k_compact_i32<<<cdiv(nIn, 256), 256, 0, st>>>(dFlags, dOffs, nIn, dMatIn, S.triMat);
                w->launches++;
                r = check_cuda(cudaStreamSynchronize(st), "triangle materials");
            }
            cudaFree(dMatIn);
            if (r != CQ_OK) {
                cudaEventDestroy(e0);
                cudaEventDestroy(e1);
                return done(r);
            }
        }
        k_init_bounds<<<1, 32, 0, st>>>(dBounds);
        k_centroid_bounds<<<cdiv(n, 256), 256, 0, st>>>(S.worldPos, S.indices, n, dBounds);
        k_morton<<<cdiv(n, 256), 256, 0, st>>>(S.worldPos, S.indices, n, dBounds, dKeys, S.sortedTri);
        w->launches += 4;
        rc = use_classic_sort() ? radix_sort_pairs_classic(w, dKeys, S.sortedTri, dKeysTmp, dValsTmp, n, dHist)
                                : radix_sort_pairs_onesweep(w, dKeys, S.sortedTri, dKeysTmp, dValsTmp, n, dHist, histWords);
        if (rc == CQ_OK) rc = build_tree(w, S, dKeys, st);
        if (rc == CQ_OK) { // for the dirty-subtree refit: where every triangle sits, and clean marking counters
            k_invert_sorted<<<cdiv(n, 256), 256, 0, st>>>(S.sortedTri, n, S.slotOfTri);
            w->launches++;
            rc = check_cuda(cudaMemsetAsync(S.expect, 0, sizeof(int32_t) * (size_t)n, st), "expect");
        }
    } else {
        rc = build_tree(w, S, nullptr, st);
    }
    cudaEventRecord(e1, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (rc == CQ_OK) rc = check_cuda(e, "build sync");
    float ms = 0;
    if (rc == CQ_OK && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) w->buildMs += ms;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return done(rc);
}

// ---------------------------------------------------------------- coherent processing order for big worlds
// Queries arrive in arbitrary order; on a world that does not fit the caches (10 M triangles = 1.1 GB of nodes
// + triangles) neighbouring lanes then touch unrelated subtrees.  For such worlds the persistent kernels fetch
// their work units through `order[]`, the units' indices sorted by the 30-bit Morton code of their position
// (same onesweep sort as the build).  Results are written to the units' own slots, so the order is invisible.
__global__ void k_order_keys(const unsigned char *__restrict__ base, size_t stride, int isDouble, int n,
                             const SetHeader *__restrict__ hdr, uint32_t *__restrict__ keys, uint32_t *__restrict__ vals) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned char *p = base + (size_t)i * stride;
    float x, y, z;
    if (isDouble) {
        const double *d = reinterpret_cast<const double *>(p);
        x = (float)d[0], y = (float)d[1], z = (float)d[2];
    } else {
        const float *f = reinterpret_cast<const float *>(p);
        x = f[0], y = f[1], z = f[2];
    }
    SetHeader h = *hdr;
    const f3 lo = {h.lo[0], h.lo[1], h.lo[2]}, hi = {h.hi[0], h.hi[1], h.hi[2]};
    keys[i] = morton30_adaptive(mk3(x, y, z), lo, hi - lo);
    vals[i] = (uint32_t)i;
}

const uint32_t *make_unit_order(cq_world *w, const void *dUnits, size_t stride, bool positionIsDouble, int n, cudaStream_t st) {
    if (n < (1 << 16) || w->set[0].nTris < (1 << 18)) return nullptr; // small world / batch: everything is cache resident
    const int tiles = cdiv(n, RS_TILE);
    const size_t sortWords = (size_t)4 * 256 * tiles + 4 + 1024 + 1;
    const size_t words = (size_t)4 * n + sortWords + 64;
    ScratchBuf &b = w->orderScratch[w->orderSeq++ & 3];
    if (words * 4 > b.cap) {
        if (check_cuda(cudaDeviceSynchronize(), "order scratch sync") != CQ_OK) return nullptr;
        for (int k = 0; k < 4; k++)
            if (ensure_scratch(w->orderScratch[k], words * 4) != CQ_OK) return nullptr;
    }
    if (scratch_acquire(w, b, st) != CQ_OK) return nullptr;
    uint32_t *keys = (uint32_t *)b.ptr, *vals = keys + n, *keysTmp = vals + n, *valsTmp = keysTmp + n, *scratch = valsTmp + n;
    k_order_keys<<<cdiv(n, 256), 256, 0, st>>>((const unsigned char *)dUnits, stride, positionIsDouble ? 1 : 0, n, w->set[0].hdr,
                                               keys, vals);
    w->launches++;
    if (radix_sort_pairs_onesweep(w, keys, vals, keysTmp, valsTmp, n, scratch, sortWords, st, false) != CQ_OK) return nullptr;
    return vals;
}

size_t sort_scratch_words(int n) { return (size_t)4 * 256 * cdiv(n, RS_TILE) + 4 + 1024 + 1; }
int sort_pairs_u32(cq_world *w, uint32_t *keys, uint32_t *vals, uint32_t *keysTmp, uint32_t *valsTmp, int n, uint32_t *scratch,
                   size_t scratchWords, cudaStream_t st) {
    return radix_sort_pairs_onesweep(w, keys, vals, keysTmp, valsTmp, n, scratch, scratchWords, st, false);
}

// ---------------------------------------------------------------- agent snapshot + grid (CQ_MAS_AGENTS)
// bounds: [0..1] min x,z  [2..3] max x,z  [4] max |v|  (ordered ints)
__global__ void k_agent_bounds_init(int *bounds) {
    if (threadIdx.x < 5) {
        const float init = threadIdx.x < 2 ? FLT_MAX : (threadIdx.x < 4 ? -FLT_MAX : 0.0f);
        bounds[threadIdx.x] = float_to_ordered(init);
    }
}
__global__ void k_agent_snapshot(const cq_character_state *__restrict__ states, int n, float dt, float gx, float gy, float gz,
                                 uint32_t flags, float4 *__restrict__ pos, float4 *__restrict__ vel, int *bounds) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    float v[5] = {FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, 0.0f};
    if (i < n) {
        const cq_character_state &S = states[i];
        d3 vd = {S.velocity[0], S.velocity[1], S.velocity[2]};
        // collectAgentStates runs after GravitySystem (system #3), so the snapshot carries the post-gravity velocity
        if ((flags & CQ_MAS_APPLY_GRAVITY) && !(S.grounded != 0 && S.grounded_near != 0))
            vd = vd + to_d3(mk3(gx, gy, gz)) * (double)dt;
        f3 p = {(float)S.position[0], (float)S.position[1], (float)S.position[2]};
        f3 vf = to_f3(vd);
        pos[i] = make_float4(p.x, p.y, p.z, __int_as_float(i));
        vel[i] = make_float4(vf.x, vf.y, vf.z, 0.0f);
        v[0] = p.x, v[1] = p.z, v[2] = p.x, v[3] = p.z;
        v[4] = sqrtf(vf.x * vf.x + vf.y * vf.y + vf.z * vf.z);
    }
    __shared__ float red[5][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        float x = v[k];
        for (int o = 16; o > 0; o >>= 1) {
            float y = __shfl_xor_sync(0xffffffffu, x, o);
            x = k < 2 ? fminf(x, y) : fmaxf(x, y);
        }
        if (lane == 0) red[k][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        const int k = threadIdx.x;
        float x = red[k][0];
        for (int wi = 1; wi < (int)(blockDim.x >> 5); wi++) x = k < 2 ? fminf(x, red[k][wi]) : fmaxf(x, red[k][wi]);
        if (k < 2) atomicMin(bounds + k, float_to_ordered(x));
        else atomicMax(bounds + k, float_to_ordered(x));
    }
}

// cell = the farthest two agents can be apart (XZ) and still touch within one step, so a sweep looks at 3x3 cells;
// any cell size is exact (the kernel derives its cell range from the actual reach), this one is just the fast one
__global__ void k_agent_grid_params(const int *bounds, float radius, float dt, AgentGridParams *out) {
    float minX = ordered_to_float(bounds[0]), minZ = ordered_to_float(bounds[1]);
    float maxX = ordered_to_float(bounds[2]), maxZ = ordered_to_float(bounds[3]);
    float vmax = ordered_to_float(bounds[4]);
    if (!(vmax >= 0.0f) || vmax > 1e18f) vmax = 1e18f;
    float cell = (2.0f * radius + 2.0f * vmax * dt) * 1.01f + 1e-3f;
    float ex = fmaxf(maxX - minX, 0.0f), ez = fmaxf(maxZ - minZ, 0.0f);
    if (!(ex < 1e30f)) ex = 1e30f;
    if (!(ez < 1e30f)) ez = 1e30f;
    const float maxDim = 32767.0f; // 15 bits per axis -> 30-bit keys, what the radix sort handles
    cell = fmaxf(cell, fmaxf(ex, ez) / (maxDim - 1.0f));
    out->originX = minX, out->originZ = minZ;
    out->cell = cell, out->invCell = 1.0f / cell;
    out->dimX = (int)fminf(floorf(ex / cell) + 1.0f, maxDim);
    out->dimZ = (int)fminf(floorf(ez / cell) + 1.0f, maxDim);
    out->maxSpeed = vmax;
    out->_pad = 0.0f;
}

__global__ void k_agent_keys(const float4 *__restrict__ pos, int n, const AgentGridParams *__restrict__ gp, uint32_t *keys,
                             uint32_t *vals) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const AgentGridParams G = *gp;
    float4 p = pos[i];
    keys[i] = (uint32_t)agent_cell(p.z, G.originZ, G.invCell, G.dimZ) * (uint32_t)G.dimX +
              (uint32_t)agent_cell(p.x, G.originX, G.invCell, G.dimX);
    vals[i] = (uint32_t)i;
}

__global__ void k_agent_gather(const uint32_t *__restrict__ vals, int n, const float4 *__restrict__ pos,
                               const float4 *__restrict__ vel, float4 *__restrict__ posS, float4 *__restrict__ velS) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t j = vals[i];
    posS[i] = pos[j];
    velS[i] = vel[j];
}

// one thread per agent: the three sorted-array ranges its 3x3 cell neighbourhood occupies (binary searches done here,
// at full occupancy, instead of by a lone lane inside the move-and-slide kernel)
__global__ void k_agent_rows(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ vals, int n,
                             const AgentGridParams *__restrict__ gp, int4 *__restrict__ rows) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int dimX = gp->dimX, dimZ = gp->dimZ;
    const uint32_t key = keys[j];
    const int iz = (int)(key / (uint32_t)dimX), ix = (int)(key % (uint32_t)dimX);
    int se[6];
    for (int dz = -1; dz <= 1; dz++) {
        int row = iz + dz, start = 0, end = 0;
        if (row >= 0 && row < dimZ) {
            const uint32_t keyLo = (uint32_t)row * (uint32_t)dimX + (uint32_t)max(ix - 1, 0);
            const uint32_t keyHi = (uint32_t)row * (uint32_t)dimX + (uint32_t)min(ix + 1, dimX - 1);
            int lo = 0, hi = n;
            while (lo < hi) { // lower_bound(keyLo)
                int mid = (lo + hi) >> 1;
                if (keys[mid] < keyLo) lo = mid + 1;
                else hi = mid;
            }
            start = lo;
            hi = n;
            while (lo < hi) { // upper_bound(keyHi)
                int mid = (lo + hi) >> 1;
                if (keys[mid] <= keyHi) lo = mid + 1;
                else hi = mid;
            }
            end = lo;
        }
        se[2 * (dz + 1)] = start, se[2 * (dz + 1) + 1] = end;
    }
    const uint32_t orig = vals[j];
    rows[2 * (size_t)orig] = make_int4(se[0], se[1], se[2], se[3]);
    rows[2 * (size_t)orig + 1] = make_int4(se[4], se[5], ix, iz);
}

int make_agent_grid(cq_world *w, const cq_character_state *dStates, int n, float radius, float dt, const float g[3],
                    uint32_t flags, cudaStream_t st, AgentGrid &out) {
    const int tiles = cdiv(n, RS_TILE);
    const size_t sortWords = (size_t)4 * 256 * tiles + 4 + 1024 + 1;
    // [pos n][vel n][posS n][velS n] float4, [rows 2n] int4, [firstHit n] float4, [keys n][vals n][keysTmp n][valsTmp n] u32, sort scratch,
    // bounds, params
    const size_t bytes = (size_t)n * 112 + ((size_t)4 * n + sortWords + 64) * 4;
    if (bytes > w->agentScratch.cap) {
        CQ_CUDA(cudaDeviceSynchronize());
        CQ_TRY(ensure_scratch(w->agentScratch, bytes));
    }
    CQ_TRY(scratch_acquire(w, w->agentScratch, st));
    float4 *pos = (float4 *)w->agentScratch.ptr, *vel = pos + n, *posS = vel + n, *velS = posS + n;
    int4 *rows = (int4 *)(velS + n);
    float4 *firstHit = (float4 *)(rows + 2 * (size_t)n);
    uint32_t *keys = (uint32_t *)(firstHit + n), *vals = keys + n, *keysTmp = vals + n, *valsTmp = keysTmp + n;
    uint32_t *scratch = valsTmp + n;
    int *bounds = (int *)(scratch + sortWords);
    AgentGridParams *gp = (AgentGridParams *)(bounds + 8);
    k_agent_bounds_init<<<1, 32, 0, st>>>(bounds);
    k_agent_snapshot<<<cdiv(n, 256), 256, 0, st>>>(dStates, n, dt, g[0], g[1], g[2], flags, pos, vel, bounds);
    k_agent_grid_params<<<1, 1, 0, st>>>(bounds, radius, dt, gp);
    k_agent_keys<<<cdiv(n, 256), 256, 0, st>>>(pos, n, gp, keys, vals);
    w->launches += 4;
    CQ_TRY(radix_sort_pairs_onesweep(w, keys, vals, keysTmp, valsTmp, n, scratch, sortWords, st, false));
    k_agent_gather<<<cdiv(n, 256), 256, 0, st>>>(vals, n, pos, vel, posS, velS);
    k_agent_rows<<<cdiv(n, 256), 256, 0, st>>>(keys, vals, n, gp, rows);
    w->launches += 2;
    out.pos = posS, out.vel = velS, out.keys = keys, out.params = gp, out.rows = rows, out.firstHit = firstHit, out.n = n;
    return check_cuda(cudaGetLastError(), "agent grid");
}

// ---------------------------------------------------------------- reference order (cq_reftree.h)
// Boxes of the reference's tree, bottom-up: one thread per leaf computes boundsForRange (CollisionQuery.swift:662-677)
// from the leaf's triangles, writes it into its parent's child slot and climbs while it is the second child to arrive
// (merge = component-wise min / max, :700-702 — exact, so the arrival order does not matter).  Arrival counters are
// left at zero, so the same kernel serves every refit (BVH.refit :528-575 touches only the ancestors of moved leaves;
// refitting everything gives the same boxes).
__device__ __forceinline__ void ref_store_child_box(Node *nd, int which, f3 lo, f3 hi) { // keeps the refs in n0.w / n1.w
    float *p = reinterpret_cast<float *>(nd);
    float *l = p + (which ? 8 : 0), *h = p + (which ? 12 : 4);
    l[0] = lo.x, l[1] = lo.y, l[2] = lo.z;
    h[0] = hi.x, h[1] = hi.y, h[2] = hi.z;
}

__global__ void k_ref_fit(int nLeaves, const int32_t *__restrict__ leafRange, const int32_t *__restrict__ leafParent,
                          const int32_t *__restrict__ nodeParent, const uint32_t *__restrict__ refSlot,
                          const float4 *__restrict__ tv0, const float4 *__restrict__ tv1, const float4 *__restrict__ tv2,
                          Node *nodes, int32_t *visit, SetHeader *hdr) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nLeaves) return;
    const int range = leafRange[l], start = range >> 2, count = (range & 3) + 1;
    f3 lo = {0, 0, 0}, hi = {0, 0, 0};
    for (int k = 0; k < count; k++) {
        const uint32_t slot = refSlot[start + k];
        const f3 a = xyz(tv0[slot]), b = xyz(tv1[slot]), c = xyz(tv2[slot]);
        const f3 tlo = vmin(a, vmin(b, c)), thi = vmax(a, vmax(b, c));
        lo = k ? vmin(lo, tlo) : tlo;
        hi = k ? vmax(hi, thi) : thi;
    }
    int pw = leafParent[l];
    while (true) {
        if (pw < 0) { // the root's own box lives in the header
            hdr->lo[0] = lo.x, hdr->lo[1] = lo.y, hdr->lo[2] = lo.z;
            hdr->hi[0] = hi.x, hdr->hi[1] = hi.y, hdr->hi[2] = hi.z;
            return;
        }
        const int p = pw >> 1;
        ref_store_child_box(nodes + p, pw & 1, lo, hi);
        __threadfence();
        if (atomicAdd(&visit[p], 1) == 0) return; // first arrival: the sibling subtree is not done yet
        visit[p] = 0;
        __threadfence();
        const float4 *q = reinterpret_cast<const float4 *>(nodes + p);
        const float4 l0 = __ldcg(q), h0 = __ldcg(q + 1), l1 = __ldcg(q + 2), h1 = __ldcg(q + 3);
        lo = vmin(xyz(l0), xyz(l1));
        hi = vmax(xyz(h0), xyz(h1));
        pw = nodeParent[p];
    }
}

static int ref_fit(cq_world *w, DeviceSet &S, cudaStream_t st) {
    if (!S.refArena || S.nRefLeaves <= 0) return CQ_OK;
    k_ref_fit<<<cdiv(S.nRefLeaves, 256), 256, 0, st>>>(S.nRefLeaves, S.refLeafRange, S.refLeafParent, S.refNodeParent,
                                                     S.refSlot, S.tv0, S.tv1, S.tv2, S.refNodes, S.refVisit, S.refHdr);
    w->launches++;
    return check_cuda(cudaGetLastError(), "k_ref_fit");
}

static inline float int_bits_as_float(int v) {
    float f;
    memcpy(&f, &v, sizeof(f));
    return f;
}

// Reference order: download the sets' triangle boxes, rebuild the reference's tree on the host (cq_reftree.h), upload
// the visiting ranks (one global array, static set first like the reference's own merge of its two sets,
// CollisionQuery.swift:990-1008) and the tree itself for the ray walk.
int attach_ref_order(cq_world *w) {
    const auto t0 = std::chrono::steady_clock::now();
    cudaStream_t st = w->stream;
    const int nS = w->set[0].nTris, nD = w->set[1].nTris;
    std::vector<int32_t> rankAll((size_t)nS + nD);
    std::vector<uint32_t> encOfRank((size_t)nS + nD);
    for (int s = 0; s < 2; s++) {
        DeviceSet &S = w->set[s];
        const int n = S.nTris;
        if (n <= 0) continue;
        // triangle boxes as the device computed them (leaf boxes of the sorted order) back in the soup's numbering
        std::vector<float4> sLo(n), sHi(n), lo(n), hi(n);
        std::vector<uint32_t> sorted(n), slotOf(n);
        CQ_CUDA(cudaMemcpyAsync(sLo.data(), S.boxLo + (n - 1), sizeof(float4) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CQ_CUDA(cudaMemcpyAsync(sHi.data(), S.boxHi + (n - 1), sizeof(float4) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CQ_CUDA(cudaMemcpyAsync(sorted.data(), S.sortedTri, sizeof(uint32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CQ_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < n; k++) lo[sorted[k]] = sLo[k], hi[sorted[k]] = sHi[k], slotOf[sorted[k]] = (uint32_t)k;
        RefTree T;
        build_ref_tree(&lo[0].x, &hi[0].x, 4, n, T);
        const int off = s == 0 ? 0 : nS;
        for (int t = 0; t < n; t++) {
            rankAll[(size_t)off + t] = off + T.rank[t];
            encOfRank[(size_t)off + T.rank[t]] = ((uint32_t)s << 26) | slotOf[t];
        }
        // device form: internal nodes and leaves numbered separately
        const int nNodes = (int)T.nodes.size();
        std::vector<int32_t> idOf(nNodes);
        int nInt = 0, nLeaf = 0;
        for (int k = 0; k < nNodes; k++) idOf[k] = T.nodes[k].left >= 0 ? nInt++ : nLeaf++;
        std::vector<Node> nodes(std::max(nInt, 1));
        std::vector<int32_t> nodeParent(std::max(nInt, 1), -1), leafParent(std::max(nLeaf, 1), -1), leafRange(std::max(nLeaf, 1), 0);
        std::vector<uint32_t> refSlot(n);
        for (int p = 0; p < n; p++) refSlot[p] = slotOf[T.order[p]];
        std::vector<int32_t> leafOfTri(n);
        auto ref_of = [&](int k) { // reference to node k as a parent stores it
            const RefNode &nd = T.nodes[k];
            return nd.left >= 0 ? idOf[k] : ~((nd.start << 2) | (nd.count - 1));
        };
        int depthMax = 0; // the ray walk keeps one stack entry per level
        for (int k = 0; k < nNodes; k++) {
            if (T.nodes[k].left >= 0) continue;
            int d = 0;
            for (int q = T.nodes[k].parent; q >= 0; q = T.nodes[q].parent) d++;
            depthMax = std::max(depthMax, d);
        }
        for (int k = 0; k < nNodes; k++) {
            const RefNode &nd = T.nodes[k];
            int pw = -1;
            if (nd.parent >= 0) pw = (idOf[nd.parent] << 1) | (T.nodes[nd.parent].right == k ? 1 : 0);
            if (nd.left >= 0) {
                Node &o = nodes[idOf[k]];
                o.n0 = make_float4(0, 0, 0, int_bits_as_float(ref_of(nd.left)));
                o.n1 = make_float4(0, 0, 0, int_bits_as_float(ref_of(nd.right)));
                o.n2 = make_float4(0, 0, 0, 0), o.n3 = make_float4(0, 0, 0, 0);
                nodeParent[idOf[k]] = pw;
            } else {
                leafParent[idOf[k]] = pw;
                leafRange[idOf[k]] = (nd.start << 2) | (nd.count - 1);
                for (int q = nd.start; q < nd.start + nd.count; q++) leafOfTri[T.order[q]] = idOf[k];
            }
        }
        if (depthMax + 2 > CQ_STACK) {
            set_error("cq_world_create: the reference tree of set %d is %d levels deep (limit %d); use CQ_ORDER_CANONICAL", s, depthMax,
                      CQ_STACK - 2);
            return CQ_ERR_INVALID;
        }
        auto carve = [&](Arena &a) {
            S.refNodes = a.take<Node>(nInt);
            S.refSlot = a.take<uint32_t>(n);
            S.refNodeParent = a.take<int32_t>(nInt);
            S.refLeafParent = a.take<int32_t>(nLeaf);
            S.refLeafRange = a.take<int32_t>(nLeaf);
            S.refVisit = a.take<int32_t>(nInt);
            S.refExpect = a.take<int32_t>(nInt);
            S.refLeafMark = a.take<int32_t>(nLeaf);
            S.refLeafOfTri = a.take<int32_t>(n);
            S.refHdr = a.take<SetHeader>(1);
        };
        Arena arena;
        arena.cap = arena_layout(carve);
        CQ_CUDA(cudaMalloc((void **)&arena.base, arena.cap));
        S.refArena = arena.base;
        carve(arena);
        S.nRefInternal = nInt, S.nRefLeaves = nLeaf, S.refDepth = depthMax;
        SetHeader h;
        h.nTris = n;
        h.rootRef = ref_of(0);
        h.lo[0] = h.lo[1] = h.lo[2] = 0.0f, h.hi[0] = h.hi[1] = h.hi[2] = 0.0f;
        CQ_CUDA(cudaMemcpyAsync(S.refNodes, nodes.data(), sizeof(Node) * (size_t)std::max(nInt, 1), cudaMemcpyHostToDevice, st));
        CQ_CUDA(cudaMemcpyAsync(S.refSlot, refSlot.data(), sizeof(uint32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
        CQ_CUDA(cudaMemcpyAsync(S.refNodeParent, nodeParent.data(), sizeof(int32_t) * (size_t)std::max(nInt, 1), cudaMemcpyHostToDevice, st));
        CQ_CUDA(cudaMemcpyAsync(S.refLeafParent, leafParent.data(), sizeof(int32_t) * (size_t)std::max(nLeaf, 1), cudaMemcpyHostToDevice, st));
        CQ_CUDA(cudaMemcpyAsync(S.refLeafRange, leafRange.data(), sizeof(int32_t) * (size_t)std::max(nLeaf, 1), cudaMemcpyHostToDevice, st));
        CQ_CUDA(cudaMemsetAsync(S.refVisit, 0, sizeof(int32_t) * (size_t)std::max(nInt, 1), st));
        CQ_CUDA(cudaMemsetAsync(S.refExpect, 0, sizeof(int32_t) * (size_t)std::max(nInt, 1), st));
        CQ_CUDA(cudaMemsetAsync(S.refLeafMark, 0, sizeof(int32_t) * (size_t)std::max(nLeaf, 1), st));
        CQ_CUDA(cudaMemcpyAsync(S.refLeafOfTri, leafOfTri.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
        CQ_CUDA(cudaMemcpyAsync(S.refHdr, &h, sizeof(h), cudaMemcpyHostToDevice, st));
        CQ_TRY(ref_fit(w, S, st));
        CQ_CUDA(cudaStreamSynchronize(st)); // the host vectors above are the copies' sources
    }
    if (nS + nD > 0) {
        CQ_CUDA(cudaMalloc((void **)&w->dRank, sizeof(int32_t) * (size_t)(nS + nD)));
        CQ_CUDA(cudaMemcpy(w->dRank, rankAll.data(), sizeof(int32_t) * (size_t)(nS + nD), cudaMemcpyHostToDevice));
        CQ_CUDA(cudaMalloc((void **)&w->dEncOfRank, sizeof(uint32_t) * (size_t)(nS + nD)));
        CQ_CUDA(cudaMemcpy(w->dEncOfRank, encOfRank.data(), sizeof(uint32_t) * (size_t)(nS + nD), cudaMemcpyHostToDevice));
    }
    // the ranks travel in tv2.w: rewrite the sorted SoA now that they are known (it was gathered with rank = index)
    for (int s = 0; s < 2; s++) {
        DeviceSet &S = w->set[s];
        if (S.nTris <= 0) continue;
        k_gather_sorted<<<cdiv(S.nTris, 256), 256, 0, st>>>(S.sortedTri, S.nTris, S.worldPos, S.indices, S.triLayer, w->dRank,
                                                            s == 0 ? 0 : nS, S.tv0, S.tv1, S.tv2);
        w->launches++;
    }
    CQ_CUDA(cudaStreamSynchronize(st));
    w->refBuildMs = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return CQ_OK;
}

// TriangleMeshSet.updateTransforms + BVH.refit: re-transform the moved parts' vertices (k_update_parts), then
//   * few triangles moved (less than a quarter of the set): the dirty-subtree refit above — the updated triangles' slots,
//     their leaves and only the ancestors of those, in the LBVH, its 4-wide collapse and (reference order) the reference's
//     own tree, like BVH.refit (CollisionQuery.swift:528-575): 1 + 3 + 3 + 1 launches;
//   * otherwise: regather the whole sorted SoA and recompute every box bottom-up (same topology): 1 + 4 + 1 launches.
// Both give the same boxes (min / max are exact).  Stream-ordered on `st`, no host synchronisation.
int refit_set(cq_world *w, DeviceSet &S, const MovedPart *dTab, const std::vector<MovedPart> &rows, cudaStream_t st) {
    const int nRows = (int)rows.size();
    if (nRows == 0) return CQ_OK;
    const int nVerts = rows.back().vertBase + rows.back().nVerts, moved = rows.back().triBase + rows.back().nTris;
    k_update_parts<<<cdiv(nVerts, 256), 256, 0, st>>>(dTab, nRows, nVerts, S.localPos, S.worldPos, w->dModels);
    w->launches++;
    static const bool forceFull = getenv("CQ_REFIT_FULL") != nullptr; // A/B and the test that both paths agree
    if (forceFull || (long long)moved * 4 >= (long long)S.nTris) {
        CQ_TRY(build_tree(w, S, nullptr, st));
        return ref_fit(w, S, st); // reference order: the reference's own tree keeps its topology too (BVH.refit)
    }
    const int n = S.nTris, blocks = cdiv(moved, 256);
    k_refit_mark<<<blocks, 256, 0, st>>>(dTab, nRows, moved, S.slotOfTri, n, S.worldPos, S.indices, S.tv0, S.tv1, S.tv2, S.parent,
                                         S.boxLo, S.boxHi, S.expect);
    k_refit_climb<<<blocks, 256, 0, st>>>(dTab, nRows, moved, S.slotOfTri, n, S.nodes, S.parent, S.boxLo, S.boxHi, S.visit, S.expect,
                                          S.depthParity, S.nodes4);
    k_refit_clear<<<blocks, 256, 0, st>>>(dTab, nRows, moved, S.slotOfTri, n, S.parent, S.visit, S.expect);
    w->launches += 3;
    if (S.refArena && S.nRefLeaves > 0) {
        k_ref_refit_mark<<<blocks, 256, 0, st>>>(dTab, nRows, moved, S.refLeafOfTri, S.refLeafRange, S.refLeafParent, S.refNodeParent,
                                                 S.refSlot, S.tv0, S.tv1, S.tv2, S.refNodes, S.refLeafMark, S.refExpect, S.refHdr);
        k_ref_refit_climb<<<blocks, 256, 0, st>>>(dTab, nRows, moved, S.refLeafOfTri, S.refLeafParent, S.refNodeParent, S.refNodes,
                                                  S.refLeafMark, S.refVisit, S.refExpect, S.refHdr);
        k_ref_refit_clear<<<blocks, 256, 0, st>>>(dTab, nRows, moved, S.refLeafOfTri, S.refLeafParent, S.refNodeParent,
                                                  S.refLeafMark, S.refVisit, S.refExpect);
        w->launches += 3;
    }
    k_header<<<1, 32, 0, st>>>(n, S.boxLo, S.boxHi, S.hdr);
    w->launches++;
    return check_cuda(cudaGetLastError(), "dirty refit");
}

} // namespace cq
