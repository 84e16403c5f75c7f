// cq_reftree.h — the reference's own BVH (Game/CollisionQuery.swift:496-707), restated on the host, for ONE purpose:
// the ORDER in which the reference visits triangles.
//
// Why it exists.  Every query of the reference is a depth-first walk of its median-split tree that pushes the left
// child, then the right one (so the right subtree is visited first, :1106-1107, :965-966, :1277-1278), and keeps the
// FIRST visited triangle on exactly equal keys (strict `<` / `>`: :1084, :944, :1172) or simply the first `maxHits`
// overlaps (:1272-1274).  Which triangles are candidates does not depend on the tree (nodes are culled by box overlap
// only), so the library walks its own LBVH — but to name the same triangle as the reference on ties, and to return the
// same `maxHits` overlaps, it needs the reference's visiting rank of every triangle.  That rank is a property of the
// tree alone: subtrees are only ever skipped, never reordered.  Raycasts additionally cull by `tmin > closestT` with a
// slab test that is not conservative in floating point (:933, :1603-1631), so their answers can depend on the tree's
// boxes themselves; in reference order the ray kernel therefore walks THIS tree (as 64-byte nodes) with the reference's
// own slab test.  The library cuts the same tree on the device (cq_build.cu: attach_ref_order); this restatement is the
// reference the tests compare that build with.
//
// The split rule is restated from the Swift (spatial median of the centroid bounds along their longest axis, the
// swap-with-tail partition of :617-634, the sorted-median fallback of :637-653, leaves of <= 4 triangles); the
// implementation is this library's own: items carry their centroid so the partition streams through memory, the top
// of the tree is cut by a pool of workers (one task per node, the two halves queued as new tasks), the subtrees below
// a grain size are built in parallel into private node arrays and spliced together afterwards.  The numbering of the
// nodes is deterministic but not the reference's preorder — nothing observable depends on it.
//
// Host-only, no CUDA: tests compile it into a CPU harness (tests/hostmath/reftree.cpp).
#pragma once
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

namespace cq {

struct RefNode {
    int32_t left, right; // children (internal node), -1 / -1 for a leaf
    int32_t start, count; // leaf: its range of `order`; internal: 0, 0
    int32_t parent;       // -1 for the root
};

struct RefTree {
    std::vector<RefNode> nodes; // nodes[0] is the root (when there is any triangle)
    std::vector<int32_t> order; // position -> triangle (the reference's triOrder after the build)
    std::vector<int32_t> rank;  // triangle -> position in the reference's visiting order (0 = visited first)
    int32_t nLeaves = 0;
};

namespace reftree_detail {

struct Item { // one triangle while the tree is being cut: AABB centroid (:696-698) + its id
    float c[3];
    int32_t tri;
};

// centroid bounds of a range (:679-694), longest axis (:602-610: x wins ties over y wins ties over z), pivot (:612-617)
static inline void split_plane(const Item *it, int start, int count, int &axis, float &pivot) {
    float lo[3] = {it[start].c[0], it[start].c[1], it[start].c[2]};
    float hi[3] = {lo[0], lo[1], lo[2]};
    for (int i = start + 1; i < start + count; i++)
        for (int a = 0; a < 3; a++) {
            const float v = it[i].c[a];
            lo[a] = v < lo[a] ? v : lo[a]; // simd_min / simd_max
            hi[a] = v > hi[a] ? v : hi[a];
        }
    const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
    axis = (ex >= ey && ex >= ez) ? 0 : (ey >= ez ? 1 : 2);
    pivot = (lo[axis] + hi[axis]) * 0.5f;
}

// The reference's partition (:617-634): walk i up from the front; an element that is not `< pivot` is swapped with the
// current tail, and the element that arrives from the tail is examined next.  When everything lands on one side the
// range is (stably) sorted by the centroid along the axis and cut in the middle (:637-653).  Returns the cut.
static inline int partition_range(Item *it, int start, int count, int axis, float pivot) {
    int i = start, j = start + count - 1;
    while (i <= j) { // branch-free form of `if value < pivot { i += 1 } else { swapAt(i, j); j -= 1 }` (the outcome is a coin flip)
        const Item a = it[i], b = it[j];
        const bool lt = a.c[axis] < pivot;
        it[i] = lt ? a : b;
        it[j] = lt ? b : a;
        i += lt ? 1 : 0;
        j -= lt ? 0 : 1;
    }
    const int end = start + count;
    if (i == start || i == end) {
        std::stable_sort(it + start, it + end, [axis](const Item &a, const Item &b) { return a.c[axis] < b.c[axis]; });
        i = start + count / 2;
    }
    return i;
}

static inline int32_t add_node(std::vector<RefNode> &nodes, int32_t start, int32_t count, int32_t parent) {
    nodes.push_back(RefNode{-1, -1, start, count, parent});
    return (int32_t)nodes.size() - 1;
}

// cut one node; returns false when it is a leaf (:590-596)
static inline bool split_node(Item *it, std::vector<RefNode> &nodes, int32_t node, int32_t &leftStart, int32_t &leftCount,
                              int32_t &rightStart, int32_t &rightCount) {
    const int32_t start = nodes[node].start, count = nodes[node].count;
    if (count <= 4) return false; // leafTriangleLimit (:473)
    int axis;
    float pivot;
    split_plane(it, start, count, axis, pivot);
    const int mid = partition_range(it, start, count, axis, pivot);
    leftStart = start, leftCount = mid - start, rightStart = mid, rightCount = start + count - mid;
    return true;
}

// a whole subtree, depth-first with an explicit stack, into `nodes` (indices local to that vector; nodes[0] = its root)
static inline void build_subtree(Item *it, int32_t start, int32_t count, std::vector<RefNode> &nodes) {
    nodes.clear();
    add_node(nodes, start, count, -1);
    std::vector<int32_t> stack{0};
    while (!stack.empty()) {
        const int32_t node = stack.back();
        stack.pop_back();
        int32_t ls, lc, rs, rc;
        if (!split_node(it, nodes, node, ls, lc, rs, rc)) continue;
        const int32_t l = add_node(nodes, ls, lc, node), r = add_node(nodes, rs, rc, node);
        nodes[node].left = l, nodes[node].right = r, nodes[node].start = 0, nodes[node].count = 0;
        stack.push_back(l);
        stack.push_back(r);
    }
}

} // namespace reftree_detail

// lo / hi: triangle AABBs in the soup's numbering, `stride` floats apart (3 = packed xyz, 4 = float4 arrays).
inline void build_ref_tree(const float *lo, const float *hi, int stride, int n, RefTree &out, int threads = 0) {
    using namespace reftree_detail;
    out.nodes.clear();
    out.order.assign((size_t)n, 0);
    out.rank.assign((size_t)n, 0);
    out.nLeaves = 0;
    if (n <= 0) return;
    if (threads <= 0) threads = (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    std::vector<Item> items((size_t)n);
    {
        auto fill = [&](int a, int b) {
            for (int t = a; t < b; t++) {
                const float *l = lo + (size_t)t * stride, *h = hi + (size_t)t * stride;
                items[t].c[0] = (l[0] + h[0]) * 0.5f, items[t].c[1] = (l[1] + h[1]) * 0.5f, items[t].c[2] = (l[2] + h[2]) * 0.5f;
                items[t].tri = t;
            }
        };
        if (n < (1 << 16) || threads == 1) {
            fill(0, n);
        } else {
            std::vector<std::thread> th;
            for (int k = 0; k < threads; k++) th.emplace_back(fill, (int)((int64_t)n * k / threads), (int)((int64_t)n * (k + 1) / threads));
            for (auto &t : th) t.join();
        }
    }
    Item *it = items.data();
    // Phase A — the top of the tree (ranges above `grain` triangles): a pool of workers, one task per node; a task cuts its
    // range and queues the two halves, so the parallelism doubles with every level (the ranges are disjoint).
    // Phase B — the remaining subtrees, each built depth-first by one worker into a private node array.
    // The final numbering is made deterministic afterwards (preorder of the top, subtrees in range order).
    struct Top {
        int32_t start, count, left, right, parent;
    };
    std::vector<Top> top{Top{0, n, -1, -1, -1}};
    const int32_t grain = threads > 1 ? std::max<int32_t>(1 << 12, std::min<int32_t>(1 << 16, n / (threads * 16))) : n;
    if (n > grain) {
        std::mutex mu;
        std::condition_variable cv;
        std::vector<int32_t> queue{0};
        int outstanding = 1;
        auto worker = [&]() {
            std::unique_lock<std::mutex> lk(mu);
            for (;;) {
                cv.wait(lk, [&] { return !queue.empty() || outstanding == 0; });
                if (queue.empty()) return;
                const int32_t t = queue.back();
                queue.pop_back();
                const int32_t start = top[t].start, count = top[t].count;
                lk.unlock();
                int axis;
                float pivot;
                split_plane(it, start, count, axis, pivot);
                const int32_t mid = partition_range(it, start, count, axis, pivot);
                lk.lock();
                const int32_t l = (int32_t)top.size();
                top.push_back(Top{start, mid - start, -1, -1, t});
                top.push_back(Top{mid, start + count - mid, -1, -1, t});
                top[t].left = l, top[t].right = l + 1;
                int pushed = 0;
                for (int32_t c = l; c <= l + 1; c++)
                    if (top[c].count > grain) queue.push_back(c), pushed++;
                outstanding += pushed - 1;
                cv.notify_all();
            }
        };
        std::vector<std::thread> th;
        for (int k = 1; k < threads; k++) th.emplace_back(worker);
        worker();
        for (auto &t : th) t.join();
    }
    // deterministic numbering of the top: nested ranges sorted by (start ascending, count descending) = preorder
    std::vector<int32_t> byRange(top.size()), newIndex(top.size());
    for (size_t k = 0; k < top.size(); k++) byRange[k] = (int32_t)k;
    std::sort(byRange.begin(), byRange.end(), [&](int32_t a, int32_t b) {
        return top[a].start != top[b].start ? top[a].start < top[b].start : top[a].count > top[b].count;
    });
    for (size_t k = 0; k < byRange.size(); k++) newIndex[byRange[k]] = (int32_t)k;
    std::vector<RefNode> &nodes = out.nodes;
    nodes.resize(top.size());
    std::vector<int32_t> tips; // nodes of the top that still have to be grown into subtrees, in range order
    for (size_t k = 0; k < byRange.size(); k++) {
        const Top &t = top[byRange[k]];
        const bool cut = t.left >= 0;
        nodes[k] = RefNode{cut ? newIndex[t.left] : -1, cut ? newIndex[t.right] : -1, cut ? 0 : t.start, cut ? 0 : t.count,
                           t.parent >= 0 ? newIndex[t.parent] : -1};
        if (!cut) tips.push_back((int32_t)k);
    }
    std::vector<std::vector<RefNode>> sub(tips.size());
    {
        std::vector<size_t> bySize(tips.size());
        for (size_t k = 0; k < bySize.size(); k++) bySize[k] = k;
        std::sort(bySize.begin(), bySize.end(), [&](size_t a, size_t b) { return nodes[tips[a]].count > nodes[tips[b]].count; });
        std::atomic<size_t> nextTask{0};
        auto work = [&]() {
            for (;;) {
                const size_t k = nextTask.fetch_add(1);
                if (k >= bySize.size()) return;
                const RefNode &tip = nodes[tips[bySize[k]]];
                build_subtree(it, tip.start, tip.count, sub[bySize[k]]);
            }
        };
        const int nWorkers = (int)std::min<size_t>((size_t)threads, tips.size());
        if (nWorkers <= 1) {
            work();
        } else {
            std::vector<std::thread> th;
            for (int k = 0; k < nWorkers; k++) th.emplace_back(work);
            for (auto &t : th) t.join();
        }
    }
    // splice: a subtree's root IS its tip node; its other nodes are appended, subtrees in range order
    {
        size_t total = nodes.size();
        for (const auto &S : sub) total += S.size() - 1;
        nodes.reserve(total);
    }
    for (size_t k = 0; k < tips.size(); k++) {
        const std::vector<RefNode> &S = sub[k];
        const int32_t rootGlobal = tips[k];
        const int32_t base = (int32_t)nodes.size() - 1; // local index j >= 1 -> base + j
        auto remap = [&](int32_t j) { return j < 0 ? -1 : (j == 0 ? rootGlobal : base + j); };
        const int32_t keepParent = nodes[rootGlobal].parent;
        nodes[rootGlobal] = RefNode{remap(S[0].left), remap(S[0].right), S[0].start, S[0].count, keepParent};
        for (size_t j = 1; j < S.size(); j++)
            nodes.push_back(RefNode{remap(S[j].left), remap(S[j].right), S[j].start, S[j].count, remap(S[j].parent)});
    }
    // triOrder and the visiting rank.  The walk pops the right child first, so leaves are visited in DESCENDING order of
    // their range start and a leaf's own triangles in ascending position (:1055, :938, :1240): a triangle at position p
    // of the leaf [start, start + count) is visited after the n - (start + count) triangles of the leaves to its right.
    for (int p = 0; p < n; p++) out.order[p] = it[p].tri;
    int32_t leaves = 0;
    for (const RefNode &nd : nodes) {
        if (nd.left >= 0) continue;
        leaves++;
        for (int32_t p = nd.start; p < nd.start + nd.count; p++) out.rank[out.order[p]] = n - (nd.start + nd.count) + (p - nd.start);
    }
    out.nLeaves = leaves;
}

} // namespace cq
