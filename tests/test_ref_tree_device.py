"""The reference's tree cut on the device (csrc/cq_build.cu: attach_ref_order) against the host restatement of the
reference's build (csrc/cq_reftree.h, compiled into tests/hostmath/reftree.cpp).

CPU: the scan formulation the device uses for the swap-with-tail partition (destinations from prefix counts over a
forward and a backward stream) and for the median fallback (a stable sort on an unsigned key that merges -0 and +0)
builds the same tree as the host builder, on adversarial inputs.
GPU: cq_world_read_ref_order of real and adversarial worlds equals the host builder run on the same device-computed
triangle boxes (read back with cq_world_read_soup): same triOrder, same visiting rank, same node count, and the same
refusal of a tree too deep for the ray walk's stack."""
import importlib.util
import os

import numpy as np
import pytest

_spec = importlib.util.spec_from_file_location("_reftree_helpers", os.path.join(os.path.dirname(__file__), "test_reftree.py"))
R = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(R)
rt = R.rt  # the host builder's harness (fixture)

CQ_ERR_INVALID = -1
CQ_STACK = 64
f32 = np.float32


# ---------------------------------------------------------------- the scan formulation, in numpy

def partition_dest(keys, pivot):
    """Destination (range-local) of every element of a range under the reference's swap-with-tail loop, from prefix
    counts only; and the number of elements < pivot.  Same arithmetic as k_lv_less / k_lv_scatter."""
    n = len(keys)
    lt = (keys < pivot).astype(np.int64)
    less = np.cumsum(lt) - lt
    tot_l = int(lt.sum())
    i = np.arange(n)
    ge_f = i - less
    len_f = np.full(n + 1, n, np.int64)  # len_f[m]: elements of the first m forward runs (run m ends at the m-th >=)
    len_b = np.full(n + 1, n, np.int64)  # len_b[m]: elements of the first m backward runs (run m ends at the m-th <)
    len_f[0] = len_b[0] = 0
    g = np.nonzero(lt == 0)[0]
    len_f[ge_f[g] + 1] = g + 1
    l_ = np.nonzero(lt == 1)[0]
    len_b[tot_l - less[l_]] = n - l_
    lb = len_b[ge_f]
    fwd = i + lb < n
    less_b = tot_l - less - lt
    lf = len_f[np.minimum(less_b + 1, n)]
    dest = np.where(fwd, np.where(lt == 1, i, n - 1 - lb), np.where(lt == 1, less_b + lf - (less_b + 1), i - 1))
    return dest, tot_l


def sort_key(v):
    """The fallback's key: the float's order as an unsigned integer, -0 and +0 one key (rt_sort_key)."""
    u = np.where(v == 0, f32(0), v).astype(f32).view(np.uint32)
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def literal_partition(keys, pivot):
    a, i, j = list(range(len(keys))), 0, len(keys) - 1
    while i <= j:
        if keys[a[i]] < pivot:
            i += 1
        else:
            a[i], a[j] = a[j], a[i]
            j -= 1
    return a, i


def numpy_build(lo, hi):
    """The whole tree with the scan formulation, level by level: (order, rank, node count, depth)."""
    n = len(lo)
    c = ((lo + hi) * f32(0.5)).astype(f32)
    order = np.arange(n)
    open_, leaves, n_nodes, depth = [(0, n, 0)] if n else [], [], 1 if n else 0, 0
    while open_:
        nxt = []
        for s, cnt, d in open_:
            if cnt <= 4:
                leaves.append((s, cnt))
                depth = max(depth, d)
                continue
            cc = c[order[s:s + cnt]]
            lo_b, hi_b = cc[0].copy(), cc[0].copy()
            for v in cc[1:]:  # the host's sequential bounds (finite inputs here)
                lo_b, hi_b = np.where(v < lo_b, v, lo_b), np.where(v > hi_b, v, hi_b)
            ex = hi_b - lo_b
            axis = 0 if ex[0] >= ex[1] and ex[0] >= ex[2] else (1 if ex[1] >= ex[2] else 2)
            pivot = f32((lo_b[axis] + hi_b[axis]) * f32(0.5))
            dest, tot_l = partition_dest(cc[:, axis], pivot)
            seg = np.empty(cnt, np.int64)
            seg[dest] = order[s:s + cnt]
            if tot_l in (0, cnt):
                seg = seg[np.argsort(sort_key(c[seg, axis]), kind="stable")]
                tot_l = cnt // 2
            order[s:s + cnt] = seg
            nxt += [(s, tot_l, d + 1), (s + tot_l, cnt - tot_l, d + 1)]
            n_nodes += 2
        open_ = nxt
    rank = np.zeros(n, np.int64)
    for s, cnt in leaves:
        rank[order[s:s + cnt]] = n - (s + cnt) + np.arange(cnt)
    return order, rank, n_nodes, depth


def host_depth(nodes):
    best = 0
    for k, (l, r, s, cnt, p) in enumerate(nodes):
        if l >= 0:
            continue
        dd, q = 0, p
        while q >= 0:
            dd, q = dd + 1, nodes[q][4]
        best = max(best, dd)
    return best


def adversarial(kind, n, rng):
    """Triangle boxes (lo, hi) whose centroids stress the split rule."""
    if kind == "random":
        c = rng.uniform(-10, 10, (n, 3)).astype(f32)
    elif kind == "dupes":  # duplicate centroids
        c = rng.uniform(-10, 10, (max(n // 8, 1), 3)).astype(f32)[rng.integers(0, max(n // 8, 1), n)]
    elif kind == "ties":  # centroids on the pivot and on a few values
        c = rng.integers(0, 4, (n, 3)).astype(f32)
    elif kind == "same":  # everything on one side at every level
        c = np.tile(np.array([[1.5, -2.0, 3.0]], f32), (n, 1))
    elif kind == "signed_zero":  # -0 and +0 on the longest axis, nothing else differs: the fallback must keep their order
        c = np.zeros((n, 3), f32)
        c[:, 0] = np.where(rng.integers(0, 2, n) == 1, f32(-0.0), f32(0.0))
    elif kind == "two_values":  # adjacent floats whose midpoint rounds to the lower one: all >= pivot, sort by value
        a = f32(1.0)
        c = np.zeros((n, 3), f32)
        c[:, 0] = np.where(rng.integers(0, 2, n) == 1, np.nextafter(a, f32(2)), a)
    elif kind == "peel":  # exponentially spaced: one triangle peeled per level
        c = np.zeros((n, 3), f32)
        c[:, 0] = (f32(2.0) ** np.arange(n)).astype(f32)[rng.permutation(n)]
    else:
        raise ValueError(kind)
    return np.ascontiguousarray(c), np.ascontiguousarray(c)


def test_partition_scan_equals_literal_loop():
    rng = np.random.default_rng(5)
    for _ in range(3000):
        n = int(rng.integers(1, 60))
        keys = rng.integers(0, 10, n).astype(f32)
        pivot = f32(rng.choice([-1, 0, 3, 4.5, 5, 9, 10]))
        perm, mid = literal_partition(keys, pivot)
        dest, tot_l = partition_dest(keys, pivot)
        out = np.empty(n, np.int64)
        out[dest] = np.arange(n)
        assert out.tolist() == perm and tot_l == mid


def test_sort_key_orders_like_less_than():
    v = np.array([-np.inf, -3e38, -1.0, -1e-45, -0.0, 0.0, 1e-45, 1.0, 3e38, np.inf], f32)
    k = sort_key(v)
    assert k[4] == k[5]  # -0 and +0 are one key, as `<` sees them
    assert all(k[i] < k[i + 1] for i in range(len(v) - 1) if i != 4)


@pytest.mark.parametrize("kind,n", [(k, n) for k in ("random", "dupes", "ties", "same", "signed_zero", "two_values")
                                     for n in (1, 2, 3, 4, 5, 6, 7, 8, 9, 33, 200)] + [("peel", 20), ("peel", 40)])
def test_numpy_scan_build_equals_host_builder(rt, kind, n):
    rng = np.random.default_rng(n * 31 + len(kind))
    lo, hi = adversarial(kind, n, rng)
    order, rank, counts, nodes = R.build(rt, lo, hi, 1, want_nodes=True)
    o, r, n_nodes, depth = numpy_build(lo, hi)
    assert o.tolist() == order.tolist()
    assert r.tolist() == rank.tolist()
    assert n_nodes == counts[0] and depth == host_depth(nodes)


def test_read_ref_order_argument_checks(cq):
    L = cq.lib()
    assert L.cq_world_read_ref_order(None, 0, None, None) == CQ_ERR_INVALID


# ---------------------------------------------------------------- the device build against the host builder

def tri_world(cq, centroids_x, base=None):
    """One static part with one triangle per entry, in the plane x = const (so its box's centroid x is exactly that
    constant under the identity model); y and z are the same for every triangle unless `base` moves them."""
    n = len(centroids_x)
    pos = np.zeros((3 * n, 3), f32)
    pos[:, 0] = np.repeat(np.asarray(centroids_x, f32), 3)
    off = np.zeros((n, 3), f32) if base is None else np.asarray(base, f32)
    pos[0::3, 1:] = off[:, 1:]
    pos[1::3, 1:] = off[:, 1:] + np.array([1, 0], f32)
    pos[2::3, 1:] = off[:, 1:] + np.array([0, 1], f32)
    return [cq.scenes.part(pos, np.arange(3 * n, dtype=np.uint32), entity_id=0)]


def device_equals_host(cq, rt, parts):
    g = cq.CollisionQuery(parts)
    try:
        info = g.info()
        total_nodes = 0
        for which in (0, 1):
            nt = info["n_dynamic_triangles"] if which else info["n_static_triangles"]
            if nt == 0:
                continue
            a = g.read_soup(which)["aabbs"]
            lo, hi = np.ascontiguousarray(a[:, :3]), np.ascontiguousarray(a[:, 3:])
            order, rank, counts, _ = R.build(rt, lo, hi, 0)
            d_order, d_rank = g.read_ref_order(which)
            assert np.array_equal(d_order, order), f"set {which}: triOrder differs"
            assert np.array_equal(d_rank, rank), f"set {which}: visiting rank differs"
            total_nodes += int(counts[0])
        assert info["n_ref_nodes"] == total_nodes
        return g.read_ref_order(0)
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["mirror_hulls", "mirror_render", "semla", "cheese", "merged_c5", "terrain_1m"])
def test_device_tree_equals_host_tree_scenes(cq, rt, scene):
    S = cq.scenes
    parts = {"mirror_hulls": lambda: S.mirror_scene(use_hulls=True),
             "mirror_render": lambda: S.mirror_scene(use_hulls=False, mirror_dynamic=True),
             "semla": lambda: S.semla_scene(),
             "cheese": lambda: [S.part(S.load_asset_fixture("cheese")["positions"], S.load_asset_fixture("cheese")["indices"],
                                       S.cheese_model(S.load_asset_fixture("cheese")["transform"]), entity_id=0)],
             "merged_c5": lambda: S.merged_scene(),
             "terrain_1m": lambda: S.terrain_scene(cells=708, cell=2.0)[0]}[scene]()
    device_equals_host(cq, rt, parts)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("random", n) for n in range(1, 10)] + [("random", 5000), ("dupes", 3000),
                                                                         ("ties", 3000), ("same", 500),
                                                                         ("two_values", 40), ("two_values", 3000),
                                                                         ("peel", 50)])
def test_device_tree_equals_host_tree_adversarial(cq, rt, kind, n):
    rng = np.random.default_rng(n * 17 + len(kind))
    if kind in ("two_values", "peel", "same"):
        c, _ = adversarial(kind, n, rng)
        parts = tri_world(cq, c[:, 0])
    else:  # centroids spread in 3-D: each triangle translated by its centroid
        c, _ = adversarial(kind, n, rng)
        parts = tri_world(cq, c[:, 0], base=c)
    device_equals_host(cq, rt, parts)


@pytest.mark.gpu
def test_nan_centroid_tree_follows_the_documented_rule(cq):
    """A NaN vertex is NaN in all three world coordinates, and such a triangle passes the degenerate filter.  When it comes
    first in a range the range's bounds and pivot are NaN and the median fallback sorts a NaN key, which std::stable_sort
    leaves unordered; the device sorts NaN above +inf.  Its tree equals the numpy model of that rule on the world's own
    boxes, and two worlds agree."""
    rng = np.random.default_rng(3)
    c = rng.uniform(-10, 10, (2000, 3)).astype(f32)
    xs = c[:, 0].copy()
    xs[[0, 777]] = np.nan
    parts = tri_world(cq, xs, base=c)
    runs = []
    for _ in range(2):
        g = cq.CollisionQuery(parts)
        try:
            a = g.read_soup(0)["aabbs"]
            runs.append(g.read_ref_order(0))
        finally:
            g.close()
    assert np.isnan(a[[0, 777]]).all(axis=1).all() and not np.isnan(np.delete(a, [0, 777], axis=0)).any()
    order, rank, _, _ = numpy_build(np.ascontiguousarray(a[:, :3]), np.ascontiguousarray(a[:, 3:]))
    for o, r in runs:
        assert np.array_equal(o, order) and np.array_equal(r, rank)


@pytest.mark.gpu
def test_infinite_centroid_tree_equals_host_tree(cq, rt):
    """A vertex at x = +inf passes the degenerate filter (its cross product is not <= 1e-10) and becomes (inf, NaN, NaN) in
    world space (the model matrix multiplies it by zero too); its box's centroid is +inf in x.  Infinite centroids are
    ordinary values of the split rule (an extent inf - inf is NaN and loses every `>=` of the axis choice; the fallback's
    key orders +-inf like `<`), so the device tree equals the host builder's."""
    rng = np.random.default_rng(4)
    c = rng.uniform(-10, 10, (3000, 3)).astype(f32)
    parts = tri_world(cq, c[:, 0], base=c)
    pos = parts[0]["positions"].copy()
    pos[3 * 5, 0] = np.inf  # one vertex of triangle 5
    pos[3 * 900 + 1, 0] = -np.inf
    parts[0]["positions"] = pos
    device_equals_host(cq, rt, parts)
    g = cq.CollisionQuery(parts)
    try:  # either output may be NULL
        assert cq.lib().cq_world_read_ref_order(g.handle, 0, None, None) == 0
        assert cq.lib().cq_world_read_ref_order(g.handle, 2, None, None) == CQ_ERR_INVALID
    finally:
        g.close()


@pytest.mark.gpu
def test_too_deep_tree_is_refused_with_the_same_message(cq, rt):
    # x = 4^k: the pivot (lo + hi) / 2 lies above the second largest value, so every level peels one triangle; 134
    # values (denormals included) put the leaves far past the ray walk's stack
    xs = (np.float64(4.0) ** np.arange(-70, 64)).astype(f32)
    n = len(xs)
    xs = xs[np.random.default_rng(1).permutation(n)]
    lo = np.zeros((n, 3), f32)
    lo[:, 0] = xs
    _, _, _, nodes = R.build(rt, lo, lo.copy(), 1, want_nodes=True)
    depth = host_depth(nodes)
    assert depth + 2 > CQ_STACK
    with pytest.raises(cq.CQError, match=f"the reference tree of set 0 is {depth} levels deep \\(limit {CQ_STACK - 2}\\)"):
        cq.CollisionQuery(tri_world(cq, xs))


@pytest.mark.gpu
def test_read_ref_order_refused_in_canonical_order(cq):
    g = cq.CollisionQuery(cq.scenes.mirror_scene(use_hulls=True), order=cq.ORDER_CANONICAL)
    try:
        with pytest.raises(cq.CQError, match="canonical order"):
            g.read_ref_order(0)
    finally:
        g.close()
