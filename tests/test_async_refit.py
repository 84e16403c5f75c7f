"""cq_world_update_transforms_async: the stream-ordered transform update.  It must leave exactly what the synchronous
call leaves (both run one refit implementation: k_update_parts + a fixed number of launches per set), order itself
against launches on every stream of the world, copy the caller's arrays before returning, and never block the host on
the device.  Each GPU test compares against the synchronous path and the CPU oracle, byte for byte."""
import ctypes as C

import numpy as np
import pytest

CQ_ERR_INVALID = -1
MAX_HITS = 8


def test_null_world_is_invalid(cq):
    """Argument checks happen before any CUDA call, so they answer without a GPU."""
    L = cq.lib()
    ids = np.zeros(1, np.uint32)
    models = np.zeros(16, np.float32)
    assert L.cq_world_update_transforms_async(None, cq._ptr(ids), cq._ptr(models), 1, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_async(None, None, None, 0, None) == CQ_ERR_INVALID


# ---------------------------------------------------------------- GPU helpers
def _caller_order(hits, counts):
    """capsuleOverlapAll as its reference callers use it (stable sort by depth, Systems.swift:759)."""
    depth = np.where(np.arange(hits.shape[1])[None, :] < counts[:, None], hits["depth"], -np.inf)
    return np.take_along_axis(hits, np.argsort(-depth, axis=1, kind="stable"), axis=1)


def _dev(torch, arr):
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1).copy()).cuda()


def _host(t, dtype, shape=None):
    a = t.cpu().numpy().view(dtype)
    return a.reshape(shape) if shape is not None else a


class DeviceQueries:
    """Every query kind of the world, on device buffers, queued on one stream without synchronising."""

    def __init__(self, torch, cq, casts, rays, caps):
        self.torch, self.cq = torch, cq
        self.n = {"cast": len(casts), "ray": len(rays), "cap": len(caps)}
        self.d = {"cast": _dev(torch, casts), "ray": _dev(torch, rays), "cap": _dev(torch, caps)}

    def queue(self, g, stream):
        torch, cq, L = self.torch, self.cq, self.cq.lib()
        out = {}
        for mode in (0, 1, 2):
            o = torch.empty(self.n["cast"] * cq.CAST_HIT.itemsize, dtype=torch.uint8, device="cuda")
            g.capsule_cast_device(self.d["cast"].data_ptr(), self.n["cast"], mode, o.data_ptr(), stream)
            out[f"cast{mode}"] = o
        o = torch.empty(self.n["ray"] * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
        g.raycast_device(self.d["ray"].data_ptr(), self.n["ray"], o.data_ptr(), stream)
        out["ray"] = o
        nc = self.n["cap"]
        o = torch.empty(nc * cq.OVERLAP_HIT.itemsize, dtype=torch.uint8, device="cuda")
        cq._check(L.cq_capsule_overlap_device(g.handle, C.c_void_p(self.d["cap"].data_ptr()), nc, C.c_void_p(o.data_ptr()),
                                              C.c_void_p(stream)))
        out["overlap"] = o
        hits = torch.empty(nc * MAX_HITS * cq.OVERLAP_HIT.itemsize, dtype=torch.uint8, device="cuda")
        counts = torch.empty(nc * 4, dtype=torch.uint8, device="cuda")
        ovf = torch.empty(nc, dtype=torch.uint8, device="cuda")
        cq._check(L.cq_capsule_overlap_all_device(g.handle, C.c_void_p(self.d["cap"].data_ptr()), nc, MAX_HITS,
                                                  C.c_void_p(hits.data_ptr()), C.c_void_p(counts.data_ptr()),
                                                  C.c_void_p(ovf.data_ptr()), C.c_void_p(stream)))
        out["all"], out["counts"], out["ovf"] = hits, counts, ovf
        return out

    def fetch(self, out):
        cq = self.cq
        r = {k: _host(out[f"cast{k}"], cq.CAST_HIT) for k in (0, 1, 2)}
        r["ray"] = _host(out["ray"], cq.RAY_HIT)
        r["overlap"] = _host(out["overlap"], cq.OVERLAP_HIT)
        r["all"] = _host(out["all"], cq.OVERLAP_HIT, (-1, MAX_HITS))
        r["counts"] = _host(out["counts"], np.int32)
        r["ovf"] = _host(out["ovf"], np.uint8)
        return r


def _host_answers(g, casts, rays, caps):
    r = {k: g._cast(casts, k) for k in (0, 1, 2)}
    r["ray"] = g.raycast(rays)
    r["overlap"] = g.capsuleOverlap(caps)
    r["all"], r["counts"], r["ovf"] = g.capsuleOverlapAll(caps, MAX_HITS)
    return r


def _oracle_answers(o, order, casts, rays, caps):
    r = {k: o.capsule_cast(casts, k, order) for k in (0, 1, 2)}
    r["ray"] = o.raycast(rays, order)
    r["overlap"] = o.capsule_overlap(caps, order)
    r["all"], r["counts"], r["ovf"] = o.capsule_overlap_all(caps, MAX_HITS, order)
    return r


def _assert_same(a, b, step, what):
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), (what, step, k)


def _assert_oracle(a, ref, reference_order, step):
    for k in (0, 1, 2, "ray", "overlap", "counts"):
        assert a[k].tobytes() == ref[k].tobytes(), ("oracle", step, k)
    got = _caller_order(a["all"], a["counts"]) if reference_order else a["all"]
    assert got.tobytes() == ref["all"].tobytes(), ("oracle", step, "all")


def _terrain_boxes_scene(scenes, n_static_boxes, n_dynamic_boxes, seed, cells=120, box=3.0, spread=40.0):
    tv, ti, _ = scenes.terrain_mesh(cells=cells, cell=1.0)
    bv, bi = scenes.box_mesh(box)
    rng = np.random.default_rng(seed)
    parts = [scenes.part(tv, ti, entity_id=0)]
    spots = rng.uniform(-spread, spread, (n_static_boxes + n_dynamic_boxes, 2))
    for k, (x, z) in enumerate(spots):
        y = float(scenes.terrain_height(np.float32([x]), np.float32([z]))[0]) + 1.0
        parts.append(scenes.part(bv, bi, scenes.trs_model((x, y, z)), is_dynamic=k >= n_static_boxes, layer=2,
                                 entity_id=1 + k))
    return parts, spots


def _box_pose(scenes, rng, spots, eid, step):
    x, z = spots[eid - 1] + rng.uniform(-3, 3, 2)
    y = float(scenes.terrain_height(np.float32([x]), np.float32([z]))[0]) + 1.0 + 0.3 * step
    return scenes.trs_model((x, y, z), scenes.quat_angle_axis(0.4 * step, (0, 1, 0)))


def _order(cq, order):
    return cq.ORDER_REFERENCE if order == "reference" else cq.ORDER_CANONICAL


# ---------------------------------------------------------------- equal to the synchronous path
@pytest.mark.gpu
@pytest.mark.parametrize("path", ["dirty", "full"])
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_async_update_equals_synchronous_update(cq, orc, scenes, order, path):
    """World A refits with the synchronous call, world B with update_transforms_async on a torch stream; every step of B
    queues its device queries and one move-and-slide step on the same stream and nothing synchronises until the end.  Six
    steps alternate the static and the dynamic set.  Dirty: one box of the set moves (the dirty-subtree refit).  Full: the
    terrain or every dynamic box moves (the full fit).  Every answer, the characters and the final soup equal A's and the
    oracle's byte for byte."""
    torch = pytest.importorskip("torch")
    n_static, n_dynamic = 6, 8
    parts, spots = _terrain_boxes_scene(scenes, n_static, n_dynamic, seed=5)
    ga = cq.CollisionQuery(parts, order=_order(cq, order))
    gb = cq.CollisionQuery(parts, order=_order(cq, order))
    o = orc.OracleWorld(parts)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    casts = scenes.gen_casts(3000, lo, hi, seed=61, radius=0.6, half_height=0.7, expand=0.0)
    rays = scenes.gen_rays(6000, lo, hi, seed=62, expand=0.0)
    caps = scenes.gen_capsules(2000, lo, hi, seed=63, expand=0.0)
    rng = np.random.default_rng(7)
    xz = rng.uniform(-30, 30, (512, 2)).astype(np.float32)
    y = scenes.terrain_height(xz[:, 0], xz[:, 1]) + 4.0
    pos = np.stack([xz[:, 0], y, xz[:, 1]], 1).astype(np.float32)
    vel = rng.uniform(-6, 6, (512, 3)).astype(np.float32)
    params = cq.default_params()
    sa, so = cq.init_states(pos, vel), orc.init_states(pos, vel)
    dq = DeviceQueries(torch, cq, casts, rays, caps)
    d_states = _dev(torch, cq.init_states(pos, vel))
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    per_step, moves = [], []
    for step in range(1, 7):
        static = step % 2 == 1
        if path == "dirty":
            ids = [1 + rng.integers(0, n_static)] if static else [1 + n_static + rng.integers(0, n_dynamic)]
        else:
            ids = [0] if static else list(range(1 + n_static, 1 + n_static + n_dynamic))
        models = [scenes.trs_model((0.0, 0.1 * step, 0.05 * step)) if eid == 0 else _box_pose(scenes, rng, spots, eid, step)
                  for eid in ids]
        moves.append((ids, models))
        gb.update_transforms_async(ids, models, stream=stream.cuda_stream)
        out = dq.queue(gb, stream.cuda_stream)
        gb.move_and_slide_device(d_states.data_ptr(), len(pos), params, flags=cq.MAS_APPLY_GRAVITY, stream=stream.cuda_stream)
        with torch.cuda.stream(stream):
            out["states"] = d_states.clone()
        per_step.append(out)
    stream.synchronize()
    for step, ((ids, models), out) in enumerate(zip(moves, per_step), 1):
        ga.update_transforms(ids, models)
        o.update_transforms(ids, models)
        want = _host_answers(ga, casts, rays, caps)
        got = dq.fetch(out)
        _assert_same(got, want, step, "sync")
        _assert_oracle(got, _oracle_answers(o, ga.order, casts, rays, caps), ga.order == cq.ORDER_REFERENCE, step)
        ga.move_and_slide(sa, params)
        o.move_and_slide(so, orc.default_params(), order=ga.order)
        got_states = _host(out["states"], cq.STATE)
        assert got_states.tobytes() == sa.tobytes() == so.tobytes(), step
    for which in (0, 1):
        a, b, r = ga.read_soup(which), gb.read_soup(which), o.read_soup(which)
        for k in ("positions", "aabbs"):
            assert np.array_equal(b[k], a[k]) and np.array_equal(b[k], r[k]), (which, k)
    assert (dq.fetch(per_step[-1])["ray"]["triangle_index"] >= ga.info()["n_static_triangles"]).any()
    assert gb.info()["refit_ms"] == 0.0  # refit_ms reports synchronous updates only
    ga.close(), gb.close(), o.close()


# ---------------------------------------------------------------- launches do not grow with parts
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_launches_do_not_grow_with_moved_parts(cq, orc, scenes, order):
    """2,048 dynamic 12-triangle boxes over a terrain.  Moving 1, 64 or 1,024 of them costs a fixed handful of kernel
    launches per update (both calls), not a few per box; the answers equal the oracle's."""
    n_boxes = 2048
    parts, spots = _terrain_boxes_scene(scenes, 0, n_boxes, seed=9, box=1.0, spread=55.0)
    g = cq.CollisionQuery(parts, order=_order(cq, order))
    o = orc.OracleWorld(parts)
    rng = np.random.default_rng(11)
    lo, hi = np.float32([-60, -10, -60]), np.float32([60, 20, 60])
    casts = scenes.gen_casts(2000, lo, hi, seed=71, radius=0.5, half_height=0.5, expand=0.0)
    step = 0
    deltas = {}
    for call in ("sync", "async"):
        for n_moved in (1, 64, 1024):
            step += 1
            ids = (1 + rng.choice(n_boxes, n_moved, replace=False)).tolist()
            models = [_box_pose(scenes, rng, spots, eid, step) for eid in ids]
            g.stats(reset=True)
            if call == "sync":
                g.update_transforms(ids, models)
            else:
                g.update_transforms_async(ids, models)
            launches = g.stats()["kernel_launches"]
            deltas[(call, n_moved)] = launches
            o.update_transforms(ids, models)
            assert 1 <= launches <= 12, (call, n_moved, launches)
            # rays from above at every moved box's centre, and blocking casts
            centres = np.stack([np.asarray(m, np.float32).reshape(16)[12:15] for m in models])
            rays = np.zeros(len(ids), cq.RAY)
            rays["origin"] = centres + np.float32([0.01, 30.0, 0.02])
            rays["direction"] = (0, -1, 0)
            rays["max_distance"], rays["mask"] = 100.0, cq.LAYER_ALL
            got = g.raycast(rays)
            assert got.tobytes() == o.raycast(rays, g.order).tobytes(), (call, n_moved)
            assert (got["triangle_index"] >= g.info()["n_static_triangles"]).all()
            assert g.capsuleCastBlocking(casts).tobytes() == o.capsule_cast(casts, 1, g.order).tobytes(), (call, n_moved)
    for n_moved in (1, 64, 1024):
        assert deltas[("sync", n_moved)] == deltas[("async", n_moved)]
    assert deltas[("sync", 1)] == deltas[("sync", 64)]  # both take the dirty-subtree path
    g.close(), o.close()


# ---------------------------------------------------------------- many small dirty refits that share ancestors
def _packed_run(cq, orc, scenes, order, seed, n_updates=100):
    bv, bi = scenes.box_mesh(0.5)
    pv, pidx = scenes.plane_mesh(20.0)
    parts = [scenes.part(pv, pidx, entity_id=0)]
    grid = np.array([(x, y, z) for x in range(4) for y in range(4) for z in range(4)], np.float32) * 0.6
    for k, c in enumerate(grid):
        parts.append(scenes.part(bv, bi, scenes.trs_model(c + np.float32([0, 1, 0])), is_dynamic=True, entity_id=1 + k))
    g = cq.CollisionQuery(parts, order=_order(cq, order))
    o = orc.OracleWorld(parts)
    rng = np.random.default_rng(seed)
    corners = np.array([(x, y, z) for x in (-0.25, 0.25) for y in (-0.25, 0.25) for z in (-0.25, 0.25)], np.float32)
    casts = scenes.gen_casts(256, np.float32([-1, 0, -1]), np.float32([3, 4, 3]), seed=seed + 1, radius=0.2, half_height=0.2,
                             expand=0.0)
    out = []
    for step in range(n_updates):
        k = int(rng.integers(1, 16))  # < a quarter of the 768 triangles: the dirty-subtree path every time
        ids = (1 + rng.choice(64, k, replace=False)).tolist()
        centres = grid[np.asarray(ids) - 1] + np.float32([0, 1, 0]) + rng.uniform(-0.2, 0.2, (k, 3)).astype(np.float32)
        models = [scenes.trs_model(c, scenes.quat_angle_axis(float(rng.uniform(0, 6.28)), (0, 1, 0))) for c in centres]
        g.update_transforms_async(ids, models)
        o.update_transforms(ids, models)
        # rays aimed at the moved boxes' corners from outside the pack
        targets = (centres[:, None, :] + corners[None] * 0.9).reshape(-1, 3)
        origins = targets + rng.uniform(-1, 1, targets.shape).astype(np.float32) * 6.0
        d = targets - origins
        rays = np.zeros(len(targets), cq.RAY)
        rays["origin"], rays["direction"] = origins, d / np.linalg.norm(d, axis=1, keepdims=True)
        rays["max_distance"], rays["mask"] = 20.0, cq.LAYER_ALL
        got_r, got_c = g.raycast(rays), g.capsuleCastBlocking(casts)
        assert got_r.tobytes() == o.raycast(rays, g.order).tobytes(), step
        assert got_c.tobytes() == o.capsule_cast(casts, 1, g.order).tobytes(), step
        out += [got_r.tobytes(), got_c.tobytes()]
    out.append(g.read_soup(1)["aabbs"].tobytes())
    g.close(), o.close()
    return b"".join(out)


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_many_small_dirty_refits_sharing_ancestors(cq, orc, scenes, order):
    """64 small boxes packed so that their leaves share ancestors; 100 random dirty updates of 1..15 of them.  Rays aimed at
    the moved boxes' corners and blocking casts equal the oracle after every update (a climb that merged an ancestor
    before its dirty sibling was final would shrink a box and lose hits), and a second pass with the same seed gives the
    same bytes."""
    first = _packed_run(cq, orc, scenes, order, seed=123)
    assert _packed_run(cq, orc, scenes, order, seed=123) == first


# ---------------------------------------------------------------- the host is not blocked, and the inputs are copied
@pytest.mark.gpu
def test_async_update_does_not_block_and_copies_inputs(cq, orc, scenes):
    torch = pytest.importorskip("torch")
    parts, spots = _terrain_boxes_scene(scenes, 2, 8, seed=21)
    g = cq.CollisionQuery(parts)
    o = orc.OracleWorld(parts)
    rng = np.random.default_rng(3)
    ids = np.arange(3, 11, dtype=np.uint32)
    models = np.stack([_box_pose(scenes, rng, spots, int(e), 1) for e in ids]).astype(np.float32)
    s = torch.cuda.Stream()
    g.update_transforms_async(ids, models, stream=s.cuda_stream)  # same table size: no allocation in the timed call
    s.synchronize()
    o.update_transforms(ids, models)
    models[:] = np.stack([_box_pose(scenes, rng, spots, int(e), 2) for e in ids])
    intended = models.copy()
    with torch.cuda.stream(s):
        torch.cuda._sleep(400_000_000)
    g.update_transforms_async(ids, models, stream=s.cuda_stream)
    assert not s.query()  # the call returned while the stream was still busy
    ids[:] = 0xFFFFFFF0
    models[:] = np.nan
    o.update_transforms(np.arange(3, 11, dtype=np.uint32), intended)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    rays = scenes.gen_rays(4000, lo, hi, seed=5, expand=0.0)
    d_rays = _dev(torch, rays)
    d_out = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    g.raycast_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), s.cuda_stream)
    s.synchronize()
    assert _host(d_out, cq.RAY_HIT).tobytes() == o.raycast(rays, g.order).tobytes()
    g.close(), o.close()


# ---------------------------------------------------------------- ordering across streams
@pytest.mark.gpu
def test_async_update_is_ordered_across_streams(cq, orc, scenes):
    """Rays queued on stream A behind a sleep read the pose before the update queued next on stream B; rays queued after
    it on stream C read the new pose; a second update on A is what read_soup finally sees."""
    torch = pytest.importorskip("torch")
    parts, spots = _terrain_boxes_scene(scenes, 2, 8, seed=31)
    g = cq.CollisionQuery(parts)
    ref = cq.CollisionQuery(parts)
    rng = np.random.default_rng(4)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    rays = scenes.gen_rays(1 << 20, lo, hi, seed=6, expand=0.0)
    ids = list(range(3, 11))
    m1 = [_box_pose(scenes, rng, spots, e, 1) for e in ids]
    m2 = [_box_pose(scenes, rng, spots, e, 2) for e in ids]
    before = ref.raycast(rays)
    ref.update_transforms(ids, m1)
    after1 = ref.raycast(rays)
    ref.update_transforms(ids, m2)
    soup2 = ref.read_soup(1)
    assert before.tobytes() != after1.tobytes()
    d_rays = _dev(torch, rays)
    out_a = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    out_c = torch.empty_like(out_a)
    torch.cuda.synchronize()
    sa, sb, sc = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sa):
        torch.cuda._sleep(200_000_000)
    g.raycast_device(d_rays.data_ptr(), len(rays), out_a.data_ptr(), sa.cuda_stream)
    g.update_transforms_async(ids, m1, stream=sb.cuda_stream)
    g.raycast_device(d_rays.data_ptr(), len(rays), out_c.data_ptr(), sc.cuda_stream)
    g.update_transforms_async(ids, m2, stream=sa.cuda_stream)
    soup = g.read_soup(1)
    torch.cuda.synchronize()
    assert _host(out_a, cq.RAY_HIT).tobytes() == before.tobytes()
    assert _host(out_c, cq.RAY_HIT).tobytes() == after1.tobytes()
    for k in ("positions", "aabbs"):
        assert np.array_equal(soup[k], soup2[k]), k
    g.close(), ref.close()


# ---------------------------------------------------------------- errors change nothing
@pytest.mark.gpu
def test_async_update_errors_change_nothing(cq, orc, scenes):
    parts, spots = _terrain_boxes_scene(scenes, 2, 4, seed=41)
    g = cq.CollisionQuery(parts)
    o = orc.OracleWorld(parts)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    rays = scenes.gen_rays(4000, lo, hi, seed=8, expand=0.0)
    soup = g.read_soup(1)
    model = scenes.trs_model((1.0, 2.0, 3.0))
    with pytest.raises(cq.CQError, match="unknown entity id 99"):
        g.update_transforms_async([3, 99], [model, model])  # 3 is known: nothing of it may be applied either
    g.stats(reset=True)
    g.update_transforms_async(np.zeros(0, np.uint32), np.zeros((0, 16), np.float32))
    assert g.stats()["kernel_launches"] == 0
    after = g.read_soup(1)
    for k in ("positions", "aabbs"):
        assert np.array_equal(after[k], soup[k]), k
    assert g.raycast(rays).tobytes() == o.raycast(rays, g.order).tobytes()
    L = cq.lib()
    ids = np.zeros(1, np.uint32)
    assert L.cq_world_update_transforms_async(g.handle, cq._ptr(ids), None, 1, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_async(g.handle, cq._ptr(ids), cq._ptr(np.zeros(16, np.float32)), -1, None) == CQ_ERR_INVALID
    g.close(), o.close()
