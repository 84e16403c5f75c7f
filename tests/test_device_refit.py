"""cq_world_update_transforms_device: the transform update from device arrays, with the ids resolved and the table of
moved parts built on the GPU, and CUDA-graph capture of a fixed step's device calls.  The device call must leave exactly
what the synchronous call leaves (one refit implementation serves all three update calls), decide its errors on the
device without changing anything, cost a fixed number of launches, never block the host, and be recordable into a graph
whose replays equal uncaptured synchronous steps byte for byte."""
import ctypes as C
import importlib.util
import os
import time

import numpy as np
import pytest

# the async refit tests' scenes and query helpers (imported by path: tests/ is not a package)
_spec = importlib.util.spec_from_file_location("_async_refit_helpers", os.path.join(os.path.dirname(__file__), "test_async_refit.py"))
A = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(A)

CQ_ERR_INVALID = -1
MAX_LAUNCHES = 30


def test_device_update_argument_checks(cq):
    """NULL world, n < 0 and a NULL array with n > 0 are refused before any CUDA call, so they answer without a GPU."""
    L = cq.lib()
    p = C.c_void_p(16)  # never dereferenced: the checks come first
    assert L.cq_world_update_transforms_device(None, p, p, 1, None, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_device(None, p, p, -1, None, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_device(None, None, None, 1, None, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_device(None, None, None, 0, None, None) == CQ_ERR_INVALID
    assert "cq_world_update_transforms_device" in cq.EXPORTS


# ---------------------------------------------------------------- helpers
class DeviceUpdate:
    """Device copies of one update's ids and models (kept alive until the stream has passed the call)."""

    def __init__(self, torch, ids, models):
        self.ids = torch.from_numpy(np.asarray(ids, np.uint32).view(np.int32).copy()).cuda()
        self.models = torch.from_numpy(np.ascontiguousarray(models, np.float32).reshape(-1, 16).copy()).cuda()
        self.status = torch.full((1,), -7, dtype=torch.int32, device="cuda")
        self.n = len(ids)

    def queue(self, g, stream):
        g.update_transforms_device(self.ids.data_ptr(), self.models.data_ptr(), self.n, self.status.data_ptr(), stream)


def _soups(g):
    return [g.read_soup(w) for w in (0, 1)]


def _assert_soups_equal(a, b, what):
    for which in (0, 1):
        for k in ("positions", "aabbs"):
            assert np.array_equal(a[which][k], b[which][k]), (what, which, k)


# ---------------------------------------------------------------- equal to the synchronous path
@pytest.mark.gpu
@pytest.mark.parametrize("path", ["dirty", "full"])
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_device_update_equals_synchronous_update(cq, orc, scenes, order, path):
    """World A refits with the synchronous call, world B with the device call fed from torch tensors on a torch stream,
    followed on the same stream by every device query and one move-and-slide step; nothing synchronises until the end.
    Six steps alternate the static and the dynamic set.  Every answer, the characters and the final soup equal A's and
    the oracle's byte for byte."""
    torch = pytest.importorskip("torch")
    n_static, n_dynamic = 6, 8
    parts, spots = A._terrain_boxes_scene(scenes, n_static, n_dynamic, seed=5)
    ga = cq.CollisionQuery(parts, order=A._order(cq, order))
    gb = cq.CollisionQuery(parts, order=A._order(cq, order))
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
    dq = A.DeviceQueries(torch, cq, casts, rays, caps)
    d_states = A._dev(torch, cq.init_states(pos, vel))
    moves = []
    for step in range(1, 7):
        static = step % 2 == 1
        if path == "dirty":
            ids = [1 + rng.integers(0, n_static)] if static else [1 + n_static + rng.integers(0, n_dynamic)]
        else:
            ids = [0] if static else list(range(1 + n_static, 1 + n_static + n_dynamic))
        models = [scenes.trs_model((0.0, 0.1 * step, 0.05 * step)) if eid == 0 else A._box_pose(scenes, rng, spots, eid, step)
                  for eid in ids]
        moves.append((ids, models, DeviceUpdate(torch, ids, models)))
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    per_step = []
    for ids, models, du in moves:
        du.queue(gb, stream.cuda_stream)
        out = dq.queue(gb, stream.cuda_stream)
        gb.move_and_slide_device(d_states.data_ptr(), len(pos), params, flags=cq.MAS_APPLY_GRAVITY, stream=stream.cuda_stream)
        with torch.cuda.stream(stream):
            out["states"] = d_states.clone()
        per_step.append(out)
    stream.synchronize()
    for step, ((ids, models, du), out) in enumerate(zip(moves, per_step), 1):
        assert int(du.status.item()) == 0, step
        ga.update_transforms(ids, models)
        o.update_transforms(ids, models)
        want = A._host_answers(ga, casts, rays, caps)
        got = dq.fetch(out)
        A._assert_same(got, want, step, "sync")
        A._assert_oracle(got, A._oracle_answers(o, ga.order, casts, rays, caps), ga.order == cq.ORDER_REFERENCE, step)
        ga.move_and_slide(sa, params)
        o.move_and_slide(so, orc.default_params(), order=ga.order)
        assert A._host(out["states"], cq.STATE).tobytes() == sa.tobytes() == so.tobytes(), step
    a, b = _soups(ga), _soups(gb)
    _assert_soups_equal(a, b, "sync")
    _assert_soups_equal(a, [o.read_soup(w) for w in (0, 1)], "oracle")
    assert gb.info()["refit_ms"] == 0.0  # refit_ms reports synchronous updates only
    ga.close(), gb.close(), o.close()


# ---------------------------------------------------------------- semantics
@pytest.mark.gpu
def test_device_update_semantics(cq, orc, scenes):
    """A duplicated id takes its last model; an id shared by several parts moves all of them; a part without triangles
    is skipped; n == 0 queues no launch.  Each case equals the synchronous call, and the oracle where it has the same
    semantics: the oracle keeps one slice per entity id (the last part), so it is compared before the shared-id case
    only."""
    torch = pytest.importorskip("torch")
    parts, spots = A._terrain_boxes_scene(scenes, 1, 4, seed=13)
    bv, bi = scenes.box_mesh(2.0)
    for k, x in enumerate((-20.0, -14.0)):  # entity 50: two dynamic parts
        parts.append(scenes.part(bv, bi, scenes.trs_model((x, 12.0, 5.0)), is_dynamic=True, layer=2, entity_id=50))
    flat = np.zeros((3, 3), np.float32)  # entity 60: one degenerate triangle, filtered out: no triangles
    parts.append(scenes.part(flat, np.arange(3, dtype=np.uint32), is_dynamic=True, entity_id=60))
    ga, gb, o = cq.CollisionQuery(parts), cq.CollisionQuery(parts), orc.OracleWorld(parts)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 30, 55])
    rays = scenes.gen_rays(20000, lo, hi, seed=17, expand=0.0)
    casts = scenes.gen_casts(2000, lo, hi, seed=18, radius=0.6, half_height=0.7, expand=0.0)
    s = torch.cuda.Stream()
    rng = np.random.default_rng(19)
    m3a, m3b, m4 = A._box_pose(scenes, rng, spots, 3, 1), A._box_pose(scenes, rng, spots, 3, 2), A._box_pose(scenes, rng, spots, 4, 1)
    cases = [  # (device ids, models, the equivalent synchronous ids, models)
        ([3, 4, 3], [m3a, m4, m3b], [4, 3], [m4, m3b]),  # a duplicated id takes its last model
        ([50], [scenes.trs_model((-10.0, 9.0, -8.0))], None, None),  # an id shared by two parts moves both
        ([60, 2], [scenes.trs_model((1.0, 2.0, 3.0)), A._box_pose(scenes, rng, spots, 2, 2)], None, None),  # no triangles
    ]
    for k, (ids, models, sync_ids, sync_models) in enumerate(cases):
        du = DeviceUpdate(torch, ids, models)
        before = gb.read_soup(1)["positions"]
        torch.cuda.synchronize()
        du.queue(gb, s.cuda_stream)
        s.synchronize()
        assert int(du.status.item()) == 0
        ga.update_transforms(sync_ids or ids, sync_models or models)
        assert gb.raycast(rays).tobytes() == ga.raycast(rays).tobytes(), k
        assert gb.capsuleCastBlocking(casts).tobytes() == ga.capsuleCastBlocking(casts).tobytes(), k
        _assert_soups_equal(_soups(ga), _soups(gb), k)
        assert gb.read_models().tobytes() == ga.read_models().tobytes(), k
        if 50 in ids:  # both 8-vertex boxes of entity 50 (dynamic vertices 32..47) moved
            moved = np.any(gb.read_soup(1)["positions"] != before, axis=1)
            assert moved[32:48].all() and not moved[:32].any() and not moved[48:].any()
        if k == 0:  # before the shared-id case, after which the oracle's world differs from A's
            o.update_transforms(sync_ids, sync_models)
            assert ga.raycast(rays).tobytes() == o.raycast(rays, ga.order).tobytes()
    gb.stats(reset=True)
    du = DeviceUpdate(torch, [3], [m3a])
    gb.update_transforms_device(du.ids.data_ptr(), du.models.data_ptr(), 0, du.status.data_ptr(), s.cuda_stream)
    assert gb.stats()["kernel_launches"] == 0
    assert int(du.status.item()) == -7  # nothing was queued, not even the status write
    ga.close(), gb.close(), o.close()


# ---------------------------------------------------------------- unknown ids change nothing
@pytest.mark.gpu
def test_device_update_unknown_ids_change_nothing(cq, orc, scenes):
    torch = pytest.importorskip("torch")
    parts, spots = A._terrain_boxes_scene(scenes, 2, 4, seed=41)
    g, o = cq.CollisionQuery(parts), orc.OracleWorld(parts)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    rays = scenes.gen_rays(4000, lo, hi, seed=8, expand=0.0)
    casts = scenes.gen_casts(1000, lo, hi, seed=9, radius=0.6, half_height=0.7, expand=0.0)
    caps = scenes.gen_capsules(1000, lo, hi, seed=10, expand=0.0)
    before = (_soups(g), A._host_answers(g, casts, rays, caps), g.read_models())
    model = scenes.trs_model((1.0, 2.0, 3.0))
    bad = DeviceUpdate(torch, [3, 99], [model, model])  # 3 is known (and dynamic): nothing of it may be applied either
    torch.cuda.synchronize()
    bad.queue(g, None)
    torch.cuda.synchronize()
    g.update_transforms_device(bad.ids.data_ptr(), bad.models.data_ptr(), 2, None, None)  # no status pointer
    assert int(bad.status.item()) == 1
    _assert_soups_equal(before[0], _soups(g), "unknown id")
    A._assert_same(A._host_answers(g, casts, rays, caps), before[1], 0, "unknown id")
    assert g.read_models().tobytes() == before[2].tobytes()  # no model row was written
    good = DeviceUpdate(torch, [3, 5], [model, A._box_pose(scenes, np.random.default_rng(1), spots, 5, 1)])
    torch.cuda.synchronize()
    good.queue(g, None)
    o.update_transforms([3, 5], good.models.cpu().numpy())
    assert g.raycast(rays).tobytes() == o.raycast(rays, g.order).tobytes()
    assert int(good.status.item()) == 0
    rows = g.read_models()  # part k carries entity k in this scene
    assert rows[3].tobytes() == good.models[0].cpu().numpy().tobytes() and rows[5].tobytes() == good.models[1].cpu().numpy().tobytes()
    assert np.delete(rows, [3, 5], axis=0).tobytes() == np.delete(before[2], [3, 5], axis=0).tobytes()
    L = cq.lib()
    p = C.c_void_p(good.ids.data_ptr())
    assert L.cq_world_update_transforms_device(g.handle, p, None, 1, None, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_device(g.handle, None, p, 1, None, None) == CQ_ERR_INVALID
    assert L.cq_world_update_transforms_device(g.handle, p, p, -1, None, None) == CQ_ERR_INVALID
    g.close(), o.close()


# ---------------------------------------------------------------- a fixed number of launches
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_device_update_launch_count_is_fixed(cq, orc, scenes, order):
    """2,048 dynamic boxes over a terrain: moving 1, 64 or 1,024 of them costs the same number of launches (28 in
    reference order, 20 in canonical order: 2 + 13 or 9 per set), and the answers equal the oracle's."""
    torch = pytest.importorskip("torch")
    n_boxes = 2048
    parts, spots = A._terrain_boxes_scene(scenes, 0, n_boxes, seed=9, box=1.0, spread=55.0)
    g, o = cq.CollisionQuery(parts, order=A._order(cq, order)), orc.OracleWorld(parts)
    rng = np.random.default_rng(11)
    lo, hi = np.float32([-60, -10, -60]), np.float32([60, 20, 60])
    casts = scenes.gen_casts(2000, lo, hi, seed=71, radius=0.5, half_height=0.5, expand=0.0)
    deltas = []
    for step, n_moved in enumerate((1, 64, 1024), 1):
        ids = (1 + rng.choice(n_boxes, n_moved, replace=False)).tolist()
        models = [A._box_pose(scenes, rng, spots, eid, step) for eid in ids]
        du = DeviceUpdate(torch, ids, models)
        torch.cuda.synchronize()
        g.stats(reset=True)
        du.queue(g, None)
        deltas.append(g.stats()["kernel_launches"])
        o.update_transforms(ids, models)
        centres = np.stack([np.asarray(m, np.float32).reshape(16)[12:15] for m in models])
        rays = np.zeros(len(ids), cq.RAY)
        rays["origin"] = centres + np.float32([0.01, 30.0, 0.02])
        rays["direction"] = (0, -1, 0)
        rays["max_distance"], rays["mask"] = 100.0, cq.LAYER_ALL
        got = g.raycast(rays)
        assert got.tobytes() == o.raycast(rays, g.order).tobytes(), n_moved
        assert (got["triangle_index"] >= g.info()["n_static_triangles"]).all()
        assert g.capsuleCastBlocking(casts).tobytes() == o.capsule_cast(casts, 1, g.order).tobytes(), n_moved
    assert deltas[0] == deltas[1] == deltas[2] == (28 if order == "reference" else 20), deltas
    assert deltas[0] <= MAX_LAUNCHES
    g.close(), o.close()


# ---------------------------------------------------------------- no host block, ordering across streams
@pytest.mark.gpu
def test_device_update_does_not_block_and_is_ordered(cq, orc, scenes):
    """The call returns while its stream still sleeps.  An update on stream B queued after rays on stream A does not
    overtake them; rays queued on A after the update see the new trees."""
    torch = pytest.importorskip("torch")
    parts, spots = A._terrain_boxes_scene(scenes, 2, 8, seed=31)
    g, ref = cq.CollisionQuery(parts), cq.CollisionQuery(parts)
    rng = np.random.default_rng(4)
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    rays = scenes.gen_rays(1 << 20, lo, hi, seed=6, expand=0.0)
    ids = list(range(3, 11))
    m1 = [A._box_pose(scenes, rng, spots, e, 1) for e in ids]
    m0 = [A._box_pose(scenes, rng, spots, e, 0) for e in ids]
    warm = DeviceUpdate(torch, ids, m0)  # loads the kernels: the timed call below measures the enqueue only
    torch.cuda.synchronize()
    warm.queue(g, None)
    ref.update_transforms(ids, m0)
    before = ref.raycast(rays)
    ref.update_transforms(ids, m1)
    after = ref.raycast(rays)
    assert before.tobytes() != after.tobytes()
    du = DeviceUpdate(torch, ids, m1)
    d_rays = A._dev(torch, rays)
    out_a = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    out_a2 = torch.empty_like(out_a)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(sa):
        torch.cuda._sleep(200_000_000)
    g.raycast_device(d_rays.data_ptr(), len(rays), out_a.data_ptr(), sa.cuda_stream)
    with torch.cuda.stream(sb):
        torch.cuda._sleep(50_000_000)
    t0 = time.perf_counter()
    du.queue(g, sb.cuda_stream)
    dt = time.perf_counter() - t0
    assert not sb.query() and not sa.query()  # returned while both streams were still busy
    assert dt < 0.02, dt
    g.raycast_device(d_rays.data_ptr(), len(rays), out_a2.data_ptr(), sa.cuda_stream)
    torch.cuda.synchronize()
    assert A._host(out_a, cq.RAY_HIT).tobytes() == before.tobytes()
    assert A._host(out_a2, cq.RAY_HIT).tobytes() == after.tobytes()
    _assert_soups_equal(_soups(ref), _soups(g), "ordered")
    g.close(), ref.close()


# ---------------------------------------------------------------- CUDA-graph capture of a fixed step
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_fixed_step_graph_capture(cq, orc, scenes, order):
    """One uncaptured warm-up step, then a torch.cuda.CUDAGraph of: device update -> move-and-slide on the crowd's
    resident records with a platform -> rays -> blocking casts.  20 replays, each after new models were written into the
    same device buffer, equal uncaptured synchronous steps of world A byte for byte.  Under the capture, a call that would
    grow scratch and cq_agent_separation_device are refused and the capture stays usable.  After the replays, uncaptured
    async updates and queries on another stream still work (no captured world event is left behind)."""
    torch = pytest.importorskip("torch")
    n_static, n_dynamic = 4, 6
    parts, spots = A._terrain_boxes_scene(scenes, n_static, n_dynamic, seed=77)
    ga, gb = cq.CollisionQuery(parts, order=A._order(cq, order)), cq.CollisionQuery(parts, order=A._order(cq, order))
    lo, hi = np.float32([-55, -10, -55]), np.float32([55, 20, 55])
    rays = scenes.gen_rays(8000, lo, hi, seed=81, expand=0.0)
    casts = scenes.gen_casts(2000, lo, hi, seed=82, radius=0.6, half_height=0.7, expand=0.0)
    rng = np.random.default_rng(83)
    xz = rng.uniform(-30, 30, (256, 2)).astype(np.float32)
    pos = np.stack([xz[:, 0], scenes.terrain_height(xz[:, 0], xz[:, 1]) + 3.0, xz[:, 1]], 1).astype(np.float32)
    vel = rng.uniform(-6, 6, (256, 3)).astype(np.float32)
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    g3 = np.float32([0.0, -98.0, 0.0])
    bv, _ = scenes.box_mesh(3.0)
    platform = scenes.platform_record(bv, scenes.trs_model((5.0, 2.0, 5.0)), (5.0, 2.0, 5.0), (5.2, 2.0, 5.0))
    platform = np.ascontiguousarray(platform, cq.PLATFORM)
    ids = [1 + n_static + k for k in range(0, n_dynamic, 2)] + [1]  # three dynamic boxes and one static one
    pose = lambda step: np.stack([A._box_pose(scenes, rng, spots, e, step) for e in ids]).astype(np.float32)
    sa = cq.init_states(pos, vel)
    crowd = cq.Crowd(gb, cq.init_states(pos, vel))
    d_ids = torch.from_numpy(np.asarray(ids, np.uint32).view(np.int32).copy()).cuda()
    d_models = torch.zeros((len(ids), 16), dtype=torch.float32, device="cuda")
    d_status = torch.zeros(1, dtype=torch.int32, device="cuda")
    d_rays, d_casts = A._dev(torch, rays), A._dev(torch, casts)
    out_r = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    out_c = torch.empty(len(casts) * cq.CAST_HIT.itemsize, dtype=torch.uint8, device="cuda")
    L = cq.lib()

    def step_b(stream):
        gb.update_transforms_device(d_ids.data_ptr(), d_models.data_ptr(), len(ids), d_status.data_ptr(), stream)
        cq._check(L.cq_move_and_slide_device_ex(gb.handle, C.c_void_p(crowd.device_states), crowd.n, cq._ptr(params),
                                                C.c_float(1.0 / 60.0), cq._ptr(g3), cq.MAS_APPLY_GRAVITY, cq._ptr(platform), 1,
                                                C.c_void_p(stream)))
        gb.raycast_device(d_rays.data_ptr(), len(rays), out_r.data_ptr(), stream)
        gb.capsule_cast_device(d_casts.data_ptr(), len(casts), cq.CAST_BLOCKING, out_c.data_ptr(), stream)

    def step_a(models):
        ga.update_transforms(ids, models)
        ga.move_and_slide(sa, params, platforms=platform)
        return ga.raycast(rays), ga.capsuleCastBlocking(casts)

    def check(step, want_r, want_c):
        assert A._host(out_r, cq.RAY_HIT).tobytes() == want_r.tobytes(), step
        assert A._host(out_c, cq.CAST_HIT).tobytes() == want_c.tobytes(), step
        assert crowd.read().tobytes() == sa.tobytes(), step
        assert int(d_status.item()) == 0, step

    m = pose(0)
    d_models.copy_(torch.from_numpy(m))
    torch.cuda.synchronize()
    step_b(torch.cuda.current_stream().cuda_stream)  # warm-up: sizes every scratch block
    torch.cuda.synchronize()
    check(0, *step_a(m))
    big = A._dev(torch, np.repeat(casts, 64))
    big_out = torch.empty(len(casts) * 64 * cq.CAST_HIT.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    graph, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=cs):
        st = torch.cuda.current_stream().cuda_stream
        step_b(st)
        with pytest.raises(cq.CQError, match="make one uncaptured call of this size first"):  # more lanes: more node scratch
            gb.capsule_cast_device(big.data_ptr(), len(casts) * 64, cq.CAST_BLOCKING, big_out.data_ptr(), st)
        with pytest.raises(cq.CQError, match="cannot be captured"):
            gb.agent_separation_device(crowd.device_states, crowd.n, params, stream=st)
    # a refused captured call leaves uncaptured calls alone: host batches and a crowd step work as before
    assert gb.raycast(rays).tobytes() == ga.raycast(rays).tobytes()
    assert gb.capsuleCastBlocking(casts).tobytes() == ga.capsuleCastBlocking(casts).tobytes()
    crowd.step(None, params, platforms=platform)
    ga.move_and_slide(sa, params, platforms=platform)
    assert crowd.read().tobytes() == sa.tobytes()
    for step in range(1, 21):
        if step == 11:
            # an uncaptured call that outgrows the node scratch the graph recorded: the graph's blocks must survive it
            gb.capsule_cast_device(big.data_ptr(), len(casts) * 64, cq.CAST_BLOCKING, big_out.data_ptr(), None)
            torch.cuda.synchronize()
            big_hits = A._host(big_out, cq.CAST_HIT)
            assert big_hits.tobytes() == ga.capsuleCastBlocking(np.repeat(casts, 64)).tobytes()
        m = pose(step)
        d_models.copy_(torch.from_numpy(m))
        graph.replay()
        torch.cuda.synchronize()
        check(step, *step_a(m))
    # uncaptured work on another stream after the replays
    s2 = torch.cuda.Stream()
    m = pose(21)
    gb.update_transforms_async(ids, m, stream=s2.cuda_stream)
    ga.update_transforms(ids, m)
    gb.raycast_device(d_rays.data_ptr(), len(rays), out_r.data_ptr(), s2.cuda_stream)
    s2.synchronize()
    assert A._host(out_r, cq.RAY_HIT).tobytes() == ga.raycast(rays).tobytes()
    _assert_soups_equal(_soups(ga), _soups(gb), "after replays")
    del graph
    crowd.close(), ga.close(), gb.close()


# ---------------------------------------------------------------- many small dirty refits that share ancestors
def _packed_run_device(torch, cq, orc, scenes, order, seed, n_updates=100):
    bv, bi = scenes.box_mesh(0.5)
    pv, pidx = scenes.plane_mesh(20.0)
    parts = [scenes.part(pv, pidx, entity_id=0)]
    grid = np.array([(x, y, z) for x in range(4) for y in range(4) for z in range(4)], np.float32) * 0.6
    for k, c in enumerate(grid):
        parts.append(scenes.part(bv, bi, scenes.trs_model(c + np.float32([0, 1, 0])), is_dynamic=True, entity_id=1 + k))
    g, o = cq.CollisionQuery(parts, order=A._order(cq, order)), orc.OracleWorld(parts)
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
        du = DeviceUpdate(torch, ids, models)
        du.queue(g, None)
        o.update_transforms(ids, models)
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
def test_many_small_device_dirty_refits(cq, orc, scenes, order):
    """100 random device updates of 1..15 of 64 packed boxes whose leaves share ancestors match the oracle after every
    update, and a second pass with the same seed gives the same bytes."""
    torch = pytest.importorskip("torch")
    first = _packed_run_device(torch, cq, orc, scenes, order, seed=321)
    assert _packed_run_device(torch, cq, orc, scenes, order, seed=321) == first
