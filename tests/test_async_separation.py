"""cq_agent_separation_device_async: agent separation queued on a stream with every outcome decided on the device (the
drift retry, the grid overflow, a stalled schedule), so that the reference's whole fixed step can be captured in a CUDA
graph.  The call must leave exactly what the synchronous calls and the oracle leave, change nothing when it fails,
never block the host, respect the ordering contract of transform updates, cost a fixed number of launches, and record
into a graph whose replays equal uncaptured synchronous steps byte for byte."""
import ctypes as C
import importlib.util
import os
import time

import numpy as np
import pytest

# device-buffer helpers of the async refit tests (imported by path: tests/ is not a package)
_spec = importlib.util.spec_from_file_location("_async_refit_helpers", os.path.join(os.path.dirname(__file__), "test_async_refit.py"))
A = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(A)

CQ_ERR_INVALID = -1


def launches_per_call(iterations):  # include/cq.h: 3 + 23 per sweep
    return 3 + 23 * max(1, iterations)


def test_async_separation_argument_checks(cq):
    """NULL world, NULL params, n < 0 and a NULL states pointer with n > 0 are refused before any CUDA call, so they
    answer without a GPU."""
    L = cq.lib()
    p = C.c_void_p(16)  # never dereferenced: the checks come first (a non-NULL world too, so each check is reached)
    args = lambda w, st, n, params: (w, st, n, params, None, 2, C.c_float(0.2), C.c_float(0.1), 1, None, None)
    assert L.cq_agent_separation_device_async(*args(None, p, 4, p)) == CQ_ERR_INVALID
    assert L.cq_agent_separation_device_async(*args(p, p, 4, None)) == CQ_ERR_INVALID
    assert L.cq_agent_separation_device_async(*args(p, p, -1, p)) == CQ_ERR_INVALID
    assert L.cq_agent_separation_device_async(*args(p, None, 4, p)) == CQ_ERR_INVALID
    assert "cq_agent_separation_device_async" in cq.EXPORTS
    assert (cq.SEP_STATUS_OK, cq.SEP_STATUS_GRID, cq.SEP_STATUS_DRIFT, cq.SEP_STATUS_STALLED) == (0, 1, 2, 3)


# ---------------------------------------------------------------- scenes
def _crowd_params(cq):
    p = cq.default_params()
    p["radius"], p["half_height"] = 0.4, 0.5
    p["skin_width"], p["snap_distance"] = 0.08, 0.3
    return p


def _dense_crowd(cq, scenes, n=2500, seed=21):
    """The crowd of test_agent_separation_sequential_semantics: 45% footprint coverage on a terrain with three walls,
    mixed mass weights including immovable agents."""
    tparts, _ = scenes.terrain_scene(cells=96, cell=1.5, seed=5)
    bv, bi = scenes.box_mesh(6.0)
    walls = [scenes.part(bv, bi, scenes.trs_model((x, float(scenes.terrain_height(np.float32([x]), np.float32([z]), 5)[0]), z)),
                         entity_id=10 + k) for k, (x, z) in enumerate([(-8.0, 3.0), (9.0, -6.0), (2.0, 12.0)])]
    rng = np.random.default_rng(seed)
    half = np.sqrt(n * np.pi * 0.4 ** 2 / 0.45) / 2
    x, z = rng.uniform(-half, half, n), rng.uniform(-half, half, n)
    y = scenes.terrain_height(x, z, 5) + np.float32(0.9 + 0.05) + rng.uniform(0, 0.2, n)
    pos = np.stack([x, y, z], axis=1).astype(np.float32)
    ang = rng.uniform(0, 2 * np.pi, n)
    walk = (np.stack([np.cos(ang), np.zeros(n), np.sin(ang)], axis=1) * rng.uniform(1, 7, (n, 1))).astype(np.float32)
    mass = rng.choice(np.float32([1.0, 3.0, 500.0, 0.0]), n, p=[0.6, 0.25, 0.1, 0.05])
    return tparts + walls, pos, walk, mass


def _pusher_rows(n_rows=40, y=-3.0 + 0.9 + 0.05, z0=-60.0):
    """The drift scene of test_agent_separation_sequential_semantics: per row 8 immovable pushers, then a light agent
    they shove more than two cells before its own turn, then a bystander."""
    rows = []
    for r in range(n_rows):
        zr = 3.0 * r + z0
        rows += [[-0.3 + 0.4 * k, y, zr] for k in range(8)] + [[0.0, y, zr], [3.38, y, zr + 0.3]]
    return np.float32(rows), np.tile(np.float32([0.0] * 8 + [1.0, 1.0]), n_rows)


def _flat(scenes):
    fv, fi = scenes.plane_mesh(80.0)
    return [scenes.part(fv, fi, scenes.trs_model((0, -3, 0)), entity_id=0)]


class DeviceCrowd:
    """Character records, mass weights and a status word in device memory."""

    def __init__(self, torch, cq, states, mass=None):
        self.cq, self.n = cq, len(states)
        self.states = A._dev(torch, states)
        self.mass = None if mass is None else torch.from_numpy(np.ascontiguousarray(mass, np.float32)).cuda()
        self.status = torch.full((1,), -7, dtype=torch.int32, device="cuda")

    def separate(self, g, params, stream=None, **kw):
        g.agent_separation_device_async(self.states.data_ptr(), self.n, params,
                                        None if self.mass is None else self.mass.data_ptr(),
                                        d_status_ptr=self.status.data_ptr(), stream=stream, **kw)

    def read(self):
        return A._host(self.states, self.cq.STATE)


# ---------------------------------------------------------------- equal to the synchronous call and the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("use_query", [True, False])
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_async_separation_equals_sync_and_oracle(cq, orc, scenes, order, use_query):
    """5 crowd steps (move-and-slide with agent CCD, then separation) of the dense crowd.  World A runs the synchronous
    batch calls, world B the device calls on device records with the async separation, sweeps alternating between 1 and
    2.  After every step B's records equal A's and the oracle's byte for byte, and the status is 0."""
    torch = pytest.importorskip("torch")
    parts, pos, walk, mass = _dense_crowd(cq, scenes)
    ga, gb = cq.CollisionQuery(parts, order=A._order(cq, order)), cq.CollisionQuery(parts, order=A._order(cq, order))
    o = orc.OracleWorld(parts)
    p = _crowd_params(cq)
    sa, so = cq.init_states(pos, walk), orc.init_states(pos, walk)
    dc = DeviceCrowd(torch, cq, cq.init_states(pos, walk), mass)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    for step in range(5):
        it = 2 if step % 2 == 0 else 1
        gb.move_and_slide_device(dc.states.data_ptr(), dc.n, p, flags=3, stream=s.cuda_stream)
        dc.separate(gb, p, s.cuda_stream, iterations=it, use_query=use_query)
        ga.move_and_slide(sa, p, flags=3)
        ga.agent_separation(sa, p, mass_weight=mass, iterations=it, use_query=use_query)
        o.move_and_slide(so, p, flags=3, order=ga.order, n_threads=8)
        o.agent_separation(so, p, mass_weight=mass, iterations=it, use_query=use_query, order=ga.order, n_threads=8)
        s.synchronize()
        assert int(dc.status.item()) == cq.SEP_STATUS_OK, step
        got = dc.read()
        assert got.tobytes() == sa.tobytes(), ("sync", step)
        assert got.tobytes() == so.tobytes(), ("oracle", step)
        new = sa.copy()
        for rec in (sa, so, new):
            rec["velocity"][:, 0] = walk[:, 0]
            rec["velocity"][:, 2] = walk[:, 2]
        dc.states.copy_(A._dev(torch, new))
        torch.cuda.synchronize()
    ga.close(), gb.close(), o.close()


# ---------------------------------------------------------------- the drift retry, decided on the device
@pytest.mark.gpu
@pytest.mark.parametrize("use_query", [False, True])
def test_async_separation_drift_retry(cq, orc, scenes, use_query):
    torch = pytest.importorskip("torch")
    flat = _flat(scenes)
    g, o = cq.CollisionQuery(flat), orc.OracleWorld(flat)
    p = _crowd_params(cq)
    rows, dmass = _pusher_rows()
    dc = DeviceCrowd(torch, cq, cq.init_states(rows), dmass)
    b = orc.init_states(rows)
    torch.cuda.synchronize()
    dc.separate(g, p, use_query=use_query)
    o.agent_separation(b, p, mass_weight=dmass, iterations=2, use_query=use_query, order=g.order)
    torch.cuda.synchronize()
    assert int(dc.status.item()) == cq.SEP_STATUS_OK
    got = dc.read()
    assert got.tobytes() == b.tobytes()
    assert (got["position"][8::10, 0] > 2.0).all()  # every light agent was pushed more than two cells: R = 1 failed
    g.close(), o.close()


# ---------------------------------------------------------------- all-or-nothing errors
@pytest.mark.gpu
def test_async_separation_grid_overflow_changes_nothing(cq, orc, scenes):
    """Two agents 1e5 m apart on both axes span 1e10 cells of 1 m: status CQ_SEP_STATUS_GRID and not one byte of the
    records changes; the synchronous call still reports CQ_ERR_INVALID with its message; a valid call right after on
    the same world writes status 0 and the oracle's result."""
    torch = pytest.importorskip("torch")
    flat = _flat(scenes)
    g, o = cq.CollisionQuery(flat), orc.OracleWorld(flat)
    p = _crowd_params(cq)
    far = cq.init_states(np.float32([[-5e4, -2.05, -5e4], [5e4, -2.05, 5e4]]), np.float32([[1, 0, 0], [0, 0, 1]]))
    before = far.tobytes()
    dc = DeviceCrowd(torch, cq, far)
    torch.cuda.synchronize()
    dc.separate(g, p)
    torch.cuda.synchronize()
    assert int(dc.status.item()) == cq.SEP_STATUS_GRID
    assert dc.read().tobytes() == before
    host = far.copy()
    with pytest.raises(cq.CQError, match=r"the crowd spans more than 2\^31 grid cells of 1.000 m") as e:
        g.agent_separation(host, p)
    assert f"libcq error {CQ_ERR_INVALID}:" in str(e.value)
    assert host.tobytes() == before
    with pytest.raises(cq.CQError, match=r"2\^31 grid cells"):
        g.agent_separation_device(dc.states.data_ptr(), dc.n, p)
    assert dc.read().tobytes() == before
    rows, dmass = _pusher_rows(4)
    ok = DeviceCrowd(torch, cq, cq.init_states(rows), dmass)
    b = orc.init_states(rows)
    torch.cuda.synchronize()
    ok.separate(g, p)
    o.agent_separation(b, p, mass_weight=dmass, order=g.order)
    torch.cuda.synchronize()
    assert int(ok.status.item()) == cq.SEP_STATUS_OK
    assert ok.read().tobytes() == b.tobytes()
    g.close(), o.close()


# ---------------------------------------------------------------- no host block
@pytest.mark.gpu
def test_async_separation_does_not_block(cq, orc, scenes):
    torch = pytest.importorskip("torch")
    parts, pos, walk, mass = _dense_crowd(cq, scenes)
    g, ref = cq.CollisionQuery(parts), cq.CollisionQuery(parts)
    p = _crowd_params(cq)
    warm = DeviceCrowd(torch, cq, cq.init_states(pos, walk), mass)  # sizes the scratch and instantiates the graphs
    torch.cuda.synchronize()
    warm.separate(g, p)
    torch.cuda.synchronize()
    dc = DeviceCrowd(torch, cq, cq.init_states(pos, walk), mass)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
    t0 = time.perf_counter()
    dc.separate(g, p, s.cuda_stream)
    dt = time.perf_counter() - t0
    assert not s.query()  # returned while the stream was still busy
    assert dt < 0.05, dt
    s.synchronize()
    assert int(dc.status.item()) == cq.SEP_STATUS_OK
    want = cq.init_states(pos, walk)
    ref.agent_separation(want, p, mass_weight=mass)
    assert dc.read().tobytes() == want.tobytes()
    g.close(), ref.close()


# ---------------------------------------------------------------- ordered against transform updates
@pytest.mark.gpu
def test_async_separation_ordered_after_update(cq, orc, scenes):
    """update_transforms_async on stream 1 (queued behind a sleep) moves a wall into a pushed crowd; the use_query
    separation queued next on stream 2 must see the moved wall: its vetoes equal the oracle's with the wall moved, which
    differ from those with the wall where it was."""
    torch = pytest.importorskip("torch")
    bv, bi = scenes.box_mesh(4.0)
    wall0, wall1 = scenes.trs_model((30.0, -1.0, 0.0)), scenes.trs_model((2.6, -1.0, 0.0))
    parts = _flat(scenes) + [scenes.part(bv, bi, wall0, is_dynamic=True, entity_id=5)]
    g, o, o_still = cq.CollisionQuery(parts), orc.OracleWorld(parts), orc.OracleWorld(parts)
    p = _crowd_params(cq)
    rows, dmass = _pusher_rows(12, z0=-1.0)
    rows[:, 2] *= 0.1  # rows 0.3 m apart in z: all of them within reach of the wall's side
    dc = DeviceCrowd(torch, cq, cq.init_states(rows), dmass)
    want, still = orc.init_states(rows), orc.init_states(rows)
    o.update_transforms([5], [wall1])
    o.agent_separation(want, p, mass_weight=dmass, order=g.order)
    o_still.agent_separation(still, p, mass_weight=dmass, order=g.order)
    assert want.tobytes() != still.tobytes()  # the moved wall vetoes pushes
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(100_000_000)
    g.update_transforms_async([5], [wall1], stream=s1.cuda_stream)
    dc.separate(g, p, s2.cuda_stream)
    torch.cuda.synchronize()
    assert int(dc.status.item()) == cq.SEP_STATUS_OK
    assert dc.read().tobytes() == want.tobytes()
    g.close(), o.close(), o_still.close()


# ---------------------------------------------------------------- a fixed number of launches
@pytest.mark.gpu
@pytest.mark.parametrize("iterations", [1, 2])
def test_async_separation_launch_count_is_fixed(cq, orc, scenes, iterations):
    """A crowd without drift, the drift scene and the grid overflow cost the launches cq.h states, whatever happened."""
    torch = pytest.importorskip("torch")
    flat = _flat(scenes)
    g = cq.CollisionQuery(flat)
    p = _crowd_params(cq)
    rows, dmass = _pusher_rows()
    rng = np.random.default_rng(3)
    calm = np.stack([rng.uniform(-30, 30, 400), np.full(400, -2.05), rng.uniform(-30, 30, 400)], 1).astype(np.float32)
    far = np.float32([[-5e4, -2.05, -5e4], [5e4, -2.05, 5e4]])
    deltas = {}
    for name, pos, mass, want in (("calm", calm, None, cq.SEP_STATUS_OK), ("drift", rows, dmass, cq.SEP_STATUS_OK),
                                  ("grid", far, None, cq.SEP_STATUS_GRID)):
        dc = DeviceCrowd(torch, cq, cq.init_states(pos), mass)
        torch.cuda.synchronize()
        dc.separate(g, p, iterations=iterations)  # warm-up: scratch growth and graph instantiation are not launches either
        torch.cuda.synchronize()
        g.stats(reset=True)
        dc.separate(g, p, iterations=iterations)
        deltas[name] = g.stats()["kernel_launches"]
        torch.cuda.synchronize()
        assert int(dc.status.item()) == want, name
    assert set(deltas.values()) == {launches_per_call(iterations)}, deltas
    g.close()


# ---------------------------------------------------------------- CUDA-graph capture of the whole fixed step
@pytest.mark.gpu
def test_fixed_step_with_separation_graph_capture(cq, orc, scenes):
    """One uncaptured warm-up step, then a torch.cuda.CUDAGraph of the reference's whole fixed step: device update of a
    moving box -> move-and-slide (gravity, agent CCD, a platform) on a crowd's resident records -> async separation ->
    rays.  Under the capture, a separation larger than any uncaptured one and cq_agent_separation_device are refused and
    the capture stays usable.  20 replays, each after new models were written into the same buffer, equal the uncaptured
    synchronous sequence update -> move-and-slide -> separation -> rays of world A byte for byte, with status 0.  Before
    some replays the pusher rows are put back in both worlds, so that those replays take the drift retry."""
    torch = pytest.importorskip("torch")
    bv, bi = scenes.box_mesh(3.0)
    parts = _flat(scenes) + [scenes.part(bv, bi, scenes.trs_model((-20.0, -1.5, 20.0)), is_dynamic=True, layer=2, entity_id=3)]
    ga, gb = cq.CollisionQuery(parts), cq.CollisionQuery(parts)
    rng = np.random.default_rng(91)
    rows, rmass = _pusher_rows(20, z0=-60.0)
    m = 1600  # a dense crowd (~45% coverage) beside the rows
    half = np.sqrt(m * np.pi * 0.4 ** 2 / 0.45) / 2
    xz = rng.uniform(-half, half, (m, 2)).astype(np.float32) + np.float32([0.0, 25.0])
    crowd_pos = np.concatenate([rows, np.stack([xz[:, 0], np.full(m, -2.05, np.float32), xz[:, 1]], 1)])
    n = len(crowd_pos)
    vel = np.zeros((n, 3), np.float32)
    vel[len(rows):] = rng.uniform(-5, 5, (m, 3)) * np.float32([1, 0, 1])
    mass = np.concatenate([rmass, rng.choice(np.float32([1.0, 3.0, 0.0]), m, p=[0.7, 0.25, 0.05])])
    p = np.ascontiguousarray(_crowd_params(cq), cq.PARAMS)
    g3 = np.float32([0.0, -98.0, 0.0])
    platform = np.ascontiguousarray(scenes.platform_record(bv, scenes.trs_model((-20.0, -1.5, 20.0)), (-20.0, -1.5, 20.0),
                                                           (-19.8, -1.5, 20.0)), cq.PLATFORM)
    lo, hi = np.float32([-40, -4, -40]), np.float32([40, 4, 40])
    rays = scenes.gen_rays(4000, lo, hi, seed=92, expand=0.0)
    pose = lambda step: np.float32(scenes.trs_model((-20.0 + 0.5 * step, -1.5 + 0.1 * (step % 3), 20.0))).reshape(1, 16)
    sa = cq.init_states(crowd_pos, vel)
    crowd = cq.Crowd(gb, cq.init_states(crowd_pos, vel))
    d_ids = torch.tensor([3], dtype=torch.int32, device="cuda")
    d_models = torch.zeros((1, 16), dtype=torch.float32, device="cuda")
    d_upd, d_sep = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.full((1,), -7, dtype=torch.int32, device="cuda")
    d_mass = torch.from_numpy(mass).cuda()
    d_rays = A._dev(torch, rays)
    out_r = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    L = cq.lib()

    def step_b(stream, n_sep=n):
        gb.update_transforms_device(d_ids.data_ptr(), d_models.data_ptr(), 1, d_upd.data_ptr(), stream)
        cq._check(L.cq_move_and_slide_device_ex(gb.handle, C.c_void_p(crowd.device_states), n, cq._ptr(p), C.c_float(1.0 / 60.0),
                                                cq._ptr(g3), cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS, cq._ptr(platform), 1,
                                                C.c_void_p(stream)))
        gb.agent_separation_device_async(crowd.device_states, n_sep, p, d_mass.data_ptr(), d_status_ptr=d_sep.data_ptr(),
                                         stream=stream)
        gb.raycast_device(d_rays.data_ptr(), len(rays), out_r.data_ptr(), stream)

    def step_a(models):
        ga.update_transforms([3], models)
        ga.move_and_slide(sa, p, flags=cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS, platforms=platform)
        ga.agent_separation(sa, p, mass_weight=mass)
        return ga.raycast(rays)

    def check(step, want_r):
        assert int(d_upd.item()) == 0 and int(d_sep.item()) == cq.SEP_STATUS_OK, step
        assert crowd.read().tobytes() == sa.tobytes(), step
        assert A._host(out_r, cq.RAY_HIT).tobytes() == want_r.tobytes(), step

    m0 = pose(0)
    d_models.copy_(torch.from_numpy(m0))
    torch.cuda.synchronize()
    step_b(torch.cuda.current_stream().cuda_stream)  # warm-up: sizes every scratch block
    torch.cuda.synchronize()
    check(0, step_a(m0))
    bigger = torch.zeros((n + 4096) * cq.STATE.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    graph, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=cs):
        st = torch.cuda.current_stream().cuda_stream
        step_b(st)
        with pytest.raises(cq.CQError, match="make one uncaptured call of this size first"):
            gb.agent_separation_device_async(bigger.data_ptr(), n + 4096, p, stream=st)
        with pytest.raises(cq.CQError, match="cannot be captured"):
            gb.agent_separation_device(crowd.device_states, n, p, stream=st)
    drifted = 0
    for step in range(1, 21):
        if step % 5 == 0:  # put the pusher rows back: their light agents are shoved more than two cells again
            rec = crowd.read()
            fresh = cq.init_states(rows)
            rec[:len(rows)], sa[:len(rows)] = fresh, fresh
            torch.cuda.synchronize()
            crowd.write(rec)
        m1 = pose(step)
        d_models.copy_(torch.from_numpy(m1))
        graph.replay()
        torch.cuda.synchronize()
        check(step, step_a(m1))
        if step % 5 == 0 and (sa["position"][8:len(rows):10, 0] > 2.0).all():
            drifted += 1
    assert drifted == 4, f"only {drifted} of 4 replays took the drift retry (pushed agents moved less than two cells)"
    # the graph's blocks survive an uncaptured call that outgrows them, and uncaptured work continues
    big = cq.init_states(np.concatenate([crowd_pos, crowd_pos[:4096] + np.float32([0, 0, 90])]))
    bd = DeviceCrowd(torch, cq, big)
    torch.cuda.synchronize()
    bd.separate(gb, p)
    graph.replay()
    torch.cuda.synchronize()
    check(21, step_a(pose(20)))
    del graph
    crowd.close(), ga.close(), gb.close()
