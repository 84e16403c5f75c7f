"""Kinematic platforms on the device: cq_world_platforms_device builds platform records from the world's vertices on the
GPU, and cq_move_and_slide_device_platforms reads them from device memory when its kernels run.  Together they let a
captured fixed step carry characters with the records of each replay's frame instead of the frame of the capture.  The
records must equal scenes.platform_record (meshWorldAABB) of the current models, the step must equal the host-array call
and the oracle byte for byte at any platform count, and a replayed graph must equal uncaptured steps."""
import ctypes as C
import importlib.util
import os
import subprocess

import numpy as np
import pytest

# device-buffer helpers of the async refit tests (imported by path: tests/ is not a package)
_spec = importlib.util.spec_from_file_location("_async_refit_helpers", os.path.join(os.path.dirname(__file__), "test_async_refit.py"))
A = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(A)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CQ_ERR_INVALID = -1
UNKNOWN_ID = 12345


def test_device_platforms_argument_checks(cq):
    """NULL world, negative counts and NULL arrays with a positive count are refused before any CUDA call, so they
    answer without a GPU."""
    L = cq.lib()
    p = C.c_void_p(16)  # never dereferenced: the checks come first (a non-NULL world too, so each check is reached)
    assert L.cq_world_platforms_device(None, p, p, 1, p, None, None) == CQ_ERR_INVALID
    assert L.cq_world_platforms_device(p, p, p, -1, p, None, None) == CQ_ERR_INVALID
    assert L.cq_world_platforms_device(p, None, p, 1, p, None, None) == CQ_ERR_INVALID
    assert L.cq_world_platforms_device(p, p, None, 1, p, None, None) == CQ_ERR_INVALID
    assert L.cq_world_platforms_device(p, p, p, 1, None, None, None) == CQ_ERR_INVALID
    g = np.zeros(3, np.float32)
    mas = lambda w, st, n, params, grav, plat, n_plat: L.cq_move_and_slide_device_platforms(
        w, st, n, params, C.c_float(1.0 / 60.0), grav, 1, plat, n_plat, None)
    assert mas(None, p, 4, p, cq._ptr(g), p, 1) == CQ_ERR_INVALID
    assert mas(p, p, -1, p, cq._ptr(g), p, 1) == CQ_ERR_INVALID
    assert mas(p, None, 4, p, cq._ptr(g), p, 1) == CQ_ERR_INVALID
    assert mas(p, p, 4, None, cq._ptr(g), p, 1) == CQ_ERR_INVALID
    assert mas(p, p, 4, p, None, p, 1) == CQ_ERR_INVALID
    assert mas(p, p, 4, p, cq._ptr(g), p, -1) == CQ_ERR_INVALID
    assert mas(p, p, 4, p, cq._ptr(g), None, 1) == CQ_ERR_INVALID
    assert mas(p, p, 4, p, cq._ptr(g), None, 100000) == CQ_ERR_INVALID
    assert "cq_move_and_slide_device_platforms" in cq.lib().cq_last_error().decode()
    assert "cq_world_platforms_device" in cq.EXPORTS and "cq_move_and_slide_device_platforms" in cq.EXPORTS


CPP_PROBE = r"""
// The C++ mirror hands the device platform calls' arguments to the library unchanged, and the host-array moveAndSlide
// overload still reaches the host-array call.  The world and the calls are stubbed here (these definitions take
// precedence over libcq.so's), so no GPU is needed.
#include <cstdio>
#include "CollisionQuery.hpp"

static int seen = 0;
static const void *seenPtr = nullptr;
static int32_t seenN = 0;
static uint32_t seenFlags = 0;
extern "C" int cq_world_create_ex(const cq_mesh_part *, int32_t, const cq_world_options *, cq_world **out) {
    static int dummy;
    *out = reinterpret_cast<cq_world *>(&dummy);
    return CQ_OK;
}
extern "C" void cq_world_destroy(cq_world *) {}
extern "C" int cq_world_platforms_device(cq_world *, const uint32_t *ids, const float *, int32_t n, cq_platform *out,
                                         int32_t *status, void *stream) {
    seen = 1, seenPtr = out, seenN = n;
    return ids && status == nullptr && stream == (void *)0x30 ? CQ_OK : CQ_ERR_INVALID;
}
extern "C" int cq_move_and_slide_device_platforms(cq_world *, cq_character_state *, int32_t, const cq_controller_params *, float,
                                                  const float *, uint32_t flags, const cq_platform *d_platforms,
                                                  int32_t n_platforms, void *) {
    seen = 2, seenPtr = d_platforms, seenN = n_platforms, seenFlags = flags;
    return CQ_OK;
}
extern "C" int cq_move_and_slide_batch_ex(cq_world *, cq_character_state *, int32_t, const cq_controller_params *, float,
                                          const float *, uint32_t, const cq_platform *platforms, int32_t n_platforms) {
    seen = 3, seenPtr = platforms, seenN = n_platforms;
    return CQ_OK;
}

int main() {
    cqhost::CollisionQuery q(std::vector<cq_mesh_part>{});
    static uint32_t ids[1] = {7};
    static float deltas[3] = {0, 0, 0};
    static cq_platform recs[3];
    if (!q.platformsDevice(ids, deltas, 3, recs, nullptr, (void *)0x30) || seen != 1 || seenPtr != recs || seenN != 3) return 1;
    static cq_controller_params p{};
    static cq_character_state s{};
    const float g[3] = {0, -98, 0};
    if (!q.moveAndSlide(&s, 1, p, 1.0f / 60.0f, g, cqhost::DevicePlatforms{recs, 1000}, true) || seen != 2 || seenPtr != recs ||
        seenN != 1000 || seenFlags != (CQ_MAS_APPLY_GRAVITY | CQ_MAS_AGENTS))
        return 2;
    if (!q.moveAndSlide(&s, 1, p, 1.0f / 60.0f, g, recs, 2, false) || seen != 3 || seenN != 2) return 3;
    std::printf("ok\n");
    return 0;
}
"""


def test_cpp_wrapper_device_platforms(cq, tmp_path):
    cq.build()
    src = tmp_path / "device_platforms_probe.cpp"
    src.write_text(CPP_PROBE)
    exe = tmp_path / "device_platforms_probe"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "swift-game-engine_b200", "cpp"),
                        str(src), "-L" + cq.CSRC, "-lcq", "-Wl,-rpath," + cq.CSRC, "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stdout, r.stderr)


# ---------------------------------------------------------------- scenes and helpers
T0 = [np.float32([0, -1.0, 0]), np.float32([12, -1.0, 0])]  # elevator, mover (entity ids 1 and 2)
OFFSET7 = np.float32([5.0, 0.0, 0.0])  # entity 7's second part, in its local frame


def _platform_scene(scenes):
    """The elevator-and-mover scene of test_kinematic_platforms_carry_and_push, plus entity 7 (two dynamic parts), entity
    8 (a static-set box) and entity 9 (one degenerate triangle, filtered out: no triangles)."""
    bv, bi = scenes.box_mesh(4.0)
    sv, si = scenes.box_mesh(2.0)
    v, i = scenes.plane_mesh(80.0)
    parts = [scenes.part(v, i, scenes.trs_model((0, -3, 0)), entity_id=0),
             scenes.part(bv, bi, scenes.trs_model(T0[0]), is_dynamic=True, entity_id=1),
             scenes.part(bv, bi, scenes.trs_model(T0[1]), is_dynamic=True, entity_id=2),
             scenes.part(sv, si, scenes.trs_model((-20, 5, -20)), is_dynamic=True, entity_id=7),
             scenes.part(sv + OFFSET7, si, scenes.trs_model((-20, 5, -20)), is_dynamic=True, entity_id=7),
             scenes.part(sv, si, scenes.trs_model((20, 4, 20)), entity_id=8),
             scenes.part(np.zeros((3, 3), np.float32), np.arange(3, dtype=np.uint32), is_dynamic=True, entity_id=9)]
    local = {1: bv, 2: bv, 7: np.concatenate([sv, sv + OFFSET7]), 8: sv}
    return parts, local


def _crowd(rng, n, capsule_half):
    """Characters on the plane (y = -3) around both platforms, those above a platform standing on its top (y = 1)."""
    pos = np.stack([rng.uniform(-6, 18, n), np.full(n, -3.0 + capsule_half + 0.05), rng.uniform(-5, 5, n)], axis=1).astype(np.float32)
    on_top = (np.abs(pos[:, 0]) < 2) & (np.abs(pos[:, 2]) < 2) | (np.abs(pos[:, 0] - 12) < 2) & (np.abs(pos[:, 2]) < 2)
    pos[on_top, 1] = 1.0 + capsule_half + 0.05
    vel = (rng.uniform(-3, 3, (n, 3)) * [1, 0, 1]).astype(np.float32)
    return pos, vel, on_top


def _empty_record():
    r = np.zeros(1, np.dtype([("aabb_min", "<f4", 3), ("aabb_max", "<f4", 3), ("delta", "<f4", 3)]))
    r["aabb_min"], r["aabb_max"] = np.inf, -np.inf
    return r


def _assert_records_equal(got, want, what):
    """Boxes and deltas compared with float == (min / max may pick either sign of a zero coordinate)."""
    for k in ("aabb_min", "aabb_max", "delta"):
        assert np.array_equal(got[k], want[k]), (what, k, got[k], want[k])


def _extra_platforms(rng, n):
    """n synthetic platform records over the crowd's area: a third carry or push with a non-zero motion, a third do not
    move, a third are empty (inert) boxes."""
    rec = np.zeros(n, np.dtype([("aabb_min", "<f4", 3), ("aabb_max", "<f4", 3), ("delta", "<f4", 3)]))
    c = np.stack([rng.uniform(-6, 18, n), rng.uniform(-3.5, -1.5, n), rng.uniform(-5, 5, n)], 1).astype(np.float32)
    h = rng.uniform(0.5, 2.0, (n, 3)).astype(np.float32)
    rec["aabb_min"], rec["aabb_max"] = c - h, c + h
    back = np.arange(n)[::-1]
    rec["delta"] = (rng.uniform(-0.1, 0.1, (n, 3)) * (back % 3 == 0)[:, None]).astype(np.float32)
    empty = back % 3 == 2
    rec["aabb_min"][empty], rec["aabb_max"][empty] = np.inf, -np.inf
    # the last record carries the characters standing on the plane between x = 2.5 and 9.5, and its motion is longer than
    # any other record's, so it wins their carry (the longest delta among the platforms stood on): a record past the
    # host-array cap that certainly matters
    rec[-1] = ((4.0, -4.0, -2.0), (8.0, -2.5, 2.0), (0.25, 0.1, 0.0))
    return rec


# ---------------------------------------------------------------- 1. device records equal host records
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_device_platform_records_equal_host_records(cq, orc, scenes, order):
    """After a host update, an async update on another stream and a device update on the same stream, the device records
    of [elevator, mover, two-part entity, static entity, entity without triangles, unknown id] equal scenes.platform_record
    on the current models (float ==), deltas equal the inputs, the triangle-less and unknown ids give inert empty
    records (the unknown one with a zero delta), and the status is the number of unknown ids."""
    torch = pytest.importorskip("torch")
    parts, local = _platform_scene(scenes)
    g = cq.CollisionQuery(parts, order=A._order(cq, order))
    rng = np.random.default_rng(5)
    ids = [1, 2, 7, 8, 9, UNKNOWN_ID]
    models = {1: parts[1]["model"], 2: parts[2]["model"], 7: parts[3]["model"], 8: parts[5]["model"]}
    d_ids = torch.from_numpy(np.asarray(ids, np.uint32).view(np.int32).copy()).cuda()
    d_out = torch.zeros(len(ids) * cq.PLATFORM.itemsize, dtype=torch.uint8, device="cuda")
    d_status = torch.full((1,), -7, dtype=torch.int32, device="cuda")
    deltas = rng.uniform(-0.2, 0.2, (4, len(ids), 3)).astype(np.float32)
    d_deltas = torch.from_numpy(deltas).cuda()  # uploaded once: no synchronisation between an update and the call below
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def pose(step):
        q = scenes.quat_angle_axis(0.3 * step, (0, 1, 0))
        return {1: scenes.trs_model(T0[0] + np.float32([0, 0.08 * step, 0])),
                2: scenes.trs_model(T0[1] + np.float32([0.12 * step, 0, 0]), q),
                7: scenes.trs_model((-20 + step, 5, -20), q, (1.0, 1.5, 0.5)),
                8: scenes.trs_model((20, 4 + 0.3 * step, 20), q)}

    def check(what, phase, stream):
        g.platforms_device(d_ids.data_ptr(), d_deltas[phase].data_ptr(), len(ids), d_out.data_ptr(), d_status.data_ptr(),
                           stream.cuda_stream if stream is not None else None)
        torch.cuda.synchronize()
        got = A._host(d_out, cq.PLATFORM)
        for k, e in enumerate(ids):
            if e in local:
                want = scenes.platform_record(local[e], models[e], (0, 0, 0), deltas[phase, k])
            else:
                want = _empty_record()
                want["delta"] = deltas[phase, k] if e == 9 else 0.0
            _assert_records_equal(got[k:k + 1], want, (what, e))
        assert int(d_status.item()) == 1, what
        assert not (got["aabb_min"][4:] <= got["aabb_max"][4:]).any()  # empty boxes: inert
        return got

    torch.cuda.synchronize()
    check("creation", 0, None)
    m = pose(1)
    g.update_transforms([1, 2, 7, 8], [m[e] for e in (1, 2, 7, 8)])
    models.update(m)
    check("host update", 1, None)
    m = pose(2)
    with torch.cuda.stream(s1):
        torch.cuda._sleep(50_000_000)
    g.update_transforms_async([1, 7], [m[1], m[7]], stream=s1.cuda_stream)
    models[1], models[7] = m[1], m[7]
    check("async update on another stream", 2, s2)
    m = pose(3)
    upd = torch.from_numpy(np.asarray([2, 8], np.uint32).view(np.int32).copy()).cuda()
    d_models = torch.from_numpy(np.stack([m[2], m[8]]).astype(np.float32)).cuda()
    torch.cuda.synchronize()
    g.update_transforms_device(upd.data_ptr(), d_models.data_ptr(), 2, None, s2.cuda_stream)
    models[2], models[8] = m[2], m[8]
    check("device update on the same stream", 3, s2)
    # n == 0 queues nothing, not even the status write; a NULL status pointer is accepted
    d_status.fill_(-7)
    torch.cuda.synchronize()
    g.stats(reset=True)
    g.platforms_device(d_ids.data_ptr(), d_ids.data_ptr(), 0, d_out.data_ptr(), d_status.data_ptr())
    assert g.stats()["kernel_launches"] == 0 and int(d_status.item()) == -7
    zeros = torch.zeros(len(ids) * 3, device="cuda")
    torch.cuda.synchronize()
    g.platforms_device(d_ids.data_ptr(), zeros.data_ptr(), len(ids), d_out.data_ptr())
    torch.cuda.synchronize()
    assert (A._host(d_out, cq.PLATFORM)["delta"] == 0).all()
    g.close()


# ---------------------------------------------------------------- 2. move-and-slide parity with the host-array call
def _mas_run(cq, orc, scenes, torch, n_platforms, flags, steps=6):
    """`steps` steps of the elevator-and-mover crowd: one world steps device records A with the host-array call and B
    with the device-platform call, the oracle steps its own; returns the three after every step."""
    parts, local = _platform_scene(scenes)
    g, o = cq.CollisionQuery(parts), orc.OracleWorld(parts)
    rng = np.random.default_rng(3)
    n = 3000 if not flags & cq.MAS_AGENTS else 1200
    pos, vel, _ = _crowd(rng, n, 2.5)
    so = orc.init_states(pos, vel)
    da, db = A._dev(torch, cq.init_states(pos, vel)), A._dev(torch, cq.init_states(pos, vel))
    extra = _extra_platforms(rng, n_platforms - 2) if n_platforms > 2 else None
    so_drop = orc.init_states(pos, vel) if n_platforms > 64 else None  # the oracle without the last record
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    g3 = np.float32([0.0, -98.0, 0.0])
    L = cq.lib()
    prev = [t.copy() for t in T0]
    out = []
    for step in range(1, steps + 1):
        cur = [T0[0] + np.float32([0, 0.08 * step, 0]), T0[1] + np.float32([0.12 * step, 0, 0])]
        models = [scenes.trs_model(c) for c in cur]
        g.update_transforms([1, 2], models)
        o.update_transforms([1, 2], models)
        plats = np.concatenate([scenes.platform_record(local[1 + k], models[k], prev[k], cur[k]) for k in range(2)])
        if extra is not None:
            plats = np.concatenate([plats, extra])
        plats = np.ascontiguousarray(plats, cq.PLATFORM)
        d_plats = A._dev(torch, plats)
        torch.cuda.synchronize()
        if len(plats) <= 64:
            cq._check(L.cq_move_and_slide_device_ex(g.handle, C.c_void_p(da.data_ptr()), n, cq._ptr(params), C.c_float(1.0 / 60.0),
                                                    cq._ptr(g3), flags, cq._ptr(plats), len(plats), None))
        g.move_and_slide_device_platforms(db.data_ptr(), n, params, d_plats.data_ptr(), len(plats), flags=flags)
        o.move_and_slide(so, orc.default_params(), flags=flags, platforms=plats, order=g.order, n_threads=8)
        if so_drop is not None:
            o.move_and_slide(so_drop, orc.default_params(), flags=flags, platforms=plats[:-1], order=g.order, n_threads=8)
        torch.cuda.synchronize()
        out.append((A._host(da, cq.STATE).copy() if len(plats) <= 64 else None, A._host(db, cq.STATE).copy(), so.copy()))
        prev = cur
    g.close(), o.close()
    return out, so_drop


@pytest.mark.gpu
@pytest.mark.parametrize("agents", [False, True])
@pytest.mark.parametrize("n_platforms", [2, 64])
def test_device_platforms_move_and_slide_equals_host_array(cq, orc, scenes, n_platforms, agents):
    """6 steps with 2 and with 64 platforms, with and without CQ_MAS_AGENTS: the device-platform call equals the
    host-array call with the same records and the oracle byte for byte, and characters were carried."""
    torch = pytest.importorskip("torch")
    flags = cq.MAS_APPLY_GRAVITY | (cq.MAS_AGENTS if agents else 0)
    out, _ = _mas_run(cq, orc, scenes, torch, n_platforms, flags)
    for step, (a, b, o) in enumerate(out, 1):
        assert b.tobytes() == a.tobytes(), ("host array", step)
        assert b.tobytes() == o.tobytes(), ("oracle", step)
    assert (out[-1][1]["position"][:, 1] > 2.0).sum() > 20  # the elevator's and the mover's riders went up with them


# ---------------------------------------------------------------- 3. beyond the host-array cap
@pytest.mark.gpu
@pytest.mark.parametrize("n_platforms", [65, 1000])
def test_device_platforms_beyond_host_cap(cq, orc, scenes, n_platforms):
    """65 and 1,000 platforms (most inert, some carrying and pushing): records equal the oracle's byte for byte, while
    the host-array call still refuses more than 64."""
    torch = pytest.importorskip("torch")
    out, dropped = _mas_run(cq, orc, scenes, torch, n_platforms, cq.MAS_APPLY_GRAVITY)
    for step, (_, b, o) in enumerate(out, 1):
        assert b.tobytes() == o.tobytes(), ("oracle", step)
    assert dropped.tobytes() != out[-1][2].tobytes()  # the record past the cap carried characters
    parts, _ = _platform_scene(scenes)
    g = cq.CollisionQuery(parts)
    d = A._dev(torch, cq.init_states(np.zeros((4, 3), np.float32)))
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    g3 = np.float32([0.0, -98.0, 0.0])
    rc = cq.lib().cq_move_and_slide_device_ex(g.handle, C.c_void_p(d.data_ptr()), 4, cq._ptr(params), C.c_float(1.0 / 60.0),
                                              cq._ptr(g3), 1, cq._ptr(np.zeros(65, cq.PLATFORM)), 65, None)
    assert rc == CQ_ERR_INVALID
    g.close()


# ---------------------------------------------------------------- 4. a captured fixed step with moving platforms
def _crowd_params(cq):
    p = cq.default_params()
    p["radius"], p["half_height"] = 0.4, 0.5
    p["skin_width"], p["snap_distance"] = 0.08, 0.3
    return np.ascontiguousarray(p, cq.PARAMS)


@pytest.mark.gpu
def test_fixed_step_with_moving_platforms_graph_capture(cq, orc, scenes):
    """One uncaptured warm-up, then a torch.cuda.CUDAGraph of: device update of the platforms' models -> platforms_device
    -> move_and_slide_device_platforms (gravity, agents) -> agent_separation_device_async -> rays.  20 replays; before
    each, new models and deltas are written into the same buffers: the elevator goes up for 10 frames then down, the mover
    goes +x then back.  After every replay the records and the hits equal uncaptured synchronous steps of world A that use
    host records from scenes.platform_record, byte for byte, and the riders of the elevator followed it both ways."""
    torch = pytest.importorskip("torch")
    parts, local = _platform_scene(scenes)
    ga, gb = cq.CollisionQuery(parts), cq.CollisionQuery(parts)
    p = _crowd_params(cq)
    rng = np.random.default_rng(17)
    pos, vel, on_top = _crowd(rng, 200, 0.9)  # ~40% footprint coverage
    riders = on_top & (np.abs(pos[:, 0]) < 2)  # on the elevator
    n = len(pos)
    sa = cq.init_states(pos, vel)
    d_states = A._dev(torch, cq.init_states(pos, vel))
    lo, hi = np.float32([-8, -4, -6]), np.float32([20, 4, 6])
    rays = scenes.gen_rays(4000, lo, hi, seed=92, expand=0.0)
    d_rays = A._dev(torch, rays)
    out_r = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    ids = [1, 2]
    d_ids = torch.from_numpy(np.asarray(ids, np.uint32).view(np.int32).copy()).cuda()
    d_models = torch.zeros((2, 16), dtype=torch.float32, device="cuda")
    d_deltas = torch.zeros((2, 3), dtype=torch.float32, device="cuda")
    d_plats = torch.zeros(2 * cq.PLATFORM.itemsize, dtype=torch.uint8, device="cuda")
    d_upd, d_pst = torch.full((1,), -7, dtype=torch.int32, device="cuda"), torch.full((1,), -7, dtype=torch.int32, device="cuda")
    d_sep = torch.full((1,), -7, dtype=torch.int32, device="cuda")
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS

    def translations(frame):  # up 10 frames then down; +x 10 frames then back
        k = frame if frame <= 10 else 20 - frame
        return [T0[0] + np.float32([0, 0.08 * k, 0]), T0[1] + np.float32([0.12 * k, 0, 0])]

    def step_b(stream):
        gb.update_transforms_device(d_ids.data_ptr(), d_models.data_ptr(), 2, d_upd.data_ptr(), stream)
        gb.platforms_device(d_ids.data_ptr(), d_deltas.data_ptr(), 2, d_plats.data_ptr(), d_pst.data_ptr(), stream)
        gb.move_and_slide_device_platforms(d_states.data_ptr(), n, p, d_plats.data_ptr(), 2, flags=flags, stream=stream)
        gb.agent_separation_device_async(d_states.data_ptr(), n, p, d_status_ptr=d_sep.data_ptr(), stream=stream)
        gb.raycast_device(d_rays.data_ptr(), len(rays), out_r.data_ptr(), stream)

    def frame_inputs(frame):
        prev, cur = translations(frame - 1) if frame > 0 else translations(0), translations(frame)
        models = [scenes.trs_model(c) for c in cur]
        plats = np.concatenate([scenes.platform_record(local[1 + k], models[k], prev[k], cur[k]) for k in range(2)])
        d_models.copy_(torch.from_numpy(np.stack(models).astype(np.float32)))
        d_deltas.copy_(torch.from_numpy(np.ascontiguousarray(plats["delta"], np.float32)))
        return models, np.ascontiguousarray(plats, cq.PLATFORM)

    def step_a(models, plats):
        ga.update_transforms(ids, models)
        ga.move_and_slide(sa, p, flags=flags, platforms=plats)
        ga.agent_separation(sa, p)
        return ga.raycast(rays)

    def check(frame, want_r):
        assert int(d_upd.item()) == 0 and int(d_pst.item()) == 0 and int(d_sep.item()) == cq.SEP_STATUS_OK, frame
        assert A._host(d_states, cq.STATE).tobytes() == sa.tobytes(), frame
        assert A._host(out_r, cq.RAY_HIT).tobytes() == want_r.tobytes(), frame

    models, plats = frame_inputs(0)
    torch.cuda.synchronize()
    step_b(torch.cuda.current_stream().cuda_stream)  # warm-up: sizes every scratch block
    torch.cuda.synchronize()
    check(0, step_a(models, plats))
    graph, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=cs):
        step_b(torch.cuda.current_stream().cuda_stream)
    rider_y = [float(np.median(sa["position"][riders, 1]))]
    for frame in range(1, 21):
        models, plats = frame_inputs(frame)
        graph.replay()
        torch.cuda.synchronize()
        check(frame, step_a(models, plats))
        rider_y.append(float(np.median(A._host(d_states, cq.STATE)["position"][riders, 1])))
    assert riders.sum() >= 5
    # a graph with the records of its capture would carry the riders up on every replay
    assert rider_y[10] > rider_y[0] + 0.6 and rider_y[20] < rider_y[10] - 0.6, rider_y
    del graph
    ga.close(), gb.close()


# ---------------------------------------------------------------- 5. launch counts
@pytest.mark.gpu
@pytest.mark.parametrize("agents", [False, True])
def test_device_platforms_launch_counts(cq, orc, scenes, agents):
    """platforms_device costs one launch whatever n is; the device-platform move-and-slide costs what the host-array call
    costs."""
    torch = pytest.importorskip("torch")
    parts, _ = _platform_scene(scenes)
    g = cq.CollisionQuery(parts)
    rng = np.random.default_rng(8)
    pos, vel, _ = _crowd(rng, 500, 2.5)
    d = A._dev(torch, cq.init_states(pos, vel))
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    g3 = np.float32([0.0, -98.0, 0.0])
    flags = cq.MAS_APPLY_GRAVITY | (cq.MAS_AGENTS if agents else 0)
    plats = np.ascontiguousarray(_extra_platforms(rng, 64), cq.PLATFORM)
    d_plats = A._dev(torch, plats)
    L = cq.lib()
    costs = {}
    for n_ids in (1, 6, 5000):
        ids = np.resize(np.uint32([1, 2, 7, 8, 9, UNKNOWN_ID]), n_ids)
        d_ids = torch.from_numpy(ids.view(np.int32).copy()).cuda()
        d_deltas = torch.zeros(n_ids * 3, dtype=torch.float32, device="cuda")
        d_out = torch.zeros(n_ids * cq.PLATFORM.itemsize, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        g.stats(reset=True)
        g.platforms_device(d_ids.data_ptr(), d_deltas.data_ptr(), n_ids, d_out.data_ptr())
        costs[n_ids] = g.stats()["kernel_launches"]
    assert set(costs.values()) == {1}, costs
    for k in range(2):  # the first round also sizes the scratch
        g.stats(reset=True)
        cq._check(L.cq_move_and_slide_device_ex(g.handle, C.c_void_p(d.data_ptr()), len(pos), cq._ptr(params), C.c_float(1.0 / 60.0),
                                                cq._ptr(g3), flags, cq._ptr(plats), len(plats), None))
        host = g.stats(reset=True)["kernel_launches"]
        g.move_and_slide_device_platforms(d.data_ptr(), len(pos), params, d_plats.data_ptr(), len(plats), flags=flags)
        dev = g.stats()["kernel_launches"]
        assert dev == host >= (2 if agents else 1), (k, host, dev)
    torch.cuda.synchronize()
    g.close()
