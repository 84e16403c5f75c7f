"""cq_world_rebuild: a world rebuilt in place from new parts answers every call exactly as a fresh world made from those
parts; a failed rebuild leaves it answering as before; crowds survive; launches queued before the rebuild see the old
geometry; the device entity index is rebuilt; under capture the call is refused and records nothing."""
import ctypes as C

import numpy as np
import pytest

CQ_ERR_INVALID = -1


def test_rebuild_argument_checks(cq):
    L = cq.lib()
    assert L.cq_world_rebuild(None, None, 0, None) == CQ_ERR_INVALID
    assert L.cq_world_read_ref_order(None, 2, None, None) == CQ_ERR_INVALID


def _scenes(scenes):
    p1 = scenes.mirror_scene(use_hulls=False, mirror_dynamic=True)  # ground + render mesh in the dynamic set
    p2 = scenes.semla_scene()                                         # ground + Semla, static
    lo1, hi1 = scenes.scene_aabb(p1)
    lo2, hi2 = scenes.scene_aabb(p2)
    return p1, p2, np.minimum(lo1, lo2), np.maximum(hi1, hi2)


def fingerprint(cq, scenes, g, lo, hi):
    """Every kind of answer the world gives, as bytes (info without its timing fields)."""
    rays = scenes.gen_rays(4096, lo, hi, seed=11)
    casts = scenes.gen_casts(4096, lo, hi, seed=12)
    caps = scenes.gen_capsules(2048, lo, hi, seed=13)
    pos, vel = scenes.gen_c3_characters(1024, seed=14)
    plat = np.zeros(1, cq.PLATFORM)
    plat["aabb_min"], plat["aabb_max"], plat["delta"] = (-12, -4, 0), (-8, -2, 6), (0.05, 0.0, 0.0)
    out = []
    for f in (g.raycast(rays, with_flags=True), g.capsuleCast(casts, with_flags=True),
              g.capsuleCastBlocking(casts, with_flags=True), g.capsuleOverlap(caps, with_flags=True)):
        out += [f[0].tobytes(), f[1].tobytes()]
    for m in (8, 16):
        out += [np.asarray(x).tobytes() for x in g.capsuleOverlapAll(caps, m)]
    params = cq.default_params()
    for flags in (cq.MAS_APPLY_GRAVITY, cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS):
        s = cq.init_states(pos, vel)
        g.move_and_slide(s, params, flags=flags, platforms=plat)
        g.move_and_slide(s, params, flags=flags)
        out.append(s.tobytes())
    s = cq.init_states(pos, vel)
    g.agent_separation(s, params)
    out.append(s.tobytes())
    info = g.info()
    for k in ("build_ms", "refit_ms", "ref_order_ms"):
        info.pop(k)
    out.append(repr(sorted(info.items())).encode())
    for which in (0, 1):
        out += [v.tobytes() for v in g.read_soup(which).values()]
        if g.order == cq.ORDER_REFERENCE:
            out += [v.tobytes() for v in g.read_ref_order(which)]
    out.append(g.read_models().tobytes())
    return out


def fresh(cq, parts, order):
    g = cq.CollisionQuery(parts, order=order)
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_rebuild_equals_fresh_world(cq, scenes, order):
    order = cq.ORDER_REFERENCE if order == "reference" else cq.ORDER_CANONICAL
    p1, p2, lo, hi = _scenes(scenes)
    want = {}
    for name, p in (("p1", p1), ("p2", p2)):
        f = fresh(cq, p, order)
        want[name] = fingerprint(cq, scenes, f, lo, hi)
        f.close()
    g = cq.CollisionQuery(p1, order=order)
    try:
        assert fingerprint(cq, scenes, g, lo, hi) == want["p1"]
        g.rebuild(p2)
        assert fingerprint(cq, scenes, g, lo, hi) == want["p2"]
        g.rebuild(p1)
        assert fingerprint(cq, scenes, g, lo, hi) == want["p1"]
    finally:
        g.close()


@pytest.mark.gpu
def test_failed_rebuild_leaves_the_world_unchanged(cq, scenes):
    p1, p2, lo, hi = _scenes(scenes)
    g = cq.CollisionQuery(p1)
    try:
        before = fingerprint(cq, scenes, g, lo, hi)
        bad = [dict(p) for p in p2]
        idx = np.array(bad[1]["indices"], np.uint32).copy()
        idx[7] = 10 ** 7
        bad[1]["indices"] = idx
        with pytest.raises(cq.CQError, match="part 1 index 10000000 out of range"):
            g.rebuild(bad)
        assert fingerprint(cq, scenes, g, lo, hi) == before
    finally:
        g.close()


@pytest.mark.gpu
def test_crowd_survives_rebuild(cq, scenes):
    p1, p2, _, _ = _scenes(scenes)
    pos, vel = scenes.gen_c3_characters(4096, seed=21)
    params = cq.default_params()
    g = cq.CollisionQuery(p1)
    crowd = cq.Crowd(g, cq.init_states(pos, vel))
    try:
        crowd.step(None, params)
        records = crowd.read().copy()
        g.rebuild(p2)
        assert crowd.read().tobytes() == records.tobytes()
        f = cq.CollisionQuery(p2)
        want = records.copy()
        for _ in range(3):
            crowd.step(None, params)
            f.move_and_slide(want, params)
        assert crowd.read().tobytes() == want.tobytes()
        f.close()
    finally:
        crowd.close()
        g.close()


@pytest.mark.gpu
def test_queued_device_work_sees_the_old_world(cq, scenes):
    torch = pytest.importorskip("torch")
    p1, p2, lo, hi = _scenes(scenes)
    rays = scenes.gen_rays(1 << 18, lo, hi, seed=31)
    ref = cq.CollisionQuery(p1)
    want = ref.raycast(rays)
    ref.close()
    g = cq.CollisionQuery(p1)
    try:
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_out = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
        s = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(50_000_000)  # keeps the raycast queued while the rebuild runs on the host
            g.raycast_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), s.cuda_stream)
        g.rebuild(p2)
        s.synchronize()
        assert d_out.cpu().numpy().view(cq.RAY_HIT).tobytes() == want.tobytes()
    finally:
        g.close()


@pytest.mark.gpu
def test_device_update_after_rebuild_uses_the_new_entities(cq, scenes):
    torch = pytest.importorskip("torch")
    p1, p2, _, _ = _scenes(scenes)
    p1 = [dict(p, entity_id=100 + k) for k, p in enumerate(p1)]  # ids 100.. only in P1
    p2 = [dict(p, entity_id=200 + k) for k, p in enumerate(p2)]  # ids 200.. only in P2
    g = cq.CollisionQuery(p1)
    f = cq.CollisionQuery(p2)
    try:
        g.rebuild(p2)
        moved = np.array(p2[1]["model"], np.float32).reshape(16).copy()
        moved[13] += 0.5
        models = torch.from_numpy(np.stack([moved, moved]).astype(np.float32)).cuda()
        status = torch.zeros(1, dtype=torch.int32, device="cuda")

        def soups_equal():
            return all(all(a[k].tobytes() == b[k].tobytes() for k in a)
                       for a, b in ((g.read_soup(w), f.read_soup(w)) for w in (0, 1)))

        # an update naming an id only P1 had is refused as a whole (unknown ids make the update change nothing)
        ids = torch.tensor(np.array([201, 101], np.uint32).view(np.int32)).cuda()
        g.update_transforms_device(ids.data_ptr(), models.data_ptr(), 2, status.data_ptr())
        torch.cuda.synchronize()
        assert int(status.item()) == 1
        assert soups_equal()
        # an id of P2 resolves to P2's part
        ids = torch.tensor(np.array([201], np.uint32).view(np.int32)).cuda()
        status.zero_()
        g.update_transforms_device(ids.data_ptr(), models.data_ptr(), 1, status.data_ptr())
        torch.cuda.synchronize()
        assert int(status.item()) == 0
        f.update_transforms(np.array([201], np.uint32), moved.reshape(1, 16))
        assert soups_equal()
    finally:
        g.close()
        f.close()


@pytest.mark.gpu
def test_rebuild_under_capture_is_refused(cq, scenes):
    torch = pytest.importorskip("torch")
    rt = C.CDLL("libcudart.so.12")
    p1, p2, lo, hi = _scenes(scenes)
    rays = scenes.gen_rays(4096, lo, hi, seed=41)
    g = cq.CollisionQuery(p1)
    try:
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_out = torch.empty(len(rays) * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
        cs = torch.cuda.Stream()
        g.raycast_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), cs.cuda_stream)  # sizes scratch, meets cs
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=cs):
            st = torch.cuda.current_stream().cuda_stream
            g.raycast_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), st)
            status, gid, gr = C.c_int(0), C.c_ulonglong(0), C.c_void_p()
            deps, ndeps, before, after = C.c_void_p(), C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
            assert rt.cudaStreamGetCaptureInfo_v2(C.c_void_p(st), C.byref(status), C.byref(gid), C.byref(gr), C.byref(deps),
                                                  C.byref(ndeps)) == 0
            assert rt.cudaGraphGetNodes(gr, None, C.byref(before)) == 0
            with pytest.raises(cq.CQError, match="cq_world_rebuild cannot be captured"):
                g.rebuild(p2)
            assert rt.cudaGraphGetNodes(gr, None, C.byref(after)) == 0
            assert after.value == before.value
        d_out.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().view(cq.RAY_HIT).tobytes() == g.raycast(rays).tobytes()
    finally:
        g.close()
