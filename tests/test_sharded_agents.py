"""A CQ_MAS_AGENTS crowd moved in slices: cq_agent_snapshot_device writes every slice's snapshot records into its range of
one crowd-wide array, and cq_move_and_slide_device_agents moves one slice against the whole array.  Every slice
snapshotted, then each moved, must give the records of one whole-crowd CQ_MAS_AGENTS call byte for byte (and so the
oracle's), on one GPU in any number of slices, inside a CUDA graph, through a process-per-GPU group and through
cq_multi_move_and_slide_batch_ex on every visible GPU."""
import ctypes as C
import importlib.util
import os
import subprocess

import numpy as np
import pytest

_spec = importlib.util.spec_from_file_location("_device_platform_helpers",
                                               os.path.join(os.path.dirname(__file__), "test_device_platforms.py"))
DP = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(DP)
A = DP.A  # device-buffer helpers (_dev, _host, _order)
_spec = importlib.util.spec_from_file_location("_capture_refusal_helpers",
                                               os.path.join(os.path.dirname(__file__), "test_capture_refusal.py"))
CR = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(CR)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CQ_OK, CQ_ERR_INVALID = 0, -1
STATE_BYTES, SNAP_BYTES = 168, 32
LAUNCHES_SNAPSHOT = 1  # include/cq.h
LAUNCHES_AGENTS, LAUNCHES_UNIT_ORDER = 14, 7


# ---------------------------------------------------------------- CPU: argument checks and the C++ mirror
def test_sharded_agents_argument_checks(cq):
    """Every refusal comes before any CUDA call, so a fake (never dereferenced) world pointer answers without a GPU; so
    does n == 0, which queues nothing."""
    L = cq.lib()
    p = C.c_void_p(16)
    g = cq._ptr(np.zeros(3, np.float32))
    dt = C.c_float(1.0 / 60.0)
    snap = lambda w, st, n, out, grav=g: L.cq_agent_snapshot_device(w, st, n, dt, grav, 3, out, None)
    assert snap(None, p, 4, p) == CQ_ERR_INVALID
    assert snap(p, p, -1, p) == CQ_ERR_INVALID
    assert snap(p, None, 4, p) == CQ_ERR_INVALID
    assert snap(p, p, 4, None) == CQ_ERR_INVALID
    assert snap(p, p, 4, p, None) == CQ_ERR_INVALID
    assert snap(p, p, 4, C.c_void_p(24)) == CQ_ERR_INVALID  # read as float4 pairs: 16-byte alignment
    assert snap(p, None, 0, None) == CQ_OK

    def mas(w=p, st=p, n=4, agents=p, n_agents=8, first=2, params=p, grav=g, flags=3, plat=None, n_plat=0):
        return L.cq_move_and_slide_device_agents(w, st, n, agents, n_agents, first, params, dt, grav, flags, plat, n_plat, None)

    assert mas(w=None) == CQ_ERR_INVALID
    assert mas(flags=1) == CQ_ERR_INVALID  # without CQ_MAS_AGENTS
    assert mas(n=-1) == CQ_ERR_INVALID
    assert mas(n_agents=-1, n=0, first=0) == CQ_ERR_INVALID
    assert mas(first=-1) == CQ_ERR_INVALID
    assert mas(first=5) == CQ_ERR_INVALID  # 5 + 4 > 8
    assert mas(first=2 ** 31 - 1, n=2, n_agents=2 ** 31 - 1) == CQ_ERR_INVALID  # the sum is taken in 64 bits
    assert mas(st=None) == CQ_ERR_INVALID
    assert mas(agents=None) == CQ_ERR_INVALID
    assert mas(agents=C.c_void_p(40)) == CQ_ERR_INVALID
    assert mas(params=None) == CQ_ERR_INVALID
    assert mas(grav=None) == CQ_ERR_INVALID
    assert mas(n_plat=-1) == CQ_ERR_INVALID
    assert mas(n_plat=3) == CQ_ERR_INVALID  # NULL platforms
    assert "cq_move_and_slide_device_agents" in L.cq_last_error().decode()
    assert mas(n=0, st=None, first=8) == CQ_OK
    assert mas(n=0, st=None, agents=None, n_agents=0, first=0) == CQ_OK

    multi = lambda mw=p, st=p, n=4, params=p, grav=g, plat=None, n_plat=0: L.cq_multi_move_and_slide_batch_ex(
        mw, st, n, params, dt, grav, 3, plat, n_plat)
    assert multi(mw=None) == CQ_ERR_INVALID
    assert multi(n=-1) == CQ_ERR_INVALID
    assert multi(st=None) == CQ_ERR_INVALID
    assert multi(params=None) == CQ_ERR_INVALID
    assert multi(grav=None) == CQ_ERR_INVALID
    assert multi(plat=p, n_plat=65) == CQ_ERR_INVALID
    assert multi(n_plat=2) == CQ_ERR_INVALID
    assert multi(n_plat=-1) == CQ_ERR_INVALID
    for s in ("cq_agent_snapshot_device", "cq_move_and_slide_device_agents", "cq_multi_move_and_slide_batch_ex"):
        assert s in cq.EXPORTS
    assert cq.AGENT_SNAPSHOT.itemsize == SNAP_BYTES


CPP_PROBE = r"""
// The C++ mirror hands the sliced-crowd calls' arguments to the library unchanged.  The world and the calls are stubbed
// here (these definitions take precedence over libcq.so's), so no GPU is needed.
#include <cstdio>
#include "CollisionQuery.hpp"

static int seen = 0;
static const void *seenStates = nullptr, *seenSnap = nullptr, *seenPlat = nullptr;
static int32_t seenN = 0, seenAgents = 0, seenFirst = 0, seenNPlat = 0;
static uint32_t seenFlags = 0;
static void *seenStream = nullptr;
extern "C" int cq_world_create_ex(const cq_mesh_part *, int32_t, const cq_world_options *, cq_world **out) {
    static int dummy;
    *out = reinterpret_cast<cq_world *>(&dummy);
    return CQ_OK;
}
extern "C" void cq_world_destroy(cq_world *) {}
extern "C" int cq_agent_snapshot_device(cq_world *, const cq_character_state *s, int32_t n, float, const float *, uint32_t flags,
                                        cq_agent_snapshot *out, void *stream) {
    seen = 1, seenStates = s, seenN = n, seenFlags = flags, seenSnap = out, seenStream = stream;
    return CQ_OK;
}
extern "C" int cq_move_and_slide_device_agents(cq_world *, cq_character_state *s, int32_t n, const cq_agent_snapshot *a,
                                               int32_t nAgents, int32_t first, const cq_controller_params *, float, const float *,
                                               uint32_t flags, const cq_platform *pl, int32_t nPl, void *stream) {
    seen = 2, seenStates = s, seenN = n, seenSnap = a, seenAgents = nAgents, seenFirst = first, seenFlags = flags, seenPlat = pl;
    seenNPlat = nPl, seenStream = stream;
    return CQ_OK;
}

int main() {
    cqhost::CollisionQuery q(std::vector<cq_mesh_part>{});
    static cq_character_state s[8];
    static cq_agent_snapshot snap[20];
    static cq_platform pl[3];
    const float g[3] = {0, -98, 0};
    if (!q.agentSnapshotDevice(s, 8, 1.0f / 60.0f, g, snap + 4, true, (void *)0x30) || seen != 1 || seenStates != s || seenN != 8 ||
        seenSnap != snap + 4 || seenFlags != (CQ_MAS_APPLY_GRAVITY | CQ_MAS_AGENTS) || seenStream != (void *)0x30)
        return 1;
    static cq_controller_params p{};
    if (!q.moveAndSlideAgents(s, 8, snap, 20, 4, p, 1.0f / 60.0f, g, cqhost::DevicePlatforms{pl, 3}, false, (void *)0x40) ||
        seen != 2 || seenStates != s || seenN != 8 || seenSnap != snap || seenAgents != 20 || seenFirst != 4 || seenPlat != pl ||
        seenNPlat != 3 || seenFlags != CQ_MAS_AGENTS || seenStream != (void *)0x40)
        return 2;
    if (!q.moveAndSlideAgents(s, 8, snap, 20, 12, p, 1.0f / 60.0f, g) || seenPlat != nullptr || seenNPlat != 0 ||
        seenFlags != (CQ_MAS_APPLY_GRAVITY | CQ_MAS_AGENTS))
        return 3;
    std::printf("ok\n");
    return 0;
}
"""


def test_cpp_wrapper_sharded_agents(cq, tmp_path):
    cq.build()
    src = tmp_path / "sharded_agents_probe.cpp"
    src.write_text(CPP_PROBE)
    exe = tmp_path / "sharded_agents_probe"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "swift-game-engine_b200", "cpp"),
                        str(src), "-L" + cq.CSRC, "-lcq", "-Wl,-rpath," + cq.CSRC, "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stdout, r.stderr)


# ---------------------------------------------------------------- scenes
def _crowd_params(cq):
    p = cq.default_params()
    p["radius"], p["half_height"] = 0.4, 0.5
    p["skin_width"], p["snap_distance"] = 0.08, 0.3
    return np.ascontiguousarray(p, cq.PARAMS)


def _walkers(scenes, n=3000, seed=11):
    """The crowd of test_agents_capsule_capsule_ccd: n walkers at ~35% footprint coverage on a terrain."""
    parts, half_world = scenes.terrain_scene(cells=96, cell=1.5, seed=5)
    rng = np.random.default_rng(seed)
    half = min(np.sqrt(n * np.pi * 0.4 ** 2 / 0.35) / 2, half_world - 4.0)
    x, z = rng.uniform(-half, half, n), rng.uniform(-half, half, n)
    y = scenes.terrain_height(x, z, 5) + np.float32(0.9 + 0.05) + rng.uniform(0, 0.3, n)
    pos = np.stack([x, y, z], axis=1).astype(np.float32)
    ang = rng.uniform(0, 2 * np.pi, n)
    walk = (np.stack([np.cos(ang), np.zeros(n), np.sin(ang)], axis=1) * rng.uniform(2, 9, (n, 1))).astype(np.float32)
    return parts, pos, walk


def _carried(scenes, m=1500, seed=12):
    """Walkers on a plane, many carried several grid cells away by one large platform (the kernel's fallback search)."""
    fv, fi = scenes.plane_mesh(80.0)
    parts = [scenes.part(fv, fi, scenes.trs_model((0, -3, 0)), entity_id=0)]
    rng = np.random.default_rng(seed)
    pos = np.stack([rng.uniform(-16, 16, m), np.full(m, -3.0 + 0.9 + 0.05), rng.uniform(-16, 16, m)], axis=1).astype(np.float32)
    ang = rng.uniform(0, 2 * np.pi, m)
    walk = (np.stack([np.cos(ang), np.zeros(m), np.sin(ang)], axis=1) * rng.uniform(2, 9, (m, 1))).astype(np.float32)
    plat = np.zeros(1, [("aabb_min", "<f4", 3), ("aabb_max", "<f4", 3), ("delta", "<f4", 3)])
    plat["aabb_min"], plat["aabb_max"], plat["delta"] = (-6, -4, -6), (6, -3, 6), (3.0, 0.0, 0.7)
    return parts, pos, walk, plat


def _cuts(n, k, seed):
    """k ragged slices of [0, n); for k > 1 one of them is empty."""
    if k == 1:
        return [0, n]
    if k == 2:
        return [0, n, n]
    rng = np.random.default_rng(seed)
    inner = sorted(rng.choice(np.arange(1, n), k - 2, replace=False).tolist())
    inner.insert(rng.integers(0, len(inner) + 1), inner[0])
    cuts = [0] + sorted(inner) + [n]
    assert len(cuts) == k + 1 and any(a == b for a, b in zip(cuts, cuts[1:]))
    return cuts


def _sliced_step(g, d_states, d_snap, n, cuts, params, flags, d_plats=None, n_plats=0, stream=None, reverse=False):
    """Snapshot every slice, then move every slice (in reverse order when asked: the order must not matter)."""
    sl = list(zip(cuts, cuts[1:]))
    for lo, hi in sl:
        g.agent_snapshot_device(d_states.data_ptr() + lo * STATE_BYTES, hi - lo, d_snap.data_ptr() + lo * SNAP_BYTES,
                                flags=flags, stream=stream)
    for lo, hi in (sl[::-1] if reverse else sl):
        g.move_and_slide_device_agents(d_states.data_ptr() + lo * STATE_BYTES, hi - lo, d_snap.data_ptr(), n, lo, params,
                                       flags=flags, d_platforms_ptr=d_plats.data_ptr() if d_plats is not None else None,
                                       n_platforms=n_plats, stream=stream)


_ORACLE = {}


def _oracle_walkers(cq, orc, scenes, order, steps=8):
    """The oracle's records after every step of the walkers, walk intent re-applied, and how many moves an agent hit
    decided (computed once per world order)."""
    if order in _ORACLE:
        return _ORACLE[order]
    parts, pos, walk = _walkers(scenes)
    o = orc.OracleWorld(parts)
    p = _crowd_params(cq)
    so = orc.init_states(pos, walk)
    out, agent_hits = [], 0
    for _ in range(steps):
        ghost = so.copy()
        o.move_and_slide(so, p, flags=3, order=A._order(cq, order), n_threads=8)
        o.move_and_slide(ghost, p, flags=1, order=A._order(cq, order), n_threads=8)
        agent_hits += int((ghost["position"] != so["position"]).any(axis=1).sum())
        out.append(so.copy())
        so["velocity"][:, 0], so["velocity"][:, 2] = walk[:, 0], walk[:, 2]
    o.close()
    _ORACLE[order] = (out, agent_hits)
    return _ORACLE[order]


# ---------------------------------------------------------------- GPU: slices on one device
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3, 7])
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_slices_equal_whole_crowd_call(cq, orc, scenes, order, k):
    """The walkers (3,000 at 35% coverage, 8 steps, walk intent re-applied) and the platform-carried crowd, split into k
    ragged slices (one empty for k > 1): after every step the records equal the whole-crowd CQ_MAS_AGENTS call and the
    oracle byte for byte, and agent hits decided at least a quarter of the moves."""
    torch = pytest.importorskip("torch")
    parts, pos, walk = _walkers(scenes)
    n = len(pos)
    g = cq.CollisionQuery(parts, order=A._order(cq, order))
    p = _crowd_params(cq)
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS
    want, agent_hits = _oracle_walkers(cq, orc, scenes, order)
    assert agent_hits > n // 4
    cuts = _cuts(n, k, seed=100 + k)
    d_s, d_w = A._dev(torch, cq.init_states(pos, walk)), A._dev(torch, cq.init_states(pos, walk))
    d_snap = torch.zeros(n * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    for step in range(len(want)):
        torch.cuda.synchronize()
        _sliced_step(g, d_s, d_snap, n, cuts, p, flags, reverse=step % 2 == 1)
        g.move_and_slide_device_platforms(d_w.data_ptr(), n, p, None, 0, flags=flags)
        torch.cuda.synchronize()
        got, whole = A._host(d_s, cq.STATE).copy(), A._host(d_w, cq.STATE).copy()
        assert got.tobytes() == whole.tobytes(), ("whole-crowd call", step)
        assert got.tobytes() == want[step].tobytes(), ("oracle", step)
        for s in (got, whole):
            s["velocity"][:, 0], s["velocity"][:, 2] = walk[:, 0], walk[:, 2]
        d_s.copy_(A._dev(torch, got)), d_w.copy_(A._dev(torch, whole))
    g.close()
    # carried far from their snapshot cells by a platform read from device memory
    parts, fpos, fwalk, plat = _carried(scenes)
    m = len(fpos)
    g2, o2 = cq.CollisionQuery(parts, order=A._order(cq, order)), orc.OracleWorld(parts)
    plat = np.ascontiguousarray(plat, cq.PLATFORM)
    d_plat = A._dev(torch, plat)
    cuts = _cuts(m, k, seed=200 + k)
    d_s, d_w = A._dev(torch, cq.init_states(fpos, fwalk)), A._dev(torch, cq.init_states(fpos, fwalk))
    d_snap = torch.zeros(m * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    so = orc.init_states(fpos, fwalk)
    for step in range(3):
        torch.cuda.synchronize()
        _sliced_step(g2, d_s, d_snap, m, cuts, p, flags, d_plat, 1)
        g2.move_and_slide_device_platforms(d_w.data_ptr(), m, p, d_plat.data_ptr(), 1, flags=flags)
        o2.move_and_slide(so, p, flags=3, platforms=plat, order=g2.order, n_threads=8)
        torch.cuda.synchronize()
        got = A._host(d_s, cq.STATE)
        assert got.tobytes() == A._host(d_w, cq.STATE).tobytes(), ("whole-crowd call, carried", step)
        assert got.tobytes() == so.tobytes(), ("oracle, carried", step)
    assert (np.abs(A._host(d_s, cq.STATE)["position"][:, 0] - fpos[:, 0]) > 2.5).sum() > 50
    g2.close(), o2.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_platforms", [2, 100])
def test_slices_with_device_platforms(cq, orc, scenes, n_platforms):
    """The elevator-and-mover scene of the device-platform tests with 2 and with 100 platform records (beyond the 64 of
    the host-array calls), 1,200 agents in 3 slices: equal to the whole-crowd call and to the oracle after every step."""
    torch = pytest.importorskip("torch")
    parts, local = DP._platform_scene(scenes)
    g, o = cq.CollisionQuery(parts), orc.OracleWorld(parts)
    rng = np.random.default_rng(3)
    n = 1200
    pos, vel, _ = DP._crowd(rng, n, 2.5)
    extra = DP._extra_platforms(rng, n_platforms - 2) if n_platforms > 2 else np.zeros(0, cq.PLATFORM)
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS
    d_s, d_w = A._dev(torch, cq.init_states(pos, vel)), A._dev(torch, cq.init_states(pos, vel))
    d_snap = torch.zeros(n * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    so = orc.init_states(pos, vel)
    cuts = [0, 517, 518, n]
    prev = [t.copy() for t in DP.T0]
    for step in range(1, 6):
        cur = [DP.T0[0] + np.float32([0, 0.08 * step, 0]), DP.T0[1] + np.float32([0.12 * step, 0, 0])]
        models = [scenes.trs_model(c) for c in cur]
        g.update_transforms([1, 2], models)
        o.update_transforms([1, 2], models)
        plats = [scenes.platform_record(local[1 + k], models[k], prev[k], cur[k]) for k in range(2)]
        plats = np.ascontiguousarray(np.concatenate([np.ascontiguousarray(r, cq.PLATFORM) for r in plats] + [extra]), cq.PLATFORM)
        d_plats = A._dev(torch, plats)
        torch.cuda.synchronize()
        _sliced_step(g, d_s, d_snap, n, cuts, params, flags, d_plats, len(plats))
        g.move_and_slide_device_platforms(d_w.data_ptr(), n, params, d_plats.data_ptr(), len(plats), flags=flags)
        o.move_and_slide(so, orc.default_params(), flags=flags, platforms=plats, order=g.order, n_threads=8)
        torch.cuda.synchronize()
        got = A._host(d_s, cq.STATE)
        assert got.tobytes() == A._host(d_w, cq.STATE).tobytes(), ("whole-crowd call", step)
        assert got.tobytes() == so.tobytes(), ("oracle", step)
        prev = cur
    assert (A._host(d_s, cq.STATE)["position"][:, 1] > 2.0).sum() > 20  # riders went up with the elevator
    g.close(), o.close()


@pytest.mark.gpu
def test_sliced_step_graph_capture(cq, scenes):
    """A torch.cuda.CUDAGraph of one sliced step (snapshots of 3 slices, then their moves) replayed 10 times equals
    uncaptured whole-crowd steps byte for byte; a sliced move of a larger crowd than any uncaptured call is refused
    under capture and adds no node to the graph."""
    torch = pytest.importorskip("torch")
    rt = C.CDLL("libcudart.so.12")
    parts, pos, walk = _walkers(scenes, n=1000, seed=21)
    big_parts, big_pos, big_walk = _walkers(scenes, n=2000, seed=22)
    n, nb = len(pos), len(big_pos)
    g = cq.CollisionQuery(parts)
    p = _crowd_params(cq)
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS
    cuts = [0, 333, 334, n]
    d_s, d_w = A._dev(torch, cq.init_states(pos, walk)), A._dev(torch, cq.init_states(pos, walk))
    d_snap = torch.zeros(n * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    d_big = A._dev(torch, cq.init_states(big_pos, big_walk))
    d_big_snap = torch.zeros(nb * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _sliced_step(g, d_s, d_snap, n, cuts, p, flags, stream=torch.cuda.current_stream().cuda_stream)  # sizes the scratch
    g.move_and_slide_device_platforms(d_w.data_ptr(), n, p, None, 0, flags=flags)
    torch.cuda.synchronize()
    assert A._host(d_s, cq.STATE).tobytes() == A._host(d_w, cq.STATE).tobytes()
    graph, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=cs):
        st = torch.cuda.current_stream().cuda_stream
        _sliced_step(g, d_s, d_snap, n, cuts, p, flags, stream=st)
        nodes = CR._captured_nodes(rt, st)
        with pytest.raises(cq.CQError, match="make one uncaptured call of this size first"):
            g.move_and_slide_device_agents(d_big.data_ptr(), nb, d_big_snap.data_ptr(), nb, 0, p, flags=flags, stream=st)
        assert CR._captured_nodes(rt, st) == nodes
    d_s.copy_(d_w)
    for replay in range(10):
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()  # the replay and the world's own stream share the agent-grid scratch
        g.move_and_slide_device_platforms(d_w.data_ptr(), n, p, None, 0, flags=flags)
        torch.cuda.synchronize()
        assert A._host(d_s, cq.STATE).tobytes() == A._host(d_w, cq.STATE).tobytes(), replay
    del graph
    g.close()


@pytest.mark.gpu
def test_multi_world_agents_on_the_visible_gpus(cq, scenes):
    """cq_multi_move_and_slide_batch_ex on every visible GPU (one is enough): a prime crowd (ragged shards), 3 steps with
    agents, then 3 without agents but with a platform: byte-equal to the single-GPU call."""
    import torch
    n_gpus = torch.cuda.device_count()
    parts, pos, walk = _walkers(scenes, n=3001, seed=31)
    group = cq.Group.local(n_gpus)
    mw, g = cq.MultiWorld(group, parts), cq.CollisionQuery(parts)
    p = _crowd_params(cq)
    a, b = cq.init_states(pos, walk), cq.init_states(pos, walk)
    for step in range(3):
        mw.move_and_slide_ex(a, p, flags=cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS)
        g.move_and_slide(b, p, flags=cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS)
        assert a.tobytes() == b.tobytes(), step
    mw.close(), g.close()
    parts, fpos, fwalk, plat = _carried(scenes, m=1009)
    mw, g = cq.MultiWorld(group, parts), cq.CollisionQuery(parts)
    plat = np.ascontiguousarray(plat, cq.PLATFORM)
    for flags in (cq.MAS_APPLY_GRAVITY, cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS):
        a, b = cq.init_states(fpos, fwalk), cq.init_states(fpos, fwalk)
        for step in range(3):
            mw.move_and_slide_ex(a, p, flags=flags, platforms=plat)
            g.move_and_slide(b, p, flags=flags, platforms=plat)
            assert a.tobytes() == b.tobytes(), (flags, step)
    with pytest.raises(cq.CQError):  # the call without platforms still refuses agents
        mw.move_and_slide(a, p, flags=cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS)
    mw.close(), g.close()
    group.close()


@pytest.mark.gpu
def test_rank_group_flow(cq, scenes):
    """The process-per-GPU flow with a group of one rank: snapshot the rank's shard, cq_group_gather_records of the
    32-byte records, move the shard against the gathered snapshot; equal to the whole-crowd call."""
    import torch
    torch.cuda.set_device(0)
    parts, pos, walk = _walkers(scenes, n=2003, seed=41)
    n = len(pos)
    g = cq.CollisionQuery(parts)
    p = _crowd_params(cq)
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS
    rg = cq.Group.rank(1, 0, cq.Group.unique_id())
    lo, hi = cq.shard_range(n, rg.size, 0)
    d_s, d_w = A._dev(torch, cq.init_states(pos, walk)), A._dev(torch, cq.init_states(pos, walk))
    d_local = torch.zeros((hi - lo) * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    d_all = torch.zeros(n * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    for step in range(3):
        g.agent_snapshot_device(d_s.data_ptr() + lo * STATE_BYTES, hi - lo, d_local.data_ptr(), flags=flags, stream=st.cuda_stream)
        rg.gather_records(d_local.data_ptr(), n, SNAP_BYTES, d_all.data_ptr(), st.cuda_stream)
        g.move_and_slide_device_agents(d_s.data_ptr() + lo * STATE_BYTES, hi - lo, d_all.data_ptr(), n, lo, p, flags=flags,
                                       stream=st.cuda_stream)
        st.synchronize()
        g.move_and_slide_device_platforms(d_w.data_ptr(), n, p, None, 0, flags=flags)
        torch.cuda.synchronize()
        assert A._host(d_s, cq.STATE).tobytes() == A._host(d_w, cq.STATE).tobytes(), step
    rg.close()
    g.close()


@pytest.mark.gpu
def test_sharded_agents_launch_counts(cq, scenes):
    """What include/cq.h states: a snapshot is one launch; a sliced move is 14 launches, plus 7 for the processing order
    when the slice has >= 65,536 characters on a world of >= 262,144 static triangles, whatever the crowd's size, the
    same as the whole-crowd call on that many characters."""
    torch = pytest.importorskip("torch")
    parts, _ = scenes.terrain_scene(cells=384, cell=1.0)  # 294,912 static triangles
    g = cq.CollisionQuery(parts)
    rng = np.random.default_rng(51)
    n = 70000
    xz = rng.uniform(-150, 150, (n, 2)).astype(np.float32)
    pos = np.stack([xz[:, 0], scenes.terrain_height(xz[:, 0], xz[:, 1]) + 1.2, xz[:, 1]], 1).astype(np.float32)
    vel = (rng.uniform(-4, 4, (n, 3)) * np.float32([1, 0, 1])).astype(np.float32)
    p = _crowd_params(cq)
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS
    d_s = A._dev(torch, cq.init_states(pos, vel))
    d_snap = torch.zeros(n * SNAP_BYTES, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for rnd in range(2):  # the first round also sizes the scratch
        g.stats(reset=True)
        g.agent_snapshot_device(d_s.data_ptr(), n, d_snap.data_ptr(), flags=flags)
        assert g.stats(reset=True)["kernel_launches"] == LAUNCHES_SNAPSHOT
        for lo, cnt, want in ((0, 1000, LAUNCHES_AGENTS), (1000, 66000, LAUNCHES_AGENTS + LAUNCHES_UNIT_ORDER),
                              (n - 1, 1, LAUNCHES_AGENTS)):
            g.move_and_slide_device_agents(d_s.data_ptr() + lo * STATE_BYTES, cnt, d_snap.data_ptr(), n, lo, p, flags=flags)
            assert g.stats(reset=True)["kernel_launches"] == want, (rnd, lo, cnt)
        g.move_and_slide_device_agents(d_s.data_ptr(), 0, d_snap.data_ptr(), n, n, p, flags=flags)
        g.agent_snapshot_device(d_s.data_ptr(), 0, d_snap.data_ptr(), flags=flags)
        assert g.stats(reset=True)["kernel_launches"] == 0
        for cnt, want in ((1000, LAUNCHES_AGENTS), (66000, LAUNCHES_AGENTS + LAUNCHES_UNIT_ORDER)):
            g.move_and_slide_device_platforms(d_s.data_ptr(), cnt, p, None, 0, flags=flags)
            assert g.stats(reset=True)["kernel_launches"] == want, ("whole-crowd call", cnt)
    torch.cuda.synchronize()
    g.close()
