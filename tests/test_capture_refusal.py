"""A device call refused under CUDA-graph capture because it would have to grow scratch enqueues nothing: the graph being
captured has as many nodes after the refused call as before it, and the graph still replays to the results of an
uncaptured step.  Covered: more cast lanes than any uncaptured call (node scratch), a raycast that needs a larger unit
order, move-and-slide with CQ_MAS_AGENTS on a larger crowd (agent grid) and the async agent separation on a larger crowd."""
import ctypes as C

import numpy as np
import pytest

N_RAYS = 1 << 16  # with >= 2^18 static triangles the rays are run in a unit order (make_unit_order)
N_CASTS = 500
N_CROWD = 512


def _dev(torch, arr):
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1).copy()).cuda()


def _host(t, dtype):
    return t.cpu().numpy().view(dtype)


def _captured_nodes(rt, stream):
    """Nodes of the graph a capture is recording on `stream`.  cudaStreamGetCaptureInfo_v2 is the entry point the CUDA 12
    headers call cudaStreamGetCaptureInfo (the unsuffixed symbol keeps the CUDA 11 signature)."""
    status, gid, graph = C.c_int(0), C.c_ulonglong(0), C.c_void_p()
    deps, ndeps, nodes = C.c_void_p(), C.c_size_t(0), C.c_size_t(0)
    assert rt.cudaStreamGetCaptureInfo_v2(C.c_void_p(stream), C.byref(status), C.byref(gid), C.byref(graph), C.byref(deps),
                                          C.byref(ndeps)) == 0
    assert status.value == 1  # cudaStreamCaptureStatusActive
    assert rt.cudaGraphGetNodes(graph, None, C.byref(nodes)) == 0
    return nodes.value


@pytest.mark.gpu
def test_refused_captured_calls_enqueue_nothing(cq, scenes):
    torch = pytest.importorskip("torch")
    rt = C.CDLL("libcudart.so.12")
    parts, _ = scenes.terrain_scene(cells=384, cell=1.0)  # 294,912 static triangles
    g = cq.CollisionQuery(parts)
    lo, hi = np.float32([-60, -15, -60]), np.float32([60, 20, 60])
    rays = scenes.gen_rays(2 * N_RAYS, lo, hi, seed=101, expand=0.0)
    casts = scenes.gen_casts(64 * N_CASTS, lo, hi, seed=102, radius=0.5, half_height=0.5, expand=0.0)
    rng = np.random.default_rng(103)
    xz = rng.uniform(-16, 16, (2 * N_CROWD, 2)).astype(np.float32)
    pos = np.stack([xz[:, 0], scenes.terrain_height(xz[:, 0], xz[:, 1]) + 3.0, xz[:, 1]], 1).astype(np.float32)
    vel = (rng.uniform(-6, 6, (2 * N_CROWD, 3)) * np.float32([1, 0, 1])).astype(np.float32)
    states = cq.init_states(pos, vel)
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS

    d_rays, d_casts = _dev(torch, rays), _dev(torch, casts)
    out_r = torch.zeros(2 * N_RAYS * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    out_c = torch.zeros(64 * N_CASTS * cq.CAST_HIT.itemsize, dtype=torch.uint8, device="cuda")
    d_crowd = _dev(torch, states[:N_CROWD])
    d_big = _dev(torch, states)
    d_sep = torch.full((1,), -7, dtype=torch.int32, device="cuda")

    def step(st):
        g.raycast_device(d_rays.data_ptr(), N_RAYS, out_r.data_ptr(), st)
        g.capsule_cast_device(d_casts.data_ptr(), N_CASTS, cq.CAST_BLOCKING, out_c.data_ptr(), st)
        g.move_and_slide_device(d_crowd.data_ptr(), N_CROWD, params, flags=flags, stream=st)
        g.agent_separation_device_async(d_crowd.data_ptr(), N_CROWD, params, d_status_ptr=d_sep.data_ptr(), stream=st)

    def results():
        torch.cuda.synchronize()
        return (_host(out_r, cq.RAY_HIT)[:N_RAYS].tobytes(), _host(out_c, cq.CAST_HIT)[:N_CASTS].tobytes(),
                _host(d_crowd, cq.STATE).tobytes(), int(d_sep.item()))

    # the uncaptured step sizes every scratch block and gives the results a replay must equal
    torch.cuda.synchronize()
    step(torch.cuda.current_stream().cuda_stream)
    want = results()
    assert want[3] == cq.SEP_STATUS_OK

    refused = {
        "cast lanes": lambda st: g.capsule_cast_device(d_casts.data_ptr(), 64 * N_CASTS, cq.CAST_BLOCKING, out_c.data_ptr(), st),
        "ray order": lambda st: g.raycast_device(d_rays.data_ptr(), 2 * N_RAYS, out_r.data_ptr(), st),
        "agent grid": lambda st: g.move_and_slide_device(d_big.data_ptr(), 2 * N_CROWD, params, flags=flags, stream=st),
        "separation": lambda st: g.agent_separation_device_async(d_big.data_ptr(), 2 * N_CROWD, params, stream=st),
    }
    graph, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=cs):
        st = torch.cuda.current_stream().cuda_stream
        empty = _captured_nodes(rt, st)
        step(st)
        nodes = _captured_nodes(rt, st)
        assert nodes > empty  # the count sees what a call enqueues
        for what, call in refused.items():
            with pytest.raises(cq.CQError, match="make one uncaptured call of this size first"):
                call(st)
            assert _captured_nodes(rt, st) == nodes, what

    d_crowd.copy_(_dev(torch, states[:N_CROWD]))
    out_r.zero_(), out_c.zero_(), d_sep.fill_(-7)
    torch.cuda.synchronize()
    graph.replay()
    assert results() == want
    del graph
    g.close()
