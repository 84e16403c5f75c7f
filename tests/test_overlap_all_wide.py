"""capsuleOverlapAll with maxHits above eight (CollisionQuery.swift:148-157 accepts any maxHits): the wide path of
cq_capsule_overlap_all_* (a heap of winners in the caller's output slots, a sort pass and an emit pass) against the CPU
oracle, against the eight-hit kernel, under CUDA-graph capture, in both counting modes and through the chunked host call.
The C++ wrapper's pass-through of maxHits is checked without a GPU."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("triangle_index", "depth", "position", "normal", "triangle_normal")
WIDE_LAUNCHES = 3  # include/cq.h: pool kernel, sort, emit


def _caller_order(hits, counts):
    """What every caller of capsuleOverlapAll in the reference does with the result (Systems.swift:759): a stable sort by
    depth, deepest first.  The oracle's C wrapper emits that order; in reference order the library returns the hits the
    way the reference itself returns them — in visiting order — so the comparison sorts the library's rows the same way."""
    depth = np.where(np.arange(hits.shape[1])[None, :] < counts[:, None], hits["depth"], -np.inf)
    idx = np.argsort(-depth, axis=1, kind="stable")
    return np.take_along_axis(hits, idx, axis=1)


def _check_vs_oracle(g, o, orc, c, max_hits):
    got, gcnt, gov = g.capsuleOverlapAll(c, max_hits)
    ref, rcnt, rov = o.capsule_overlap_all(c, max_hits, g.order)
    assert got.shape == (len(c), max_hits)
    assert np.array_equal(gcnt, rcnt) and np.array_equal(gov, rov)
    nil = np.arange(max_hits)[None, :] >= gcnt[:, None]
    assert (got["triangle_index"][nil] == -1).all() and (got["depth"][nil] == 0).all()
    if g.order == orc.ORDER_REFERENCE:
        got = _caller_order(got, gcnt)
    for f in FIELDS:
        assert np.array_equal(got[f], ref[f]), (max_hits, f)
    return gcnt, gov


def _capsules(name, parts, scenes, seed=8):
    lo, hi = scenes.scene_aabb(parts[1:])
    return scenes.gen_capsules(6000 if name == "hulls" else 600, lo, hi, seed=seed)


@pytest.fixture(scope="module", params=["hulls-reference", "hulls-canonical", "render-reference", "render-canonical"])
def world(request, cq, orc, scenes):
    name, order = request.param.split("-")
    parts = scenes.mirror_scene(use_hulls=name == "hulls")
    g = cq.CollisionQuery(parts, order=cq.ORDER_REFERENCE if order == "reference" else cq.ORDER_CANONICAL)
    o = orc.OracleWorld(parts)
    yield name, parts, g, o
    g.close()
    o.close()


@pytest.mark.gpu
def test_wide_bit_exact_vs_oracle(world, scenes, orc):
    name, parts, g, o = world
    c = _capsules(name, parts, scenes)
    shares = {}
    for max_hits in (9, 16, 64, 257):
        gcnt, gov = _check_vs_oracle(g, o, orc, c, max_hits)
        shares[max_hits] = float(gov.mean())
        assert (gcnt > 0).sum() > len(c) // 20
    if name == "render":  # the kept list really overflows, and really holds more than the eight-hit kernel could
        assert shares[9] > 0.2 and shares[16] > 0.2, shares
        assert shares[257] < 1.0, shares


@pytest.mark.gpu
def test_wide_prefix_equals_eight_hit_kernel(world, scenes):
    """Both results are sorted lists of the same order rule, so the first eight rows of a wide call are the eight-hit call."""
    name, parts, g, o = world
    c = _capsules(name, parts, scenes, seed=9)
    narrow, ncnt, nov = g.capsuleOverlapAll(c, 8)
    for max_hits in (9, 40):
        wide, wcnt, _ = g.capsuleOverlapAll(c, max_hits)
        assert np.array_equal(np.minimum(wcnt, 8), ncnt)
        assert np.array_equal(nov, (wcnt > 8).astype(np.uint8))
        assert wide[:, :8].tobytes() == narrow.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["reference", "canonical"])
def test_wide_static_and_dynamic_sets(cq, orc, scenes, order):
    """Render mirror in the dynamic set over the static ground: in reference order the static set is visited first, so a
    kept list longer than a query's static overlaps runs on into the dynamic set."""
    parts = scenes.mirror_scene(use_hulls=False, mirror_dynamic=True)
    g = cq.CollisionQuery(parts, order=cq.ORDER_REFERENCE if order == "reference" else cq.ORDER_CANONICAL)
    o = orc.OracleWorld(parts)
    try:
        n_static = g.info()["n_static_triangles"]
        assert n_static > 0 and g.info()["n_dynamic_triangles"] > 0
        lo, hi = scenes.scene_aabb(parts[1:])
        lo = lo.copy()
        lo[1] = -2.0  # reach down to the ground plane
        c = scenes.gen_capsules(800, lo, hi, seed=12)
        for max_hits in (12, 48):
            gcnt, _ = _check_vs_oracle(g, o, orc, c, max_hits)
            got, _, _ = g.capsuleOverlapAll(c, max_hits)
            kept = np.arange(max_hits)[None, :] < gcnt[:, None]
            tri = got["triangle_index"]
            both = ((kept & (tri < n_static)).any(axis=1) & (kept & (tri >= n_static)).any(axis=1))
            assert both.sum() > 0, max_hits
    finally:
        g.close()
        o.close()


def _torch():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available()
    return torch


def _dev(torch, arr):
    return torch.from_numpy(np.frombuffer(arr.tobytes(), np.uint8).copy()).cuda()


def _host(t, dtype, shape=None):
    a = np.frombuffer(t.cpu().numpy().tobytes(), dtype)
    return a if shape is None else a.reshape(shape)


class _DeviceCall:
    def __init__(self, torch, cq, n, max_hits):
        self.n, self.max_hits, self.cq = n, max_hits, cq
        self.q = torch.empty(n * cq.CAPSULE.itemsize, dtype=torch.uint8, device="cuda")
        self.out = torch.full((n * max_hits * cq.OVERLAP_HIT.itemsize,), 0xAB, dtype=torch.uint8, device="cuda")
        self.counts = torch.full((n,), -7, dtype=torch.int32, device="cuda")
        self.overflow = torch.full((n,), 0xCD, dtype=torch.uint8, device="cuda")

    def enqueue(self, g, stream):
        g.capsule_overlap_all_device(self.q.data_ptr(), self.n, self.max_hits, self.out.data_ptr(), self.counts.data_ptr(),
                                     self.overflow.data_ptr(), stream)

    def read(self):
        return (_host(self.out, self.cq.OVERLAP_HIT, (self.n, self.max_hits)), self.counts.cpu().numpy(),
                self.overflow.cpu().numpy())


@pytest.mark.gpu
def test_wide_device_call_capture_and_launch_count(world, cq, scenes):
    torch = _torch()
    name, parts, g, o = world
    c0, c1, c2 = (_capsules(name, parts, scenes, seed=s) for s in (20, 21, 22))
    max_hits = 24
    d = _DeviceCall(torch, cq, len(c0), max_hits)
    d.q.copy_(_dev(torch, c0))
    torch.cuda.synchronize()
    g.stats(reset=True)
    d.enqueue(g, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert g.stats()["kernel_launches"] == WIDE_LAUNCHES
    want = g.capsuleOverlapAll(c0, max_hits)
    for a, b in zip(d.read(), want):
        assert a.tobytes() == b.tobytes()
    # the eight-hit kernel is still one launch
    g.stats(reset=True)
    g.capsuleOverlapAll(c0[:100], 8)
    assert g.stats()["kernel_launches"] == 1
    # captured once, replayed with new capsules written into the same input buffer
    g.stats(reset=True)
    graph, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=cs):
        d.enqueue(g, torch.cuda.current_stream().cuda_stream)
    assert g.stats()["kernel_launches"] == WIDE_LAUNCHES
    for cap in (c1, c2):
        d.q.copy_(_dev(torch, cap))
        graph.replay()
        torch.cuda.synchronize()
        want = g.capsuleOverlapAll(cap, max_hits)
        for a, b in zip(d.read(), want):
            assert a.tobytes() == b.tobytes()
    assert g.stats()["kernel_launches"] == WIDE_LAUNCHES + 2 * WIDE_LAUNCHES  # replays are not counted; two host calls are
    del graph


@pytest.mark.gpu
def test_wide_counting_modes(world, cq, scenes, orc):
    name, parts, g, o = world
    c = _capsules(name, parts, scenes, seed=30)
    max_hits = 20
    st = orc.Stats()
    o.capsule_overlap_all(c, max_hits, orc.ORDER_REFERENCE, 1, st)
    try:
        g.set_counting(cq.COUNT_REFERENCE)
        g.resetStats()
        ref_mode = g.capsuleOverlapAll(c, max_hits)
        r = g.stats()
        assert r["candidates"] == st.candidates
        assert r["distance_evals"] > 0 and r["kernel_launches"] == WIDE_LAUNCHES
        g.set_counting(cq.COUNT_PATH)
        g.resetStats()
        path_mode = g.capsuleOverlapAll(c, max_hits)
        p = g.stats()
    finally:
        g.set_counting(False)
    plain = g.capsuleOverlapAll(c, max_hits)
    for a, b, x in zip(ref_mode, path_mode, plain):
        assert a.tobytes() == b.tobytes() == x.tobytes()
    for k in ("nodes_visited", "candidates", "distance_evals"):
        assert 0 < p[k] <= r[k], k


@pytest.mark.gpu
def test_wide_chunked_host_call_equals_device_call(cq, scenes):
    """A host call whose records exceed CQ_OVERLAP_ALL_CHUNK_BYTES runs in several chunks; the answer is the device call's."""
    torch = _torch()
    parts = scenes.mirror_scene(use_hulls=True)
    g = cq.CollisionQuery(parts)
    try:
        lo, hi = scenes.scene_aabb(parts[1:])
        max_hits = 300
        n = cq.OVERLAP_ALL_CHUNK_BYTES // (max_hits * cq.OVERLAP_HIT.itemsize) * 2 + 1234  # two full chunks and a part
        c = scenes.gen_capsules(n, lo, hi, seed=40)
        got = g.capsuleOverlapAll(c, max_hits)
        assert got[0].nbytes > 2 * cq.OVERLAP_ALL_CHUNK_BYTES and (got[1] > 0).sum() > n // 20
        d = _DeviceCall(torch, cq, n, max_hits)
        d.q.copy_(_dev(torch, c))
        d.enqueue(g, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        for a, b in zip(d.read(), got):
            assert a.tobytes() == b.tobytes()
        del d
    finally:
        g.close()


CPP_PROBE = r"""
// capsuleOverlapAll of the C++ mirror hands maxHits to the library unchanged and gives it room for maxHits records.  The
// world and the query are stubbed here (these definitions take precedence over libcq.so's), so no GPU is needed.
#include <cstdio>
#include "CollisionQuery.hpp"

static int seenMaxHits = 0;
extern "C" int cq_world_create_ex(const cq_mesh_part *, int32_t, const cq_world_options *, cq_world **out) {
    static int dummy;
    *out = reinterpret_cast<cq_world *>(&dummy);
    return CQ_OK;
}
extern "C" void cq_world_destroy(cq_world *) {}
extern "C" int cq_world_triangle_material(const cq_world *, int32_t, cq_material *m) {
    m->mu_s = 0.8f, m->mu_k = 0.6f, m->flatten_ground = 0;
    return CQ_OK;
}
extern "C" int cq_capsule_overlap_all_batch(cq_world *, const cq_capsule *, int32_t n, int32_t max_hits, cq_overlap_hit *out,
                                            int32_t *counts, uint8_t *) {
    seenMaxHits = max_hits;
    for (int32_t k = 0; k < n * max_hits; k++) { // every record the caller must have room for
        out[k] = cq_overlap_hit{};
        out[k].depth = 1.0f + (float)k;
        out[k].triangle_index = k;
    }
    counts[0] = max_hits;
    return CQ_OK;
}

int main() {
    cqhost::CollisionQuery q(std::vector<cq_mesh_part>{});
    auto hits = q.capsuleOverlapAll({0, 0, 0}, 1.0f, 1.0f, 32);
    if (seenMaxHits != 32 || hits.size() != 32 || hits[31].triangleIndex != 31) {
        std::printf("maxHits %d, %zu hits\n", seenMaxHits, hits.size());
        return 1;
    }
    hits = q.capsuleOverlapAll({0, 0, 0}, 1.0f, 1.0f, 0); // max(1, maxHits)
    if (seenMaxHits != 1 || hits.size() != 1) return 2;
    std::printf("ok\n");
    return 0;
}
"""


def test_cpp_wrapper_passes_max_hits_through(cq, tmp_path):
    cq.build()
    src = tmp_path / "overlap_all_probe.cpp"
    src.write_text(CPP_PROBE)
    exe = tmp_path / "overlap_all_probe"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "swift-game-engine_b200", "cpp"),
                        str(src), "-L" + cq.CSRC, "-lcq", "-Wl,-rpath," + cq.CSRC, "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stdout, r.stderr)
