"""CPU-side checks: the oracle against its committed golden trajectory, the C-ABI library's symbol table,
the *.static.json loader (host-only), and the host-side sharding logic under gloo (world_size 2)."""
import ctypes
import json
import os
import re
import shutil
import importlib
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _c1(scenes, orc, order):
    w = orc.OracleWorld(scenes.c1_scene())
    s = orc.init_states(scenes.C1_STARTS)
    p = orc.default_params()
    return scenes.c1_run(lambda st: w.move_and_slide(st, p, order=order), s, 600, scenes.C1_SPEEDS)


@pytest.mark.parametrize("name", ["reference", "canonical"])
def test_oracle_reproduces_golden_c1_trajectory(orc, scenes, name):
    """Config C1 (BASELINE.json): characters driven 600 fixed steps over the demo's static world."""
    z = np.load(os.path.join(GOLDEN, "c1_trajectory.npz"))
    rec = _c1(scenes, orc, orc.ORDER_REFERENCE if name == "reference" else orc.ORDER_CANONICAL)
    for k in rec.dtype.names:
        assert np.array_equal(rec[k], z[f"{name}_{k}"]), k
    # sanity of the recorded behaviour: the demo player lands and then stays grounded
    assert rec["grounded"][:, 0].sum() > 500 and rec["position"][-1, 0, 1] == pytest.approx(-0.45, abs=0.1)


def test_reference_vs_canonical_order_divergence_is_bounded(scenes):
    """Visiting order only matters through exact ties; over 600 frames the two oracle modes stay within a
    fraction of the capsule radius (reported, SURVEY.md §8d 'trajectory divergence')."""
    z = np.load(os.path.join(GOLDEN, "c1_trajectory.npz"))
    d = np.linalg.norm(z["reference_position"] - z["canonical_position"], axis=2)
    assert (d[:, [0, 1, 3]] == 0).all()
    assert d.max() < 0.5


def test_libcq_exports_every_declared_symbol(cq):
    """The C-ABI library loads (no GPU needed for that) and exports exactly what include/cq.h declares."""
    cq.build()
    lib = ctypes.CDLL(cq.LIB_PATH)
    header = open(cq.HEADER).read()
    declared = sorted(set(re.findall(r"\b(cq_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 30
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert sorted(cq.EXPORTS) == declared
    lib.cq_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.cq_version()
    out = subprocess.run(["cuobjdump", "-lelf", cq.LIB_PATH], capture_output=True, text=True)
    if out.returncode == 0:
        assert "sm_100a" in out.stdout


def test_record_layouts_match_header(cq):
    assert cq.STATE.itemsize == 168 and cq.PARAMS.itemsize == 52 and cq.CAST.itemsize == 40
    assert cq.CAST_HIT.itemsize == 44 and cq.OVERLAP_HIT.itemsize == 44 and cq.RAY.itemsize == 32
    assert cq.RAY_HIT.itemsize == 32 and cq.CAPSULE.itemsize == 24
    assert ctypes.sizeof(cq.MeshPart) == 112
    # the per-triangle materials were carved out of the reserved words of cq_world_options: its size must not move
    assert ctypes.sizeof(cq.WorldOptions) == 32 and cq.SURFACE_MATERIAL.itemsize == 12 and ctypes.sizeof(cq.TriangleMaterials) == 16


def test_no_cpu_fallback_without_gpu(cq):
    """Without a CUDA device the product must fail loudly (CQ_ERR_CUDA), never answer from the CPU."""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    with pytest.raises(cq.CQError):
        cq.CollisionQuery(cq.scenes.mirror_scene(True))


def _write_static_json(path, asset):
    doc = {"version": 1, "meshes": [{
        "name": asset["name"], "transform": [float(x) for x in np.asarray(asset["transform"]).reshape(4, 4).T.reshape(16)],
        "mesh": {"positions": [float(x) for x in asset["positions"].reshape(-1)], "normals": [], "uvs": [],
                 "indices": [int(i) for i in asset["indices"]],
                 "submeshes": [{"start": 0, "count": int(len(asset["indices"])), "material": "m"}]},
        "collisionHulls": [{"positions": [float(x) for x in hp.reshape(-1)], "indices": [int(i) for i in hi]}
                           for hp, hi in asset["hulls"]]}]}
    json.dump(doc, open(path, "w"))


def test_static_mesh_loader_round_trip(cq, scenes, tmp_path):
    """StaticMeshLoader (StaticMeshLoader.swift:30-197): schema, double->float narrowing, row-major ->
    column-major transform, hulls; checked against Python's json module on a file in the reference's schema."""
    a = scenes.load_mirror_fixture()
    p = tmp_path / "ornate_mirror.static.json"
    _write_static_json(str(p), a)
    got = cq.StaticMeshAsset(str(p))
    assert len(got.parts) == 1
    part = got.parts[0]
    assert part["name"] == a["name"]
    assert np.array_equal(part["transform"], a["transform"])
    assert np.array_equal(part["positions"], a["positions"]) and np.array_equal(part["indices"], a["indices"])
    assert len(part["hulls"]) == 2
    for (gp, gi), (hp, hi) in zip(part["hulls"], a["hulls"]):
        assert np.array_equal(gp, hp) and np.array_equal(gi, hi)


def test_static_mesh_loader_reference_asset(cq, scenes):
    """The reference's own asset file, when the reference tree is present (build container only)."""
    src = "/root/reference/Game/ornate_mirror.static.json"
    if not os.path.exists(src):
        pytest.skip("reference tree not present on this box")
    part = cq.StaticMeshAsset(src).parts[0]
    a = scenes.load_mirror_fixture()
    assert part["positions"].shape == (8978, 3) and part["indices"].shape == (42738,)
    assert np.array_equal(part["positions"], a["positions"]) and np.array_equal(part["transform"], a["transform"])
    assert [h[1].shape[0] // 3 for h in part["hulls"]] == [40, 36]


def test_static_mesh_loader_errors(cq, tmp_path):
    with pytest.raises(cq.CQError, match="-3"):  # missing file -> CQ_ERR_IO (the reference returns nil)
        cq.StaticMeshAsset(str(tmp_path / "nope.json"))
    bad = tmp_path / "bad.json"
    bad.write_text('{"version": 1, "meshes": [ {"name": "x", ')
    with pytest.raises(cq.CQError, match="-4"):
        cq.StaticMeshAsset(str(bad))
    # invalid parts are skipped, not fatal (StaticMeshLoader.swift:53-61)
    ok = tmp_path / "skip.json"
    ok.write_text(json.dumps({"version": 1, "meshes": [
        {"name": "noidx", "transform": [], "mesh": {"positions": [0, 0, 0, 1, 0, 0, 0, 1, 0], "normals": [], "uvs": [], "indices": []}},
        {"name": "badpos", "transform": [], "mesh": {"positions": [0, 0], "normals": [], "uvs": [], "indices": [0, 1, 2]}},
        {"name": "good", "transform": [], "mesh": {"positions": [0, 0, 0, 1, 0, 0, 0, 1, 0], "normals": [], "uvs": [], "indices": [0, 1, 2]}}]}))
    a = cq.StaticMeshAsset(str(ok))
    assert [p["name"] for p in a.parts] == ["good"]
    assert np.array_equal(a.parts[0]["transform"], np.eye(4, dtype=np.float32).reshape(16))  # identity when not 16 values



def _doc(positions="[0, 0, 0, 1, 0, 0, 0, 1, 0]", indices="[0, 1, 2]", version="1", extra="", tail=""):
    return ('{"version": %s, %s"meshes": [{"name": "t", "transform": [], "mesh": {"positions": %s, "normals": [], '
            '"uvs": [], "indices": %s}}]}%s' % (version, extra, positions, indices, tail))


def test_static_mesh_loader_is_strict_json(cq, tmp_path):
    """JSONDecoder semantics at the edges (StaticMeshLoader.swift:35-42: any decode error -> nil): numbers follow the
    RFC 8259 grammar (no nan / inf / hex / leading '+' / leading zeros / bare '.'), nothing may follow the document,
    `version` is an Int, indices are UInt32 — while unknown keys may hold anything, including arrays that start with a
    number and go on with something else."""
    f = tmp_path / "d.json"

    def load(text):
        f.write_text(text)
        return cq.StaticMeshAsset(str(f))

    for good in (_doc(), _doc(positions="[-0, 0.0, 0e0, 1E+0, 0, 0, 0, 1.0e-0, 0]"),
                 _doc(extra='"extras": [1, "two", {"three": [3, [4, null, true]]}, -5.5e-1], '),
                 _doc(extra='"n": null, "s": "a\\u00e9\\n\\"q\\"", "deep": [[[[[[[[1]]]]]]]], '),
                 "  \n\t" + _doc(tail="  \n ")):
        a = load(good)
        assert len(a.parts) == 1 and a.parts[0]["indices"].tolist() == [0, 1, 2]
    p = load(_doc(positions="[-0, 0.0, 0e0, 1E+0, 0, 0, 0, 1.0e-0, 0]")).parts[0]["positions"]
    assert p.tolist() == [[0, 0, 0], [1, 0, 0], [0, 1, 0]] and np.signbit(p[0, 0])
    for bad_number in ("nan", "NaN", "inf", "-inf", "Infinity", "+1", "01", "1.", ".5", "0x10", "1e", "1e+", "-", "1.e3", "--1"):
        with pytest.raises(cq.CQError, match="-4"):
            load(_doc(positions="[0, 0, 0, 1, 0, 0, 0, %s, 0]" % bad_number))
        with pytest.raises(cq.CQError, match="-4"):
            load(_doc(positions="[%s, 0, 0, 1, 0, 0, 0, 1, 0]" % bad_number))
    for bad in (_doc(tail="x"), _doc(tail="{}"), _doc(version="1.5"), _doc(version='"1"'), _doc(indices="[0, 1, 2.5]"),
                _doc(indices="[0, 1, -2]"), _doc(indices="[0, 1, 4294967296]"), _doc(indices='[0, 1, "2"]'),
                _doc(positions="[0, 0, 0, 1, 0, 0, 0, 1, 0,]"), _doc(positions='"nope"'), _doc(extra='"s": "\\u12G4", '),
                "[" * 100 + "]" * 100, '{"version": 1, "meshes": [' + "[" * 200 + "]" * 200 + "]}", "", "   ", "nul"):
        with pytest.raises(cq.CQError, match="-4"):
            load(bad)
    assert load(_doc(indices="[0, 1, 4294967295]")).parts[0]["indices"].tolist() == [0, 1, 4294967295]  # the loader does not range-check


def test_static_mesh_loader_survives_mutated_documents(cq, tmp_path):
    """Robustness: 4,000 random byte-level mutations (flips, deletions, insertions of structural characters, truncations)
    of a valid document either load or fail with CQ_ERR_PARSE — never anything else, never a crash — and whatever loads
    is self-consistent (whole triangles of in-range floats)."""
    rng = np.random.default_rng(7)
    base = _doc(positions="[0.5, -1.25e1, 3, 1, 0, 0, 0, 1, 0, 2, 2, 2]", indices="[0, 1, 2, 2, 1, 3]",
                extra='"collisionHullsNote": [1, "x"], ').replace(
        '"indices": [0, 1, 2, 2, 1, 3]}', '"indices": [0, 1, 2, 2, 1, 3], "submeshes": [{"start": 0, "count": 6, "material": "m"}]}, '
        '"collisionHulls": [{"positions": [0, 0, 0, 1, 0, 0, 0, 1, 0], "indices": [0, 1, 2]}]').encode()
    f = tmp_path / "m.json"
    f.write_bytes(base)
    assert len(cq.StaticMeshAsset(str(f)).parts[0]["hulls"]) == 1
    alphabet = b'{}[]",:.-+eE0123456789 \\ntu\x00\xff'
    loaded = 0
    for _ in range(4000):
        doc = bytearray(base)
        for _ in range(int(rng.integers(1, 4))):
            kind, at = int(rng.integers(0, 4)), int(rng.integers(0, len(doc)))
            if kind == 0:
                doc[at] = alphabet[int(rng.integers(0, len(alphabet)))]
            elif kind == 1:
                del doc[at:at + int(rng.integers(1, 6))]
            elif kind == 2:
                doc[at:at] = bytes([alphabet[int(rng.integers(0, len(alphabet)))]])
            else:
                del doc[at:]
            if not doc:
                break
        f.write_bytes(bytes(doc))
        try:
            a = cq.StaticMeshAsset(str(f))
        except cq.CQError as e:
            assert "libcq error -4" in str(e), str(e)
            continue
        loaded += 1
        for part in a.parts:
            assert part["positions"].shape[1] == 3 and len(part["positions"]) > 0 and len(part["indices"]) > 0
    assert 0 < loaded < 4000



def test_fbx_regenerator_reproduces_shipped_asset_and_fixtures(cq, scenes, tmp_path):
    """SURVEY.md §8f-1 (tools/fbx_to_static_mesh.py, build container only — it reads /root/reference): the Blender-free FBX
    reader reproduces the one asset whose JSON ships (ornate_mirror: 14,246 triangles, local AABB, transform, and — with
    Blender's quad-flip rule — more than 99.5% of the triangles as the same vertex-position triples), the committed Semla /
    17-Cheese fixtures are what `--fixtures` generates under that same Blender rule (Semla's FBX is all triangles, so only
    17-Cheese's quads depend on it), and the JSON the tool writes goes through the product's own loader unchanged."""
    if not os.path.exists("/root/reference/ExternalResources/17-Cheese.fbx"):
        pytest.skip("reference tree not present on this box")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import fbx_to_static_mesh as fbx
    assert fbx.validate_against_mirror()
    mine = fbx.load_geometry(os.path.join(fbx.REF, "ornate-mirror/source/ornate_mirror.fbx"))[0]
    ref = json.load(open("/root/reference/Game/ornate_mirror.static.json"))["meshes"][0]

    from scipy.spatial import cKDTree
    mine_pos = np.asarray(mine["positions"], np.float64).reshape(-1, 3)
    tree = cKDTree(mine_pos)

    def triangle_keys(pos, idx):  # order-free identity of a triangle: its corners as ids of the nearest regenerated vertex
        d, ids = tree.query(np.asarray(pos, np.float64).reshape(-1, 3))
        assert d.max() < 2e-5  # every shipped vertex position exists in the regenerated mesh (JSON text rounding only)
        return {tuple(sorted(tri)) for tri in ids[np.asarray(idx).reshape(-1, 3)].tolist()}
    a, b = triangle_keys(mine_pos, mine["indices"]), triangle_keys(ref["mesh"]["positions"], ref["mesh"]["indices"])
    assert len(a & b) >= 0.995 * len(b), (len(a & b), len(a), len(b))  # the rest: n-gons, which Blender poly-fills
    for name, rel in (("semla", "semla/source/Semla.fbx"), ("cheese", "17-Cheese.fbx")):
        part = fbx.load_geometry(os.path.join(fbx.REF, rel), "blender")
        dst = tmp_path / (name + ".npz")
        fbx.save_fixture(part, str(dst))
        new, old = np.load(dst), np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        assert sorted(new.files) == sorted(old.files)
        for k in new.files:
            assert np.array_equal(new[k], old[k]), (name, k)
    out = tmp_path / "semla.static.json"
    assert fbx.main([os.path.join(fbx.REF, "semla/source/Semla.fbx"), str(out)]) == 0
    loaded = cq.StaticMeshAsset(str(out)).parts[0]
    fixture = scenes.load_asset_fixture("semla")  # same vertices and hulls; the quads' diagonals follow the Blender rule
    assert np.array_equal(loaded["positions"], fixture["positions"]) and loaded["indices"].shape == fixture["indices"].shape
    assert len(loaded["hulls"]) == len(fixture["hulls"]) >= 1
    for (lp, li), (fp, fi) in zip(loaded["hulls"], fixture["hulls"]):
        assert np.array_equal(lp, fp) and np.array_equal(li, fi)


_GLOO_WORKER = r"""
import os, sys, importlib
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from oracle import oracle as orc
sc = importlib.import_module("swift-game-engine_b200.scenes")
shard = importlib.import_module("swift-game-engine_b200.shard")
dist.init_process_group("gloo")
rank, ws = dist.get_rank(), dist.get_world_size()
w = orc.OracleWorld(sc.mirror_scene(True))
for n in (3000, 2001, 1):   # equal shards (one all_gather_into_tensor), ragged shards, fewer units than ranks
    pos, vel = sc.gen_c3_characters(n, seed=7)
    lo, hi = shard.rank_range(n, rank, ws)   # contiguous rank ranges, mesh replicated (SURVEY.md §8e)
    s = orc.init_states(pos[lo:hi], vel[lo:hi])
    if hi > lo:
        w.move_and_slide(s, orc.default_params())
    mine = torch.from_numpy(np.frombuffer(s.tobytes(), np.uint8).copy())
    got = shard.gather_records(mine, n, orc.STATE.itemsize)
    full = orc.init_states(pos, vel)
    w.move_and_slide(full, orc.default_params())
    assert got.numpy().tobytes() == full.tobytes(), "sharded result differs from the single-rank result (n=%d)" % n
    assert shard.records_from_bytes(got, orc.STATE)["position"].shape == (n, 3)
assert sum(shard.shard_sizes(10, 4)) == 10 and shard.shard_sizes(2, 4).count(0) == 2
if rank == 0:
    print("GLOO_OK")
dist.destroy_process_group()
"""


def test_sharded_characters_equal_single_rank_gloo(tmp_path):
    """Multi-GPU plan on CPU: characters split into contiguous rank ranges, world replicated, results gathered;
    the gathered states must equal the unsharded run byte for byte (world_size 2, gloo)."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    # --standalone: the rendezvous takes a free local port, so runs on a shared host do not collide
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node=2",
                          str(script), ROOT],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GLOO_OK" in out.stdout


def test_header_is_plain_c_and_cpp_mirror_compiles(tmp_path):
    """include/cq.h must be a C header (no C++/torch types in the signatures); the C++ host mirror of the
    reference class must compile against it."""
    r = subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-x", "c", os.path.join(ROOT, "include", "cq.h")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    src = tmp_path / "use.cpp"
    src.write_text('#include "%s"\nint main(){ cqhost::Float3 a{0,0,0}; (void)a; static_assert(sizeof(cq_world_options) == 32 && sizeof(cq_surface_material) == 12 && sizeof(cq_triangle_materials) == 16, "ABI"); return sizeof(cq_character_state)==168 ? 0 : 1; }\n'
                   % os.path.join(ROOT, "swift-game-engine_b200", "cpp", "CollisionQuery.hpp"))
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_native_example_links_and_fails_loudly_without_a_gpu(cq, scenes, tmp_path):
    """examples/cq_walk.cpp — the boundary used from compiled host code (loader + cpp/CollisionQuery.hpp + libcq.so): it
    must build and link with a plain g++, load an asset in the reference's schema, and, on a box without a CUDA device,
    stop with the library's own error (exit 4) instead of computing anything on the CPU.  On a GPU box it runs the walk."""
    cq.build()
    exe = tmp_path / "cq_walk"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", os.path.join(ROOT, "examples", "cq_walk.cpp"), "-L" + cq.CSRC,
                        "-lcq", "-Wl,-rpath," + cq.CSRC, "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert subprocess.run([str(exe)], capture_output=True).returncode == 2
    r = subprocess.run([str(exe), str(tmp_path / "missing.static.json")], capture_output=True, text=True)
    assert r.returncode == 3 and "missing json" in r.stderr
    asset = tmp_path / "ornate_mirror.static.json"
    _write_static_json(str(asset), scenes.load_mirror_fixture())
    r = subprocess.run([str(exe), str(asset), "256", "3"], capture_output=True, text=True, timeout=300)
    assert "2 part(s), 78 triangles with the ground plane" in r.stdout
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        assert r.returncode == 0 and "256 characters x 3 steps" in r.stdout, r.stderr
    else:
        assert r.returncode == 4 and "cq_world_create: CUDA error" in r.stderr, (r.returncode, r.stderr)


def test_multi_gpu_example_links_and_group_api_without_a_gpu(cq, tmp_path):
    """examples/cq_multi_gpu.cpp (all GPUs of a box from compiled host code: cq_group_*, cq_world_create_multi, the NCCL
    gather) must build against include/cq.h and libcq.so alone and stop with exit 4 on a box without a CUDA device.  The
    host half of the group API works anywhere: cq_shard_range tiles a batch exactly like shard.rank_range, NCCL is loaded
    at run time (no link-time dependency), a local group without devices is refused with CQ_ERR_CUDA."""
    cq.build()
    shard = importlib.import_module("swift-game-engine_b200.shard")
    for n in (0, 1, 7, 8, 1000, (1 << 23) + 5):
        for ws in (1, 2, 3, 8):
            got = [cq.shard_range(n, ws, r) for r in range(ws)]
            assert got == [shard.rank_range(n, r, ws) for r in range(ws)]
            assert got[0][0] == 0 and got[-1][1] == n and all(a[1] == b[0] for a, b in zip(got, got[1:]))
    assert cq.shard_range(10, 0, 0) == (0, 0) and cq.shard_range(10, 2, 5) == (0, 0)
    needed = subprocess.run(["ldd", cq.LIB_PATH], capture_output=True, text=True).stdout
    assert "nccl" not in needed and "libcudart" not in needed and "torch" not in needed
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not available")
    exe = tmp_path / "cq_multi_gpu"
    r = subprocess.run(["nvcc", "-std=c++17", "-O1", "-Wno-deprecated-gpu-targets", os.path.join(ROOT, "examples", "cq_multi_gpu.cpp"),
                        "-L" + cq.CSRC, "-lcq", "-Xlinker", "-rpath", "-Xlinker", cq.CSRC, "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if not have_gpu:
        r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
        assert r.returncode == 4 and "no usable CUDA device" in r.stderr
        with pytest.raises(cq.CQError):
            cq.Group.local(1)


class _RecorderWorld:
    """Stands in for the CUDA query object so the service policy can be tested without a GPU."""
    log = []

    def __init__(self, parts):
        self.parts = parts
        _RecorderWorld.log.append(("build", [p["entity_id"] for p in parts], [bool(p["is_dynamic"]) for p in parts]))

    def updateStaticTransforms(self, ids, models):
        _RecorderWorld.log.append(("static", list(ids)))

    def updateDynamicTransforms(self, ids, models):
        _RecorderWorld.log.append(("dynamic", list(ids)))

    def close(self):
        pass


def test_collision_query_service_rebuild_vs_refit_policy(cq, scenes):
    """CollisionQueryService.update (SceneServices.swift:52-169): what triggers a rebuild, what a refit."""
    v, i = scenes.plane_mesh(10.0)
    bv, bi = scenes.box_mesh(2.0)
    ents = [dict(entity_id=0, positions=v, indices=i, body_type="static"),
            dict(entity_id=1, positions=bv, indices=bi, translation=(0, 1, 0), body_type="kinematic"),
            dict(entity_id=2, positions=bv, indices=bi, translation=(4, 1, 0)),
            dict(entity_id=3, positions=bv, indices=bi, collides=False)]
    _RecorderWorld.log = []
    svc = cq.CollisionQueryService(world_factory=_RecorderWorld)
    svc.update(ents)
    assert svc.last_action == "rebuild" and _RecorderWorld.log[-1] == ("build", [0, 1, 2], [False, True, False])
    svc.update(ents)
    assert svc.last_action == "none"
    ents[1]["translation"] = (0, 1.5, 0)  # kinematic platform moved -> dynamic refit
    svc.update(ents)
    assert svc.last_action == "refit" and _RecorderWorld.log[-1] == ("dynamic", [1])
    ents[2]["rotation"] = tuple(scenes.quat_angle_axis(0.3, (0, 1, 0)))  # body-less entity -> static refit
    svc.update(ents)
    assert _RecorderWorld.log[-1] == ("static", [2])
    ents[2]["translation"] = (4, 1 + 5e-4, 0)  # squared delta 2.5e-7 <= 1e-6: below the threshold
    svc.update(ents)
    assert svc.last_action == "none"
    n_builds = sum(1 for x in _RecorderWorld.log if x[0] == "build")
    for mutate in (lambda: ents[2].__setitem__("dirty", True), lambda: ents[1].__setitem__("body_type", "dynamic"),
                   lambda: ents[3].__setitem__("collides", True), lambda: ents[0].__setitem__("indices", i[:3]),
                   lambda: svc.markDirty()):
        mutate()
        svc.update(ents)
        n_builds += 1
        assert svc.last_action == "rebuild" and sum(1 for x in _RecorderWorld.log if x[0] == "build") == n_builds
    svc.update(ents, active_ids={0, 1})  # active set changed -> rebuild with the filtered entities
    assert _RecorderWorld.log[-1][0] == "build" and _RecorderWorld.log[-1][1] == [0, 1]


_CPP_SERVICE_DRIVER = r"""
#include <cstdio>
#include "%(hdr)s"
using namespace cqhost;
struct Recorder {  // stands in for the CUDA query object (no device needed)
    explicit Recorder(const std::vector<cq_mesh_part> &parts) {
        std::printf("build");
        for (auto &p : parts) std::printf(" %%u:%%d", p.entity_id, (int)p.is_dynamic);
        std::printf("\n");
    }
    bool updateTransforms(const std::vector<uint32_t> &ids, const std::vector<float> &models) {
        std::printf("refit");
        for (auto id : ids) std::printf(" %%u", id);
        std::printf(" | %%.9g %%.9g %%.9g\n", models[12], models[13], models[14]);
        return true;
    }
};
static const char *name(CollisionQueryServiceT<Recorder>::Action a) {
    return a == CollisionQueryServiceT<Recorder>::Action::None ? "none" : a == CollisionQueryServiceT<Recorder>::Action::Refit ? "refit" : "rebuild";
}
int main() {
    static const float quad[12] = {-5, 0, -5, 5, 0, -5, 5, 0, 5, -5, 0, 5};
    static const uint32_t quadIdx[6] = {0, 2, 1, 0, 3, 2};
    std::vector<MeshEntity> e(4);
    for (int k = 0; k < 4; k++) e[k].id = k, e[k].positions = quad, e[k].n_verts = 4, e[k].indices = quadIdx, e[k].n_indices = 6;
    e[0].bodyType = BodyType::Static;
    e[1].bodyType = BodyType::Kinematic, e[1].translation = {0, 1, 0};
    e[2].translation = {4, 1, 0};
    e[3].collides = false;
    CollisionQueryServiceT<Recorder> svc;
    auto step = [&](const CollisionQueryServiceT<Recorder>::ActiveSet &a = std::nullopt) { svc.update(e, a); std::printf("-> %%s\n", name(svc.lastAction())); };
    step();                                   // first update: rebuild
    step();                                   // nothing changed
    e[1].translation = {0, 1.5f, 0}; step();  // kinematic platform moved -> dynamic refit
    e[2].rotation[1] = 0.14943813f, e[2].rotation[3] = 0.98877108f; step();  // body-less entity turned -> static refit
    e[2].translation = {4, 1.0005f, 0}; step();  // squared delta 2.5e-7 <= 1e-6: below the threshold
    e[2].dirty = true; step();
    e[1].bodyType = BodyType::Dynamic; step();
    e[3].collides = true; step();
    e[0].n_indices = 3; step();
    svc.markDirty(); step();
    step(std::set<uint32_t>{0, 1});           // active set changed -> rebuild with the filtered entities
    step(std::set<uint32_t>{0, 1});
    // model matrix of a general TRS and the streaming set
    MeshEntity t; t.translation = {1.5f, -2.25f, 3.0f}; t.scale = {2.0f, 0.5f, 1.25f};
    t.rotation[0] = 0.18257419f, t.rotation[1] = 0.36514837f, t.rotation[2] = 0.54772256f, t.rotation[3] = 0.73029674f;
    float m[16]; modelMatrix(t, m);
    std::printf("model");
    for (float v : m) std::printf(" %%.9g", v);
    std::printf("\n");
    std::vector<MeshEntity> far(3);
    far[0].id = 10, far[0].translation = {255.9f, 0, 0};
    far[1].id = 11, far[1].translation = {1300.0f, 0, 0};
    far[2].id = 12, far[2].translation = {-1281.0f, 0, 600.0f};
    const double player[3] = {10.0, 0.0, 0.0};
    std::printf("active");
    for (auto id : activeEntityIDs(player, far)) std::printf(" %%u", id);
    std::printf("\n");
    return 0;
}
"""


def test_cpp_service_mirror_makes_the_reference_decisions(cq, scenes, tmp_path):
    """cpp/CollisionQueryService.hpp — the compiled-language host mirror of SceneServices.swift:33-207 and of the streaming
    active set: the scenario of the Python policy test above through the C++ class with a recorder in place of the CUDA
    query object (no device needed), action by action; its modelMatrix against scenes.trs_model; chunk membership."""
    src = tmp_path / "svc.cpp"
    src.write_text(_CPP_SERVICE_DRIVER % {"hdr": os.path.join(ROOT, "swift-game-engine_b200", "cpp", "CollisionQueryService.hpp")})
    exe = tmp_path / "svc"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines()
    actions = [ln[3:] for ln in out if ln.startswith("-> ")]
    assert actions == ["rebuild", "none", "refit", "refit", "none", "rebuild", "rebuild", "rebuild", "rebuild", "rebuild", "rebuild", "none"]
    events = [ln for ln in out if ln.startswith(("build", "refit"))]
    assert events[0] == "build 0:0 1:1 2:0"                      # entity 3 does not collide; the kinematic body is dynamic
    assert events[1].startswith("refit 1 |") and events[2].startswith("refit 2 |")
    assert events[1].split("|")[1].split() == ["0", "1.5", "0"]  # the refit carries the new model matrix
    assert events[5] == "build 0:0 1:1 2:0 3:0"                  # entity 3 collides now
    assert events[-1] == "build 0:0 1:1"                         # the active set filters the entities
    model = np.float32([float(x) for x in next(ln for ln in out if ln.startswith("model")).split()[1:]])
    want = scenes.trs_model((1.5, -2.25, 3.0), (0.18257419, 0.36514837, 0.54772256, 0.73029674), (2.0, 0.5, 1.25))
    assert np.allclose(model, want, atol=1e-6)
    # chunks of 512 m centred on multiples of 512, Chebyshev radius 2 around the player's chunk 0: x = 1300 is chunk 3 (out),
    # x = -1281 is chunk -3 (out) ... -1281 + 256 = -1025 -> floor(-2.002) = -3
    assert next(ln for ln in out if ln.startswith("active")).split()[1:] == ["10"]


def test_active_chunk_set_drives_rebuilds(cq, scenes):
    """ActiveChunkSystem (Systems.swift:2354-2396) + WorldPosition.fromWorld (Components.swift:58-69): 512 m chunks
    centred on multiples of 512, Chebyshev radius 2; a player crossing a chunk border changes the active set, and the
    changed set is what makes CollisionQueryService rebuild (SceneServices.swift:55-58)."""
    ch, lo = cq.world_to_chunk([[255.9, -256.0, 256.0], [-256.1, 767.9, 0.0]])
    assert ch.tolist() == [[0, 0, 1], [-1, 1, 0]]
    assert np.allclose(lo, [[255.9, -256.0, -256.0], [255.9, 255.9, 0.0]])
    assert np.allclose(cq.chunk_to_world(ch, lo), [[255.9, -256.0, 256.0], [-256.1, 767.9, 0.0]])
    bv, bi = scenes.box_mesh(2.0)
    ents = [dict(entity_id=k, positions=bv, indices=bi, translation=(512.0 * k, 0, 0)) for k in range(8)]
    ents.append(dict(entity_id=100, translation=(0, 0, 0)))  # a mesh-less entity (e.g. the player itself)
    acs = cq.ActiveChunkSet()
    active, static = acs.update((10.0, 0.0, 0.0), ents)
    assert active == {0, 1, 2, 100} and static == {0, 1, 2}
    _RecorderWorld.log = []
    svc = cq.CollisionQueryService(world_factory=_RecorderWorld)
    meshes = ents[:8]
    svc.update(meshes, active_ids=static)
    assert _RecorderWorld.log[-1][:2] == ("build", [0, 1, 2])
    active, static = acs.update((250.0, 0.0, 0.0), ents)  # same chunk: same set, nothing to do
    svc.update(meshes, active_ids=static)
    assert svc.last_action == "none"
    active, static = acs.update((260.0, 0.0, 0.0), ents)  # crossed into chunk 1: entity 3 streams in
    assert static == {0, 1, 2, 3} and acs.center_chunk.tolist() == [1, 0, 0]
    svc.update(meshes, active_ids=static)
    assert svc.last_action == "rebuild" and _RecorderWorld.log[-1][1] == [0, 1, 2, 3]
    active, static = acs.update((512.0 * 5, 0.0, 0.0), ents)
    assert static == {3, 4, 5, 6, 7}
    acs.radius_chunks = -3  # max(radiusChunks, 0)
    assert acs.update((512.0 * 5, 0.0, 0.0), ents)[1] == {5}


def test_transform_helpers_against_scipy(scenes):
    """TransformComponent.modelMatrix = T * (R(quat) * S) (Components.swift:26-44) and the simd quaternion conventions of
    SURVEY.md §A.1 as scenes.py restates them (host-only scene-recipe code shared by oracle and GPU): checked against
    scipy's Rotation — rotation matrices, Hamilton products, angle-axis construction and the matrix -> (T, quat, S) round
    trip used to re-pose the demo assets."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(17)
    for _ in range(200):
        axis = rng.standard_normal(3)
        axis /= np.linalg.norm(axis)
        angle = rng.uniform(-np.pi, np.pi)
        q = scenes.quat_angle_axis(angle, axis)  # (ix, iy, iz, r) like simd_quatf
        want = Rotation.from_rotvec(axis * angle)
        assert np.allclose(np.asarray(q, np.float64), want.as_quat(), atol=1e-6) or np.allclose(-np.asarray(q, np.float64), want.as_quat(), atol=1e-6)
        assert np.allclose(scenes.quat_to_mat3(q), want.as_matrix(), atol=1e-6)
        q2 = scenes.quat_angle_axis(rng.uniform(-3, 3), (0.0, 1.0, 0.0))
        prod = scenes.quat_mul(q, q2)
        assert np.allclose(scenes.quat_to_mat3(prod), want.as_matrix() @ Rotation.from_quat(np.asarray(q2, np.float64)).as_matrix(), atol=1e-5)
        t, s = rng.uniform(-20, 20, 3), rng.uniform(0.2, 8.0, 3)
        m = scenes.trs_model(t, q, s).reshape(4, 4).T  # column-major flat -> m[row][col]
        assert np.allclose(m[:3, :3], want.as_matrix() * s[None, :], atol=1e-5) and np.allclose(m[:3, 3], t, atol=1e-6)
        assert np.allclose(m[3], [0, 0, 0, 1])
        t2, q3, s2 = scenes.transform_from_matrix(scenes.trs_model(t, q, s))
        assert np.allclose(t2, t, atol=1e-5) and np.allclose(s2, s, atol=1e-4)
        assert np.allclose(scenes.quat_to_mat3(q3), want.as_matrix(), atol=1e-5)
    # the loader's row-major file order -> simd's column-major (StaticMeshLoader.swift:127-134)
    rowmajor = np.arange(16, dtype=np.float32)
    assert np.array_equal(scenes.rowmajor_to_colmajor(rowmajor).reshape(4, 4), rowmajor.reshape(4, 4).T)


def test_sass_breakdown_tool_accounts_for_every_instruction(cq):
    """tools/sass_breakdown.py (the evidence behind DESIGN.md §10's code-size and per-region tables): on the shipped
    k_move_and_slide it must find every region by its function definition (no region may silently vanish when the sources
    move) and its per-region counts must add up to the kernel's instruction count."""
    import re
    import shutil
    if shutil.which("nvdisasm") is None or shutil.which("cuobjdump") is None:
        pytest.skip("CUDA binary utilities not available")
    cq.build()
    obj = os.path.join(cq.CSRC, "cq_mas.o")
    if not os.path.exists(obj):
        pytest.skip("object files not kept on this box")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sass_breakdown.py"), obj, "k_move_and_slideILb0ELb0ELb0E"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    total = int(re.search(r"(\d+) instructions", r.stdout).group(1))
    by_region = r.stdout.split("by region:")[1]
    counts = [int(m.group(1)) for m in re.finditer(r"^\s+(\d+)\s+[\d.]+ KB  \S", by_region, re.M)]
    assert total > 3000 and sum(counts) == total
    for label in ("controller logic", "pool: posting queries", "pool: cooperative walk", "pool: job pickup", "pool: pair state machine",
                  "pool: commit", "pool: main loop", "closest_point_on_triangle", "vertical-axis specialisations",
                  "segment_triangle_distance body"):
        assert label in by_region, label
    assert "other:" not in by_region
