"""B200 batched collision-query engine — Python host binding over the C ABI (include/cq.h).

The product is `csrc/libcq.so` (hand-written CUDA for sm_100a behind a C ABI).  This
module is a thin ctypes mirror of the reference's `CollisionQuery` class
(Game/CollisionQuery.swift:54-160) so tests and bench.py read like calls on the
reference API.  There is NO CPU fallback: importing works without a GPU (so the
symbol table can be checked), but every compute call fails loudly if the CUDA
library or a device is missing.

The directory name contains a '-', so import it with
    importlib.import_module("swift-game-engine_b200")
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import scenes, shard  # noqa: F401  (re-export)
from .service import ActiveChunkSet, CollisionQueryService, chunk_to_world, world_to_chunk  # noqa: E402,F401

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# CQ_LIB: another build of the same library (A/B runs of kernel variants: tools/ab_e2e.py, bench.py); build() then leaves it alone
LIB_PATH = os.environ.get("CQ_LIB") or os.path.join(CSRC, "libcq.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "cq.h")

# ---- record layouts of include/cq.h -------------------------------------------------------------
RAY = scenes.RAY
CAST = scenes.CAST
CAPSULE = scenes.CAPSULE
RAY_HIT = np.dtype([("distance", "<f4"), ("position", "<f4", 3), ("normal", "<f4", 3), ("triangle_index", "<i4")])
CAST_HIT = np.dtype([("toi", "<f4"), ("position", "<f4", 3), ("normal", "<f4", 3),
                     ("triangle_normal", "<f4", 3), ("triangle_index", "<i4")])
OVERLAP_HIT = np.dtype([("depth", "<f4"), ("position", "<f4", 3), ("normal", "<f4", 3),
                        ("triangle_normal", "<f4", 3), ("triangle_index", "<i4")])
PARAMS = np.dtype([("radius", "<f4"), ("half_height", "<f4"), ("skin_width", "<f4"), ("ground_snap_skin", "<f4"),
                   ("snap_distance", "<f4"), ("fall_probe_distance", "<f4"), ("ground_snap_max_speed", "<f4"),
                   ("ground_snap_max_toi", "<f4"), ("ground_snap_max_step", "<f4"),
                   ("ground_sweep_max_step", "<f4"), ("max_slide_iterations", "<i4"), ("min_ground_dot", "<f4"),
                   ("collision_mask", "<u4")])
STATE = np.dtype([("position", "<f8", 3), ("velocity", "<f8", 3), ("ground_normal", "<f4", 3),
                  ("ground_distance", "<f4"), ("side_contact_normal", "<f4", 3), ("ground_triangle_index", "<i4"),
                  ("ground_transition_frames", "<i4"), ("side_contact_frames", "<i4"), ("manifold_frames", "<i4"),
                  ("manifold_count", "<i4"), ("manifold_triangles", "<i4", 4), ("manifold_normals", "<f4", (4, 3)),
                  ("grounded", "u1"), ("grounded_near", "u1"), ("ground_sliding", "u1"), ("_pad", "u1", 5)])
assert STATE.itemsize == 168 and CAST.itemsize == 40 and CAST_HIT.itemsize == 44 and RAY.itemsize == 32

CROWD_POSE = np.dtype([("position", "<f8", 3), ("velocity", "<f8", 3), ("ground_triangle_index", "<i4"), ("grounded", "u1"),
                       ("grounded_near", "u1"), ("ground_sliding", "u1"), ("_pad", "u1")])
assert CROWD_POSE.itemsize == 56
PLATFORM = np.dtype([("aabb_min", "<f4", 3), ("aabb_max", "<f4", 3), ("delta", "<f4", 3)])
CAST_ALL, CAST_BLOCKING, CAST_GROUND = 0, 1, 2
MAS_APPLY_GRAVITY = 1
MAS_AGENTS = 2  # characters of the batch collide with each other (capsule-capsule CCD)
LAYER_ALL = 0xFFFFFFFF


class MeshPart(C.Structure):
    _fields_ = [("positions_xyz", C.c_void_p), ("indices", C.c_void_p), ("n_verts", C.c_int32),
                ("n_indices", C.c_int32), ("model", C.c_float * 16), ("layer", C.c_uint32), ("mu_s", C.c_float),
                ("mu_k", C.c_float), ("flatten_ground", C.c_uint8), ("is_dynamic", C.c_uint8), ("_pad", C.c_uint16),
                ("entity_id", C.c_uint32)]


class WorldInfo(C.Structure):
    _fields_ = [("n_static_triangles", C.c_int32), ("n_dynamic_triangles", C.c_int32),
                ("n_static_vertices", C.c_int32), ("n_dynamic_vertices", C.c_int32),
                ("n_static_nodes", C.c_int32), ("n_dynamic_nodes", C.c_int32), ("n_parts", C.c_int32),
                ("device", C.c_int32), ("build_ms", C.c_float), ("refit_ms", C.c_float), ("order", C.c_int32),
                ("ref_order_ms", C.c_float), ("n_ref_nodes", C.c_int32), ("_reserved", C.c_int32)]


class TriangleMaterials(C.Structure):  # cq_triangle_materials
    _fields_ = [("entity_id", C.c_uint32), ("n", C.c_int32), ("materials", C.c_void_p)]


class WorldOptions(C.Structure):
    _fields_ = [("order", C.c_int32), ("n_triangle_materials", C.c_int32), ("triangle_materials", C.c_void_p),
                ("_reserved", C.c_int32 * 4)]


# cq_surface_material: StaticMeshComponent.triangleMaterials entries (a part dict may carry "triangle_materials": (T, 3)
# rows of mu_s, mu_k, flatten_ground — used when T equals the part's triangle count, ignored otherwise, as the reference does)
SURFACE_MATERIAL = np.dtype([("mu_s", "<f4"), ("mu_k", "<f4"), ("flatten_ground", "u1"), ("_pad", "u1", (3,))])


def _world_options(parts, order, keep):
    """cq_world_options for `parts`: the order rule + the per-triangle materials some part dicts carry."""
    opt = WorldOptions()
    lib().cq_world_options_default(C.byref(opt))
    opt.order = int(order)
    per_tri = [(int(p.get("entity_id", i)), surface_materials(p["triangle_materials"]))
               for i, p in enumerate(parts) if p.get("triangle_materials") is not None]
    if per_tri:
        tm = (TriangleMaterials * len(per_tri))()
        for k, (eid, mats) in enumerate(per_tri):
            keep.append(mats)
            tm[k].entity_id, tm[k].n, tm[k].materials = eid, len(mats), mats.ctypes.data
        keep.append(tm)
        opt.n_triangle_materials, opt.triangle_materials = len(per_tri), C.addressof(tm)
    return opt


def surface_materials(rows):
    rows = np.asarray(rows, np.float32).reshape(-1, 3)
    out = np.zeros(len(rows), SURFACE_MATERIAL)
    out["mu_s"], out["mu_k"], out["flatten_ground"] = rows[:, 0], rows[:, 1], rows[:, 2] != 0
    return out


ORDER_REFERENCE, ORDER_CANONICAL = 0, 1  # include/cq.h: which of several exactly equal candidates a query names
COUNT_OFF, COUNT_REFERENCE, COUNT_PATH = 0, 1, 2  # include/cq.h: cq_world_set_counting modes
HIT_TIE, HIT_OVERFLOW = 1, 2


class Material(C.Structure):
    _fields_ = [("mu_s", C.c_float), ("mu_k", C.c_float), ("flatten_ground", C.c_int32)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("queries", "nodes_visited", "candidates", "distance_evals",
                                          "kernel_launches")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


EXPORTS = [
    "cq_world_create", "cq_world_create_ex", "cq_world_options_default", "cq_world_destroy", "cq_world_get_info", "cq_world_update_transforms",
    "cq_world_update_transforms_async", "cq_world_read_soup",
    "cq_world_triangle_material", "cq_static_mesh_load", "cq_static_mesh_free", "cq_static_mesh_part_count",
    "cq_static_mesh_part_name", "cq_static_mesh_part_transform", "cq_static_mesh_hull_count",
    "cq_static_mesh_geometry", "cq_raycast_batch", "cq_capsule_cast_batch", "cq_capsule_overlap_batch",
    "cq_capsule_overlap_all_batch", "cq_raycast_batch_ex", "cq_capsule_cast_batch_ex", "cq_capsule_overlap_batch_ex",
    "cq_raycast_device_ex", "cq_capsule_cast_device_ex", "cq_capsule_overlap_device_ex", "cq_raycast_device", "cq_capsule_cast_device", "cq_capsule_overlap_device",
    "cq_capsule_overlap_all_device", "cq_controller_params_default", "cq_character_state_init",
    "cq_move_and_slide_batch", "cq_move_and_slide_device", "cq_move_and_slide_batch_ex",
    "cq_move_and_slide_device_ex", "cq_agent_separation_batch", "cq_agent_separation_device",
    "cq_world_set_counting", "cq_world_read_counters",
    "cq_crowd_create", "cq_crowd_destroy", "cq_crowd_size", "cq_crowd_step", "cq_crowd_read", "cq_crowd_write",
    "cq_crowd_device_states",
    "cq_shard_range", "cq_group_unique_id", "cq_group_create_rank", "cq_group_create_local", "cq_group_destroy",
    "cq_group_size", "cq_group_rank", "cq_group_device", "cq_group_gather_records", "cq_group_gather_records_local",
    "cq_group_synchronize", "cq_world_create_multi", "cq_multi_world_destroy", "cq_multi_world_size",
    "cq_multi_world_replica", "cq_multi_update_transforms", "cq_multi_raycast_batch", "cq_multi_capsule_cast_batch",
    "cq_multi_move_and_slide_batch",
    "cq_host_alloc", "cq_host_free", "cq_last_error", "cq_version",
]
GROUP_ID_BYTES = 128


class CQError(RuntimeError):
    pass


def build(force=False, verbose=False):
    """Compile csrc/libcq.so for sm_100a with the committed Makefile (nvcc cross-compiles without a GPU)."""
    if os.environ.get("CQ_LIB"):
        return LIB_PATH
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", ".cpp"))]
    srcs.append(HEADER)
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", CSRC, "-j8"] + ([] if verbose else ["-s"])
        subprocess.check_call(cmd)
    return LIB_PATH


_lib = None


def lib():
    """Load libcq.so (must have been built: build() / __graft_entry__.build()).  Raises if missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CQError(f"{LIB_PATH} is missing: run __graft_entry__.build() (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        vp, i32, u32, f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_float
        L.cq_last_error.restype = C.c_char_p
        L.cq_version.restype = C.c_char_p
        L.cq_host_alloc.restype = vp
        L.cq_host_alloc.argtypes = [C.c_size_t]
        L.cq_host_free.argtypes = [vp]
        L.cq_world_create.argtypes = [vp, i32, C.POINTER(vp)]
        L.cq_world_create_ex.argtypes = [vp, i32, vp, C.POINTER(vp)]
        L.cq_world_options_default.argtypes = [vp]
        L.cq_raycast_batch_ex.argtypes = [vp, vp, i32, vp, vp]
        L.cq_capsule_cast_batch_ex.argtypes = [vp, vp, i32, i32, vp, vp]
        L.cq_capsule_overlap_batch_ex.argtypes = [vp, vp, i32, vp, vp]
        L.cq_raycast_device_ex.argtypes = [vp, vp, i32, vp, vp, vp]
        L.cq_capsule_cast_device_ex.argtypes = [vp, vp, i32, i32, vp, vp, vp]
        L.cq_capsule_overlap_device_ex.argtypes = [vp, vp, i32, vp, vp, vp]
        L.cq_world_destroy.argtypes = [vp]
        L.cq_world_get_info.argtypes = [vp, C.POINTER(WorldInfo)]
        L.cq_world_update_transforms.argtypes = [vp, vp, vp, i32]
        L.cq_world_update_transforms_async.argtypes = [vp, vp, vp, i32, vp]
        L.cq_world_read_soup.argtypes = [vp, i32, vp, vp, vp, vp, vp]
        L.cq_world_triangle_material.argtypes = [vp, i32, C.POINTER(Material)]
        L.cq_static_mesh_load.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.cq_static_mesh_free.argtypes = [vp]
        L.cq_static_mesh_part_count.argtypes = [vp]
        L.cq_static_mesh_part_name.restype = C.c_char_p
        L.cq_static_mesh_part_name.argtypes = [vp, i32]
        L.cq_static_mesh_part_transform.argtypes = [vp, i32, vp]
        L.cq_static_mesh_hull_count.argtypes = [vp, i32]
        L.cq_static_mesh_geometry.argtypes = [vp, i32, i32, C.POINTER(vp), C.POINTER(i32), C.POINTER(vp),
                                              C.POINTER(i32)]
        L.cq_raycast_batch.argtypes = [vp, vp, i32, vp]
        L.cq_capsule_cast_batch.argtypes = [vp, vp, i32, i32, vp]
        L.cq_capsule_overlap_batch.argtypes = [vp, vp, i32, vp]
        L.cq_capsule_overlap_all_batch.argtypes = [vp, vp, i32, i32, vp, vp, vp]
        L.cq_raycast_device.argtypes = [vp, vp, i32, vp, vp]
        L.cq_capsule_cast_device.argtypes = [vp, vp, i32, i32, vp, vp]
        L.cq_capsule_overlap_device.argtypes = [vp, vp, i32, vp, vp]
        L.cq_capsule_overlap_all_device.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp]
        L.cq_controller_params_default.argtypes = [vp]
        L.cq_character_state_init.argtypes = [vp, vp, vp]
        L.cq_move_and_slide_batch.argtypes = [vp, vp, i32, vp, f32, vp, u32]
        L.cq_move_and_slide_device.argtypes = [vp, vp, i32, vp, f32, vp, u32, vp]
        L.cq_move_and_slide_batch_ex.argtypes = [vp, vp, i32, vp, f32, vp, u32, vp, i32]
        L.cq_move_and_slide_device_ex.argtypes = [vp, vp, i32, vp, f32, vp, u32, vp, i32, vp]
        L.cq_agent_separation_batch.argtypes = [vp, vp, i32, vp, vp, i32, f32, f32, i32]
        L.cq_agent_separation_device.argtypes = [vp, vp, i32, vp, vp, i32, f32, f32, i32, vp]
        L.cq_crowd_create.argtypes = [vp, vp, i32, C.POINTER(vp)]
        L.cq_crowd_destroy.argtypes = [vp]
        L.cq_crowd_size.argtypes = [vp]
        L.cq_crowd_step.argtypes = [vp, vp, vp, f32, vp, u32, vp, i32, vp]
        L.cq_crowd_read.argtypes = [vp, vp]
        L.cq_crowd_write.argtypes = [vp, vp]
        L.cq_crowd_device_states.argtypes = [vp]
        L.cq_crowd_device_states.restype = vp
        i64, sz = C.c_int64, C.c_size_t
        L.cq_shard_range.restype = None
        L.cq_shard_range.argtypes = [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]
        L.cq_group_unique_id.argtypes = [vp]
        L.cq_group_create_rank.argtypes = [i32, i32, vp, C.POINTER(vp)]
        L.cq_group_create_local.argtypes = [i32, vp, C.POINTER(vp)]
        L.cq_group_destroy.argtypes = [vp]
        L.cq_group_destroy.restype = None
        L.cq_group_size.argtypes = [vp]
        L.cq_group_rank.argtypes = [vp]
        L.cq_group_device.argtypes = [vp, i32]
        L.cq_group_gather_records.argtypes = [vp, vp, i64, sz, vp, vp]
        L.cq_group_gather_records_local.argtypes = [vp, vp, i64, sz, vp, vp]
        L.cq_group_synchronize.argtypes = [vp]
        L.cq_world_create_multi.argtypes = [vp, vp, i32, vp, C.POINTER(vp)]
        L.cq_multi_world_destroy.argtypes = [vp]
        L.cq_multi_world_destroy.restype = None
        L.cq_multi_world_size.argtypes = [vp]
        L.cq_multi_world_replica.argtypes = [vp, i32]
        L.cq_multi_world_replica.restype = vp
        L.cq_multi_update_transforms.argtypes = [vp, vp, vp, i32]
        L.cq_multi_raycast_batch.argtypes = [vp, vp, i32, vp]
        L.cq_multi_capsule_cast_batch.argtypes = [vp, vp, i32, i32, vp]
        L.cq_multi_move_and_slide_batch.argtypes = [vp, vp, i32, vp, f32, vp, u32]
        L.cq_world_set_counting.argtypes = [vp, i32]
        L.cq_world_read_counters.argtypes = [vp, C.POINTER(Counters), i32]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise CQError(f"libcq error {rc}: {lib().cq_last_error().decode(errors='replace')}")


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def default_params(**over):
    p = np.zeros(1, PARAMS)
    lib().cq_controller_params_default(_ptr(p))
    for k, v in over.items():
        p[k] = v
    return p


def init_states(positions, velocities=None):
    positions = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
    n = positions.shape[0]
    vel = None if velocities is None else np.ascontiguousarray(velocities, np.float32).reshape(-1, 3)
    s = np.zeros(n, STATE)
    L = lib()
    for i in range(n) if n <= 4096 else ():
        L.cq_character_state_init(C.c_void_p(s.ctypes.data + i * STATE.itemsize), _ptr(positions[i]),
                                  _ptr(vel[i]) if vel is not None else None)
    if n > 4096:  # vectorised equivalent of cq_character_state_init
        s["position"] = positions.astype(np.float64)
        if vel is not None:
            s["velocity"] = vel.astype(np.float64)
        s["ground_normal"] = (0, 1, 0)
        s["ground_distance"] = np.finfo(np.float32).max
        s["ground_triangle_index"] = -1
    return s


class PinnedArray:
    """numpy view over cq_host_alloc'ed (page-locked) memory."""

    def __init__(self, shape, dtype):
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        self._p = lib().cq_host_alloc(max(n, 1))
        if not self._p:
            raise CQError("cq_host_alloc failed (no CUDA device?)")
        buf = (C.c_char * max(n, 1)).from_address(self._p)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p:
            self.array = None
            lib().cq_host_free(self._p)
            self._p = None


class StaticMeshAsset:
    """StaticMeshLoader.loadStaticMeshAsset(named:) (StaticMeshLoader.swift:30-125) through the C ABI.
    Returns None-like failure as CQError with the code (the reference returns nil and prints)."""

    def __init__(self, path):
        h = C.c_void_p()
        _check(lib().cq_static_mesh_load(os.fsencode(path), C.byref(h)))
        self._h = h
        L = lib()
        self.parts = []
        for p in range(L.cq_static_mesh_part_count(h)):
            tr = np.zeros(16, np.float32)
            _check(L.cq_static_mesh_part_transform(h, p, _ptr(tr)))

            def geom(hull):
                pp, ip, nv, ni = C.c_void_p(), C.c_void_p(), C.c_int32(), C.c_int32()
                _check(L.cq_static_mesh_geometry(h, p, hull, C.byref(pp), C.byref(nv), C.byref(ip), C.byref(ni)))
                pos = np.ctypeslib.as_array(C.cast(pp, C.POINTER(C.c_float)), (nv.value * 3,)).copy().reshape(-1, 3)
                idx = np.ctypeslib.as_array(C.cast(ip, C.POINTER(C.c_uint32)), (ni.value,)).copy()
                return pos, idx

            pos, idx = geom(-1)
            hulls = [geom(k) for k in range(L.cq_static_mesh_hull_count(h, p))]
            self.parts.append({"name": L.cq_static_mesh_part_name(h, p).decode(), "transform": tr,
                               "positions": pos, "indices": idx, "hulls": hulls})
        L.cq_static_mesh_free(h)
        self._h = None


class CollisionQuery:
    """Mirror of the reference's `final class CollisionQuery` (CollisionQuery.swift:54-160), batched.

    parts: list of dicts as produced by scenes.part(): the (TransformComponent, StaticMeshComponent,
    body type) of every collidable entity, in entity-id order.
    Batch methods take numpy record arrays (host) and return numpy record arrays; `*_device` methods
    take raw device pointers (e.g. torch tensor .data_ptr()) and enqueue on a CUDA stream."""

    def __init__(self, parts, order=ORDER_REFERENCE):
        """order: ORDER_REFERENCE (default: exact ties and overlap-all overflow resolved in the reference's own visiting
        order, raycasts walk the reference's own tree) or ORDER_CANONICAL (tree-independent rule); include/cq.h."""
        self._keep = []
        self.order = order
        arr = (MeshPart * max(len(parts), 1))()
        for i, p in enumerate(parts):
            pos = np.ascontiguousarray(p["positions"], np.float32).reshape(-1, 3)
            idx = np.ascontiguousarray(p["indices"], np.uint32).reshape(-1)
            self._keep += [pos, idx]
            arr[i].positions_xyz = pos.ctypes.data
            arr[i].indices = idx.ctypes.data
            arr[i].n_verts = pos.shape[0]
            arr[i].n_indices = idx.shape[0]
            m = np.asarray(p["model"], np.float32).reshape(16)
            for k in range(16):
                arr[i].model[k] = float(m[k])
            arr[i].layer = int(p.get("layer", 1))
            arr[i].mu_s = float(p.get("mu_s", 0.8))
            arr[i].mu_k = float(p.get("mu_k", 0.6))
            arr[i].flatten_ground = int(bool(p.get("flatten_ground", False)))
            arr[i].is_dynamic = int(bool(p.get("is_dynamic", False)))
            arr[i].entity_id = int(p.get("entity_id", i))
        h = C.c_void_p()
        opt = _world_options(parts, order, self._keep)
        _check(lib().cq_world_create_ex(C.byref(arr), len(parts), C.byref(opt), C.byref(h)))
        self._h = h
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            lib().cq_world_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def info(self):
        i = WorldInfo()
        _check(lib().cq_world_get_info(self._h, C.byref(i)))
        return {n: getattr(i, n) for n, _ in WorldInfo._fields_}

    def read_soup(self, which=0):
        inf = self.info()
        nv = inf["n_dynamic_vertices"] if which else inf["n_static_vertices"]
        nt = inf["n_dynamic_triangles"] if which else inf["n_static_triangles"]
        pos = np.zeros((nv, 3), np.float32)
        idx = np.zeros((nt, 3), np.uint32)
        aabb = np.zeros((nt, 6), np.float32)
        lay = np.zeros(nt, np.uint32)
        par = np.zeros(nt, np.int32)
        _check(lib().cq_world_read_soup(self._h, which, _ptr(pos), _ptr(idx), _ptr(aabb), _ptr(lay), _ptr(par)))
        return {"positions": pos, "indices": idx, "aabbs": aabb, "layers": lay, "parts": par}

    def triangle_material(self, triangle_index):
        m = Material()
        _check(lib().cq_world_triangle_material(self._h, int(triangle_index), C.byref(m)))
        return {"mu_s": m.mu_s, "mu_k": m.mu_k, "flatten_ground": bool(m.flatten_ground)}

    # updateStaticTransforms / updateDynamicTransforms (CollisionQuery.swift:69-83)
    def update_transforms(self, entity_ids, models):
        ids = np.ascontiguousarray(entity_ids, np.uint32)
        m = np.ascontiguousarray(models, np.float32).reshape(-1, 16)
        assert m.shape[0] == ids.shape[0]
        _check(lib().cq_world_update_transforms(self._h, _ptr(ids), _ptr(m), len(ids)))

    updateStaticTransforms = update_transforms
    updateDynamicTransforms = update_transforms

    def update_transforms_async(self, entity_ids, models, stream=None):
        """cq_world_update_transforms_async: the same update queued on `stream` (a cudaStream_t handle such as
        torch.cuda.Stream().cuda_stream; None = the world's own stream) without synchronising.  The arrays are copied
        before the call returns; every later call on the world, on any stream, sees the new pose."""
        ids = np.ascontiguousarray(entity_ids, np.uint32)
        m = np.ascontiguousarray(models, np.float32).reshape(-1, 16)
        assert m.shape[0] == ids.shape[0]
        _check(lib().cq_world_update_transforms_async(self._h, _ptr(ids), _ptr(m), len(ids), C.c_void_p(stream) if stream else None))

    # raycast(origin:direction:maxDistance:mask:) (CollisionQuery.swift:85)
    def raycast(self, rays, with_flags=False):
        """with_flags: also return the per-query HIT_* flag bytes (cq_raycast_batch_ex)."""
        rays = np.ascontiguousarray(rays, RAY)
        out = np.zeros(len(rays), RAY_HIT)
        flags = np.zeros(len(rays), np.uint8)
        _check(lib().cq_raycast_batch_ex(self._h, _ptr(rays), len(rays), _ptr(out), _ptr(flags) if with_flags else None))
        return (out, flags) if with_flags else out

    def _cast(self, q, mode, with_flags=False):
        q = np.ascontiguousarray(q, CAST)
        out = np.zeros(len(q), CAST_HIT)
        flags = np.zeros(len(q), np.uint8)
        _check(lib().cq_capsule_cast_batch_ex(self._h, _ptr(q), len(q), mode, _ptr(out), _ptr(flags) if with_flags else None))
        return (out, flags) if with_flags else out

    def capsuleCast(self, q, with_flags=False):  # CollisionQuery.swift:96
        return self._cast(q, CAST_ALL, with_flags)

    def capsuleCastBlocking(self, q, with_flags=False):  # CollisionQuery.swift:109
        return self._cast(q, CAST_BLOCKING, with_flags)

    def capsuleCastGround(self, q, with_flags=False):  # CollisionQuery.swift:122 (minNormalY = q["min_normal_y"])
        return self._cast(q, CAST_GROUND, with_flags)

    def capsuleOverlap(self, q, with_flags=False):  # CollisionQuery.swift:137
        q = np.ascontiguousarray(q, CAPSULE)
        out = np.zeros(len(q), OVERLAP_HIT)
        flags = np.zeros(len(q), np.uint8)
        _check(lib().cq_capsule_overlap_batch_ex(self._h, _ptr(q), len(q), _ptr(out), _ptr(flags) if with_flags else None))
        return (out, flags) if with_flags else out

    def capsuleOverlapAll(self, q, max_hits=8):  # CollisionQuery.swift:148
        q = np.ascontiguousarray(q, CAPSULE)
        max_hits = max(1, int(max_hits))
        out = np.zeros((len(q), max_hits), OVERLAP_HIT)
        counts = np.zeros(len(q), np.int32)
        overflow = np.zeros(len(q), np.uint8)
        _check(lib().cq_capsule_overlap_all_batch(self._h, _ptr(q), len(q), max_hits, _ptr(out), _ptr(counts),
                                                  _ptr(overflow)))
        return out, counts, overflow

    # KinematicMoveStopSystem.fixedUpdate body for a batch (Systems.swift:1842-1901)
    def move_and_slide(self, states, params, dt=1.0 / 60.0, gravity=(0.0, -98.0, 0.0), flags=MAS_APPLY_GRAVITY,
                       platforms=None):
        """platforms: optional PLATFORM record array (kinematic platforms: world AABB + motion of this step)."""
        assert states.dtype == STATE and states.flags["C_CONTIGUOUS"]
        params = np.ascontiguousarray(params, PARAMS)
        g = np.asarray(gravity, np.float32)
        pl = np.ascontiguousarray(platforms if platforms is not None else np.zeros(0, PLATFORM), PLATFORM)
        _check(lib().cq_move_and_slide_batch_ex(self._h, _ptr(states), len(states), _ptr(params), C.c_float(dt), _ptr(g),
                                                flags, _ptr(pl), len(pl)))
        return states

    def agent_separation(self, states, params, mass_weight=None, iterations=2, separation_margin=0.2, height_margin=0.1,
                         use_query=True):
        """AgentSeparationSystem.fixedUpdate over the batch (Systems.swift:1906-2210), in place, sequential semantics."""
        assert states.dtype == STATE and states.flags["C_CONTIGUOUS"]
        params = np.ascontiguousarray(params, PARAMS)
        mw = None if mass_weight is None else np.ascontiguousarray(mass_weight, np.float32)
        assert mw is None or len(mw) == len(states)
        _check(lib().cq_agent_separation_batch(self._h, _ptr(states), len(states), _ptr(params),
                                               None if mw is None else _ptr(mw), iterations, separation_margin,
                                               height_margin, 1 if use_query else 0))
        return states

    def agent_separation_device(self, d_states_ptr, n, params, d_mass_weight_ptr=None, iterations=2, separation_margin=0.2,
                                height_margin=0.1, use_query=True, stream=None):
        params = np.ascontiguousarray(params, PARAMS)
        _check(lib().cq_agent_separation_device(self._h, C.c_void_p(d_states_ptr), n, _ptr(params),
                                                C.c_void_p(d_mass_weight_ptr) if d_mass_weight_ptr else None, iterations,
                                                separation_margin, height_margin, 1 if use_query else 0,
                                                C.c_void_p(stream) if stream else None))

    def move_and_slide_device(self, d_states_ptr, n, params, dt=1.0 / 60.0, gravity=(0.0, -98.0, 0.0),
                              flags=MAS_APPLY_GRAVITY, stream=None):
        params = np.ascontiguousarray(params, PARAMS)
        g = np.asarray(gravity, np.float32)
        _check(lib().cq_move_and_slide_device(self._h, C.c_void_p(d_states_ptr), n, _ptr(params), C.c_float(dt),
                                              _ptr(g), flags, C.c_void_p(stream) if stream else None))

    def capsule_cast_device(self, d_q_ptr, n, mode, d_out_ptr, stream=None):
        _check(lib().cq_capsule_cast_device(self._h, C.c_void_p(d_q_ptr), n, mode, C.c_void_p(d_out_ptr),
                                            C.c_void_p(stream) if stream else None))

    def raycast_device(self, d_rays_ptr, n, d_out_ptr, stream=None):
        _check(lib().cq_raycast_device(self._h, C.c_void_p(d_rays_ptr), n, C.c_void_p(d_out_ptr),
                                       C.c_void_p(stream) if stream else None))

    # CollisionQuery.stats / resetStats (CollisionQuery.swift:61-67)
    def set_counting(self, mode):
        """False / COUNT_OFF; True / COUNT_REFERENCE: `candidates` equals the reference's capsuleCandidateCount;
        COUNT_PATH: the counters of the path as shipped (bestT-based culling active) — see cq.h."""
        _check(lib().cq_world_set_counting(self._h, int(mode)))

    def stats(self, reset=False):
        c = Counters()
        _check(lib().cq_world_read_counters(self._h, C.byref(c), int(reset)))
        return c.as_dict()

    def resetStats(self):
        self.stats(reset=True)


def _mesh_parts(parts, keep):
    arr = (MeshPart * max(len(parts), 1))()
    for i, p in enumerate(parts):
        pos = np.ascontiguousarray(p["positions"], np.float32).reshape(-1, 3)
        idx = np.ascontiguousarray(p["indices"], np.uint32).reshape(-1)
        keep += [pos, idx]
        arr[i].positions_xyz = pos.ctypes.data
        arr[i].indices = idx.ctypes.data
        arr[i].n_verts = pos.shape[0]
        arr[i].n_indices = idx.shape[0]
        m = np.asarray(p["model"], np.float32).reshape(16)
        for k in range(16):
            arr[i].model[k] = float(m[k])
        arr[i].layer = int(p.get("layer", 1))
        arr[i].mu_s = float(p.get("mu_s", 0.8))
        arr[i].mu_k = float(p.get("mu_k", 0.6))
        arr[i].flatten_ground = int(bool(p.get("flatten_ground", False)))
        arr[i].is_dynamic = int(bool(p.get("is_dynamic", False)))
        arr[i].entity_id = int(p.get("entity_id", i))
    return arr


def shard_range(n_units, n_ranks, rank):
    """cq_shard_range: the contiguous range [lo, hi) of `rank` (the same rule as shard.rank_range)."""
    lo, hi = C.c_int64(), C.c_int64()
    lib().cq_shard_range(n_units, n_ranks, rank, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


class Group:
    """The GPUs of one box (include/cq.h: cq_group_*).  Group.local(n) = one process driving n devices;
    Group.rank(n_ranks, rank, id) = one process per GPU (the 128-byte id comes from Group.unique_id() on rank 0)."""

    def __init__(self, handle):
        self._h = handle

    @staticmethod
    def unique_id():
        buf = np.zeros(GROUP_ID_BYTES, np.uint8)
        _check(lib().cq_group_unique_id(_ptr(buf)))
        return buf

    @classmethod
    def rank(cls, n_ranks, rank, uid):
        uid = np.ascontiguousarray(uid, np.uint8)
        assert uid.shape == (GROUP_ID_BYTES,)
        h = C.c_void_p()
        _check(lib().cq_group_create_rank(n_ranks, rank, _ptr(uid), C.byref(h)))
        return cls(h)

    @classmethod
    def local(cls, n_gpus, devices=None):
        dv = None if devices is None else np.ascontiguousarray(devices, np.int32)
        h = C.c_void_p()
        _check(lib().cq_group_create_local(n_gpus, None if dv is None else _ptr(dv), C.byref(h)))
        return cls(h)

    @property
    def handle(self):
        return self._h

    @property
    def size(self):
        return lib().cq_group_size(self._h)

    def gather_records(self, d_local_ptr, n_units, record_bytes, d_all_ptr, stream=None):
        """Process-per-GPU groups: NCCL all-gather of this rank's shard of the result records into d_all (device)."""
        _check(lib().cq_group_gather_records(self._h, C.c_void_p(d_local_ptr), n_units, record_bytes, C.c_void_p(d_all_ptr),
                                             C.c_void_p(stream) if stream else None))

    def gather_records_local(self, d_local_ptrs, n_units, record_bytes, d_all_ptrs, streams=None):
        n = self.size
        loc = (C.c_void_p * n)(*[C.c_void_p(int(p)) for p in d_local_ptrs])
        al = (C.c_void_p * n)(*[C.c_void_p(int(p)) for p in d_all_ptrs])
        st = None if streams is None else (C.c_void_p * n)(*[C.c_void_p(int(p)) for p in streams])
        _check(lib().cq_group_gather_records_local(self._h, loc, n_units, record_bytes, al, st))

    def synchronize(self):
        _check(lib().cq_group_synchronize(self._h))

    def close(self):
        if getattr(self, "_h", None):
            lib().cq_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiWorld:
    """cq_world_create_multi: the world replicated on every device of a local Group; host batches are sharded over the
    replicas (contiguous ranges, one worker thread per device).  Same results as CollisionQuery, byte for byte."""

    def __init__(self, group, parts, order=ORDER_REFERENCE):
        keep = []
        arr = _mesh_parts(parts, keep)
        opt = _world_options(parts, order, keep)
        h = C.c_void_p()
        _check(lib().cq_world_create_multi(group.handle, C.byref(arr), len(parts), C.byref(opt), C.byref(h)))
        self._h, self._group, self.order = h, group, order

    def close(self):
        if getattr(self, "_h", None):
            lib().cq_multi_world_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def replica(self, i):
        return lib().cq_multi_world_replica(self._h, i)

    def update_transforms(self, entity_ids, models):
        ids = np.ascontiguousarray(entity_ids, np.uint32)
        m = np.ascontiguousarray(models, np.float32).reshape(-1, 16)
        _check(lib().cq_multi_update_transforms(self._h, _ptr(ids), _ptr(m), len(ids)))

    def raycast(self, rays):
        rays = np.ascontiguousarray(rays, RAY)
        out = np.zeros(len(rays), RAY_HIT)
        _check(lib().cq_multi_raycast_batch(self._h, _ptr(rays), len(rays), _ptr(out)))
        return out

    def capsule_cast(self, q, mode=CAST_ALL):
        q = np.ascontiguousarray(q, CAST)
        out = np.zeros(len(q), CAST_HIT)
        _check(lib().cq_multi_capsule_cast_batch(self._h, _ptr(q), len(q), mode, _ptr(out)))
        return out

    def move_and_slide(self, states, params, dt=1.0 / 60.0, gravity=(0.0, -98.0, 0.0), flags=MAS_APPLY_GRAVITY):
        assert states.dtype == STATE and states.flags["C_CONTIGUOUS"]
        params = np.ascontiguousarray(params, PARAMS)
        g = np.asarray(gravity, np.float32)
        _check(lib().cq_multi_move_and_slide_batch(self._h, _ptr(states), len(states), _ptr(params), C.c_float(dt), _ptr(g), flags))
        return states


class Crowd:
    """Resident crowd (include/cq.h: cq_crowd_*): the character records live in HBM between steps; `step` moves
    velocities in and poses out.  Same results as CollisionQuery.move_and_slide on the same records, bit for bit."""

    def __init__(self, world, states):
        assert states.dtype == STATE and states.flags["C_CONTIGUOUS"]
        self._world = world  # keeps the world alive: a crowd must be destroyed before its world
        h = C.c_void_p()
        _check(lib().cq_crowd_create(world.handle, _ptr(states), len(states), C.byref(h)))
        self._h = h
        self.n = len(states)

    def close(self):
        if getattr(self, "_h", None):
            lib().cq_crowd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step(self, velocity, params, dt=1.0 / 60.0, gravity=(0.0, -98.0, 0.0), flags=MAS_APPLY_GRAVITY, platforms=None,
             pose_out=None):
        """velocity: (n, 3) float64 array or None (keep the stored velocities); pose_out: CROWD_POSE array of n records
        or None.  Returns pose_out."""
        params = np.ascontiguousarray(params, PARAMS)
        g = np.asarray(gravity, np.float32)
        pl = np.ascontiguousarray(platforms if platforms is not None else np.zeros(0, PLATFORM), PLATFORM)
        if velocity is not None:
            assert velocity.dtype == np.float64 and velocity.shape == (self.n, 3) and velocity.flags["C_CONTIGUOUS"]
        if pose_out is not None:
            assert pose_out.dtype == CROWD_POSE and pose_out.shape == (self.n,) and pose_out.flags["C_CONTIGUOUS"]
        _check(lib().cq_crowd_step(self._h, None if velocity is None else _ptr(velocity), _ptr(params), C.c_float(dt), _ptr(g),
                                   flags, _ptr(pl) if len(pl) else None, len(pl), None if pose_out is None else _ptr(pose_out)))
        return pose_out

    def read(self):
        out = np.zeros(self.n, STATE)
        _check(lib().cq_crowd_read(self._h, _ptr(out)))
        return out

    def write(self, states):
        assert states.dtype == STATE and states.shape == (self.n,) and states.flags["C_CONTIGUOUS"]
        _check(lib().cq_crowd_write(self._h, _ptr(states)))

    @property
    def device_states(self):
        return lib().cq_crowd_device_states(self._h)
