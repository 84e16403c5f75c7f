"""Transform updates on one GPU: cq_world_update_transforms against cq_world_update_transforms_async.  Prints one JSON
line and writes it to --out (default profiles/r4_refit_async_probe.json).

  c5         the scene and ray count of `bench.py --only c5` (16,777,216 rays, the mirror spinning in the dynamic set):
             ms per step of "refit + rays" with the synchronous call, and with the async call queued on the ray stream
             (CUDA events around the loop, builds alternated --rounds times); the last step's hit records of the two
             loops are compared byte for byte.  ray_ms = one ray batch alone, refit_ms = the synchronous refit's own
             device time.
  platforms  the bench terrain plus 4,096 dynamic 12-triangle boxes; per update N random boxes move (N = 256: the
             dirty-subtree refit; N = 1,024 = a quarter of the set's triangles: the full fit), in both orders:
             kernel launches per update (cq_world_read_counters), ms per update of the synchronous call (host wall time,
             the call synchronises) and of the async call (CUDA events around back-to-back updates on one stream, and
             the host time of one call).
  parent     --parent-tree DIR: the platforms figure of another checkout (its own package and libcq.so, already built),
             run in a subprocess; it has the synchronous call only.

Usage: python tools/refit_async_probe.py [--steps K] [--warmup W] [--rounds R] [--parent-tree DIR] [--out PATH]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_package(tree):
    sys.path.insert(0, tree)
    sys.dont_write_bytecode = True
    return importlib.import_module("swift-game-engine_b200")


def gpu_identity():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "not read"
    return out


def measure_c5(cq, torch, steps, warmup, rounds):
    sc = cq.scenes
    parts = sc.merged_scene(mirror_dynamic=True)
    a = sc.load_mirror_fixture()
    base_t, base_q, base_s = sc.transform_from_matrix(sc.mirror_model(a["transform"]))
    mirror_id = parts[-1]["entity_id"]
    lo, hi = sc.scene_aabb(parts[1:])
    n = 1 << 24
    rays = sc.gen_rays(n, lo, hi, seed=0xC0111DE5, max_distance=100.0, expand=5.0, y_range=(0.0, 12.0))
    d_r = torch.from_numpy(np.frombuffer(rays.tobytes(), np.uint8).copy()).cuda()
    d_out = torch.empty(n * cq.RAY_HIT.itemsize, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    st = stream.cuda_stream

    def pose(angle):
        return sc.trs_model(base_t, sc.quat_mul(sc.quat_angle_axis(np.radians(angle), (0, 1, 0)), base_q), base_s)

    def loop(call):
        world = cq.CollisionQuery(parts)
        update = world.update_transforms if call == "sync" else (lambda i, m: world.update_transforms_async(i, m, stream=st))
        angle = 0.0
        for _ in range(warmup):
            angle += 1.0
            update([mirror_id], [pose(angle)])
            world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), st)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        refit = []
        e0.record(stream)
        for _ in range(steps):
            angle += 1.0
            update([mirror_id], [pose(angle)])
            world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), st)
            if call == "sync":
                refit.append(world.info()["refit_ms"])
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        last = d_out.cpu().numpy().tobytes()
        e0.record(stream)
        world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), st)
        e1.record(stream)
        torch.cuda.synchronize()
        ray_ms = e0.elapsed_time(e1)
        world.close()
        return ms, last, ray_ms, (float(np.mean(refit)) if refit else None)

    res = {"sync_ms_per_step": [], "async_ms_per_step": [], "ray_ms": [], "sync_refit_ms": []}
    same = True
    for _ in range(rounds):
        ms_s, last_s, ray_s, refit_s = loop("sync")
        ms_a, last_a, ray_a, _ = loop("async")
        same = same and last_s == last_a
        res["sync_ms_per_step"].append(round(ms_s, 4))
        res["async_ms_per_step"].append(round(ms_a, 4))
        res["ray_ms"] += [round(ray_s, 4), round(ray_a, 4)]
        res["sync_refit_ms"].append(round(refit_s, 4))
    res["last_step_hits_identical"] = same
    res.update(rays=n, steps=steps, warmup=warmup, rounds=rounds)
    return res


def measure_platforms(cq, torch, steps, warmup, sync_only):
    sc = cq.scenes
    tv, ti, half = sc.terrain_mesh()
    bv, bi = sc.box_mesh(2.0)
    rng = np.random.default_rng(0xB0C5)
    n_boxes = 4096
    spots = rng.uniform(-0.9 * half, 0.9 * half, (n_boxes, 2)).astype(np.float32)
    heights = sc.terrain_height(spots[:, 0], spots[:, 1]) + 2.0
    parts = [sc.part(tv, ti, entity_id=0)]
    for k in range(n_boxes):
        parts.append(sc.part(bv, bi, sc.trs_model((spots[k, 0], heights[k], spots[k, 1])), is_dynamic=True, entity_id=1 + k))
    stream = torch.cuda.Stream()
    st = stream.cuda_stream
    out = {"boxes": n_boxes, "terrain_triangles": int(len(ti) // 3), "steps": steps, "warmup": warmup}

    def moves(n_moved, count, seed):
        r = np.random.default_rng(seed)
        res = []
        for s in range(count):
            ids = (1 + r.choice(n_boxes, n_moved, replace=False)).astype(np.uint32)
            lift = np.float32(0.1 * (s % 7))
            models = np.stack([sc.trs_model((spots[i - 1, 0], heights[i - 1] + lift, spots[i - 1, 1]),
                                            sc.quat_angle_axis(0.05 * s, (0, 1, 0))) for i in ids]).astype(np.float32)
            res.append((ids, models))
        return res

    for order_name, order in (("reference", cq.ORDER_REFERENCE), ("canonical", cq.ORDER_CANONICAL)):
        world = cq.CollisionQuery(parts, order=order)
        for n_moved in (256, 1024):
            seq = moves(n_moved, warmup + steps, seed=n_moved)
            row = {}
            for call in ("sync",) if sync_only else ("sync", "async"):
                for ids, models in seq[:warmup]:
                    world.update_transforms(ids, models)
                torch.cuda.synchronize()
                world.stats(reset=True)
                if call == "sync":
                    t0 = time.perf_counter()
                    refit = []
                    for ids, models in seq[warmup:]:
                        world.update_transforms(ids, models)
                        refit.append(world.info()["refit_ms"])
                    row["sync_ms_per_update"] = round((time.perf_counter() - t0) * 1e3 / steps, 4)
                    row["sync_refit_ms"] = round(float(np.mean(refit)), 4)
                else:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    t0 = time.perf_counter()
                    for ids, models in seq[warmup:]:
                        world.update_transforms_async(ids, models, stream=st)
                    host = time.perf_counter() - t0
                    e1.record(stream)
                    torch.cuda.synchronize()
                    row["async_ms_per_update"] = round(e0.elapsed_time(e1) / steps, 4)
                    row["async_host_ms_per_call"] = round(host * 1e3 / steps, 4)
                row[f"{call}_launches_per_update"] = world.stats()["kernel_launches"] / steps
            out[f"{order_name}_moved{n_moved}"] = row
        world.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parent-tree", default=None, help="checkout of another commit with its libcq.so built")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_refit_async_probe.json"))
    ap.add_argument("--platforms-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--sync-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--tree", default=ROOT, help=argparse.SUPPRESS)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("refit_async_probe: no CUDA device (the library has no CPU path)")
    cq = load_package(args.tree)
    if args.tree == ROOT:
        cq.build()
    if args.platforms_only:
        print(json.dumps(measure_platforms(cq, torch, args.steps, args.warmup, args.sync_only)))
        return
    line = {"probe": "refit_async", **gpu_identity()}
    line["platforms"] = measure_platforms(cq, torch, args.steps, args.warmup, False)
    if args.parent_tree:
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--platforms-only", "--sync-only", "--tree",
                            os.path.abspath(args.parent_tree), "--steps", str(args.steps), "--warmup", str(args.warmup)],
                           capture_output=True, text=True, env={**os.environ, "PYTHONDONTWRITEBYTECODE": "1"})
        if p.returncode != 0:
            raise SystemExit(f"parent run failed:\n{p.stderr[-4000:]}")
        line["parent_platforms"] = json.loads(p.stdout.strip().splitlines()[-1])
    line["c5"] = measure_c5(cq, torch, args.steps, args.warmup, args.rounds)
    text = json.dumps(line)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
