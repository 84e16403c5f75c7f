"""Transform updates on one GPU: cq_world_update_transforms_async (host arrays) against cq_world_update_transforms_device
(device arrays), and a CUDA graph of a fixed step.  Prints one JSON line and writes it to --out (default
profiles/r5_refit_device_probe.json).

  platforms  the bench terrain plus 4,096 dynamic 12-triangle boxes; per update N random boxes move (N = 256: the
             dirty-subtree refit; N = 1,024 = a quarter of the set's triangles: the full fit), in both orders.  For the
             async and the device call: kernel launches per update (cq_world_read_counters), device ms per update (CUDA
             events around back-to-back updates on one stream) and host ms per call (wall time of the enqueue loop).
  c5         the scene and ray count of `bench.py --only c5` (16,777,216 rays, the mirror spinning in the dynamic set):
             ms per step of "refit + rays" three ways: uncaptured with the async update, uncaptured with the device
             update, and one captured torch.cuda.CUDAGraph (device update + ray batch) replayed; CUDA events around the
             loop, builds alternated --rounds times.  The last step's hit records of the three loops are compared byte
             for byte.  host_ms = host time of the enqueue loop per step.

Usage: python tools/refit_device_probe.py [--steps K] [--warmup W] [--rounds R] [--out PATH]
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from refit_async_probe import gpu_identity  # noqa: E402


def load_package():
    sys.path.insert(0, ROOT)
    sys.dont_write_bytecode = True
    return importlib.import_module("swift-game-engine_b200")


def measure_platforms(cq, torch, steps, warmup):
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
            dev = [(torch.from_numpy(ids.view(np.int32)).cuda(), torch.from_numpy(m).cuda()) for ids, m in seq]
            row = {}
            for call in ("async", "device"):
                def update(k):
                    if call == "async":
                        world.update_transforms_async(seq[k][0], seq[k][1], stream=st)
                    else:
                        world.update_transforms_device(dev[k][0].data_ptr(), dev[k][1].data_ptr(), n_moved, None, st)
                for k in range(warmup):
                    update(k)
                torch.cuda.synchronize()
                world.stats(reset=True)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                t0 = time.perf_counter()
                for k in range(warmup, warmup + steps):
                    update(k)
                host = time.perf_counter() - t0
                e1.record(stream)
                torch.cuda.synchronize()
                row[f"{call}_ms_per_update"] = round(e0.elapsed_time(e1) / steps, 4)
                row[f"{call}_host_ms_per_call"] = round(host * 1e3 / steps, 4)
                row[f"{call}_launches_per_update"] = world.stats()["kernel_launches"] / steps
            out[f"{order_name}_moved{n_moved}"] = row
        world.close()
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
    d_id = torch.tensor([mirror_id], dtype=torch.int32).cuda()
    d_model = torch.zeros(16, dtype=torch.float32, device="cuda")  # the buffer the device update (and the graph) reads
    stream = torch.cuda.Stream()
    st = stream.cuda_stream

    def pose(angle):
        return sc.trs_model(base_t, sc.quat_mul(sc.quat_angle_axis(np.radians(angle), (0, 1, 0)), base_q), base_s)

    host_poses = [np.asarray(pose(float(k + 1)), np.float32).reshape(16) for k in range(warmup + steps)]
    d_poses = torch.from_numpy(np.stack(host_poses)).cuda()  # step k copies its pose into d_model on the device

    def loop(call):
        world = cq.CollisionQuery(parts)
        graph = None

        def device_step():
            cur = torch.cuda.current_stream().cuda_stream
            world.update_transforms_device(d_id.data_ptr(), d_model.data_ptr(), 1, None, cur)
            world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), cur)

        def step(k, captured):
            if call == "async":
                world.update_transforms_async([mirror_id], [host_poses[k]], stream=st)
                world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), st)
                return
            d_model.copy_(d_poses[k])
            graph.replay() if captured else device_step()

        with torch.cuda.stream(stream):
            for k in range(warmup):
                step(k, False)
            torch.cuda.synchronize()
            if call == "graph":
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=stream):
                    device_step()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            t0 = time.perf_counter()
            for k in range(warmup, warmup + steps):
                step(k, call == "graph")
            host = time.perf_counter() - t0
            e1.record(stream)
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        last = d_out.cpu().numpy().tobytes()
        del graph
        world.close()
        return ms, host * 1e3 / steps, last

    res = {k: [] for k in ("async_ms_per_step", "device_ms_per_step", "graph_ms_per_step",
                           "async_host_ms", "device_host_ms", "graph_host_ms")}
    same = True
    for _ in range(rounds):
        lasts = []
        for call in ("async", "device", "graph"):
            ms, host, last = loop(call)
            res[f"{call}_ms_per_step"].append(round(ms, 4))
            res[f"{call}_host_ms"].append(round(host, 4))
            lasts.append(last)
        same = same and lasts[0] == lasts[1] == lasts[2]
    res["last_step_hits_identical"] = same
    res.update(rays=n, steps=steps, warmup=warmup, rounds=rounds)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_refit_device_probe.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("refit_device_probe: no CUDA device (the library has no CPU path)")
    cq = load_package()
    cq.build()
    line = {"probe": "refit_device", **gpu_identity()}
    line["platforms"] = measure_platforms(cq, torch, args.steps, args.warmup)
    line["c5"] = measure_c5(cq, torch, args.steps, args.warmup, args.rounds)
    text = json.dumps(line)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
