"""Kinematic platforms read from device memory on one GPU: cq_move_and_slide_device_ex (host-array records in the kernel
arguments) against cq_move_and_slide_device_platforms (records in device memory), and a captured CUDA graph of the
fixed step that rebuilds its records on the device.  Prints one JSON line and writes it to --out (default
profiles/r8_platforms_device_probe.json), with the card's name and power limit read in the same run.

Scene: the C3 hulls world of bench.py (ornate mirror's 2 collision hulls + the ground plane) with P dynamic 1 m boxes as
kinematic platforms, and --chars C3 characters (default 1,048,576).  The first min(P, 16) boxes stand in the characters'
8 x 8 m region, sunk into the ground so that the characters above them ride on them; the others stand outside the region
(their records pass the delta test and fail the overlap test, as a far platform does).  Every platform moves by a
non-zero delta; the models stay put, so every variant sees the same world and the same records on every step.

Variants, for P = 2 and 64 (host arrays hold at most 64) and P = 1,024 (device records only):
  host    cq_move_and_slide_device_ex with the records of scenes.platform_record (host array);
  device  cq_move_and_slide_device_platforms with the same records in a device buffer;
  graph   one torch.cuda.CUDAGraph of cq_world_update_transforms_device (all P models) -> cq_world_platforms_device ->
          cq_move_and_slide_device_platforms, replayed.
ms per step = CUDA events around --steps steps after --warmup uncaptured warm-up steps; the variants alternate within
each of --rounds rounds, every one from the same initial records, and the final records of every variant are compared
byte for byte.  platforms_device_us = CUDA events around --steps back-to-back cq_world_platforms_device calls.

Usage: python tools/platforms_device_probe.py [--steps K] [--warmup W] [--rounds R] [--chars N] [--out PATH]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from refit_async_probe import gpu_identity  # noqa: E402

G3 = np.float32([0.0, -98.0, 0.0])
DT = 1.0 / 60.0


def load_package():
    sys.path.insert(0, ROOT)
    sys.dont_write_bytecode = True
    return importlib.import_module("swift-game-engine_b200")


def platform_scene(cq, n_platforms):
    sc = cq.scenes
    parts = sc.mirror_scene(use_hulls=True)
    bv, bi = sc.box_mesh(1.0)
    rng = np.random.default_rng(0xB1A7)
    inside = min(n_platforms, 16)
    xz = np.concatenate([np.stack([rng.uniform(-13.5, -6.5, inside), rng.uniform(1.0, 8.0, inside)], 1),
                         np.stack([rng.uniform(-38, 38, n_platforms - inside), rng.uniform(-38, -12, n_platforms - inside)], 1)])
    ids = np.arange(1000, 1000 + n_platforms, dtype=np.uint32)
    models = np.stack([sc.trs_model((x, -3.05, z)) for x, z in xz]).astype(np.float32)
    for k in range(n_platforms):
        parts.append(sc.part(bv, bi, models[k], is_dynamic=True, entity_id=int(ids[k])))
    deltas = np.stack([rng.uniform(-0.02, 0.02, n_platforms), rng.uniform(0.0, 0.01, n_platforms),
                       rng.uniform(-0.02, 0.02, n_platforms)], 1).astype(np.float32)
    deltas[:, 1] += np.float32(0.001)  # every platform moves: none is skipped by the delta test
    records = np.concatenate([sc.platform_record(bv, models[k], (0, 0, 0), deltas[k]) for k in range(n_platforms)])
    return parts, ids, models, deltas, np.ascontiguousarray(records, cq.PLATFORM)


def measure(cq, torch, n_platforms, chars, steps, warmup, rounds):
    parts, ids, models, deltas, records = platform_scene(cq, n_platforms)
    g = cq.CollisionQuery(parts)
    pos, vel = cq.scenes.gen_c3_characters(chars, seed=0xC0111DE3)
    init = torch.from_numpy(cq.init_states(pos, vel).view(np.uint8)).cuda()
    d_states = torch.empty_like(init)
    d_ids = torch.from_numpy(ids.view(np.int32).copy()).cuda()
    d_models = torch.from_numpy(models).cuda()
    d_deltas = torch.from_numpy(deltas).cuda()
    d_plats = torch.from_numpy(records.view(np.uint8).copy()).cuda()  # the device variant's records
    d_graph_plats = torch.zeros_like(d_plats)  # written by cq_world_platforms_device inside the graph
    d_status = torch.full((2,), -7, dtype=torch.int32, device="cuda")
    params = np.ascontiguousarray(cq.default_params(), cq.PARAMS)
    L = cq.lib()
    stream = torch.cuda.Stream()
    st = stream.cuda_stream

    def host_step():
        cq._check(L.cq_move_and_slide_device_ex(g.handle, C.c_void_p(d_states.data_ptr()), chars, cq._ptr(params), C.c_float(DT),
                                                cq._ptr(G3), cq.MAS_APPLY_GRAVITY, cq._ptr(records), n_platforms, C.c_void_p(st)))

    def device_step():
        g.move_and_slide_device_platforms(d_states.data_ptr(), chars, params, d_plats.data_ptr(), n_platforms, stream=st)

    def graph_step(s):
        g.update_transforms_device(d_ids.data_ptr(), d_models.data_ptr(), n_platforms, d_status.data_ptr(), s)
        g.platforms_device(d_ids.data_ptr(), d_deltas.data_ptr(), n_platforms, d_graph_plats.data_ptr(), d_status.data_ptr() + 4, s)
        g.move_and_slide_device_platforms(d_states.data_ptr(), chars, params, d_graph_plats.data_ptr(), n_platforms, stream=s)

    d_states.copy_(init)
    torch.cuda.synchronize()
    for _ in range(warmup):  # sizes every scratch block before the capture
        graph_step(st)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        graph_step(torch.cuda.current_stream().cuda_stream)

    variants = {"device": device_step, "graph": lambda: graph.replay()}
    if n_platforms <= 64:
        variants = {"host": host_step, **variants}
    names = list(variants)
    ms = {k: [] for k in names}
    final = {}
    for r in range(rounds):
        for name in names[r % len(names):] + names[:r % len(names)]:
            run = variants[name]
            d_states.copy_(init)
            torch.cuda.synchronize()
            with torch.cuda.stream(stream):
                for _ in range(warmup):
                    run()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(steps):
                    run()
                e1.record(stream)
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / steps)
            got = d_states.cpu().numpy().tobytes()
            final.setdefault(name, got)
            assert final[name] == got, (n_platforms, name, "rounds differ")
    statuses = d_status.cpu().numpy().tolist()
    # cq_world_platforms_device alone
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        for _ in range(warmup):
            g.platforms_device(d_ids.data_ptr(), d_deltas.data_ptr(), n_platforms, d_graph_plats.data_ptr(), None, st)
        e0.record(stream)
        for _ in range(steps):
            g.platforms_device(d_ids.data_ptr(), d_deltas.data_ptr(), n_platforms, d_graph_plats.data_ptr(), None, st)
        e1.record(stream)
    torch.cuda.synchronize()
    dev_records = d_graph_plats.cpu().numpy().view(cq.PLATFORM)
    records_equal = all(np.array_equal(dev_records[k], records[k]) for k in ("aabb_min", "aabb_max", "delta"))
    same = len({final[k] for k in names}) == 1
    del graph
    g.close()
    row = {"platforms": n_platforms, "ms_per_step": {k: [round(v, 4) for v in ms[k]] for k in names},
           "ms_per_step_median": {k: round(float(np.median(ms[k])), 4) for k in names},
           "platforms_device_us": round(e0.elapsed_time(e1) / steps * 1000.0, 2),
           "final_records_identical": same, "device_records_equal_host_records": records_equal,
           "statuses_update_platforms": statuses}
    if not same or not records_equal:
        raise SystemExit(f"platforms_device_probe: results differ: {row}")
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--chars", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_platforms_device_probe.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("platforms_device_probe: no CUDA device (the library has no CPU path)")
    cq = load_package()
    cq.build()
    line = {"probe": "platforms_device", **gpu_identity(), "characters": args.chars, "steps": args.steps, "warmup": args.warmup,
            "rounds": args.rounds, "scene": "C3 hulls + P dynamic 1 m boxes as kinematic platforms"}
    line["runs"] = [measure(cq, torch, p, args.chars, args.steps, args.warmup, args.rounds) for p in (2, 64, 1024)]
    text = json.dumps(line)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
