"""Reference-order build time: this checkout's device cut of the reference's tree against another built checkout of the
repository (for example an earlier commit with the host builder), alternated on the same box.

    python tools/ref_tree_probe.py --old path/to/other/checkout --out profiles/r9_ref_tree_probe.json

Worlds: the 10 M-triangle C4 terrain and the C5 merged scene.  Each (library, world) pair runs in its own subprocess and
creates the world `--creates` times; the libraries alternate `--rounds` times.  Reported per run: ref_order_ms
(cq_world_info: wall time of the reference-order build inside creation), build_ms (LBVH kernels) and the wall time of
cq_world_create, and (where the checkout has it) cq_world_rebuild of the same world.  The card's name and power limit are recorded with the numbers.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def scene(sc, name, cache):
    import numpy as np
    if name == "c5":
        return sc.merged_scene()
    path = os.path.join(cache, "terrain.npz")
    if not os.path.exists(path):
        pos, idx, _ = sc.terrain_mesh()
        np.savez(path, pos=pos, idx=idx)
    z = np.load(path)
    return [sc.part(z["pos"], z["idx"], entity_id=0)]


def worker(root, name, creates, cache):
    sys.path.insert(0, os.path.abspath(root))
    cq = importlib.import_module("swift-game-engine_b200")
    parts = scene(cq.scenes, name, cache)
    out = []
    for _ in range(creates):
        t0 = time.perf_counter()
        g = cq.CollisionQuery(parts)
        wall = (time.perf_counter() - t0) * 1e3
        i = g.info()
        out.append({"create_ms": wall, "ref_order_ms": i["ref_order_ms"], "build_ms": i["build_ms"],
                    "n_ref_nodes": i["n_ref_nodes"], "n_triangles": i["n_static_triangles"] + i["n_dynamic_triangles"]})
        if hasattr(g, "rebuild"):  # cq_world_rebuild to the same parts, against the destroy + create above
            t0 = time.perf_counter()
            g.rebuild(parts)
            out[-1]["rebuild_ms"] = (time.perf_counter() - t0) * 1e3
        g.close()
    print(json.dumps(out))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old", required=True)
    ap.add_argument("--new", default=ROOT)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--creates", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", nargs=3, help=argparse.SUPPRESS)
    ap.add_argument("--cache", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        worker(a.worker[0], a.worker[1], int(a.worker[2]), a.cache)
        return
    cache = tempfile.mkdtemp(prefix="cq_ref_tree_probe_")
    res = {"card": card(), "rounds": a.rounds, "creates_per_run": a.creates, "runs": []}
    for r in range(a.rounds):
        for lib, tag in ((a.old, "old"), (a.new, "new")) if r % 2 == 0 else ((a.new, "new"), (a.old, "old")):
            for name in ("terrain_10m", "c5"):
                p = subprocess.run([sys.executable, __file__, "--old", a.old, "--cache", cache, "--worker", lib,
                                    "c5" if name == "c5" else "terrain", str(a.creates)], capture_output=True, text=True)
                if p.returncode:
                    raise RuntimeError(p.stderr[-2000:])
                runs = json.loads(p.stdout.strip().splitlines()[-1])
                res["runs"].append({"round": r, "lib": tag, "world": name, "creates": runs})
                print(tag, name, [(round(x["ref_order_ms"], 2), round(x["create_ms"], 1)) for x in runs], flush=True)
    summary = {}
    for name in ("terrain_10m", "c5"):
        for tag in ("old", "new"):
            xs = [c for run in res["runs"] if run["world"] == name and run["lib"] == tag for c in run["creates"][1:]]
            summary[f"{name}/{tag}"] = {k: statistics.median(c[k] for c in xs) for k in ("ref_order_ms", "create_ms", "build_ms")}
            summary[f"{name}/{tag}"]["n_ref_nodes"] = xs[0]["n_ref_nodes"]
            if "rebuild_ms" in xs[0]:
                summary[f"{name}/{tag}"]["rebuild_ms"] = statistics.median(c["rebuild_ms"] for c in xs)
    res["median_excluding_first_create"] = summary
    print(json.dumps(summary, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f)


if __name__ == "__main__":
    main()
