"""capsuleOverlapAll beyond eight hits on one GPU: the eight-hit kernel (max_hits <= 8) against the wide path (max_hits > 8,
cq_capsule_overlap_all_device), and the wide path forced at max_hits = 8 next to the eight-hit kernel.  Prints one JSON
line and writes it to --out (default profiles/r7_overlap_all_probe.json).

Workloads, 1,048,576 gen_capsules(seed=8) each (radius 1.5, half height 1.0) over the mirror's box:
  render  the 14,246-triangle mirror render mesh + ground plane (tools/profile_extra.py overlap): nearly every query
          overflows at 8
  hulls   the two collision hulls + ground plane: few overlaps per query, so a fifth of the queries overflow at 32 and none at 128
max_hits in {8, 9, 32, 128}; 8 runs the eight-hit kernel, the others the wide path.  wide_at_8 is the same call at
max_hits = 8 on a build of this commit with -DCQ_OVL_WIDE_ABOVE=0 (every call takes the wide path), loaded from
--wide0-lib (tools/build_variant.sh wide0 "-DCQ_OVL_WIDE_ABOVE=0" builds swift-game-engine_b200/csrc/libcq_wide0.so);
its records, counts and overflow flags are compared byte for byte with the eight-hit kernel's.

Method: device-resident inputs and outputs, CUDA events around each call.  Every variant gets --warmup calls first; then
--rounds rounds, each timing --reps calls of every variant in turn (alternated).  Reported per variant: the median call
time of each round, mean hits per query and the share of queries that overflowed.  The card's name and power limit are
read in the same run.

Usage: python tools/overlap_all_probe.py [--wide0-lib PATH] [--rounds R] [--reps K] [--warmup W] [--out PATH]
"""
import argparse
import importlib
import importlib.util
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from refit_async_probe import gpu_identity  # noqa: E402

N = 1 << 20
MAX_HITS = (8, 9, 32, 128)


def load_with_lib(lib_path, name):
    """A second copy of the package bound to another build of libcq.so (CQ_LIB is read when the package loads)."""
    pkg = os.path.join(ROOT, "swift-game-engine_b200")
    old = os.environ.get("CQ_LIB")
    os.environ["CQ_LIB"] = lib_path
    try:
        spec = importlib.util.spec_from_file_location(name, os.path.join(pkg, "__init__.py"), submodule_search_locations=[pkg])
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    finally:
        if old is None:
            del os.environ["CQ_LIB"]
        else:
            os.environ["CQ_LIB"] = old
    return mod


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--wide0-lib", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_overlap_all_probe.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("overlap_all_probe: no CUDA device")
    cq = importlib.import_module("swift-game-engine_b200")
    cq.build()
    wide0 = load_with_lib(os.path.abspath(args.wide0_lib), "cq_wide0") if args.wide0_lib else None
    sc = cq.scenes
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)  # (a NULL stream argument would mean the world's own stream, not the timed one)
    torch.cuda.set_stream(stream)
    st = stream.cuda_stream
    line = {"probe": "overlap_all_probe", **gpu_identity(), "n": N, "rounds": args.rounds, "reps": args.reps,
            "warmup": args.warmup, "unit": "ms per call (median of reps), per round", "workloads": {}}
    d_out = torch.empty(N * max(MAX_HITS) * cq.OVERLAP_HIT.itemsize, dtype=torch.uint8, device=dev)
    d_cnt = torch.empty(N, dtype=torch.int32, device=dev)
    d_ov = torch.empty(N, dtype=torch.uint8, device=dev)
    for mesh in ("render", "hulls"):
        parts = sc.mirror_scene(use_hulls=mesh == "hulls")
        lo, hi = sc.scene_aabb(parts[1:])
        c = sc.gen_capsules(N, lo, hi, seed=8)
        d_c = torch.from_numpy(np.frombuffer(c.tobytes(), np.uint8).copy()).to(dev)
        worlds = {"this": cq.CollisionQuery(parts)}
        if wide0 is not None:
            worlds["wide0"] = wide0.CollisionQuery(parts)
        variants = [(f"max_hits_{m}", "this", m) for m in MAX_HITS]
        if wide0 is not None:
            variants.append(("wide_at_8", "wide0", 8))

        def call(world, m):
            worlds[world].capsule_overlap_all_device(d_c.data_ptr(), N, m, d_out.data_ptr(), d_cnt.data_ptr(), d_ov.data_ptr(), st)

        res = {v: {"path": "eight-hit kernel" if (w == "this" and m <= 8) else "wide", "ms": []} for v, w, m in variants}
        snap = {}
        for v, w, m in variants:  # warm-up, answers and their digest
            for _ in range(args.warmup):
                call(w, m)
            torch.cuda.synchronize()
            cnt = d_cnt.cpu().numpy()
            res[v]["mean_hits"] = round(float(cnt.mean()), 3)
            res[v]["overflow_share"] = round(float(d_ov.float().mean()), 4)
            if m == 8:
                snap[v] = (d_out[:N * 8 * cq.OVERLAP_HIT.itemsize].cpu().numpy().tobytes(), cnt.tobytes(), d_ov.cpu().numpy().tobytes())
        if "wide_at_8" in snap:
            res["wide_at_8"]["equals_eight_hit_kernel"] = snap["wide_at_8"] == snap["max_hits_8"]
        for _ in range(args.rounds):
            for v, w, m in variants:
                ts = []
                for _ in range(args.reps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    call(w, m)
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                res[v]["ms"].append(round(float(np.median(ts)), 3))
        if wide0 is None:
            res["wide_at_8"] = {"ms": "not measured (no --wide0-lib)"}
        line["workloads"][mesh] = {"triangles": worlds["this"].info()["n_static_triangles"], "variants": res}
        for g in worlds.values():
            g.close()
        del d_c
    s = json.dumps(line)
    print(s)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
