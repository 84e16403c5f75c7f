"""Agent separation on one GPU: the synchronous call (cq_agent_separation_device, which waits for the device once per
call) against cq_agent_separation_device_async and a captured CUDA graph of the whole crowd step.  Prints one JSON line
and writes it to --out (default profiles/r6_sep_async_probe.json).

Workload: bench.py's separation leg (`--only terrain --agents C --separation`): the 10 M-triangle terrain and 1,048,576
agents whose footprints cover C = 10% and 30% of a square.  One crowd step = move-and-slide with CQ_MAS_APPLY_GRAVITY |
CQ_MAS_AGENTS, then 2 separation sweeps, on device-resident records.

Device time.  Variants, alternated --rounds times, each run starting from the same records (--warmup steps, then
--steps timed with CUDA events around every step):
  a_parent_sync  cq_agent_separation_device of the parent build (--parent-pkg: a package directory built from the
                 parent commit; skipped when not given)
  b_sync         cq_agent_separation_device of this build
  b_r1_sync      the same from a build that queues only the R = 1 attempt of each sweep (--r1-pkg: this commit with the
                 attempt loop of launch_agent_separation cut to R = 1; skipped when not given).  It differs from b_sync
                 only by the three skipped attempts per sweep, so b_sync - b_r1_sync is their cost
  c_async        cq_agent_separation_device_async of this build
  c_graph        one torch.cuda.CUDAGraph of the step (move-and-slide + async separation), replayed
The final records of every run are compared byte for byte.

Host time per call (host_ms), two ways:
  back_to_back   the timed loop above: nothing bounds how far the host runs ahead, so once the stream's launch queue is
                 full every enqueue waits for the device; the move-and-slide enqueue is timed beside the separation one
                 to show that back-pressure
  unsaturated    the stream is synchronised before every step, the move-and-slide is queued, then the separation call
                 (or, for the graph, the replay after the synchronisation) is timed alone
Drift retries: --r1-pkg's build fails a sweep that drifts more than one cell (CQ_SEP_STATUS_DRIFT) instead of retrying
it, so every step is replayed with host synchronisation on this build, and before each separation the R = 1 build
separates a copy of the same records: a step whose copy fails took the retry.  That pass's final records and those of
the same pass on the parent build are compared with the timed runs'.

Usage: python tools/sep_async_probe.py [--steps K] [--warmup W] [--rounds R] [--parent-pkg DIR] [--r1-pkg DIR] [--out PATH]
"""
import argparse
import importlib
import importlib.util
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from refit_async_probe import gpu_identity  # noqa: E402

import bench  # noqa: E402  (the workload of the separation leg)

N = 1 << 20


def load_package(path, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(path, "__init__.py"), submodule_search_locations=[path])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def measure(cq, others, torch, coverage, steps, warmup, rounds):
    parts, pos, vel = bench.make_workload(cq, "terrain", N, 0, coverage)
    params = bench.controller_params(cq, "terrain")
    flags = cq.MAS_APPLY_GRAVITY | cq.MAS_AGENTS
    worlds = {"new": cq.CollisionQuery(parts)}
    for k, mod in others.items():
        worlds[k] = mod.CollisionQuery(parts)
    world_of = {"a_parent_sync": "parent", "b_r1_sync": "r1"}
    snap = torch.from_numpy(cq.init_states(pos, vel).view(np.uint8).copy()).cuda()
    d = snap.clone()
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = torch.cuda.Stream()
    st = stream.cuda_stream
    host = {"mas": [], "sep": []}

    def step(variant, sync_first=False):
        w = worlds[world_of.get(variant, "new")]
        if sync_first:
            stream.synchronize()
        t0 = time.perf_counter()
        w.move_and_slide_device(d.data_ptr(), N, params, bench.DT, bench.GRAVITY, flags, st)
        t1 = time.perf_counter()
        if variant == "c_async":
            w.agent_separation_device_async(d.data_ptr(), N, params, d_status_ptr=status.data_ptr(), stream=st)
        else:
            w.agent_separation_device(d.data_ptr(), N, params, stream=st)
        t2 = time.perf_counter()
        host["mas"].append(t1 - t0)
        host["sep"].append(t2 - t1)

    graph = None

    def replay(sync_first=False):
        if sync_first:
            stream.synchronize()
        t0 = time.perf_counter()
        with torch.cuda.stream(stream):
            graph.replay()
        host["sep"].append(time.perf_counter() - t0)

    def run(variant):
        nonlocal graph
        d.copy_(snap)
        torch.cuda.synchronize()
        if variant == "c_graph" and graph is None:  # captured once, after an uncaptured step sized the scratch
            step("c_async")
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                cs = torch.cuda.current_stream().cuda_stream
                worlds["new"].move_and_slide_device(d.data_ptr(), N, params, bench.DT, bench.GRAVITY, flags, cs)
                worlds["new"].agent_separation_device_async(d.data_ptr(), N, params, d_status_ptr=status.data_ptr(),
                                                            stream=cs)
            d.copy_(snap)
            torch.cuda.synchronize()
        go = replay if variant == "c_graph" else (lambda: step(variant))
        for _ in range(warmup):
            with torch.cuda.stream(stream):
                go()
        stream.synchronize()
        host["mas"].clear(), host["sep"].clear()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            with torch.cuda.stream(stream):
                a.record()
                go()
                b.record()
        stream.synchronize()
        ms = [a.elapsed_time(b) for a, b in evs]
        if variant in ("c_async", "c_graph"):
            assert int(status.item()) == 0, (variant, int(status.item()))
        t = {"ms_mean": float(np.mean(ms)), "host_ms_sep": 1e3 * float(np.mean(host["sep"]))}
        if host["mas"]:
            t["host_ms_mas"] = 1e3 * float(np.mean(host["mas"]))
        return t, d.cpu().numpy().tobytes()

    variants = [v for v in ("a_parent_sync", "b_sync", "b_r1_sync", "c_async", "c_graph") if world_of.get(v, "new") in worlds]
    res = {v: [] for v in variants}
    finals = {}
    for r in range(rounds):
        for v in variants:
            t, rec = run(v)
            res[v].append(t)
            finals.setdefault(v, rec)
            assert finals[v] == rec, ("not repeatable", v)
    ref = finals["b_sync"]
    out = {"coverage": coverage, "agents": N, "steps": steps, "warmup": warmup, "rounds": rounds,
           "records_identical": {v: finals[v] == ref for v in variants}, "variants": {}}
    for v in variants:
        ms = [t["ms_mean"] for t in res[v]]
        out["variants"][v] = {"ms_per_step_by_round": ms, "ms_per_step_mean": float(np.mean(ms)),
                              "spread_ms": float(max(ms) - min(ms))}
    for v in ("c_async", "c_graph"):  # host time per call, back to back and with an idle stream
        bb = {"separation_or_replay": [t["host_ms_sep"] for t in res[v]]}
        if v == "c_async":
            bb["move_and_slide"] = [t["host_ms_mas"] for t in res[v]]
        d.copy_(snap)
        torch.cuda.synchronize()
        host["mas"].clear(), host["sep"].clear()
        for _ in range(steps):
            if v == "c_graph":
                replay(sync_first=True)
            else:
                with torch.cuda.stream(stream):
                    step(v, sync_first=True)
        stream.synchronize()
        out["variants"][v]["host_ms"] = {"back_to_back": bb, "unsaturated": {
            "separation_or_replay_mean": 1e3 * float(np.mean(host["sep"])),
            "separation_or_replay_max": 1e3 * float(np.max(host["sep"]))}}
    if "r1" in worlds:  # drift retries (see the module docstring)
        probe = torch.empty_like(d)
        d.copy_(snap)
        torch.cuda.synchronize()
        retried = []
        for k in range(warmup + steps):
            worlds["new"].move_and_slide_device(d.data_ptr(), N, params, bench.DT, bench.GRAVITY, flags, st)
            stream.synchronize()
            probe.copy_(d)
            torch.cuda.synchronize()
            try:
                worlds["r1"].agent_separation_device(probe.data_ptr(), N, params, stream=st)
            except Exception as e:  # noqa: BLE001  the R = 1 build reports a drift as an error
                assert "drifted" in str(e), e
                retried.append(k)
            worlds["new"].agent_separation_device(d.data_ptr(), N, params, stream=st)
        out["drift_retry_steps"] = {"steps": warmup + steps, "with_retry": len(retried), "which": retried}
        out["records_identical"]["stepwise_pass"] = d.cpu().numpy().tobytes() == ref
    if "parent" in worlds:  # the same host-synchronised pass on the parent build
        w = worlds["parent"]
        d.copy_(snap)
        torch.cuda.synchronize()
        for _ in range(warmup + steps):
            w.move_and_slide_device(d.data_ptr(), N, params, bench.DT, bench.GRAVITY, flags, st)
            stream.synchronize()
            w.agent_separation_device(d.data_ptr(), N, params, stream=st)
        out["records_identical"]["parent_stepwise_pass"] = d.cpu().numpy().tobytes() == ref
    for w in worlds.values():
        w.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--coverage", type=float, nargs="+", default=[0.1, 0.3])
    ap.add_argument("--parent-pkg", default=None, help="package directory built from the parent commit (variant a)")
    ap.add_argument("--r1-pkg", default=None, help="package directory built with only the R = 1 attempt queued")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_sep_async_probe.json"))
    args = ap.parse_args()
    import torch
    cq = importlib.import_module("swift-game-engine_b200")
    others = {}
    if args.parent_pkg:
        others["parent"] = load_package(os.path.abspath(args.parent_pkg), "cq_parent")
    if args.r1_pkg:
        others["r1"] = load_package(os.path.abspath(args.r1_pkg), "cq_r1")
    line = {"probe": "sep_async", **gpu_identity(), "results": []}
    for c in args.coverage:
        line["results"].append(measure(cq, others, torch, c, args.steps, args.warmup, args.rounds))
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
