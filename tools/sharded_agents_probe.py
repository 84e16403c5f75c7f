"""An agent crowd (CQ_MAS_AGENTS) moved across the GPUs of one box: every GPU snapshots its shard
(cq_agent_snapshot_device), one NCCL all-gather makes the 32-byte snapshot records whole on every GPU
(cq_group_gather_records_local), every GPU builds the crowd's grid and moves its shard (cq_move_and_slide_device_agents).
Prints one JSON line and writes it to --out (default profiles/r10_sharded_agents_probe.json), with the card's name and
power limit read in the same run.

Workload: bench.py --agents 0.1 (its make_workload: the 10 M-triangle terrain, walkers whose footprints cover 10% of a
square in its middle), one world per GPU, one CUDA stream per GPU, every call enqueued from this thread.
  weak    --per-gpu agents per GPU (default 1,048,576) at N = each of --gpus;
  strong  --per-gpu agents in all, sharded by cq_shard_range over N;
  single  cq_move_and_slide_device with CQ_MAS_AGENTS on GPU 0 for the same crowd (the 1-GPU step), beside each case.
ms per step = CUDA events around --steps steps after --warmup steps, per GPU; the max over the GPUs is reported.  Phases
(snapshot, gather, move call) from events between them, averaged over the steps, max over the GPUs.  The move call is
split into the processing-order sort, the grid build and the move kernels (k_agent_first_hit + k_move_and_slide) by a
torch.profiler pass over one more step, run after the timed rounds.  The sharded and single variants alternate within each
of --rounds rounds, every round from the same initial records.  At the strong size the final records of the sharded run
and of the single call are compared byte for byte (after the rounds: warm-up + steps of each, same initial records).

Usage: python tools/sharded_agents_probe.py [--gpus 1,2,4,8] [--per-gpu N] [--steps K] [--warmup W] [--rounds R] [--out PATH]
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
import bench  # noqa: E402  (the workload of bench.py --agents, reused as it is)
from refit_async_probe import gpu_identity  # noqa: E402

COVERAGE = 0.1
FLAGS = 3  # CQ_MAS_APPLY_GRAVITY | CQ_MAS_AGENTS
SNAP = 32
STATE = 168


class Sharded:
    """The crowd's shards, one per GPU of a local group of the first n_gpus devices."""

    def __init__(self, cq, torch, worlds, n_gpus, states):
        self.cq, self.torch, self.n_gpus, self.n = cq, torch, n_gpus, len(states)
        self.group = cq.Group.local(n_gpus)
        self.worlds = worlds[:n_gpus]
        self.shards, self.states, self.snaps, self.streams = [], [], [], []
        for i in range(n_gpus):
            lo, hi = cq.shard_range(self.n, n_gpus, i)
            self.shards.append((lo, hi))
            with torch.cuda.device(i):
                self.states.append(torch.empty((hi - lo) * STATE, dtype=torch.uint8, device=f"cuda:{i}"))
                self.snaps.append(torch.empty(self.n * SNAP, dtype=torch.uint8, device=f"cuda:{i}"))
                self.streams.append(torch.cuda.Stream(device=i))
        self.load(states)

    def load(self, states):
        for i, (lo, hi) in enumerate(self.shards):
            self.states[i].copy_(self.torch.from_numpy(states[lo:hi].view(np.uint8).reshape(-1)))
        self.sync()

    def sync(self):
        for i in range(self.n_gpus):
            self.torch.cuda.synchronize(i)

    def step(self, params, ev=None):
        """ev: per GPU, four events recorded before the snapshot, after it, after the gather and after the move."""
        def rec(i, k):
            if ev is not None:
                ev[i][k].record(self.streams[i])
        for i, (lo, hi) in enumerate(self.shards):
            with self.torch.cuda.device(i):
                rec(i, 0)
                self.worlds[i].agent_snapshot_device(self.states[i].data_ptr(), hi - lo, self.snaps[i].data_ptr() + lo * SNAP,
                                                     bench.DT, bench.GRAVITY, FLAGS, self.streams[i].cuda_stream)
                rec(i, 1)
        local = [self.snaps[i].data_ptr() + lo * SNAP for i, (lo, _) in enumerate(self.shards)]
        self.group.gather_records_local(local, self.n, SNAP, [s.data_ptr() for s in self.snaps],
                                        [s.cuda_stream for s in self.streams])
        for i, (lo, hi) in enumerate(self.shards):
            with self.torch.cuda.device(i):
                rec(i, 2)
                self.worlds[i].move_and_slide_device_agents(self.states[i].data_ptr(), hi - lo, self.snaps[i].data_ptr(), self.n,
                                                            lo, params, bench.DT, bench.GRAVITY, FLAGS,
                                                            stream=self.streams[i].cuda_stream)
                rec(i, 3)

    def records(self):
        self.sync()
        return np.concatenate([s.cpu().numpy().view(self.cq.STATE) for s in self.states])

    def close(self):
        self.group.close()


def time_sharded(sh, params, steps, warmup):
    torch = sh.torch
    for _ in range(warmup):
        sh.step(params)
    sh.sync()
    ev = [[[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(sh.n_gpus)] for _ in range(steps)]
    for s in range(steps):
        sh.step(params, [ev[s][i] for i in range(sh.n_gpus)])
    sh.sync()
    per_gpu = []
    for i in range(sh.n_gpus):
        total = ev[0][i][0].elapsed_time(ev[-1][i][3]) / steps
        ph = [np.mean([ev[s][i][k].elapsed_time(ev[s][i][k + 1]) for s in range(steps)]) for k in range(3)]
        per_gpu.append({"ms_per_step": total, "snapshot_ms": ph[0], "gather_ms": ph[1], "move_call_ms": ph[2]})
    return {k: max(p[k] for p in per_gpu) for k in per_gpu[0]}


def time_single(cq, torch, world, d_states, n, params, steps, warmup):
    with torch.cuda.device(0):
        st = torch.cuda.Stream(device=0)
        for _ in range(warmup):
            world.move_and_slide_device(d_states.data_ptr(), n, params, bench.DT, bench.GRAVITY, FLAGS, st.cuda_stream)
        torch.cuda.synchronize(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(steps):
            world.move_and_slide_device(d_states.data_ptr(), n, params, bench.DT, bench.GRAVITY, FLAGS, st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize(0)
        return e0.elapsed_time(e1) / steps


def profile_split(torch, sh, params):
    """One sharded step under torch.profiler: the move call's kernels per GPU, in launch order, split into the processing
    order (kernels before k_agent_bounds_init), the grid (k_agent_bounds_init .. k_agent_rows) and the move kernels."""
    from torch.profiler import ProfilerActivity, profile
    sh.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sh.step(params)
        sh.sync()
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    out = []
    for i in range(sh.n_gpus):
        ks = sorted([e for e in kern if e.device_index == i], key=lambda e: e.time_range.start)
        names = [e.name for e in ks]
        try:
            a = next(k for k, nm in enumerate(names) if "k_agent_bounds_init" in nm)
            b = max(k for k, nm in enumerate(names) if "k_agent_rows" in nm)
            s = min(k for k, nm in enumerate(names) if "k_agent_snapshot" in nm)
        except (StopIteration, ValueError):
            out.append(None)
            continue
        us = lambda sel: sum(e.time_range.elapsed_us() for e in sel) / 1000.0
        gather = [e for e in ks[s + 1:a] if "nccl" in e.name.lower()]
        order = [e for e in ks[s + 1:a] if "nccl" not in e.name.lower()]
        out.append({"order_sort_ms": us(order), "grid_build_ms": us(ks[a:b + 1]),
                    "move_kernels_ms": us([e for e in ks[b + 1:] if "k_agent_first_hit" in e.name or "k_move_and_slide" in e.name]),
                    "gather_kernels_ms": us(gather)})
    ok = [o for o in out if o]
    return {k: max(o[k] for o in ok) for k in ok[0]} if ok else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--per-gpu", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_sharded_agents_probe.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_agents_probe: no CUDA device (the library has no CPU path)")
    cq = importlib.import_module("swift-game-engine_b200")
    cq.build()
    visible = torch.cuda.device_count()
    counts = [g for g in (int(x) for x in args.gpus.split(",")) if g <= visible]
    params = np.ascontiguousarray(bench.controller_params(cq, "terrain"), cq.PARAMS)
    parts, _ = bench.terrain_parts(cq)
    worlds = []
    for i in range(max(counts)):
        with torch.cuda.device(i):
            worlds.append(cq.CollisionQuery(parts))
    line = {"probe": "sharded_agents", **gpu_identity(), "visible_gpus": visible, "steps": args.steps, "warmup": args.warmup,
            "rounds": args.rounds, "workload": bench.workload_name("terrain", args.per_gpu, COVERAGE), "cases": []}
    cases = [("weak", n, n * args.per_gpu) for n in counts] + [("strong", n, args.per_gpu) for n in counts if n > 1]
    for kind, n_gpus, n in cases:
        _, pos, vel = bench.make_workload(cq, "terrain", n, 0, COVERAGE)
        init = cq.init_states(pos, vel)
        sh = Sharded(cq, torch, worlds, n_gpus, init)
        with torch.cuda.device(0):
            d_single = torch.empty(n * STATE, dtype=torch.uint8, device="cuda:0")
        rounds = []
        for r in range(args.rounds):
            sh.load(init)
            t = time_sharded(sh, params, args.steps, args.warmup)
            d_single.copy_(torch.from_numpy(init.view(np.uint8).reshape(-1)))
            t["single_gpu_ms_per_step"] = time_single(cq, torch, worlds[0], d_single, n, params, args.steps, args.warmup)
            rounds.append(t)
        case = {"kind": kind, "gpus": n_gpus, "agents": n, "agents_per_gpu_max": max(hi - lo for lo, hi in sh.shards),
                "rounds": rounds, "median": {k: float(np.median([x[k] for x in rounds])) for k in rounds[0]}}
        if kind == "strong" or n_gpus == 1:  # both variants ran rounds x (warm-up + steps) from the same records
            case["records_equal_single_gpu"] = sh.records().tobytes() == d_single.cpu().numpy().tobytes()
        case["move_call_split"] = profile_split(torch, sh, params)
        line["cases"].append(case)
        print(json.dumps({k: case[k] for k in ("kind", "gpus", "agents", "median")}), flush=True)
        sh.close()
        del d_single
    text = json.dumps(line)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
