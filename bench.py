#!/usr/bin/env python
"""bench.py — move-and-slide capsule queries/sec (BASELINE.json metric), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--only NAME] [--no-extras]
                  [--dump-outputs DIR]

Headline workload (config C3 of BASELINE.json / SURVEY.md §8d): 1,048,576 characters per GPU, one fixed step of
the reference's KinematicMoveStopSystem body each (gravity -> decay -> velocity gate -> depenetration ->
<= 4 blocking slide casts -> ground snap/fall/offset probes -> snap/friction -> writeback) over the
ornate_mirror.static.json collision hulls at their demo placement + the 80x80 ground plane.  The world is created in
CQ_ORDER_REFERENCE (the library's default): every answer, exact ties included, is the one the reference's own tree
and visiting order give.

A "step" = one pass of the hot path over the whole batch; state is carried from step to step as in the engine.
  value  device-resident throughput (CUDA events on the launch stream, max over ranks);
  e2e    the same step through the public host-pointer C ABI with pinned HOST buffers, copies inside the timed region.
         Headline e2e = cq_crowd_step (records resident in HBM — they are private to KinematicMoveStopSystem in the
         reference too — velocities in, poses out); e2e.full_record = cq_move_and_slide_batch moving all 168 bytes of
         every record both ways.
  extra  the other BASELINE.json configurations at their named sizes, each with value / roofline / e2e:
         terrain (the north-star target scene: move-and-slide over the 10 M-triangle terrain), render (C3 on the
         14 k-triangle render mesh), c2 (65,536 sweeps vs Semla), c4 (8,388,608 blocking sweeps over the terrain),
         c5 (16,777,216 rays + a refit per step).  With N > 1 the sharded legs run through the library's own NCCL
         group (cq_group_*): c3_strong (1,048,576 characters in total), c4 (8,388,608 sweeps in total, the all-gather
         of the hit records INSIDE the timed region, collective_ms beside it), c5 (16,777,216 rays in total).

Multi-GPU: units are sharded across ranks (contiguous ranges), mesh + trees are replicated, no data-path collective in
the move-and-slide step (weak scaling); torch.distributed is plumbing for the barrier, the max-over-ranks and the
broadcast of the 128-byte NCCL id.

Every configuration times exactly K steps.  --dump-outputs DIR writes the character records of the headline path as
they stand after its last timed step (rank 0's characters) as DIR/<field>.npy; the inputs are seeded, so two builds run
with the same arguments can be compared output for output (see dump_outputs).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark leaves nothing in it

# Libraries (NCCL, torch) may print to stdout; the contract is ONE JSON line there.  Keep the real stdout aside
# and send everything else to stderr.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def bind_to_gpu_numa_node(local_rank):
    """Best effort: run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node its GPU hangs
    off, so that 8 ranks do not push all their PCIe traffic through one socket's memory."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


CHARS_PER_GPU = 1 << 20
SEED = 0xC0111DE3
DT = 1.0 / 60.0
GRAVITY = (0.0, -98.0, 0.0)
FP32_PEAK_TINST = 148 * 128 * 1.965e9 / 1e12  # lanes x clock: issue ceiling with FMA off (1 flop / lane / clk)
DUMP_LIMIT = 64_000_000  # --dump-outputs: bytes of all the .npy files together
DUMP_SEED = 0xC0111DE6


def dump_outputs(out_dir, records, skip=("_pad",)):
    """--dump-outputs: every field of `records` as out_dir/<field>.npy.  Float fields keep their precision; integer and
    flag fields become float64, which holds every 32-bit value exactly.  When all records would not fit in DUMP_LIMIT, a
    fixed, seeded sample of them is written (the same records in every run of the same size); record_index.npy holds
    which records were written, in ascending order."""
    names = [f for f in records.dtype.names if f not in skip]

    def as_float(a):
        return a.astype(a.dtype if a.dtype.kind == "f" else np.float64)

    per_record = 8 + sum(as_float(records[f][:1]).itemsize * int(np.prod(records.dtype[f].shape)) for f in names)
    keep = min(len(records), (DUMP_LIMIT - 256 * (len(names) + 1)) // per_record)  # 256: room for each .npy header
    idx = np.arange(len(records)) if keep == len(records) else \
        np.sort(np.random.default_rng(DUMP_SEED).choice(len(records), keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "record_index.npy"), idx.astype(np.float64))
    for f in names:
        np.save(os.path.join(out_dir, f + ".npy"), as_float(records[f][idx]))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(kernel, config):
    """DRAM bytes per unit of the dominant kernel from the committed `ncu --set full` captures (profiles/r2_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum of one launch divided by the units it processed)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))[kernel][config]["dram_bytes_per_unit"]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        # "under load" = samples whose power draw is above the idle floor (the first samples precede the first launch)
        if power:
            thr = min(power) + 0.25 * (max(power) - min(power))
            loaded = [c for c, p in zip(sm, power) if p >= thr] or sm
        else:
            loaded = sm
        return {"sm_mhz": float(np.median(loaded)) if loaded else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "samples_under_load": len(loaded),
                "reasons": sorted(reasons)}


TERRAIN_PARAMS = dict(radius=0.4, half_height=0.5, skin_width=0.08)  # human-scale capsule (SURVEY.md §7, §8d C4)
_TERRAIN = {}


def terrain_parts(cq, cells=2236):
    """The 10 M-triangle procedural terrain (generated once per process: 2 s of numpy)."""
    if cells not in _TERRAIN:
        _TERRAIN[cells] = cq.scenes.terrain_scene(cells=cells, cell=2.0)
    return _TERRAIN[cells]


def make_workload(cq, mesh, n, rank, agents=0.0, cells=2236):
    if mesh == "terrain":  # the north-star target scene: 10 M-triangle procedural terrain, walkers all over it
        parts, half = terrain_parts(cq, cells)
        rng = np.random.default_rng(SEED + 77 + rank)
        span = half - 10
        if agents > 0:  # a crowd: the walkers' footprints cover `agents` of a square in the middle of the terrain
            span = min(span, float(np.sqrt(n * np.pi * TERRAIN_PARAMS["radius"] ** 2 / agents)) / 2)
        x = rng.uniform(-span, span, (n, 2))
        y = cq.scenes.terrain_height(x[:, 0], x[:, 1]) + np.float32(0.9 + 0.2)
        pos = np.stack([x[:, 0], y, x[:, 1]], axis=1).astype(np.float32)
        heading, speed = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 4.5, n)
        vel = np.stack([np.cos(heading) * speed, np.zeros(n), np.sin(heading) * speed], axis=1).astype(np.float32)
        return parts, pos, vel
    parts = cq.scenes.mirror_scene(use_hulls=(mesh == "hulls"))
    pos, vel = cq.scenes.gen_c3_characters(n, seed=SEED + rank)
    return parts, pos, vel


def controller_params(mod, mesh):
    return mod.default_params(**TERRAIN_PARAMS) if mesh == "terrain" else mod.default_params()


def workload_name(mesh, n, agents=0.0, separation=False):
    if mesh == "terrain":
        crowd = (f"; every character a solid agent (capsule-capsule CCD against a pre-step snapshot of the others), "
                 f"crowd footprint coverage {agents:g}") if agents > 0 else ""
        if separation:
            crowd += ", followed by AgentSeparationSystem (2 sequential pair-resolution sweeps + slide + snap)"
        return (f"target scene: {n} characters/GPU x 1 move-and-slide fixed step over the procedural terrain of "
                "9,999,392 triangles (cell 2 m), human-scale controller r=0.4 hh=0.5 skin 0.08, dt=1/60, gravity on" + crowd)
    tri = "2 collision hulls (76 tris) + ground plane (2 tris)" if mesh == "hulls" else \
        "render mesh (14,211 tris after the area filter) + ground plane (2 tris)"
    return (f"C3: {n} characters/GPU x 1 move-and-slide fixed step (<=4 slide casts + ground probes), "
            f"ornate_mirror.static.json {tri}, default controller r=1.5 hh=1.0, dt=1/60, gravity on")


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The reference's CPU implementation of the path (the oracle port: no swiftc exists here, see
    DESIGN.md) on this box's host cores, all threads, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as orc
    cq = importlib.import_module("swift-game-engine_b200")  # scenes only (numpy); no CUDA call is made
    cores = os.cpu_count() or 1
    n = args.ref_sample or {"hulls": CHARS_PER_GPU, "render": 65536, "terrain": 262144}[args.mesh]
    mas_flags = 1
    if args.agents > 0:  # the reference's agent loop is O(n^2): a smaller crowd of the SAME density
        n = args.ref_sample or 32768
        mas_flags = 3
    parts, pos, vel = make_workload(cq, args.mesh, n, 0, args.agents)
    w = orc.OracleWorld(parts)
    s = orc.init_states(pos, vel)
    p = controller_params(orc, args.mesh)

    def ref_step():
        w.move_and_slide(s, p, DT, GRAVITY, mas_flags, orc.ORDER_REFERENCE, cores)
        if args.separation:
            w.agent_separation(s, p, order=orc.ORDER_REFERENCE, n_threads=cores)

    for _ in range(args.warmup):
        ref_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref_step()
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = f"{n} of {CHARS_PER_GPU} characters per step, {args.steps} steps, state carried"
    if args.agents > 0:
        sample = (f"a crowd of {n} characters at the same density (the reference tests every agent against every other: "
                  f"its cost per character grows with the crowd), {args.steps} steps, state carried")
    line = {
        "impl": "reference", "metric": "move_and_slide_queries_per_sec", "value": value, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.mesh, CHARS_PER_GPU, args.agents, args.separation), "mesh": args.mesh,
                   "reference_impl": "C++ restatement of CollisionQuery.swift + Systems.swift move-and-slide "
                                     "(oracle/), reference BVH + DFS order; not swiftc-compiled"},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------ shared plumbing
class Ctx:
    """One process per GPU: torch for device memory / streams / the process group, nothing else."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.ws = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.lrank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the CUDA path has no CPU fallback")
        torch.cuda.set_device(self.lrank)
        self.dev = torch.device("cuda", self.lrank)
        self.numa = bind_to_gpu_numa_node(self.lrank)
        if self.ws > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        # an explicit (non-default) stream: the library's NULL-stream convention means "the world's own stream", and
        # torch.cuda.Event only sees torch's current stream, so make both the same real stream
        self.tstream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.tstream)
        self.stream = self.tstream.cuda_stream
        assert self.stream != 0
        self.cq = importlib.import_module("swift-game-engine_b200")
        self.cq.build()
        self.group = None

    def barrier(self):
        if self.ws > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def red(self, x, op="max"):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.ws > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def nccl_group(self):
        """The library's own NCCL communicator over the ranks (cq_group_create_rank): rank 0 makes the 128-byte id,
        torch.distributed ships it."""
        if self.group is None:
            uid = self.cq.Group.unique_id() if self.rank == 0 else np.zeros(self.cq.GROUP_ID_BYTES, np.uint8)
            t = self.torch.from_numpy(uid.copy()).to(self.dev)
            if self.ws > 1:
                self.dist.broadcast(t, 0)
            self.group = self.cq.Group.rank(self.ws, self.rank, t.cpu().numpy())
        return self.group

    def up(self, a):
        return self.torch.from_numpy(np.frombuffer(a.tobytes(), np.uint8).copy()).to(self.dev)

    def events(self):
        return self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)

    def close(self):
        if self.group is not None:
            self.group.close()
        if self.ws > 1:
            self.dist.destroy_process_group()


def time_steps(ctx, step, steps, warmup, sampler=None, keep_loaded=0.0):
    """W warm-up steps, then K steps between a barrier + synchronize on both sides, CUDA events around every step and
    around the whole region; returns (total ms max over ranks, mean per-step ms of this rank)."""
    torch = ctx.torch
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    evs = [ctx.events() for _ in range(steps)]
    ctx.barrier()
    if sampler:
        sampler.start()
    t0, t1 = ctx.events()
    t0.record()
    for k in range(steps):
        evs[k][0].record()
        step()
        evs[k][1].record()
    t1.record()
    ctx.barrier()
    if keep_loaded > 0:
        # the timed region lasts tens of milliseconds, shorter than one nvidia-smi sampling period: keep the identical
        # load running (untimed) until the sampler has seen the GPU under it for a while
        t_load = time.perf_counter()
        while time.perf_counter() - t_load < keep_loaded:
            for _ in range(4):
                step()
            torch.cuda.synchronize()
    total_ms = ctx.red(t0.elapsed_time(t1))
    step_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    return total_ms, step_ms


def roofline_block(kernel, kernel_ms, algo_bytes, evals, per_query, traffic):
    peak, peak_src = load_peaks()
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
         "peak_source": peak_src, "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": algo_bytes,
         "per_query": per_query}
    if evals is not None:
        tf = 430.0 * evals / (kernel_ms * 1e-3) / 1e12
        r["fp32_secondary"] = {"note": "the narrow phase is FP32-issue bound, not HBM bound (SURVEY.md §8d): ~430 flop per "
                                       "distance evaluation, FMA contraction off for bit-parity",
                               "achieved_tflops": tf, "peak_tflops_nominal": FP32_PEAK_TINST, "frac": tf / FP32_PEAK_TINST}
    return r


# ------------------------------------------------------------------------------------------ move-and-slide (C3 / terrain)
def measure_mas(ctx, args, mesh, n, steps, warmup, cpu_baseline=True, clocks=True, full_record_e2e=True, dump_dir=None):
    """One move-and-slide configuration: device-resident value, roofline, e2e legs, optional CPU baseline.  dump_dir: where
    rank 0 writes its character records as the last timed step left them (dump_outputs)."""
    cq, torch = ctx.cq, ctx.torch
    agents = args.agents if mesh == "terrain" else 0.0
    parts, pos, vel = make_workload(cq, mesh, n, ctx.rank, agents, args.cells)
    mas_flags = cq.MAS_APPLY_GRAVITY | (cq.MAS_AGENTS if agents > 0 else 0)
    t0 = time.perf_counter()
    world = cq.CollisionQuery(parts, order=args.order)
    create_s = time.perf_counter() - t0
    info = world.info()
    params = controller_params(cq, mesh)
    states0 = cq.init_states(pos, vel)
    nbytes = states0.nbytes
    # device-resident state (168 B x 1 M characters = 176 MB per GPU > the 126 MB L2, so no explicit L2 flush is needed)
    d_states = ctx.up(states0)
    stream = ctx.stream
    separation = args.separation and agents > 0

    def step_device():
        world.move_and_slide_device(d_states.data_ptr(), n, params, DT, GRAVITY, mas_flags, stream)
        if separation:  # the reference's fixed step runs AgentSeparationSystem right after the kinematic move
            world.agent_separation_device(d_states.data_ptr(), n, params, stream=stream)

    sampler = ClockSampler(ctx.lrank) if clocks else None
    for _ in range(warmup):
        step_device()
    torch.cuda.synchronize()
    snapshot = d_states.clone()
    world.resetStats()
    total_ms, kernel_ms = time_steps(ctx, step_device, steps, 0, sampler)
    launches = world.stats()["kernel_launches"]
    after_timed = d_states.clone()
    if clocks:  # keep the identical load running (untimed) until nvidia-smi has seen the GPU under it for ~0.7 s
        t_load = time.perf_counter()
        while time.perf_counter() - t_load < 0.7:
            for _ in range(8):
                step_device()
            torch.cuda.synchronize()
    clk = sampler.stop() if sampler else None
    if clk is not None:
        clk["window"] = "timed region + 0.7 s of the same steps right after it (untimed)"
    value = n * ctx.ws * steps / (total_ms * 1e-3)

    # algorithmic bytes of exactly these K steps: replay them from the snapshot with the counting build
    d_states.copy_(snapshot)
    world.set_counting(cq.COUNT_PATH)
    world.resetStats()
    for _ in range(steps):
        step_device()
    torch.cuda.synchronize()
    ctr = world.stats(reset=True)
    world.set_counting(False)
    final_np = np.frombuffer(after_timed.cpu().numpy().tobytes(), dtype=cq.STATE)  # state after the K timed steps

    def same_state(a):  # every field but `_pad` (the counting build leaves per-character evaluation counts there)
        return all(np.array_equal(a[f], final_np[f]) for f in cq.STATE.names if f != "_pad")

    replay_same = same_state(np.frombuffer(d_states.cpu().numpy().tobytes(), dtype=cq.STATE))
    state_bytes = 2 * cq.STATE.itemsize  # state in + state out
    algo = (n * state_bytes * steps + 32 * ctr["nodes_visited"] + 52 * ctr["candidates"]) / steps
    per_query = {"nodes": ctr["nodes_visited"] / (n * steps), "candidates": ctr["candidates"] / (n * steps),
                 "distance_evals": ctr["distance_evals"] / (n * steps), "bvh_traversals": ctr["queries"] / (n * steps)}
    tr = measured_traffic("k_move_and_slide", mesh)
    roofline = roofline_block("k_move_and_slide", kernel_ms, algo, ctr["distance_evals"] / steps, per_query,
                              tr * n if tr is not None else None)

    snap_np = np.frombuffer(snapshot.cpu().numpy().tobytes(), dtype=cq.STATE).copy()
    e2e = {}
    # e2e, headline: the resident crowd (records stay in HBM; velocities in, poses out; pinned host buffers).  Every step
    # uploads the velocities the host holds — here the ones the previous step's pose reported, which is what a host whose
    # steering systems changed nothing would send, and what makes the run comparable with the device-resident replay.
    if not separation:
        crowd = cq.Crowd(world, snap_np.copy())
        h_vel = cq.PinnedArray((n, 3), np.float64)
        h_pose = cq.PinnedArray((n,), cq.CROWD_POSE)
        h_vel.array[:] = snap_np["velocity"]
        crowd.step(h_vel.array, params, DT, GRAVITY, mas_flags, pose_out=h_pose.array)  # warm the pipeline
        crowd.write(snap_np.copy())
        h_vel.array[:] = snap_np["velocity"]
        ctx.barrier()
        crowd_s = 0.0
        for _ in range(steps):
            t0 = time.perf_counter()
            crowd.step(h_vel.array, params, DT, GRAVITY, mas_flags, pose_out=h_pose.array)  # synchronous: H2D + kernels + D2H
            crowd_s += time.perf_counter() - t0
            # the host's own systems between two steps (here: carry the velocity the pose reported) are not the API's time
            h_vel.array[:] = h_pose.array["velocity"]
        crowd_s = ctx.red(crowd_s)
        ctx.barrier()
        same_crowd = same_state(crowd.read())
        e2e = {"value": n * ctx.ws * steps / crowd_s, "unit": "queries/s", "h2d_bytes_per_step": n * 24 * ctx.ws,
               "d2h_bytes_per_step": n * cq.CROWD_POSE.itemsize * ctx.ws, "ms_per_step": crowd_s / steps * 1e3,
               "api": "cq_crowd_step (records resident in HBM; 24 B of velocity in, 56 B of pose out per character; "
                      "pinned host buffers; chunked copy/compute overlap)",
               "matches_device_path": same_crowd}
        crowd.close()
        h_vel.free()
        h_pose.free()
    if full_record_e2e or separation:
        pinned = cq.PinnedArray((n,), cq.STATE)
        pinned.array[:] = snap_np
        world.move_and_slide(pinned.array, params, DT, GRAVITY, mas_flags)  # warm the staging buffers
        if separation:
            world.agent_separation(pinned.array, params)
        pinned.array[:] = snap_np
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            world.move_and_slide(pinned.array, params, DT, GRAVITY, mas_flags)
            if separation:
                world.agent_separation(pinned.array, params)
        torch.cuda.synchronize()
        full_s = ctx.red(time.perf_counter() - t0)
        ctx.barrier()
        full = {"value": n * ctx.ws * steps / full_s, "unit": "queries/s", "h2d_bytes_per_step": nbytes * ctx.ws,
                "d2h_bytes_per_step": nbytes * ctx.ws, "ms_per_step": full_s / steps * 1e3,
                "api": "cq_move_and_slide_batch (all 168 bytes of every record both ways; pinned, chunked copy/compute overlap)",
                "matches_device_path": same_state(pinned.array)}
        pinned.free()
        if e2e:
            e2e["full_record"] = full
        else:
            e2e = full
    grounded_frac = float(final_np["grounded"].mean())

    cpu = None
    if cpu_baseline and ctx.rank == 0 and ctx.ws == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        cores = os.cpu_count() or 1
        ns = min({"hulls": CHARS_PER_GPU, "render": 65536, "terrain": 262144}[mesh], n)
        ow = orc.OracleWorld(parts)
        what = f"first {ns} of the {n} characters"
        if agents > 0:
            # the reference tests every agent against every other (O(n^2)): time a sub-crowd of the SAME density,
            # the characters inside a centred square holding ~32768 of them
            px, pz = snap_np["position"][:, 0], snap_np["position"][:, 2]
            lim = max(np.abs(px).max(), np.abs(pz).max()) * np.sqrt(min(1.0, 32768 / n))
            sub = snap_np[(np.abs(px) <= lim) & (np.abs(pz) <= lim)].copy()
            ns = len(sub)
            what = f"the {ns} characters of a centred sub-square of the crowd (same density; the reference's agent loop is O(n^2))"
        else:
            sub = snap_np[:ns].copy()
        t0 = time.perf_counter()
        ow.move_and_slide(sub, controller_params(orc, mesh), DT, GRAVITY, 3 if agents > 0 else 1, orc.ORDER_REFERENCE, cores)
        if separation:
            ow.agent_separation(sub, controller_params(orc, mesh), order=orc.ORDER_REFERENCE, n_threads=cores)
        cdt = time.perf_counter() - t0
        cpu = {"value": ns / cdt, "unit": "queries/s", "cores": cores, "kind": "port",
               "sample": f"{what}, the first timed step, {cdt:.2f} s wall; restated reference (C++), not swiftc-compiled"}
        # parity on the way: the GPU's first timed step of the same characters must equal the reference-order oracle's
        if args.order == cq.ORDER_REFERENCE and agents == 0:
            g1 = snap_np[:ns].copy()
            world.move_and_slide(g1, params, DT, GRAVITY, mas_flags)
            cpu["gpu_step_bit_identical_to_this_run"] = bool(g1.tobytes() == sub.tobytes())
        ow.close()
    world.close()
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, final_np)
    return {
        "metric": "move_and_slide_queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": ctx.ws,
        "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(mesh, n, agents, separation), "mesh": mesh, "characters_per_gpu": n,
                   "triangles": info["n_static_triangles"] + info["n_dynamic_triangles"],
                   "order": "reference" if args.order == cq.ORDER_REFERENCE else "canonical",
                   "l2": "inputs (168 B x characters = %.0f MB per GPU) exceed the 126 MB L2; no flush" % (nbytes / 1e6),
                   "parallelism": f"queries sharded over {ctx.ws} GPU(s), mesh+BVH replicated, no collective",
                   "bvh_build_ms": info["build_ms"], "reference_order_build_ms": info["ref_order_ms"],
                   "world_create_s": create_s, "grounded_fraction_after": grounded_frac, "numa_node": ctx.numa,
                   "counting_replay_matches_timed_run": replay_same},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": int(ctx.red(launches, "sum")), "clocks": clk,
    }


# ------------------------------------------------------------------------------------------ C4: blocking sweeps over the terrain
def measure_c4(ctx, args, n_total, steps, warmup, sharded):
    """capsuleCastBlocking sweeps over the procedural 10M-triangle terrain.  sharded=False: n_total sweeps per GPU (weak);
    sharded=True: n_total sweeps in all, rank r takes cq_shard_range(n_total, ws, r), and the hit records of all ranks are
    all-gathered onto every rank INSIDE the timed region by the library's NCCL group (cq_group_gather_records)."""
    cq, torch = ctx.cq, ctx.torch
    t0 = time.perf_counter()
    parts, half = terrain_parts(cq, args.cells)
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    world = cq.CollisionQuery(parts, order=args.order)
    t_create = time.perf_counter() - t0
    info = world.info()
    lo, hi = 0, n_total
    if sharded:
        lo, hi = cq.shard_range(n_total, ctx.ws, ctx.rank)
        q_all = cq.scenes.gen_c4_casts(n_total, half, seed=0xC0111DE4, radius=args.radius, half_height=args.half_height)
        q = np.ascontiguousarray(q_all[lo:hi])
        del q_all
    else:
        q = cq.scenes.gen_c4_casts(n_total, half, seed=0xC0111DE4 + ctx.rank, radius=args.radius, half_height=args.half_height)
    n = len(q)
    units = n_total if sharded else n_total * ctx.ws
    d_q, rec = ctx.up(q), cq.CAST_HIT.itemsize
    d_out = torch.empty(n * rec, dtype=torch.uint8, device=ctx.dev)
    gather = sharded and ctx.ws > 1
    d_all = torch.empty(n_total * rec, dtype=torch.uint8, device=ctx.dev) if gather else None
    group = ctx.nccl_group() if gather else None
    stream = ctx.stream

    def step():
        world.capsule_cast_device(d_q.data_ptr(), n, cq.CAST_BLOCKING, d_out.data_ptr(), stream)
        if gather:  # the one collective of the path (DESIGN.md §6), NCCL from inside libcq.so
            group.gather_records(d_out.data_ptr(), n_total, rec, d_all.data_ptr(), stream)

    sampler = ClockSampler(ctx.lrank)
    world.resetStats()
    total_ms, step_ms = time_steps(ctx, step, steps, warmup, sampler)
    clk = sampler.stop()
    launches = world.stats()["kernel_launches"]
    value = units * steps / (total_ms * 1e-3)
    collective_ms, kernel_ms = None, total_ms / steps
    if gather:  # the collective alone and the kernel alone, same buffers, max over ranks
        def only_gather():
            group.gather_records(d_out.data_ptr(), n_total, rec, d_all.data_ptr(), stream)

        def only_cast():
            world.capsule_cast_device(d_q.data_ptr(), n, cq.CAST_BLOCKING, d_out.data_ptr(), stream)
        collective_ms = time_steps(ctx, only_gather, steps, 1)[0] / steps
        kernel_ms = time_steps(ctx, only_cast, steps, 1)[0] / steps
        mine = d_all[lo * rec:hi * rec]
        assert bool(torch.equal(mine, d_out)), "gathered records differ from the local shard"
    world.set_counting(cq.COUNT_PATH)
    world.resetStats()
    world.capsule_cast_device(d_q.data_ptr(), n, cq.CAST_BLOCKING, d_out.data_ptr(), stream)
    torch.cuda.synchronize()
    ctr = world.stats(reset=True)
    world.set_counting(False)
    hits = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=cq.CAST_HIT)
    algo = n * (40 + 44) + 32 * ctr["nodes_visited"] + 52 * ctr["candidates"]
    tr = measured_traffic("k_capsule_cast", "c4")
    roofline = roofline_block("k_capsule_cast", kernel_ms, algo, ctr["distance_evals"],
                              {k: ctr[k] / n for k in ("nodes_visited", "candidates", "distance_evals")},
                              tr * n if tr is not None else None)
    # e2e through the host-pointer API
    hq = cq.PinnedArray((n,), cq.CAST)
    hq.array[:] = q
    ho = cq.PinnedArray((n,), cq.CAST_HIT)
    L = cq.lib()
    L.cq_capsule_cast_batch(world.handle, hq.array.ctypes.data, n, cq.CAST_BLOCKING, ho.array.ctypes.data)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        rc = L.cq_capsule_cast_batch(world.handle, hq.array.ctypes.data, n, cq.CAST_BLOCKING, ho.array.ctypes.data)
        assert rc == 0
    e2e_s = ctx.red(time.perf_counter() - t0)
    same = bool(ho.array.tobytes() == hits.tobytes())
    hq.free()
    ho.free()
    cpu = None
    if ctx.rank == 0 and ctx.ws == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        cores = os.cpu_count() or 1
        t0 = time.perf_counter()
        ow = orc.OracleWorld(parts)
        t_cpu_build = time.perf_counter() - t0
        ns = min(n, 65536)
        t0 = time.perf_counter()
        ref = ow.capsule_cast(q[:ns], 1, orc.ORDER_REFERENCE, cores)
        cdt = time.perf_counter() - t0
        cpu = {"value": ns / cdt, "unit": "sweeps/s", "cores": cores, "kind": "port",
               "sample": f"first {ns} of {n} sweeps, {cdt:.2f} s; reference-BVH build {t_cpu_build:.1f} s (1 thread)",
               "gpu_bit_identical_on_the_sample": bool(ref.tobytes() == hits[:ns].tobytes())}
        ow.close()
    world.close()
    return {
        "metric": "capsule_sweeps_per_sec", "value": value, "unit": "sweeps/s", "n_gpus": ctx.ws, "steps": steps,
        "warmup": warmup, "ms_per_step": total_ms / steps, "higher_is_better": True,
        "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": (f"C4: {n_total} capsuleCastBlocking sweeps " + ("in all, sharded over the ranks, " if sharded else "per GPU ")
                                + f"over a procedural terrain of {info['n_static_triangles']} triangles (cell 2 m), "
                                f"r={args.radius} hh={args.half_height}"),
                   "triangles": info["n_static_triangles"], "bvh_build_ms": info["build_ms"],
                   "reference_order_build_ms": info["ref_order_ms"], "world_create_s": t_create, "terrain_gen_s": t_gen,
                   "hit_fraction": float((hits["triangle_index"] >= 0).mean()),
                   "l2": "triangle SoA + nodes (%.0f MB) and queries exceed the 126 MB L2" % (info["n_static_triangles"] * 112 / 1e6),
                   "e2e_matches_device_path": same,
                   "gather": (f"cq_group_gather_records (ncclAllGather inside libcq.so) of the {rec} B hit records of all ranks "
                              "inside the timed region") if gather else "none (results stay on the owning GPU)"},
        "collective_ms": collective_ms, "kernel_ms_alone": kernel_ms if gather else None,
        "roofline": roofline, "cpu_baseline": cpu,
        "e2e": {"value": units * steps / e2e_s, "unit": "sweeps/s", "h2d_bytes_per_step": units * 40,
                "d2h_bytes_per_step": units * 44, "ms_per_step": e2e_s / steps * 1e3,
                "api": "cq_capsule_cast_batch (host pointers, pinned)"},
        "gpu_launches": int(ctx.red(launches, "sum")), "clocks": clk}


# ------------------------------------------------------------------------------------------ C2: sweeps vs Semla
def measure_c2(ctx, args, n, steps, warmup):
    """Config C2: 65,536 plain capsuleCast sweeps against the Semla mesh (FBX-regenerated stand-in for the missing
    Semla.static.json) at its demo placement; a sample checked byte for byte against the reference-order oracle."""
    cq, torch = ctx.cq, ctx.torch
    sc = cq.scenes
    parts = sc.semla_scene(use_hulls=False)
    world = cq.CollisionQuery(parts, order=args.order)
    info = world.info()
    lo, hi = sc.scene_aabb(parts[1:])
    q = sc.gen_casts(n, lo, hi, seed=0xC0111DE2 + ctx.rank)  # from ~ U(AABB + 3 m), |delta| ~ U[0.05, 2], r=1.5 hh=1.0
    d_q = ctx.up(q)
    d_out = torch.empty(n * cq.CAST_HIT.itemsize, dtype=torch.uint8, device=ctx.dev)
    d_flags = torch.zeros(n, dtype=torch.uint8, device=ctx.dev)
    stream = ctx.stream
    L = cq.lib()

    def step():
        rc = L.cq_capsule_cast_device_ex(world.handle, d_q.data_ptr(), n, cq.CAST_ALL, d_out.data_ptr(), d_flags.data_ptr(), stream)
        assert rc == 0

    sampler = ClockSampler(ctx.lrank)
    world.resetStats()
    total_ms, _ = time_steps(ctx, step, steps, warmup, sampler)
    clk = sampler.stop()
    launches = world.stats()["kernel_launches"]
    ms = total_ms / steps
    world.set_counting(cq.COUNT_PATH)
    world.resetStats()
    step()
    torch.cuda.synchronize()
    ctr = world.stats(reset=True)
    world.set_counting(False)
    hits = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=cq.CAST_HIT)
    flags = d_flags.cpu().numpy()
    t0 = time.perf_counter()
    host_hits = world.capsuleCast(q)
    e2e_s = time.perf_counter() - t0
    algo = n * (40 + 44) + 32 * ctr["nodes_visited"] + 52 * ctr["candidates"]
    cpu, parity = None, None
    if ctx.rank == 0 and ctx.ws == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        cores = os.cpu_count() or 1
        ow = orc.OracleWorld(parts)
        ns = min(n, 16384)
        st = orc.Stats()
        t0 = time.perf_counter()
        ref = ow.capsule_cast(q[:ns], 0, orc.ORDER_REFERENCE, cores, st)
        cdt = time.perf_counter() - t0
        can = ow.capsule_cast(q[:ns], 0, orc.ORDER_CANONICAL, cores)
        mine = ref if args.order == cq.ORDER_REFERENCE else can
        other = can if args.order == cq.ORDER_REFERENCE else ref
        diff = hits["triangle_index"][:ns] != other["triangle_index"]
        tie = (flags[:ns] & cq.HIT_TIE).astype(bool)
        parity = {"sample": ns, "bit_exact_vs_oracle_in_the_world_order": bool(mine.tobytes() == hits[:ns].tobytes()),
                  "index_mismatch_vs_reference_order": float((ref["triangle_index"] != hits["triangle_index"][:ns]).mean()),
                  "queries_flagged_TIE": float(tie.mean()),
                  "differences_between_the_two_order_rules": float(diff.mean()),
                  "unflagged_differences": int((diff & ~tie).sum()),
                  "reference_distance_evals_per_sweep": st.distance_evals / ns}
        cpu = {"value": ns / cdt, "unit": "sweeps/s", "cores": cores, "kind": "port",
               "sample": f"first {ns} of {n} sweeps, {cdt:.2f} s wall, reference BVH + DFS order"}
        ow.close()
    world.close()
    tr = measured_traffic("k_capsule_cast", "c2")
    return {
        "metric": "capsule_sweeps_per_sec", "value": n * ctx.ws / (ms * 1e-3), "unit": "sweeps/s", "n_gpus": ctx.ws,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C2: {n} capsuleCast sweeps vs Semla render mesh ({info['n_static_triangles']} tris incl. ground), "
                               "r=1.5 hh=1.0, |delta| in [0.05, 2]", "hit_fraction": float((hits["triangle_index"] >= 0).mean()),
                   "order": "reference" if args.order == cq.ORDER_REFERENCE else "canonical",
                   "parity": parity, "e2e_matches_device_path": bool(host_hits.tobytes() == hits.tobytes())},
        "roofline": roofline_block("k_capsule_cast", ms, algo, ctr["distance_evals"],
                                   {k: ctr[k] / n for k in ("nodes_visited", "candidates", "distance_evals")},
                                   tr * n if tr is not None else None),
        "cpu_baseline": cpu,
        "e2e": {"value": n / e2e_s, "unit": "sweeps/s", "h2d_bytes_per_step": n * 40, "d2h_bytes_per_step": n * 44,
                "api": "cq_capsule_cast_batch (host pointers, pageable)"},
        "gpu_launches": int(launches), "clocks": clk}


# ------------------------------------------------------------------------------------------ C5: rays + refit
def measure_c5(ctx, args, n_total, steps, warmup, sharded):
    """Config C5: batched raycasts + a BVH refit of the spinning (dynamic-set) mirror every step."""
    cq, torch = ctx.cq, ctx.torch
    sc = cq.scenes
    parts = sc.merged_scene(mirror_dynamic=True)  # ground + 17-Cheese + Semla (FBX-regenerated stand-ins) + spinning mirror
    a = sc.load_mirror_fixture()
    base_t, base_q, base_s = sc.transform_from_matrix(sc.mirror_model(a["transform"]))
    mirror_id = parts[-1]["entity_id"]
    world = cq.CollisionQuery(parts, order=args.order)
    info = world.info()
    lo, hi = sc.scene_aabb(parts[1:])
    if sharded:
        s0, s1 = cq.shard_range(n_total, ctx.ws, ctx.rank)
        rays = np.ascontiguousarray(sc.gen_rays(n_total, lo, hi, seed=0xC0111DE5, max_distance=100.0, expand=5.0,
                                                y_range=(0.0, 12.0))[s0:s1])
    else:
        rays = sc.gen_rays(n_total, lo, hi, seed=0xC0111DE5 + ctx.rank, max_distance=100.0, expand=5.0, y_range=(0.0, 12.0))
    n = len(rays)
    units = n_total if sharded else n_total * ctx.ws
    d_r = ctx.up(rays)
    d_out = torch.empty(n * cq.RAY_HIT.itemsize, dtype=torch.uint8, device=ctx.dev)
    stream = ctx.stream
    angle = [0.0]

    def pose():
        rot = sc.quat_mul(sc.quat_angle_axis(np.radians(angle[0]), (0, 1, 0)), base_q)
        return sc.trs_model(base_t, rot, base_s)

    def step():
        angle[0] += 1.0
        world.update_transforms([mirror_id], [pose()])  # refit (synchronous: returns refit_ms)
        world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), stream)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    world.resetStats()
    sampler = ClockSampler(ctx.lrank)
    ctx.barrier()
    sampler.start()
    t0 = time.perf_counter()
    refit_ms = []
    for _ in range(steps):
        step()
        refit_ms.append(world.info()["refit_ms"])
    torch.cuda.synchronize()
    wall = ctx.red(time.perf_counter() - t0)
    ctx.barrier()
    clk = sampler.stop()
    launches = world.stats()["kernel_launches"]
    e0, e1 = ctx.events()
    e0.record()
    world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), stream)
    e1.record()
    torch.cuda.synchronize()
    ray_ms = e0.elapsed_time(e1)
    world.set_counting(cq.COUNT_PATH)
    world.resetStats()
    world.raycast_device(d_r.data_ptr(), n, d_out.data_ptr(), stream)
    torch.cuda.synchronize()
    ctr = world.stats(reset=True)
    world.set_counting(False)
    hits = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=cq.RAY_HIT)
    hit_pose = pose()
    algo = n * 64 + 32 * ctr["nodes_visited"] + 52 * ctr["candidates"]
    # e2e: the same step through the host-pointer API (refit + cq_raycast_batch, rays and hits in pinned host memory)
    hr = cq.PinnedArray((n,), cq.RAY)
    hr.array[:] = rays
    ho = cq.PinnedArray((n,), cq.RAY_HIT)
    L = cq.lib()

    def step_host():
        angle[0] += 1.0
        world.update_transforms([mirror_id], [pose()])
        rc = L.cq_raycast_batch(world.handle, hr.array.ctypes.data, n, ho.array.ctypes.data)
        assert rc == 0

    step_host()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host()
    e2e_s = ctx.red(time.perf_counter() - t0)
    hr.free()
    ho.free()
    cpu = None
    if ctx.rank == 0 and ctx.ws == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        cores = os.cpu_count() or 1
        ow = orc.OracleWorld(parts)
        t0 = time.perf_counter()
        ow.update_transforms([mirror_id], [hit_pose])  # the pose `hits` was cast at
        cpu_refit = time.perf_counter() - t0
        ns = min(n, 262144)
        t0 = time.perf_counter()
        ref = ow.raycast(rays[:ns], orc.ORDER_REFERENCE, cores)
        cdt = time.perf_counter() - t0
        cpu = {"value": ns / cdt, "unit": "rays/s", "cores": cores, "kind": "port",
               "sample": f"first {ns} of {n} rays, {cdt:.2f} s; CPU refit of the same part {cpu_refit * 1e3:.1f} ms",
               "gpu_bit_identical_on_the_sample": bool(ref.tobytes() == hits[:ns].tobytes()),
               "index_agreement": float((ref["triangle_index"] == hits["triangle_index"][:ns]).mean())}
        ow.close()
    world.close()
    tr = measured_traffic("k_raycast", "c5")
    return {
        "metric": "raycasts_per_sec_with_refit", "value": units * steps / wall, "unit": "rays/s", "n_gpus": ctx.ws,
        "steps": steps, "warmup": warmup, "ms_per_step": wall / steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C5: {n_total} raycasts " + ("in all, sharded over the ranks, " if sharded else "per GPU ") +
                               f"+ refit of the spinning mirror (dynamic set, {info['n_dynamic_triangles']} tris) each step; "
                               f"static set {info['n_static_triangles']} tris (ground + 17-Cheese + Semla render meshes regenerated "
                               "from FBX, tools/fbx_to_static_mesh.py)",
                   "order": "reference" if args.order == cq.ORDER_REFERENCE else "canonical",
                   "refit_ms_mean": float(np.mean(refit_ms)), "raycast_kernel_ms": ray_ms,
                   "hit_fraction": float((hits["triangle_index"] >= 0).mean()),
                   "timing": "host wall clock around (refit + raycast) steps, device synchronised"},
        "roofline": roofline_block("k_raycast_ref" if args.order == cq.ORDER_REFERENCE else "k_raycast", ray_ms, algo, None,
                                   {k: ctr[k] / n for k in ("nodes_visited", "candidates")}, tr * n if tr is not None else None),
        "cpu_baseline": cpu,
        "e2e": {"value": units * steps / e2e_s, "unit": "rays/s", "h2d_bytes_per_step": units * cq.RAY.itemsize,
                "d2h_bytes_per_step": units * cq.RAY_HIT.itemsize, "ms_per_step": e2e_s / steps * 1e3,
                "api": "cq_world_update_transforms + cq_raycast_batch (host pointers, pinned)"},
        "gpu_launches": int(ctx.red(launches, "sum")), "clocks": clk}


# ------------------------------------------------------------------------------------------ strong-scaling C3
def measure_c3_strong(ctx, args, n_total, steps, warmup):
    """BASELINE.json's '1M chars at 1/2/4/8': 1,048,576 characters IN ALL, rank r steps cq_shard_range(n, ws, r)."""
    cq = ctx.cq
    parts = cq.scenes.mirror_scene(use_hulls=True)
    pos, vel = cq.scenes.gen_c3_characters(n_total, seed=SEED)
    lo, hi = cq.shard_range(n_total, ctx.ws, ctx.rank)
    world = cq.CollisionQuery(parts, order=args.order)
    params = cq.default_params()
    d_states = ctx.up(cq.init_states(pos[lo:hi], vel[lo:hi]))
    n = hi - lo

    def step():
        world.move_and_slide_device(d_states.data_ptr(), n, params, DT, GRAVITY, cq.MAS_APPLY_GRAVITY, ctx.stream)

    total_ms, _ = time_steps(ctx, step, steps, warmup)
    world.close()
    return {"metric": "move_and_slide_queries_per_sec", "value": n_total * steps / (total_ms * 1e-3), "unit": "queries/s",
            "n_gpus": ctx.ws, "ms_per_step": total_ms / steps, "scaling": "strong",
            "config": {"workload": f"C3 hulls, {n_total} characters in all, sharded over {ctx.ws} GPU(s) "
                                   f"({n} on this rank), device-resident, no collective"}}


# ------------------------------------------------------------------------------------------ our arm
def _short(d):
    """An extra's record inside the headline line."""
    keep = ("metric", "value", "unit", "ms_per_step", "scaling", "collective_ms", "kernel_ms_alone", "config", "roofline",
            "cpu_baseline", "e2e", "clocks", "gpu_launches")
    return {k: d[k] for k in keep if k in d}


def run_ours(args):
    ctx = Ctx()
    cq = ctx.cq
    args.order = cq.ORDER_CANONICAL if args.order_name == "canonical" else cq.ORDER_REFERENCE
    only = args.only
    line = None
    if only in (None, "c3"):
        line = measure_mas(ctx, args, args.mesh, args.chars, args.steps, args.warmup, dump_dir=args.dump_outputs)
    extras = {}

    def extra(name, fn):
        if only not in (None, name) or (only is None and args.no_extras):
            return
        t0 = time.perf_counter()
        try:
            extras[name] = _short(fn()) if only is None else fn()
            extras[name]["bench_wall_s"] = time.perf_counter() - t0
        except Exception as e:  # an extra must never take the headline line down with it
            extras[name] = {"error": f"{type(e).__name__}: {e}", "trace": traceback.format_exc()[-1500:]}
        ctx.barrier()

    ks, kw = args.steps, 3
    multi = ctx.ws > 1
    if only is not None or (args.mesh == "hulls" and args.agents == 0):
        extra("terrain", lambda: measure_mas(ctx, args, "terrain", args.chars, ks, kw, cpu_baseline=True, clocks=False,
                                             full_record_e2e=False))
        extra("c4", lambda: measure_c4(ctx, args, args.queries or (1 << 23), ks, kw, sharded=multi))
        _TERRAIN.clear()
        if not multi:
            extra("render", lambda: measure_mas(ctx, args, "render", args.chars, ks, kw, cpu_baseline=True,
                                                clocks=False, full_record_e2e=False))
            extra("c2", lambda: measure_c2(ctx, args, args.queries or 65536, ks, kw))
        extra("c5", lambda: measure_c5(ctx, args, args.queries or (1 << 24), ks, kw, sharded=multi))
        if multi:
            extra("c3_strong", lambda: measure_c3_strong(ctx, args, CHARS_PER_GPU, ks, kw))
    if ctx.rank == 0:
        if line is None:
            line = next(iter(extras.values())) if extras else {"error": "nothing measured"}
        else:
            line["extra"] = extras
        emit(line)
    ctx.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None, choices=[None, "c3", "terrain", "render", "c2", "c4", "c5", "c3_strong"],
                    help="measure one configuration only and print its line (default: C3 headline + every extra)")
    ap.add_argument("--workload", default=None, choices=[None, "c2", "c3", "c4", "c5"], help="alias of --only")
    ap.add_argument("--no-extras", action="store_true", help="headline configuration only")
    ap.add_argument("--cells", type=int, default=2236)
    ap.add_argument("--queries", type=int, default=0)
    ap.add_argument("--radius", type=float, default=0.4)
    ap.add_argument("--half-height", type=float, default=0.5)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mesh", default="hulls", choices=["hulls", "render", "terrain"])
    ap.add_argument("--order", dest="order_name", default="reference", choices=["reference", "canonical"],
                    help="world order rule (include/cq.h); reference = the library's default")
    ap.add_argument("--chars", type=int, default=CHARS_PER_GPU)
    ap.add_argument("--separation", action="store_true",
                    help="with --agents: also run AgentSeparationSystem (exact sequential semantics) every step")
    ap.add_argument("--agents", type=float, default=0.0,
                    help="terrain mesh only: characters collide with each other; value = crowd footprint coverage (e.g. 0.1)")
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", action="store_true", help="(kept for compatibility: sharded c4 always gathers)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline path's character records as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or (args.only or args.workload) not in (None, "c3")):
        ap.error("--dump-outputs writes the move-and-slide headline's records: use it with --impl ours and no other --only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload and not args.only:
        args.only = args.workload
    if args.impl == "reference":
        return run_reference(args)
    if args.mesh != "hulls" and args.only is None:
        args.only = "c3"  # another mesh through the headline path: that configuration alone
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
