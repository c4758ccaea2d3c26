#!/usr/bin/env python
"""bench.py - env-steps/s of the cached-graph navigation hot path (step + reset + frame gather).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (CUDA, one process per GPU)
  python bench.py --impl reference [--steps K] [--warmup W]       # reference arm: CPU env classes on all host cores
  torchrun --nproc-per-node N ... bench.py --gpus N ...           # N > 1
  python bench.py --steps K --warmup W --dump-outputs DIR         # also write what the last timed step computed

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): one synthetic
thor-cached scene, 1,500 positions x 4 rotations = 6,000 states, 84x84 RGB + depth + goal frame,
4,096 envs per GPU (weak scaling: every GPU steps its own 4,096 envs, store replicated), uniform
random actions, TimeLimit 900, no curriculum by default (start states uniform over the scene, so the
4,096 envs read ~3,000 different frames per step and the gather is HBM-bound; with the reference's
initial hardness 0.01 - `--hardness 0.01` - the envs cluster around the goals and most reads hit L2).
One "step" = one vectorised step of all envs.  Rank 0 prints ONE JSON line.

Timed region: exactly K steps (`--steps K`) bracketed by a pair of CUDA events on the launching stream, preceded by
the `--mix` and the W warm-up steps (`--warmup W`), which are enqueued without waiting for them so that the region
opens with the device busy and the host ahead of it; barrier + synchronize before those and after the region.
`ms_per_step` / `value` are the region's time over K (maximised over the ranks).  NO collective, host
synchronisation or allocation sits between the two event records (`timed_blocks`, checked by
tests/test_bench_contract.py); the one NCCL call near this path - the episode-statistics all-reduce - is timed
on its own and reported as `collective_ms`.  Every input of the timed steps is seeded and the number of steps before
the region is fixed by the arguments, so the same command line steps the same envs through the same states on every
run.

`--dump-outputs DIR` writes what the last timed step computed, as seen by its caller, to DIR/<name>.npy (float32,
or float64 where float32 would not hold the values exactly; at most 64 MB in all): every observation leaf
(`obs_<leaf>`), `last_action_reward`, `reward`, `done`.  Where the observation batch is larger than that, the same
fixed, seeded sample of env rows is written for every leaf.  `--workload c5` writes the rollout builder's results
instead.  With more than one rank, rank 0 writes its own shard.
"""
import argparse
import importlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

ENVS_PER_GPU = 4096
N_CELLS, GRID = 1500, (50, 60)
MAX_EPISODE_STEPS = 900
HARDNESS = None
SCENE_SEED = 0
PLANE_BYTES = {"rgb": 84 * 84 * 3, "depth": 84 * 84, "segmentation": 84 * 84 * 3}
F_RGB, F_DEPTH, F_SEG = PLANE_BYTES["rgb"], PLANE_BYTES["depth"], PLANE_BYTES["segmentation"]
WORKLOAD = "C2 synthetic thor-cached scene: 1,500 positions x 4 rotations, 84x84 RGB+depth+goal, 4,096 envs per GPU"
METRIC = "env-steps/s (obs gather+step+reset)"
MIN_REGION_S = 0.2          # the timed region is repeated until it lasts at least this long
MAX_BLOCKS = 4000
DUMP_BYTES = 60_000_000     # --dump-outputs: array data of all files together (headers add a few hundred bytes)


def make_scene(vn, planes=("rgb", "depth")):
    return vn.scenes.make_thor_scene(N_CELLS, GRID, seed=SCENE_SEED, n_goals=4, planes=planes)


# (description, envs per GPU, observation layout, states, planes) of every BASELINE.json config - known without a GPU
WORKLOADS = {
    "c2": (WORKLOAD, ENVS_PER_GPU, "rgbd_goal"),
    "c1": ("C1 10x10 grid maze, 16 envs, 84x84 aux observation (rgb, goal, depth, seg, goal seg)", 16, "aux5"),
    "c3": ("C3 dungeon 64x64 multi-room (oriented), 65,536 envs per GPU, RGB + goal image, auto-reset", 65536, "pair"),
    "c4": ("C4 30 synthetic thor-cached scenes resident (180,000 states, 5.1 GB), 32,768 envs per GPU, RGB+depth+goal",
           32768, "rgbd_goal"),
    "rgb": ("84x84 RGB-only cached-graph nav (north_star target line), C2 scene, 4,096 envs per GPU", ENVS_PER_GPU,
            "frame"),
    "aux5": ("C2 scene with the reference's 5-tuple observation (rgb, goal, depth, seg, goal seg), 4,096 envs per GPU",
             ENVS_PER_GPU, "aux5"),
}


def make_world(vn, name):
    S = vn.scenes
    if name in ("c2", "rgb"):
        return vn.compile_world([make_scene(vn)], vn.GYM_GRAPH)
    if name == "aux5":
        return vn.compile_world([make_scene(vn, ("rgb", "depth", "segmentation"))], vn.GYM_GRAPH)
    if name == "c1":
        return vn.compile_world([S.make_maze_scene((10, 10), 0.25, 0, n_goals=1)], vn.GYM_GRAPH)
    if name == "c3":
        return vn.compile_world([S.make_dungeon_scene((64, 64), 0, oriented=True, planes=("rgb",))], vn.GYM_GRAPH)
    if name == "c4":
        scs = [S.make_thor_scene(N_CELLS, GRID, seed=k, n_goals=4, planes=("rgb", "depth"), scene_id=k) for k in range(30)]
        return vn.compile_world(scs, vn.GYM_GRAPH)
    raise ValueError(name)


def make_workload(vn, name):
    """BASELINE.json configs -> (description, world, envs per GPU, obs_layout).  configs[1] (c2) is the one
    the headline metric is quoted on; the others are secondary lines (`--workload`)."""
    desc, envs, layout = WORKLOADS[name]
    return desc, make_world(vn, name), envs, layout


def static_config(args, world_size):
    """The `config` object of the JSON line: what the workload IS, nothing that was measured - so that our arm and
    the reference arm print the SAME object for the same command line (measured rates live in `run_stats`)."""
    desc, envs, layout = WORKLOADS[args.workload]
    per_gpu = args.envs_per_gpu or envs
    hardness = None if args.hardness in (None, "none") else float(args.hardness)
    return {"workload": desc, "envs_per_gpu": per_gpu, "envs_total": per_gpu * world_size, "obs_layout": layout,
            "frame": "84x84 uint8", "actions": "uniform random over 4", "max_episode_steps": MAX_EPISODE_STEPS,
            "hardness": hardness, "auto_reset": True,
            "l2": "inputs larger than L2: store + batch rewritten every step exceed the 126 MB L2 (C2: 170 MB store + "
                  "116 MB batch); no flush needed between iterations",
            "parallelism": "env-sharded x%d, store replicated, no data-path collective" % world_size}


def layout_bytes(vn, layout):
    """(observation bytes per env-step, goal bytes per reset) of an obs layout."""
    leaves = importlib.import_module("a2cat-vn-pytorch_b200.vec_env").resolve_layout(layout)
    names = list(leaves.values()) if isinstance(leaves, dict) else (list(leaves) if isinstance(leaves, tuple) else [leaves])
    obs = sum(PLANE_BYTES[x] for x in dict.fromkeys(n for n in names if not n.startswith("goal_")))
    goal = sum(PLANE_BYTES[x[5:]] for x in dict.fromkeys(n for n in names if n.startswith("goal_")))
    return obs, goal


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs.  Construct it (nvmlInit,
    tens of ms) BEFORE the barrier that opens the timed region; `start()` only spawns the thread."""

    def __init__(self, index, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic(workload, kernel):
    """DRAM bytes (read, write) per launch of the dominant kernel from the committed ncu captures
    (profiles/roofline_traffic.json, one entry per workload), or None when that workload / kernel was not captured."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        d = json.load(open(path))
    except Exception:
        return None
    w = (d.get("workloads") or {}).get(workload)
    if not w or w.get("kernel") != kernel:
        return None
    return w


# ------------------------------------------------------------------------------------------ timed regions
def timed_blocks(make_event, run_block, n_blocks):
    """THE timed region of every device-resident number in this file: `n_blocks` back-to-back blocks, each bracketed
    by a pair of events recorded on the launching stream.  Only step launches and event records happen in here - no
    collective, no barrier, no host synchronisation, no allocation (tests/test_bench_contract.py parses this function
    and runs it under gloo with collectives that raise inside the region)."""
    events = [(make_event(), make_event()) for _ in range(n_blocks)]
    # >>> timed region
    for r in range(n_blocks):
        events[r][0].record()
        run_block(r)
        events[r][1].record()
    # <<< timed region
    return events


class Harness:
    """barrier / timing plumbing shared by every leg: barrier + synchronize on both sides of `timed_blocks`, per-block
    times maximised over the ranks AFTER the region closed."""

    def __init__(self, torch, dist, dev, world_size):
        self.torch, self.dist, self.dev, self.world_size = torch, dist, dev, world_size

    def barrier(self):
        if self.world_size > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, values):
        if self.world_size == 1:
            return [float(v) for v in values]
        t = self.torch.tensor(list(values), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def blocks(self, run_block, n_blocks, lead=None):
        """ms of each block (max over ranks).  `lead()` enqueues un-timed work between the opening barrier and the
        first event, so that the device is still busy with it when the region opens.  The events are created before
        the barrier: nothing but `lead` runs on the host between the two."""
        pool = [self.torch.cuda.Event(enable_timing=True) for _ in range(2 * n_blocks)][::-1]
        make_event = pool.pop
        self.barrier()
        if lead is not None:
            lead()
        events = timed_blocks(make_event, run_block, n_blocks)
        self.barrier()
        return self.max_over_ranks([a.elapsed_time(b) for a, b in events])

    def n_blocks_for(self, est_block_ms):
        """Blocks needed for a region of MIN_REGION_S, agreed between the ranks (max)."""
        n = int(min(MAX_BLOCKS, max(1, np.ceil(MIN_REGION_S * 1e3 / max(est_block_ms, 1e-3)))))
        return int(self.max_over_ranks([n])[0])

    def steps_per_s(self, step, n_steps, total_envs, warm=50):
        """Median-of-blocks rate of `step(i)` over blocks of `n_steps` (secondary legs)."""
        for i in range(warm):
            step(i)
        est = min(self.blocks(lambda r: [step(i) for i in range(n_steps)], 2))
        nb = self.n_blocks_for(est)
        ms = self.blocks(lambda r: [step(r * n_steps + i) for i in range(n_steps)], nb)
        med = float(np.median(ms))
        return {"value": total_envs * n_steps / (med * 1e-3), "unit": "env-steps/s", "steps": n_steps, "blocks": nb,
                "ms_per_step": med / n_steps, "ms_per_step_min": min(ms) / n_steps, "ms_per_step_max": max(ms) / n_steps}


def e2e_loop(step, n_steps, sync):
    """Wall-clock of `n_steps` host-facing steps on this rank.  The device is drained before the clock is read at both
    ends; NO barrier / collective inside (the caller puts its barrier before calling and takes the max over ranks
    afterwards)."""
    sync()
    # >>> timed region
    t0 = time.perf_counter()
    for i in range(n_steps):
        step(i)
    sync()
    dt = time.perf_counter() - t0
    # <<< timed region
    return dt


# ------------------------------------------------------------------------------------------ --dump-outputs
def obs_leaves(env):
    """(name, tensor) of every observation leaf a step of `env` hands back, in layout order, then last_action_reward."""
    lv = env.leaves
    names = list(lv) if isinstance(lv, dict) else (list(lv) if isinstance(lv, tuple) else [lv])
    obs = env._obs()
    inner, lar = obs if env.unreal_wrapper else (obs, None)
    tensors = [inner[k] for k in names] if isinstance(lv, dict) else (list(inner) if isinstance(lv, tuple) else [inner])
    out = [("obs_" + n, t) for n, t in zip(names, tensors)]
    return out + ([("last_action_reward", lar)] if lar is not None else [])


def dump_outputs(out_dir, arrays, sampled, budget=DUMP_BYTES, seed=0):
    """Writes every (name, tensor) of `arrays` to out_dir/<name>.npy: floating point as float32 (float64 stays
    float64), integers and booleans as float32, or float64 where float32 would not hold them exactly.  When all of it
    would exceed `budget` bytes, the arrays named in `sampled` (same first dimension) keep the same fixed, seeded
    sample of rows (ascending); the others are always written whole."""
    import torch
    host = []
    for name, t in arrays:
        if t.dtype in (torch.bool, torch.uint8, torch.int8, torch.int16):
            t = t.to(torch.float32)
        elif not t.is_floating_point():
            x = t.to(torch.float64)
            t = x.to(torch.float32) if torch.equal(x.to(torch.float32).to(torch.float64), x) else x
        elif t.dtype != torch.float64:
            t = t.to(torch.float32)
        host.append((name, t))
    rowed = [name in sampled for name, _ in host]
    batch = {t.shape[0] for (_, t), r in zip(host, rowed) if r}
    assert len(batch) <= 1, "sampled arrays must share their first dimension"
    batch = batch.pop() if batch else 0
    fixed = sum(t.numel() * t.element_size() for (_, t), r in zip(host, rowed) if not r)
    per_row = sum(t[0].numel() * t.element_size() for (_, t), r in zip(host, rowed) if r)
    rows = batch if per_row == 0 else min(batch, max(1, (budget - fixed) // per_row))
    if fixed + rows * per_row > budget:
        raise ValueError("--dump-outputs: %d bytes of whole arrays alone exceed %d" % (fixed, budget))
    idx = None
    if rows < batch:
        idx = np.sort(np.random.RandomState(seed).choice(batch, rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for (name, t), r in zip(host, rowed):
        if r and idx is not None:
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------ CPU arm
_CPU = {}


class _FastStart:
    """Initial placement of the CPU envs (un-timed): a uniform draw from the candidate list computed ONCE per goal -
    the distribution `sample_initial_state` has without a curriculum.  4,096 envs start in seconds instead of the
    minutes 4,096 reference-style resets take; every reset inside the timed region pays the reference's full cost."""

    def __init__(self, cands, goal_index, rng):
        self.cands, self.gi, self.rng = cands, goal_index, rng

    def __call__(self):
        pots = self.cands[self.gi]
        return 0, pots[int(self.rng.randint(len(pots)))]


def _cpu_world(n_envs, seed):
    """Oracle envs of the bench workload with the reference's cost profile (frames in RAM, per-reset
    candidate enumeration).  Built once per process (workers inherit it by fork)."""
    from oracle import envs as oenvs, vec as ovec, graph_util as gu
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    if "scene" not in _CPU:
        scene = make_scene(vn)
        _CPU["scene"] = scene
        _CPU["osc"] = oenvs.OracleScene(scene, with_all_pairs=True, cache_frames=True)
        osc = _CPU["osc"]
        _CPU["cands"] = [gu.initial_state_candidates(osc.maze, osc.graph, osc.optimal_actions, g)[0] for g in scene.goals]
    scene, osc = _CPU["scene"], _CPU["osc"]
    rng = np.random.RandomState(seed + 77)
    envs, sources = [], []
    for i in range(n_envs):
        gi = i % len(scene.goals)
        goal = scene.goals[gi]                              # one env per (scene, goal) task, dealt round-robin
        e = oenvs.GymGraphRgbdGoalEnv(osc, goals=goal)
        e.set_complexity(_CPU.get("hardness", HARDNESS))
        e.reset_source = _FastStart(_CPU["cands"], gi, rng)
        sources.append(ovec.ReferenceStyleResetSource(osc, [goal], lambda t, e=e: e.optimal_distance(), seed + i))
        tl = ovec.TimeLimit(e, MAX_EPISODE_STEPS)
        envs.append(ovec.RewardCollector(tl))
    ve = ovec.VecEnv(envs)
    ve._time_limits = [w.env for w in envs]
    ve._timed_sources = sources
    return ve


def _start(ve, seed):
    """reset() with the fast placement, then: reference-cost resets from here on, and every env at a random phase of
    its 900-step episode so that a bounded sample sees time-limit resets at the steady-state rate (1 / 900 per
    env-step) instead of none at all."""
    ve.reset()
    rng = np.random.RandomState(seed + 4242)
    for tl, src in zip(ve._time_limits, ve._timed_sources):
        tl._elapsed = int(rng.randint(0, MAX_EPISODE_STEPS))
        tl.env.reset_source = src


def _cpu_worker(conn, n_envs, seed):
    """baselines SubprocVecEnv worker protocol (SURVEY.md D1): step -> auto-reset -> send obs over a pipe."""
    ve = _cpu_world(n_envs, seed)
    while True:
        cmd, data = conn.recv()
        if cmd == "step":
            conn.send(ve.step(data)[:3])
        elif cmd == "reset":
            _start(ve, seed)
            conn.send(None)
        else:
            conn.close()
            return


def cpu_run(n_envs, steps, warmup, workers, seed=0):
    """Returns (env-steps/s, resets, seconds) of the CPU port on `workers` processes."""
    import multiprocessing as mp
    rng = np.random.RandomState(seed)
    if workers <= 1:
        ve = _cpu_world(n_envs, seed)
        _start(ve, seed)
        for _ in range(warmup):
            ve.step(rng.randint(0, 4, n_envs))
        t0 = time.perf_counter()
        nres = 0
        for _ in range(steps):
            _, _, d, _ = ve.step(rng.randint(0, 4, n_envs))
            nres += int(d.sum())
        dt = time.perf_counter() - t0
        return n_envs * steps / dt, nres, dt
    _cpu_world(0, seed)                                   # build the scene before forking
    ctx = mp.get_context("fork")
    per = [n_envs // workers + (1 if r < n_envs % workers else 0) for r in range(workers)]
    pipes, procs = [], []
    for r, n in enumerate(per):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_cpu_worker, args=(b, n, seed + 100000 * r), daemon=True)
        p.start()
        pipes.append(a)
        procs.append(p)

    def vec(cmd, acts=None):
        off = 0
        for n, c in zip(per, pipes):
            c.send((cmd, None if acts is None else acts[off:off + n]))
            off += n
        outs = [c.recv() for c in pipes]
        if cmd == "reset":
            return None
        obs = tuple(np.concatenate([o[0][0][k] for o in outs]) for k in range(3))      # parent-side stack
        return obs, np.concatenate([o[1] for o in outs]), np.concatenate([o[2] for o in outs])

    vec("reset")
    for _ in range(warmup):
        vec("step", rng.randint(0, 4, n_envs))
    t0 = time.perf_counter()
    nres = 0
    for _ in range(steps):
        _, _, d = vec("step", rng.randint(0, 4, n_envs))
        nres += int(d.sum())
    dt = time.perf_counter() - t0
    for c in pipes:
        c.send(("close", None))
    for p in procs:
        p.join(5)
    return n_envs * steps / dt, nres, dt


def reference_run(n_envs, steps, warmup, seed=0):
    """The UNMODIFIED reference classes (environments/gym_graph/graph.py GoalGymGraphAuxiliaryEnv over a ThorGridWorld
    with dense [X,Y,4,H,W,C] arrays) on the bench scene, one process: step every env, TimeLimit + auto-reset as the
    VecEnv worker does, np.stack of the C2 leaves (rgb, goal, depth).  Only where /root/reference exists (this
    container); the GPU box has no reference tree and times the oracle port instead."""
    from oracle import ref_harness as rh
    ref = rh.ref_modules()
    import io
    import pickle
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    scene = make_scene(vn, ("rgb", "depth", "segmentation"))
    X, Y = scene.maze.shape
    h, w = scene.frame_hw
    arrs = {}
    for plane, c in (("rgb", 3), ("depth", 1), ("segmentation", 3)):
        a = np.zeros((X, Y, 4, h, w, c), np.uint8)
        a[scene.cells[:, 0], scene.cells[:, 1]] = scene.plane_frames(plane).reshape(scene.n_cells, 4, h, w, c)
        arrs[plane] = a
    world = ref.thor_world.ThorGridWorld(scene.maze.copy(), arrs["rgb"], arrs["depth"], arrs["segmentation"])
    # the reference's own all-pairs routine (graph/util.py:146-176, recursive) cannot finish on a 1,500-cell scene
    # (SURVEY.md A12); the oracle's BFS gives bit-identical tables (tests/test_oracle_golden.py)
    from oracle import graph_util as gu
    world.graph, world.optimal_actions = gu.compute_shortest_path_data(scene.maze)
    import copy
    first = ref.gym_graph.GoalGymGraphAuxiliaryEnv(graph_file=io.BytesIO(pickle.dumps(world, protocol=4)),
                                                   goals=scene.goals[0], screen_size=(84, 84))
    first.graph = ref.core.GraphResize(first.graph._graph, (84, 84))     # SURVEY.md A10 quirk
    del arrs, world
    envs = []
    for i in range(n_envs):
        e = copy.copy(first)                 # same class, shared scene arrays (one 600 MB copy, not one per env)
        e.goals = scene.goals[i % len(scene.goals)]
        e._cached_goal = (None, None)
        e.set_complexity(_CPU.get("hardness", HARDNESS))
        envs.append(e)
    rng = np.random.RandomState(seed)
    obs = [e.reset() for e in envs]
    elapsed = [int(v) for v in np.random.RandomState(seed + 4242).randint(0, MAX_EPISODE_STEPS, n_envs)]

    def vec_step(actions):
        out, rew, done = [], np.zeros(n_envs, np.float32), np.zeros(n_envs, bool)
        for i, e in enumerate(envs):
            ob, r, d, info = e.step(int(actions[i]))
            elapsed[i] += 1
            if elapsed[i] >= MAX_EPISODE_STEPS:
                info["TimeLimit.truncated"] = not d
                d = True
            if d:
                ob = e.reset()
                elapsed[i] = 0
            out.append(ob)
            rew[i], done[i] = r, d
        return tuple(np.stack([o[k] for o in out]) for k in (0, 1, 2)), rew, done

    for _ in range(warmup):
        vec_step(rng.randint(0, 4, n_envs))
    t0 = time.perf_counter()
    nres = 0
    for _ in range(steps):
        _, _, d = vec_step(rng.randint(0, 4, n_envs))
        nres += int(d.sum())
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, nres, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world_size = int(os.environ.get("WORLD_SIZE", str(args.gpus or 1)))
    _CPU["hardness"] = None if args.hardness in (None, "none") else float(args.hardness)
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 64))
    steps = args.steps if args.steps else 300
    warm = args.warmup if args.warmup is not None else 5
    cfg = static_config(args, world_size)
    # Bounded sample of the workload: the configuration's own env count per GPU when K is small (the driver's
    # --steps 20: all 4,096 envs x 20 vector steps), fewer envs when K is large (<= ~100 k env-steps per leg).
    budget = args.cpu_budget
    n_multi = int(max(workers, min(cfg["envs_per_gpu"], budget // max(1, steps))))
    n_multi -= n_multi % workers
    n_single = int(max(1, min(cfg["envs_per_gpu"], (budget // 2) // max(1, steps))))
    legs = {}
    v, nres, dt = cpu_run(n_multi, steps, warm, workers)
    legs["processes_%d" % workers] = {"value": v, "envs": n_multi, "seconds": dt, "p_reset": nres / max(1, n_multi * steps)}
    v1, nres1, dt1 = cpu_run(n_single, steps, warm, 1)
    legs["process_1"] = {"value": v1, "envs": n_single, "seconds": dt1, "p_reset": nres1 / max(1, n_single * steps)}
    kind, value, used, total_dt = "port", v, workers, dt
    if v1 > v:
        value, used, total_dt = v1, 1, dt1
    from oracle import ref_harness as rh
    if rh.reference_available() and not args.port_only:
        # the unmodified reference classes, where the reference tree exists (this container, not the GPU box)
        n_ref = int(max(1, min(256, (budget // 4) // max(1, steps))))
        vr, nresr, dtr = reference_run(n_ref, steps, warm)
        legs["reference_classes_1_process"] = {"value": vr, "envs": n_ref, "seconds": dtr,
                                               "p_reset": nresr / max(1, n_ref * steps)}
        kind, value, used, total_dt = "reference", vr, 1, dtr
    port = ("oracle port of GoalGymGraphAuxiliaryEnv, %d vector steps: best of {%d envs over %d worker processes (pipes, "
            "parent-side stack), %d envs in one process (sequential + np.stack)}; per-reset candidate enumeration as in "
            "sample_initial_state, episode phases randomised to the steady state" % (steps, n_multi, workers, n_single))
    sample = port if kind == "port" else (
        "UNMODIFIED reference classes (environments/gym_graph/graph.py GoalGymGraphAuxiliaryEnv over a ThorGridWorld), "
        "%d envs x %d vector steps in one process with TimeLimit + auto-reset + np.stack; the port legs (%s) are in "
        "`legs`" % (legs["reference_classes_1_process"]["envs"], steps, port))
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "impl": "reference",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * total_dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": used, "kind": kind, "sample": sample,
                         "host_cores": cores, "legs": legs},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------ CUDA arm
def run_cuda(args):
    import torch
    import torch.distributed as dist
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    L = vn.lib
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world_size > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    H = Harness(torch, dist, dev, world_size)
    K = args.steps if args.steps else 20000
    W = args.warmup if args.warmup is not None else 200
    W = max(W, 3)
    sampler = ClockSampler(local_rank)            # nvmlInit happens here, long before the timed region

    workload, world, envs_per_gpu, layout = make_workload(vn, args.workload)
    cfg = static_config(args, world_size)
    F_OBS, F_GOAL = layout_bytes(vn, layout)
    n_total = cfg["envs_total"]
    mk = dict(device=dev, max_episode_steps=MAX_EPISODE_STEPS, unreal_wrapper=True, rank=rank, world_size=world_size,
              gather=args.gather)
    env = vn.GraphVecEnv(world, n_total, seed=1, obs_layout=layout, host_outputs=False, **mk)
    hardness = cfg["hardness"]
    _CPU["hardness"] = hardness
    env.set_complexity(hardness)
    N = env.num_envs
    # action stream resident in HBM: cyclic buffer of uniform random actions (Philox via torch generator)
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    n_rows = 2048
    actions = torch.randint(0, 4, (n_rows, N), device=dev, generator=gen, dtype=torch.int32)
    env.reset()

    graph_len = 0
    l0 = env.kernel_launches
    env.step_enqueue(actions[0], actions_ready=not args.serial)
    launches_per_step = env.kernel_launches - l0        # 1 (one fused launch) or 2 (scalar + gather)
    if args.cuda_graph:
        # launch-bound batches (C1): replay CUDA graphs of `graph_len` steps instead of 2 launches per step
        graph_len = min(64, n_rows)
        graph = env.capture_steps(actions[:graph_len])

    def device_loop(k0, k):
        """Enqueues exactly k steps: action rows k0 .. k0 + k - 1, or with --cuda-graph k // graph_len replays (rows
        0 .. graph_len - 1 each) followed by k % graph_len eager steps on rows 0, 1, ..."""
        if graph_len:
            for _ in range(k // graph_len):
                graph.replay()
            for i in range(k % graph_len):
                env.step_enqueue(actions[i], actions_ready=not args.serial)
            return
        for i in range(k0, k0 + k):
            # the action stream is pre-computed and resident: VN_STEP_ACTIONS_READY lets the scalar part of
            # step i + 1 run while the gather of step i is still copying
            env.step_enqueue(actions[i % n_rows], actions_ready=not args.serial)

    # the only collective anywhere near this path - the episode-statistics all-reduce - is exercised once here so that
    # its first-use cost (NCCL channel setup) cannot leak into anything timed later
    stats_vec = env.stats.to(torch.float64)
    if world_size > 1:
        dist.all_reduce(stats_vec)
    mark = {}

    def warm_up():
        device_loop(0, args.mix)      # un-timed: lets the state distribution settle (random-walk mixing)
        # the statistics count the warm-up and the timed steps: nothing but steps may sit between the two, or the
        # first timed step could not overlap the last warm-up gather
        env.stats.zero_()
        device_loop(0, W)
        mark["launches0"] = env.kernel_launches

    sampler.start()
    ms = H.blocks(lambda r: device_loop(W, K), 1, lead=warm_up)[0]
    clocks = sampler.stop()
    launches = (launches_per_step * K) if graph_len else env.kernel_launches - mark["launches0"]
    if args.dump_outputs and rank == 0:
        leaves = obs_leaves(env)
        dump_outputs(args.dump_outputs, leaves + [("reward", env.reward), ("done", env.done)],
                     sampled=[n for n, _ in leaves if n.startswith("obs_")])
    stats = env.episode_stats(reduce=True)
    value = n_total * K / (ms * 1e-3)
    p_reset = stats["resets"] / max(1.0, stats["steps"])
    coll = stats["collisions"] / max(1.0, stats["steps"])
    p_skip = stats["rows_skipped"] / max(1.0, stats["steps"])   # rows whose record did not change: not copied again

    # ---- the statistics all-reduce on its own (a logging-interval operation, never inside a step)
    collective_ms = None
    if world_size > 1:
        side = torch.cuda.Stream(dev)
        H.barrier()
        with torch.cuda.stream(side):
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(10):
                dist.all_reduce(stats_vec)
            c1.record()
        side.synchronize()
        collective_ms = H.max_over_ranks([c0.elapsed_time(c1) / 10])[0]

    # ---- roofline of the dominant kernel (the frame gather): instrumented pass, events around each launch alone
    peak, peak_src = measured_peak()
    import ctypes as C
    iso = None
    if launches_per_step == 2:
        Kr = 300
        es = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Kr)]
        stream = torch.cuda.current_stream(dev).cuda_stream
        env.stats.zero_()
        torch.cuda.synchronize(dev)
        for i in range(Kr):
            a = actions[(W + i) % n_rows]
            env._tick(env._c_out, env._step_flags)      # serial mode: next descriptor half, no overlap with the previous gather
            L.check(env.lib.vn_env_step_scalar(C.byref(env.dw.tables), C.byref(env._c_envs), C.byref(env._c_rules), None,
                                               a.data_ptr(), C.byref(env._c_out), stream))
            es[i][0].record()
            L.check(env.lib.vn_env_gather(C.byref(env.dw.store), C.byref(env._c_envs), C.byref(env._c_out), env.gather,
                                          stream))
            es[i][1].record()
        torch.cuda.synchronize(dev)
        gather_ms = float(np.median([a.elapsed_time(b) for a, b in es]))
        rs = env.episode_stats()
        p_reset_r = rs["resets"] / max(1.0, rs["steps"])
        p_skip_r = rs["rows_skipped"] / max(1.0, rs["steps"])
        iso_bytes = N * ((1 - p_skip_r) * 2 * F_OBS + p_reset_r * 2 * F_GOAL)
        iso = {"kernel_ms": gather_ms, "achieved": iso_bytes / (gather_ms * 1e-3) / 1e9,
               "frac": iso_bytes / (gather_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": iso_bytes,
               "how": "CUDA events around each gather launch alone (serialised, includes launch latency), median of %d" % Kr}
    # algorithmic bytes of one launch (SURVEY.md section 8(d)): one read + one write of every observation row that
    # CHANGED (rows of envs that collided hold the right frames already and are skipped, like the goal rows of envs
    # that did not reset), plus the goal rows of the envs that reset.  In the timed region the scalar part of step
    # k+1 overlaps the gather of step k, so the launch-to-launch period there IS the dominant kernel's duration in
    # situ (an upper bound of it - everything else the step does is inside).
    alg_bytes = N * ((1 - p_skip) * 2 * F_OBS + p_reset * 2 * F_GOAL)
    situ_ms = ms / K
    achieved = alg_bytes / (situ_ms * 1e-3) / 1e9
    # calibration: plain contiguous device copies of the SAME number of bytes (torch copy_, the operation the
    # measured peak was taken with, but at this kernel's size instead of 2 GiB), back to back over 4 distinct
    # (src, dst) pairs so that, like the gather in steady state, every copy starts with L2 full of the previous
    # copy's dirty lines - what a transfer of this size can sustain on this GPU
    nb = N * F_OBS
    pairs = [(torch.empty(nb, dtype=torch.uint8, device=dev).random_(0, 255),
              torch.empty(nb, dtype=torch.uint8, device=dev)) for _ in range(4)]
    for i in range(8):
        pairs[i % 4][1].copy_(pairs[i % 4][0])
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    c0.record()
    for i in range(200):
        pairs[i % 4][1].copy_(pairs[i % 4][0])
    c1.record()
    torch.cuda.synchronize(dev)
    copy_ms = c0.elapsed_time(c1) / 200
    del pairs

    if launches_per_step == 1:      # one launch per step: persistent grid (ONE host sequence word) or CTA-per-env fused
        kname = "vn_step_gather_kernel" if (env._seq_words == 1 and N > 1) else "vn_step_fused_kernel"
    else:
        kname = "vn_gather_%s_kernel" % ("ldg" if args.gather == "ldg" else "bulk")
    prof = profiled_traffic(args.workload if hardness is None else None, kname)
    traffic = (prof["dram_bytes_read_per_launch"] + prof["dram_bytes_write_per_launch"]) if prof else None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                # DRAM-counter view of the same launch: ncu dram__bytes_{read,write}.sum per steady-state launch (no
                # cache flush between launches) over THIS run's in-situ kernel time
                "dram_frac": (traffic / (situ_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "traffic_source": prof.get("source") if prof else None,
                "kernel": kname,
                "kernel_ms": situ_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "how": "in situ: CUDA events around the K timed steps / K launches (the scalar part of a step overlaps "
                       "the previous gather, so this is the gather's launch-to-launch period)",
                "rows_skipped_rate": p_skip, "isolated": iso,
                "same_size_copy_ms": copy_ms, "same_size_copy_gbs": 2 * nb / (copy_ms * 1e-3) / 1e9,
                # the DRAM rate of the gather next to what a plain copy of this size reaches on this GPU (a 36 us
                # transfer does not reach the 2 GiB copy peak either)
                "dram_rate_vs_same_size_copy": (traffic / (situ_ms * 1e-3) / 1e9) / (2 * nb / (copy_ms * 1e-3) / 1e9)
                if traffic else None}

    run_stats = {"p_reset": p_reset, "collision_rate": coll, "rows_skipped_rate": p_skip,
                 "launches_per_step": launches_per_step, "states": world.n_states, "store_bytes": env.dw.nbytes(),
                 "batch_bytes_per_step": N * F_OBS, "gather": args.gather, "mix_steps": args.mix,
                 "cuda_graph_steps": graph_len, "blocks": 1, "timed_steps_total": K,
                 "timed_region_ms": ms, "collective_ms": collective_ms}

    if args.quick:
        if rank == 0:
            emit({"value": value, "ms_per_step": ms / K, "frac": roofline["frac"], "iso": iso and iso["kernel_ms"],
                  "iso_frac": iso and iso["frac"], "p_reset": p_reset, "p_skip": p_skip,
                  "launches_per_step": launches_per_step})
        if world_size > 1:
            dist.destroy_process_group()
        return

    # ---- secondary lines (same store unless stated)
    secondary = {}
    act = lambda i: actions[i % n_rows]
    if args.workload == "c2":
        # RGB-only observation: the north-star ">= 1e9 env-steps/s on 8 GPUs for 84x84 cached-graph nav" refers to this
        # 42,336 B/step variant (SURVEY.md section 8(d))
        env_r = vn.GraphVecEnv(world, n_total, seed=3, obs_layout="frame", host_outputs=False, device_world=env.dw, **mk)
        env_r.reset()
        [env_r.step_enqueue(act(i), actions_ready=True) for i in range(300)]
        env_r.stats.zero_()
        r = H.steps_per_s(lambda i: env_r.step_enqueue(act(i), actions_ready=True), 500, n_total)
        sr = env_r.episode_stats()
        skip_r = sr["rows_skipped"] / max(1.0, sr["steps"])
        r.update({"algorithmic_bytes_per_env_step": 2 * F_RGB, "rows_skipped_rate": skip_r,
                  "frac": N * (1 - skip_r) * 2 * F_RGB / (r["ms_per_step"] * 1e-3) / 1e9 / peak,
                  "frac_if_every_row_were_copied": N * 2 * F_RGB / (r["ms_per_step"] * 1e-3) / 1e9 / peak})
        pr = profiled_traffic("rgb", kname)
        if pr:
            tr = pr["dram_bytes_read_per_launch"] + pr["dram_bytes_write_per_launch"]
            r.update({"traffic": tr, "dram_frac": tr / (r["ms_per_step"] * 1e-3) / 1e9 / peak})
        secondary["rgb_only"] = r
        del env_r
        # the same steps WITHOUT the promise that the actions were ready early - what a training loop with a GPU policy
        # between two steps gets: nothing can overlap the previous gather, VN_GATHER_AUTO runs the step as ONE launch
        env_s = vn.GraphVecEnv(world, n_total, seed=5, obs_layout=layout, host_outputs=False, device_world=env.dw, **mk)
        env_s.reset()
        [env_s.step_enqueue(act(i)) for i in range(300)]
        l0 = env_s.kernel_launches
        sr_ = H.steps_per_s(lambda i: env_s.step_enqueue(act(i)), 500, n_total)
        sr_.update({"launches_per_step": (env_s.kernel_launches - l0) / (500.0 * (sr_["blocks"] + 2) + 50),
                    "note": "serial steps (no VN_STEP_ACTIONS_READY): persistent single launch"})
        secondary["serial_steps"] = sr_
        del env_s
        # float32 CHW observations in [0, 1] - what the reference's wrappers hand to its model (TransposeImage +
        # ScaledFloatFrame, thor_cached_auxiliary.py:61-62) - converted straight from the store into persistent
        # batches (no uint8 batch in this mode): 4 bytes written per byte read
        env_f = vn.GraphVecEnv(world, n_total, seed=4, obs_layout=layout, host_outputs=False, device_world=env.dw,
                               scaled_float=True, **mk)
        env_f.reset()
        [env_f.step_enqueue(act(i), actions_ready=True) for i in range(300)]
        env_f.stats.zero_()
        f = H.steps_per_s(lambda i: env_f.step_enqueue(act(i), actions_ready=True), 200, n_total)
        fs = env_f.episode_stats()
        skip_f, reset_f = fs["rows_skipped"] / max(1.0, fs["steps"]), fs["resets"] / max(1.0, fs["steps"])
        bytes_f = N * 5 * ((1 - skip_f) * F_OBS + reset_f * F_GOAL)
        f.update({"algorithmic_bytes_per_step": bytes_f, "frac": bytes_f / (f["ms_per_step"] * 1e-3) / 1e9 / peak,
                  "note": "float32 CHW leaves (rgb, goal, depth) / 255 in persistent batches"})
        secondary["float_chw"] = f
        del env_f
        # one whole A2C / UNREAL data pass as the trainer sees it (thor_cached_auxiliary.py:30-42: num_steps = 20):
        # 20 vectorised steps that write their rollout rows themselves, then n-step returns, pixel-control rewards +
        # their back-up and reward-prediction labels, all on the device, straight from the time-major storage
        R = vn.rollout
        T_roll = 20
        rb = R.RolloutBuffer(env.dw, N, T_roll)
        v_last = torch.randn(N, device=dev)
        q_last = torch.rand(N, 400, device=dev)
        R.target_tables(env.dw, 4, (20, 20))                # per-world pixel-control table, built once

        def a2c_pass(i):
            rb.start(env)
            for t in range(T_roll):
                rb.step(env, act(i * T_roll + t), actions_ready=True)
            return rb.targets(v_last, 0.99, q_last, 0.9, 4, (20, 20), overlap=True)

        def steps_only(i):
            for t in range(T_roll):
                env.step_enqueue(act(i * T_roll + t), actions_ready=True)

        p = H.steps_per_s(a2c_pass, 10, n_total * T_roll, warm=5)
        s20 = H.steps_per_s(steps_only, 10, n_total * T_roll, warm=5)
        secondary["a2c_pass"] = {"value": p["value"], "unit": "env-steps/s", "ms_per_pass": p["ms_per_step"],
                                 "ms_20_steps_alone": s20["ms_per_step"], "blocks": p["blocks"], "num_steps": T_roll,
                                 "ratio_to_steps_alone": s20["ms_per_step"] / p["ms_per_step"],
                                 "note": "20 env steps (rollout rows written by the step kernel) + n-step returns + "
                                         "pixel-control rewards and back-up + RP labels, per pass; no torch kernels; "
                                         "returns / RP labels on a side stream next to the pixel-control chain"}

    # ---- e2e through the public VecEnv API: host actions in, host rewards/dones out, every step
    host_actions = actions[:512].cpu().numpy()
    hact = lambda i: host_actions[i % len(host_actions)]
    sync = lambda: torch.cuda.synchronize(dev)

    def e2e_of(env_x, n_steps, warm=30):
        env_x.reset()
        for i in range(warm):
            env_x.step(hact(i))
        H.barrier()
        dts = [e2e_loop(lambda i: env_x.step(hact(i)), n_steps, sync) for _ in range(3)]
        H.barrier()
        return H.max_over_ranks([float(np.median(dts))])[0], [n_total * n_steps / d for d in dts]

    env_e = vn.GraphVecEnv(world, n_total, seed=2, obs_layout=layout, host_outputs=True, device_world=env.dw, **mk)
    Ke = 2000 if N >= 1024 else 5000
    dt, per_rep = e2e_of(env_e, Ke)
    e2e = {"value": n_total * Ke / dt, "unit": "env-steps/s", "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": 20 * N,
           "steps": Ke, "repeats": 3, "this_rank_per_repeat": per_rep,
           "note": "VecEnv.step(numpy actions) -> (CUDA uint8 obs, numpy rewards, numpy dones, infos); "
                   "observations stay in HBM for the policy"}
    variants = {}
    if args.workload == "c2":
        # (a) the same call with the observation batch ALSO brought to the host as fresh numpy arrays every step - what
        # SubprocVecEnv semantics literally require for a CPU policy (PCIe-bound: 116 MB per step)
        env_n = vn.GraphVecEnv(world, n_total, seed=2, obs_layout=layout, host_outputs=True, device_world=env.dw,
                               numpy_obs=True, **mk)
        dtn, _ = e2e_of(env_n, 100, warm=5)
        variants["numpy_obs"] = {"value": n_total * 100 / dtn, "unit": "env-steps/s", "steps": 100,
                                 "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": N * (F_OBS + F_RGB) + 20 * N,
                                 "note": "obs leaves returned as numpy arrays (views of alternating pinned staging "
                                         "buffers), PCIe-bound"}
        del env_n
        # (b) the drop-in INTEGRATION.md documents: the reference's 5-tuple observation as float32 CHW in [0, 1]
        # (obs_layout='aux5', scaled_float=True), numpy actions in / numpy scalars out, observations in HBM
        world5 = make_world(vn, "aux5")
        dw5 = vn.DeviceWorld(world5, dev)
        env_a = vn.GraphVecEnv(world5, n_total, seed=2, obs_layout="aux5", host_outputs=True, device_world=dw5,
                               scaled_float=True, **mk)
        dta, _ = e2e_of(env_a, 500, warm=10)
        variants["aux5_scaled_float"] = {"value": n_total * 500 / dta, "unit": "env-steps/s", "steps": 500,
                                         "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": 20 * N,
                                         "bytes_written_per_changed_row": 4 * (F_RGB + F_DEPTH + F_SEG),
                                         "note": "INTEGRATION.md section 1 drop-in: ((rgb, goal, depth, seg, goal_seg) "
                                                 "float32 CHW / 255 CUDA, lar), numpy rewards / dones / infos"}
        env_u = vn.GraphVecEnv(world5, n_total, seed=2, obs_layout="aux5", host_outputs=True, device_world=dw5, **mk)
        dtu, _ = e2e_of(env_u, 1000, warm=10)
        variants["aux5_uint8"] = {"value": n_total * 1000 / dtu, "unit": "env-steps/s", "steps": 1000,
                                  "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": 20 * N,
                                  "note": "same 5-tuple kept as uint8 HWC (the /255 left to the first conv's loader)"}
        del env_a, env_u, dw5
        if world_size == 1:
            # (c) the reference's own run configuration (thor_cached_auxiliary.py:73-84 + :30-34): 4 envs, native 174 x 174
            # frames, 5-tuple, float32 CHW - the configuration its 106 fps log line was produced with
            sc = vn.scenes.make_thor_scene(300, (24, 30), seed=5, n_goals=4, frame_hw=(174, 174),
                                           planes=("rgb", "depth", "segmentation"))
            wn = vn.compile_world([sc], vn.GYM_GRAPH)
            env_4 = vn.GraphVecEnv(wn, 4, seed=2, obs_layout="aux5", host_outputs=True, scaled_float=True, device=dev,
                                   max_episode_steps=MAX_EPISODE_STEPS)
            env_4.set_complexity(0.01)
            a4 = np.random.RandomState(5).randint(0, 4, (512, 4)).astype(np.int32)
            env_4.reset()
            for i in range(50):
                env_4.step(a4[i % 512])
            dt4 = float(np.median([e2e_loop(lambda i: env_4.step(a4[i % 512]), 3000, sync) for _ in range(3)]))
            secondary["reference_run_config"] = {
                "value": 4 * 3000 / dt4, "unit": "env-steps/s", "us_per_vector_step": 1e6 * dt4 / 3000, "envs": 4,
                "note": "thor_cached_auxiliary.py default_args: 4 envs, 174x174 aux5 observation as float32 CHW, "
                        "hardness 0.01, through VecEnv.step(numpy); the reference logs ~106 env-steps/s for the whole "
                        "training loop at this configuration (outputs/output.txt)"}
            del env_4
    e2e["variants"] = variants

    cpu_baseline = None
    if rank == 0 and world_size == 1 and not args.no_cpu_baseline and args.workload == "c2":
        # bounded sample (10-30 s of CPU work): 32 envs x 8,000 vector steps cross the 900-step TimeLimit about nine
        # times per env, so the reference's per-reset candidate enumeration (~0.05 s each here) is included
        v, nres, cdt = cpu_run(32, 8000, 3, 1)
        cpu_baseline = {"value": v, "unit": "env-steps/s", "cores": 1, "kind": "port",
                        "sample": "32 envs x 8000 vector steps, one process, sequential + np.stack (DummyVecEnv "
                                  "equivalent), episode phases randomised, %.1f s, p_reset=%.5f"
                                  % (cdt, nres / (32 * 8000.0))}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s",
            "n_gpus": world_size, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": cfg, "run_stats": run_stats,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches * world_size, "roofline": roofline,
            "cpu_baseline": cpu_baseline, "secondary": secondary,
        }
        emit(line)
    if world_size > 1:
        dist.destroy_process_group()


def run_rollout(args):
    """BASELINE.json configs[4]: the A2C rollout builder - 128-step n-step returns + pixel-control rewards
    and their discounted back-up + reward-prediction labels / index lists (+ the 3 auxiliary targets), on a
    2^20 (env x step) batch, straight from state indices and the HBM store."""
    import torch
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    N, T = 8192, 128
    K = args.steps if args.steps else 20
    W = max(args.warmup if args.warmup is not None else 3, 3)
    scene = vn.scenes.make_thor_scene(N_CELLS, GRID, seed=SCENE_SEED, n_goals=4, planes=("rgb", "depth", "segmentation"))
    world = vn.compile_world([scene], vn.GYM_GRAPH)
    env = vn.GraphVecEnv(world, N, device=dev, seed=1, max_episode_steps=50, obs_layout="frame", host_outputs=False)
    env.set_complexity(0.05)
    env.reset()
    buf = vn.rollout.RolloutBuffer(env.dw, N, T)
    buf.start(env)
    gen = torch.Generator(device=dev).manual_seed(3)
    for _ in range(T):
        a = torch.randint(0, 4, (N,), device=dev, generator=gen, dtype=torch.int32)
        buf.step(env, a)
    v_last = torch.randn(N, device=dev, generator=gen)           # seeded like the actions: same inputs on every run
    q_last = torch.rand(N, 400, device=dev, generator=gen)

    def builder(with_aux):
        ret = buf.returns(v_last, 0.99)
        pcr = buf.pixel_control_returns(q_last, 0.9, 4, (20, 20))
        lab = buf.reward_prediction()
        aux = buf.auxiliary_targets(4, (20, 20)) if with_aux else None
        return ret, pcr, lab, aux

    last = {}

    def timed(fn, k):
        for _ in range(W):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(k):
            last["out"] = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / k

    ms_core = timed(lambda: builder(False), K)
    if args.dump_outputs:
        ret, pcr, (labels, zero, nonzero, counts), _ = last["out"]
        nz, nnz = (int(c) for c in counts.tolist())         # the position lists are valid up to their counts
        dump_outputs(args.dump_outputs, [("returns", ret), ("pixel_control_returns", pcr), ("rp_labels", labels),
                                         ("rp_zero_positions", zero[:nz]), ("rp_nonzero_positions", nonzero[:nnz])],
                     sampled=["pixel_control_returns"])
    ms_all = timed(lambda: builder(True), max(2, K // 4))
    ms_pc = timed(lambda: buf.pixel_control(4, (20, 20)), K)
    ms_ret = timed(lambda: buf.returns(v_last, 0.99), K)
    ms_rp = timed(lambda: buf.reward_prediction(), K)
    peak, peak_src = measured_peak()
    # table path: every transition reads one 1,600-byte table row and writes one 1,600-byte output row; the
    # ~2 % reset transitions read two 21,168-byte frames instead of the table row
    miss = float(buf.dones.float().mean())
    pc_bytes = N * T * (1600 + (1 - miss) * 1600 + miss * 2 * F_RGB)
    line = {
        "metric": "rollout-builder env-steps/s (n-step returns + pixel-control + back-up + RP)", "value": N * T / (ms_core * 1e-3),
        "unit": "env-steps/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms_core, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C5 A2C rollout builder: T=128, N=8,192 (2^20 env-steps), gamma .99, PC cell 4 -> 20x20, gamma_pc .9"},
        "run_stats": {"ms": {"returns": ms_ret, "pixel_control": ms_pc, "rp_labels_and_lists": ms_rp, "core_total": ms_core,
                             "with_aux_targets_total": ms_all}, "done_rate": miss},
        "roofline": {"bound": "hbm", "achieved": pc_bytes / (ms_pc * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": pc_bytes / (ms_pc * 1e-3) / 1e9 / peak, "traffic": None,
                     "kernel": "vn_transition_rows + vn_gather_rows + vn_pixel_control_list (table-driven pixel control)",
                     "kernel_ms": ms_pc, "algorithmic_bytes_per_launch": pc_bytes, "peak_source": peak_src},
        "gpu_launches": 7,
    }
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything else any library prints while the
    benchmark runs (NCCL's version banner, warnings) was diverted to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gather", default="auto", choices=["auto", "ldg", "bulk", "fused", "persistent"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--port-only", action="store_true", help="reference arm: time the oracle port even where "
                                                             "/root/reference exists")
    ap.add_argument("--cpu-budget", type=int, default=100_000, help="reference arm: env-steps per leg (bounded sample)")
    ap.add_argument("--cuda-graph", action="store_true", help="replay 64-step CUDA graphs in the device-resident loop")
    ap.add_argument("--quick", action="store_true", help="development: device-resident number + roofline only")
    ap.add_argument("--serial", action="store_true", help="development: steps without VN_STEP_ACTIONS_READY (as when a policy "
                                                          "kernel produces the actions between two steps: no overlap of the "
                                                          "scalar part with the previous gather)")
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5", "rgb", "aux5"],
                    help="BASELINE.json config; c2 is the headline, the others are secondary lines")
    ap.add_argument("--hardness", default="none", help="curriculum hardness (set_complexity); 'none' = uniform starts")
    ap.add_argument("--mix", type=int, default=1000, help="un-timed steps before warm-up")
    ap.add_argument("--envs-per-gpu", type=int, default=None, help="development: override the envs per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c5":
        run_rollout(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
