#!/usr/bin/env python
"""Cost of the geodesic-progress reward (GraphVecEnv(reward_progress=...)) on the env step at BASELINE.json configs[1]
(C2: 1,500 positions x 4 rotations, 84x84 RGB + depth + goal, 4,096 envs): device-resident steps with the rule off and
on, pipelined (VN_STEP_ACTIONS_READY, bench.py's loop) and serial (the actions produced just before each step).

Both envs share one DeviceWorld, so they read the same store and the off env's world holds the distance table as well;
the rule alone differs.  The two are timed in alternation, `--rounds` times each, each round `--steps` steps between
CUDA events after `--warmup` untimed steps; the record keeps every round and the medians.  The outputs of the two envs
are also compared: same states and dones, and rewards that differ only where the distance changed.
Usage: python tools/bench_reward_progress.py [--out FILE] [--rounds 7] [--steps 400] [--warmup 200] [--coef 0.01]"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def gpu_line():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # the numbers stay valid, the clock line is then missing from the record
        return "nvidia-smi unavailable: %s" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--coef", type=float, default=0.01)
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_reward_progress needs a CUDA device")
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    desc, world, n, layout = bench.make_workload(vn, "c2")
    kw = dict(device="cuda:0", seed=1, max_episode_steps=bench.MAX_EPISODE_STEPS, obs_layout=layout, host_outputs=False)
    off = vn.GraphVecEnv(world, n, **kw)
    on = vn.GraphVecEnv(world, n, reward_progress=args.coef, device_world=off.dw, **kw)
    envs = {"off": off, "on": on}
    gen = torch.Generator(device="cuda").manual_seed(1)
    acts = torch.randint(0, 4, (2048, n), device="cuda", generator=gen, dtype=torch.int32)

    # outputs: the rule changes rewards only, and only by coef * (distance change)
    for e in envs.values():
        e.reset()
    _, dist = off.dw.shortest_paths()
    for i in range(200):
        _, d0 = on.optimal_actions()
        task = on.task.clone()
        for e in envs.values():
            e.step_enqueue(acts[i])
        assert torch.equal(on.state, off.state) and torch.equal(on.done, off.done)
        d1 = dist[task.long(), on.info_state.long()]
        delta = torch.where((d0 < 0) | (d1 < 0), torch.zeros_like(d0), d0 - d1).float()
        assert torch.equal(on.reward, off.reward + torch.tensor(args.coef, device="cuda") * delta), i

    def timed(env, serial):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(args.warmup):
            env.step_enqueue(acts[i % 2048], actions_ready=not serial)
        e0.record()
        for i in range(args.steps):
            env.step_enqueue(acts[(args.warmup + i) % 2048], actions_ready=not serial)
        e1.record()
        torch.cuda.synchronize()
        return 1e3 * e0.elapsed_time(e1) / args.steps

    rec = {"gpu_before": gpu_line(), "workload": desc, "envs": n, "coef": args.coef, "rounds": args.rounds,
           "steps_per_round": args.steps, "warmup_per_round": args.warmup,
           "table_bytes": int(dist.numel() * dist.element_size()), "us_per_step": {}}
    for mode in ("pipelined", "serial"):
        serial = mode == "serial"
        per = {"off": [], "on": []}
        for e in envs.values():
            e.reset()
        for _ in range(args.rounds):
            for name, e in envs.items():
                per[name].append(timed(e, serial))
        rec["us_per_step"][mode] = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "rounds": v}
                                    for k, v in per.items()}
        rec["us_per_step"][mode]["mode_of_last_step"] = int(on._prev_mode)
        m = rec["us_per_step"][mode]
        m["on_minus_off_us"] = m["on"]["median"] - m["off"]["median"]
        m["on_over_off"] = m["on"]["median"] / m["off"]["median"]
    rec["gpu_after"] = gpu_line()
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
