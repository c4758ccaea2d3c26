#!/usr/bin/env python
"""Cost and throughput of the fixed episode list (GraphVecEnv.set_episodes, evaluation.evaluate_episodes) at
BASELINE.json configs[1] (C2: 1,500 positions x 4 rotations, 84x84 RGB + depth + goal, 4,096 envs).  One call records:

  * the card (name, power limit, clocks before and after);
  * `bench.py --gpus 1 --quick` `value` for this tree and, with `--parent DIR` (a checkout of the parent commit, built
    here first with its own __graft_entry__.py), for the parent, alternated `--bench-rounds` times;
  * the C2 device-resident step with no list and with a list installed (every reachable candidate start of C2's
    tasks, dealt over the 4,096 envs), pipelined (VN_STEP_ACTIONS_READY, bench.py's loop) and serial, the two envs
    alternated `--rounds` times, each round `--steps` steps between CUDA events after `--warmup` untimed steps; medians;
  * evaluate_episodes over the same list with the shortest-path policy (optimal_actions()): episodes per second (host
    clock around the whole call, which ends reading the results), steps, and SPL, which must be exactly 1.
Usage: python tools/bench_episode_list.py [--out FILE] [--parent DIR] [--rounds 7] [--steps 400] [--warmup 200]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

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


def bench_value(tree):
    """`value` of `bench.py --gpus 1 --quick` run from `tree` (its last JSON line)."""
    res = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--quick"], cwd=tree, capture_output=True,
                         text=True, timeout=1800)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    if res.returncode != 0 or not lines:
        raise RuntimeError("bench.py in %s failed (%d): %s" % (tree, res.returncode, res.stderr[-2000:]))
    return json.loads(lines[-1])["value"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--parent", default=None, help="checkout of the parent commit to compare bench.py against")
    ap.add_argument("--bench-rounds", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=200)
    args = ap.parse_args()
    rec = {"gpu_before": gpu_line()}

    # bench.py of this tree against the parent, alternated, before this process touches the device
    if args.parent:
        subprocess.run([sys.executable, "__graft_entry__.py"], cwd=args.parent, check=True, capture_output=True)
    trees = {"this": ROOT}
    if args.parent:
        trees["parent"] = os.path.abspath(args.parent)
    rec["bench_value"] = {k: [] for k in trees}
    for _ in range(args.bench_rounds):
        for k, tree in trees.items():
            rec["bench_value"][k].append(bench_value(tree))
    rec["bench_command"] = "bench.py --gpus 1 --quick"

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_episode_list needs a CUDA device")
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    EV = vn.evaluation
    desc, world, n, layout = bench.make_workload(vn, "c2")
    task, start = EV.episode_set(world, None, seed=0)
    kw = dict(device="cuda:0", seed=1, max_episode_steps=bench.MAX_EPISODE_STEPS, obs_layout=layout, host_outputs=False)
    absent = vn.GraphVecEnv(world, n, **kw)
    listed = vn.GraphVecEnv(world, n, device_world=absent.dw, **kw)
    envs = {"absent": absent, "installed": listed}
    gen = torch.Generator(device="cuda").manual_seed(1)
    acts = torch.randint(0, 4, (2048, n), device="cuda", generator=gen, dtype=torch.int32)

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

    rec.update({"workload": desc, "envs": n, "episodes_listed": int(len(task)), "rounds": args.rounds,
                "steps_per_round": args.steps, "warmup_per_round": args.warmup, "us_per_step": {}})
    for mode in ("pipelined", "serial"):
        serial = mode == "serial"
        per = {"absent": [], "installed": []}
        listed.set_episodes(task, start)
        for e in envs.values():
            e.reset()
        for _ in range(args.rounds):
            for name, e in envs.items():
                per[name].append(timed(e, serial))
        rec["us_per_step"][mode] = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "rounds": v}
                                    for k, v in per.items()}
        m = rec["us_per_step"][mode]
        m["installed_minus_absent_us"] = m["installed"]["median"] - m["absent"]["median"]
        m["installed_over_absent"] = m["installed"]["median"] / m["absent"]["median"]
        m["episodes_recorded_while_timed"] = listed.episodes_recorded
        listed.set_episodes(None)

    # evaluation throughput: every reachable candidate start of C2's tasks, shortest-path policy
    ev = vn.GraphVecEnv(world, n, device_world=absent.dw, **kw)
    policy = lambda obs: ev.optimal_actions()[0]
    EV.evaluate_episodes(ev, policy, task[:n], start[:n])            # warm-up: first launches, the policy's kernels
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = EV.evaluate_episodes(ev, policy, task, start)
    dt = time.perf_counter() - t0
    p = res.pop("per_episode")
    rec["evaluation"] = dict(res, seconds=dt, episodes_per_s=res["episodes"] / dt, env_steps=res["steps"] * n,
                             spl_is_one=bool(res["spl"] == 1.0 and (p["spl"] == 1.0).all()),
                             length_is_distance=bool((p["length"] == p["distance"]).all()))
    if not rec["evaluation"]["spl_is_one"]:
        raise SystemExit("shortest-path policy did not score SPL == 1: %s" % json.dumps(rec["evaluation"]))
    rec["gpu_after"] = gpu_line()
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
