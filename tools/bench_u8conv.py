#!/usr/bin/env python
"""vn.nn.U8Conv2d against the float path it replaces (``F.conv2d(rollout.policy_input(...))``) on the C2 world.

Sizes: "act" = 4,096 frames of an env observation batch, forward only; "update" = 81,920 frames by state index from a
[4096, 20] strided view of time-major rollout states, forward + backward.  The float path runs twice, with cuDNN's TF32
at torch's default (True) and with it off.  Reports CUDA-event medians after warm-up, the peak of
torch.cuda.max_memory_allocated over forward + backward (above what was allocated before), the per-frame byte model and
its HBM share against bench.measured_peak(), and the tensor-core rate of the fused kernels.  Then one "step + first
layer" loop: the aux5 uint8 env + U8Conv2d on the rgb and goal leaves against scaled_float=True + nn.Conv2d.

Every row also runs under torch.autocast with bf16 and fp16 (keys "ac_bf16_*" / "ac_f16_*"): U8Conv2d's one-term 16-bit
kernels against torch's own float path under the same autocast, with grad_out in the autocast dtype.  Their issued
tensor-core work is a third of the fp32 kernels' (one mma per k-step instead of three); "useful" counts the
convolution's multiply-adds alone (forward, plus as many again for the weight gradient).

With --planes it runs the plane-set cases instead: vn.nn.U8PlanesConv2d for RGB-D ((3, 1): obs rgb + depth) and
observation + goal ((3, 3): obs rgb + goal rgb, the goals from a second [4096, 20] index view) at (k 7, stride 4,
cout 32), against the float path it replaces (policy_input per plane + torch.cat + nn.Conv2d), in fp32 (TF32 on and off
for the float path) and under autocast with bf16 and fp16, with the update pass's peak memory.

    python tools/bench_u8conv.py [--reps 20] [--planes] [--out record.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402

GEOMS = {"ref_3x32_k7s4": (3, 32, 7, 4), "example_3x16_k8s4": (3, 16, 8, 4)}
ENVS, STEPS = 4096, 20
AUTOCAST = {"bf16": torch.bfloat16, "f16": torch.float16}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2]


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


PLANE_CASES = {"rgbd_3+1_32_k7s4": ((3, 1), ("rgb", "depth")), "obs_goal_3+3_32_k7s4": ((3, 3), ("rgb", "goal_rgb"))}


def planes(vn, env, dw, states, goals, reps, gen):
    """The plane-set rows: {case: {key: value}}.  "goal_rgb" is the goal leaf for the act size and the rgb plane at
    the goal indices for the update size."""
    dev = states.device
    h, w = dw.world.layout.frame_hw
    out = {}
    for name, (pcs, leaves) in PLANE_CASES.items():
        torch.manual_seed(0)
        layer = vn.nn.U8PlanesConv2d(pcs, 32, 7, stride=4).to(dev)
        conv = torch.nn.Conv2d(sum(pcs), 32, 7, stride=4).to(dev)
        conv.load_state_dict(layer.state_dict())
        oh = (h - 7) // 4 + 1
        batch = [env.goal_buf["rgb"] if lf == "goal_rgb" else env.obs_buf[lf] for lf in leaves]
        act_idx = [(env.goal if lf == "goal_rgb" else env.obs_state, "rgb" if lf == "goal_rgb" else lf)
                   for lf in leaves]
        upd = [(goals if lf == "goal_rgb" else states, "rgb" if lf == "goal_rgb" else lf) for lf in leaves]
        go = torch.randn((ENVS, STEPS, 32, oh, oh), device=dev, generator=gen)
        res = {"plane_channels": list(pcs), "act_frames": ENVS, "update_frames": ENVS * STEPS,
               "float_frame_bytes": 4 * sum(pcs) * h * w}

        def float_x(src):
            return torch.cat([vn.rollout.policy_input(dw, s, p) for s, p in src], -3)

        for tag, dtype in [("", None)] + [("ac_%s_" % t, d) for t, d in AUTOCAST.items()]:
            ac = dict(device_type="cuda", dtype=dtype or torch.float16, enabled=dtype is not None)
            g = go if dtype is None else go.to(dtype)

            def fused_update():
                layer.zero_grad(set_to_none=True)
                with torch.autocast(**ac):
                    y = layer.forward_states(dw, *upd)
                y.backward(g)

            def float_update():
                conv.zero_grad(set_to_none=True)
                with torch.autocast(**ac):
                    y = conv(float_x(upd).flatten(0, 1))
                y.backward(g.flatten(0, 1))

            with torch.no_grad(), torch.autocast(**ac):
                res[tag + "act_fused_ms"] = timed(lambda: layer(*batch), reps)
            res[tag + "update_fused_fwd_bwd_ms"] = timed(fused_update, reps)
            res[tag + "update_fused_peak_bytes"] = peak_bytes(fused_update)
            for tf32 in ((True, False) if dtype is None else (True,)):
                torch.backends.cudnn.allow_tf32 = tf32
                key = tag + ("float_tf32_%s_" % tf32 if dtype is None else "float_")
                with torch.no_grad(), torch.autocast(**ac):
                    res[key + "act_ms"] = timed(lambda: conv(float_x(act_idx)), reps)
                res[key + "update_fwd_bwd_ms"] = timed(float_update, reps)
                res[key + "update_peak_bytes"] = peak_bytes(float_update)
            torch.backends.cudnn.allow_tf32 = True
            del g
        out[name] = res
        del go
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--loop-steps", type=int, default=200)
    ap.add_argument("--planes", action="store_true", help="run the plane-set cases (U8PlanesConv2d) only")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    dev = torch.device("cuda")
    peak_gbs, peak_src = bench.measured_peak()
    scene = vn.scenes.make_thor_scene(1500, (50, 60), n_goals=4, planes=("rgb", "depth", "segmentation"))
    world = vn.compile_world([scene], vn.GYM_GRAPH)
    env = vn.GraphVecEnv(world, ENVS, seed=0, obs_layout="aux5", host_outputs=False)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(0)
    for _ in range(8):
        env.step(torch.randint(0, 4, (ENVS,), dtype=torch.int32, device=dev, generator=gen))
    dw = env.dw
    storage = torch.randint(0, world.n_states, (STEPS + 1, ENVS), dtype=torch.int32, device=dev, generator=gen)
    states = storage[:-1].t()                                  # [4096, 20] strided view, read in place
    h, w = world.layout.frame_hw
    rec = dict(gpu=gpu_info(), hbm_peak_gbs=peak_gbs, hbm_peak_source=peak_src, results={})
    if args.planes:
        goals = torch.randint(0, world.n_states, (STEPS + 1, ENVS), dtype=torch.int32, device=dev, generator=gen)
        rec["gpu_fields"] = "name, power.limit, clocks.max.sm, clocks.sm"
        rec["results"] = planes(vn, env, dw, states, goals[:-1].t(), args.reps, gen)
        line = json.dumps(rec)
        print(line)
        if args.out:
            with open(args.out, "w") as f:
                f.write(json.dumps(rec, indent=1) + "\n")
        env.close()
        return
    frame_u8 = h * w * 3
    for name, (cin, cout, k, s) in GEOMS.items():
        torch.manual_seed(0)
        layer = vn.nn.U8Conv2d(cin, cout, k, stride=s).to(dev)
        conv = torch.nn.Conv2d(cin, cout, k, stride=s).to(dev)
        conv.load_state_dict(layer.state_dict())
        oh = (h - k) // s + 1
        P, K = oh * oh, cin * k * k
        out_b = cout * P * 4
        mma_flop = 2 * 3 * ((P + 31) // 32 * 32) * ((K + 15) // 16 * 16) * cout    # issued per frame, forward
        wg_flop = 2 * 3 * ((cout + 15) // 16 * 16) * ((K + 1 + 7) // 8 * 8) * ((P + 15) // 16 * 16)
        useful = 2 * P * K * cout
        res = {}
        n = ENVS
        obs = env.obs_buf["rgb"]
        with torch.no_grad():
            t = timed(lambda: layer(obs), args.reps)
            res["act_fused_ms"] = t
            res["act_fused_bytes_per_frame"] = frame_u8 + out_b
            res["act_fused_hbm_share"] = n * (frame_u8 + out_b) / (t * 1e-3) / (peak_gbs * 1e9)
            res["act_fused_tensor_tflops_issued"] = n * mma_flop / (t * 1e-3) / 1e12
            res["act_useful_tflops"] = n * useful / (t * 1e-3) / 1e12
            for tf32 in (True, False):
                torch.backends.cudnn.allow_tf32 = tf32
                res["act_float_tf32_%s_ms" % tf32] = timed(lambda: conv(vn.rollout.policy_input(dw, env.obs_state)),
                                                          args.reps)
            torch.backends.cudnn.allow_tf32 = True
        res["act_float_bytes_per_frame"] = frame_u8 + 4 * frame_u8 + 4 * frame_u8 + out_b
        n = ENVS * STEPS
        go = torch.randn((ENVS, STEPS, cout, oh, oh), device=dev, generator=gen)

        def fused_update():
            layer.zero_grad(set_to_none=True)
            layer.forward_states(dw, states).backward(go)

        def float_update():
            conv.zero_grad(set_to_none=True)
            x = vn.rollout.policy_input(dw, states).flatten(0, 1)
            conv(x).backward(go.flatten(0, 1))

        with torch.no_grad():
            res["update_fused_fwd_ms"] = timed(lambda: layer.forward_states(dw, states), args.reps)
        t = timed(fused_update, args.reps)
        res["update_fused_fwd_bwd_ms"] = t
        res["update_fused_peak_bytes"] = peak_bytes(fused_update)
        moved = n * (2 * frame_u8 + 2 * out_b)
        res["update_fused_bytes"] = moved
        res["update_fused_hbm_share"] = moved / (t * 1e-3) / (peak_gbs * 1e9)
        res["update_fused_tensor_tflops_issued"] = n * (mma_flop + wg_flop) / (t * 1e-3) / 1e12
        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            res["update_float_tf32_%s_fwd_bwd_ms" % tf32] = timed(float_update, args.reps)
            res["update_float_tf32_%s_peak_bytes" % tf32] = peak_bytes(float_update)
        torch.backends.cudnn.allow_tf32 = True
        res["update_float_bytes_min"] = n * (frame_u8 + 4 * frame_u8 + 2 * 4 * frame_u8 + 2 * out_b)
        for tag, dtype in AUTOCAST.items():
            ac = "ac_%s_" % tag
            go_lp = go.to(dtype)

            def lp_update():
                layer.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=dtype):
                    y = layer.forward_states(dw, states)
                y.backward(go_lp)

            def lp_float_update():
                conv.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=dtype):
                    y = conv(vn.rollout.policy_input(dw, states).flatten(0, 1))
                y.backward(go_lp.flatten(0, 1))

            with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
                t = timed(lambda: layer(obs), args.reps)
                res[ac + "act_fused_ms"] = t
                res[ac + "act_fused_tensor_tflops_issued"] = ENVS * mma_flop / 3 / (t * 1e-3) / 1e12
                res[ac + "act_useful_tflops"] = ENVS * useful / (t * 1e-3) / 1e12
                res[ac + "act_float_ms"] = timed(lambda: conv(vn.rollout.policy_input(dw, env.obs_state)), args.reps)
                res[ac + "update_fused_fwd_ms"] = timed(lambda: layer.forward_states(dw, states), args.reps)
            t = timed(lp_update, args.reps)
            res[ac + "update_fused_fwd_bwd_ms"] = t
            res[ac + "update_fused_peak_bytes"] = peak_bytes(lp_update)
            res[ac + "update_fused_tensor_tflops_issued"] = n * (mma_flop + wg_flop) / 3 / (t * 1e-3) / 1e12
            res[ac + "update_useful_tflops"] = n * 2 * useful / (t * 1e-3) / 1e12
            res[ac + "update_float_fwd_bwd_ms"] = timed(lp_float_update, args.reps)
            res[ac + "update_float_peak_bytes"] = peak_bytes(lp_float_update)
            del go_lp
        rec["results"][name] = res
        del go

    # step + first layer: aux5 uint8 + U8Conv2d on rgb and goal rgb, against scaled_float=True + nn.Conv2d
    torch.manual_seed(0)
    layer = vn.nn.U8Conv2d(3, 32, 7, stride=4).to(dev)
    conv = torch.nn.Conv2d(3, 32, 7, stride=4).to(dev)
    conv.load_state_dict(layer.state_dict())
    fenv = vn.GraphVecEnv(world, ENVS, seed=0, obs_layout="aux5", host_outputs=False, scaled_float=True,
                          device_world=dw)
    fenv.reset()
    acts = torch.randint(0, 4, (args.loop_steps, ENVS), dtype=torch.int32, device=dev, generator=gen)
    loop = {}
    with torch.no_grad():
        def u8_loop():
            for i in range(args.loop_steps):
                env.step(acts[i])
                layer(env.obs_buf["rgb"])
                layer(env.goal_buf["rgb"])

        def float_loop():
            for i in range(args.loop_steps):
                fenv.step(acts[i])
                conv(fenv.float_buf["rgb"])
                conv(fenv.float_buf["goal_rgb"])

        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            ms = timed(float_loop, 3, warmup=1)
            loop["float_tf32_%s_env_steps_per_s" % tf32] = ENVS * args.loop_steps / (ms * 1e-3)
        torch.backends.cudnn.allow_tf32 = True
        ms = timed(u8_loop, 3, warmup=1)
        loop["u8_env_steps_per_s"] = ENVS * args.loop_steps / (ms * 1e-3)
        for tag, dtype in AUTOCAST.items():
            with torch.autocast("cuda", dtype=dtype):
                ms = timed(float_loop, 3, warmup=1)
                loop["ac_%s_float_env_steps_per_s" % tag] = ENVS * args.loop_steps / (ms * 1e-3)
                ms = timed(u8_loop, 3, warmup=1)
                loop["ac_%s_u8_env_steps_per_s" % tag] = ENVS * args.loop_steps / (ms * 1e-3)
    rec["step_plus_first_layer"] = loop
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")
    env.close()
    fenv.close()


if __name__ == "__main__":
    main()
