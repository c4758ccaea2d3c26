"""GPU tests of the geodesic-progress reward (GraphVecEnv(reward_progress=...), vn_rules_t.reward_progress) in every
launch mode: off it changes nothing, on it matches the oracle restatement of tests/progress_reward.py bit for bit, agrees
with the optimal_actions() distances, and reaches every output that carries a reward."""
import importlib
import math

import numpy as np
import pytest

import helpers as H
import progress_reward as P
from oracle import envs as oenvs
from oracle import graph_util as gu
from oracle import vec as ovec

pytestmark = pytest.mark.gpu

vn = importlib.import_module("a2cat-vn-pytorch_b200")
T = vn.tables
R = vn.rollout

MODES = ("ldg", "bulk", "fused", "persistent", "auto")


def f32bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def _host(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


# --------------------------------------------------------------------------- coefficient 0 changes nothing
@pytest.mark.parametrize("host_outputs", [True, False])
@pytest.mark.parametrize("gather", MODES)
def test_coefficient_zero_is_bit_identical(gather, host_outputs):
    """An env built without the keyword, one built with reward_progress=0.0 and one switched from 0.5 back to 0 (whose
    world now holds the distance table) give the same rewards, dones, last_action_reward, ep_return, statistics,
    episode infos and rollout rows, -0.0 rewards of the thor-cached rules included."""
    import torch
    for fam, scene in ((T.GYM_GRAPH, H.scenes.make_maze_scene((10, 10), 0.25, 4, n_goals=2, planes=("rgb",))),
                       (T.THOR_CACHED, H.scenes.make_maze_scene((8, 9), 0.2, 5, n_goals=1, planes=("rgb",)))):
        tasks = [(0, g) for g in scene.goals] if fam is T.GYM_GRAPH else [(0, 5), (0, 17)]
        world = T.compile_world([scene], fam, tasks=tasks)
        N = 37
        kw = dict(seed=3, max_episode_steps=9, gather=gather, host_outputs=host_outputs,
                  env_tasks=np.tile(np.array([[0, 2]], np.int32), (N, 1)), obs_layout="frame")
        envs = [vn.GraphVecEnv(world, N, **kw)]
        envs.append(vn.GraphVecEnv(world, N, reward_progress=0.0, device_world=envs[0].dw, **kw))
        envs.append(vn.GraphVecEnv(world, N, reward_progress=0.5, device_world=envs[0].dw, **kw))
        envs[2].set_reward_progress(0)
        assert envs[0].dw.tables.task_dist                     # the table exists and is simply not read
        rng = np.random.RandomState(0)
        for e in envs:
            e.reset()
        zero_sign = 0
        for t in range(60):
            a = rng.randint(0, 4, N).astype(np.int32)
            outs = [e.step(a) for e in envs]
            (_, lar0), r0, d0, i0 = outs[0]
            zero_sign += int(np.signbit(_host(r0)[_host(r0) == 0]).sum())
            for (_, lar), r, d, infos in outs[1:]:
                assert np.array_equal(f32bits(_host(r)), f32bits(_host(r0))), t
                assert np.array_equal(_host(d), _host(d0)) and torch.equal(lar, lar0), t
                assert [infos[i].get("episode") for i in range(N)] == [i0[i].get("episode") for i in range(N)], t
            for e in envs[1:]:
                assert torch.equal(e.ep_return.view(torch.int32), envs[0].ep_return.view(torch.int32))
                assert torch.equal(e.state, envs[0].state) and torch.equal(e.stats, envs[0].stats)
        assert (zero_sign > 0) == (fam is T.THOR_CACHED)
        # rollout rows written by the step kernel
        bufs = [R.RolloutBuffer(e.dw, N, 12) for e in envs]
        acts = torch.randint(0, 4, (12, N), device="cuda", dtype=torch.int32)
        for e, b in zip(envs, bufs):
            b.start(e)
            for t in range(12):
                b.step(e, acts[t], actions_ready=t > 0)
        torch.cuda.synchronize()
        for b in bufs[1:]:
            for k in ("rewards", "dones", "states", "goals", "actions"):
                x, y = getattr(b, k), getattr(bufs[0], k)
                assert torch.equal(x.view(torch.int8) if x.dtype == torch.float32 else x,
                                   y.view(torch.int8) if y.dtype == torch.float32 else y), k


# --------------------------------------------------------------------------- against the oracle restatement
def _case(kind, N, seed):
    """(world, env kwargs, inject (task, start), oracle env factory, action low) of one oracle-parity case.  Injected
    resets draw the task and any state of its scene but the goal - unreachable ones included where the maze has them;
    thor-cached starts come from the task's candidates (cached.py:41-44 asserts them)."""
    rng = np.random.RandomState(seed)
    Rn = 260
    if kind == "oriented":       # one scene, three tasks, collisions, rotations
        scene = H.scenes.make_maze_scene((9, 11), 0.3, 21, n_goals=3, planes=("rgb",))
        scs, fam = [scene], T.GYM_GRAPH
    elif kind == "multi_scene":  # MultipleGraphEnv: two un-oriented scenes, no-op actions
        scs = [H.scenes.make_maze_scene((8, 8), 0.3, 30 + k, n_goals=1, oriented=False, planes=("rgb",), scene_id=k)
               for k in range(2)]
        fam = T.SIMPLE_GRAPH
    else:                        # thor_cached: h5 action order, -0.0 step reward, collision overrides the goal reward
        scene = H.scenes.make_maze_scene((8, 9), 0.25, 40, n_goals=1, planes=("rgb",))
        scs, fam = [scene], T.THOR_CACHED
    if kind == "thor_cached":
        world = T.compile_world(scs, fam, tasks=[(0, 3), (0, 29), (0, 50)])
    else:
        world = T.compile_world(scs, fam)
    nt = len(world.tasks)
    task = rng.randint(0, nt, (N, Rn)).astype(np.int32)
    start = np.zeros((N, Rn), np.int32)
    for i in range(N):
        for k in range(Rn):
            t = world.tasks[task[i, k]]
            b = int(world.scene_base[t.scene])
            if kind == "thor_cached":
                start[i, k] = b + int(rng.choice(t.cand_state))
            else:
                s = int(rng.randint(scs[t.scene].n_states - 1))
                start[i, k] = b + (s if s < t.goal_state else s + 1)
    local = lambda i: [int(s - world.scene_base[world.scene_of_state(s)]) for s in start[i]]

    if kind == "oriented":
        osc = oenvs.OracleScene(scene)
        graph = P.oriented_graph(scene.maze)

        def make(i, coef):
            e = oenvs.GymGraphEnv(osc, goals=list(scene.goals), rewards=rewards)
            e.reset_source = H.StreamSource(task[i], np.array([scene.state_tuple(s) for s in local(i)]), Rn)
            return P.ProgressReward(e, coef, graph)
        rewards, layout, lo = (1.0, -0.01, -0.1), "frame", 0
    elif kind == "multi_scene":
        oscs = [oenvs.OracleScene(s) for s in scs]
        graphs = [P.compass_graph(s.maze) for s in scs]

        def make(i, coef):
            e = oenvs.MultipleGraphEnv(oscs, rewards=rewards)
            e.reset_source = H.StreamSource(task[i], np.array([scs[world.tasks[tk].scene].state_tuple(s)
                                                                for tk, s in zip(task[i], local(i))]), Rn)
            return P.ProgressReward(e, coef, graphs, scene_of=lambda e: e.graph_number)
        rewards, layout, lo = (1.0, -0.01, -0.1), "frame", -1
    else:
        dist, _ = gu.compute_shortest_path_data(scene.maze)
        _, h5graph, spd = gu.h5_tables(scene.maze, dist)
        goals = [int(t.goal_state) for t in world.tasks]
        graph = (list(range(scene.n_states)), lambda s: [int(n) for n in h5graph[s] if n != -1])

        def make(i, coef):
            e = oenvs.ThorCachedEnv(h5graph, np.zeros((scene.n_states, 1), np.uint8), spd, tasks=goals)
            e.reset_source = H.StreamSource(task[i], start[i], Rn)
            return P.ProgressReward(e, coef, graph, goal_of=lambda e: e._current_goal_idx,
                                    state_of=lambda e: e._current_state_idx)
        rewards, layout, lo = (1.0, 0.0, 0.0), "pair", 0
    kw = dict(max_episode_steps=11, rewards=rewards, obs_layout=layout, inject=(task, start),
              env_tasks=np.tile(np.array([[0, nt]], np.int32), (N, 1)))
    return world, kw, make, lo


@pytest.mark.parametrize("coef", [0.25, 0.01, -0.3])
@pytest.mark.parametrize("kind", ["oriented", "multi_scene", "thor_cached"])
def test_matches_the_oracle_bit_for_bit(kind, coef):
    """200 steps with injected resets in every launch mode, from the host path (numpy actions, host_outputs) and the
    device path (CUDA actions, pipelined from the second step): rewards, last_action_reward, dones, states, episode
    infos and ep_return equal the oracle restatement's bits; a non-dyadic coefficient (0.01) included."""
    import torch
    N, steps = 40, 200
    world, kw, make, lo = _case(kind, N, seed=int(coef * 1000) & 0xFFFF)
    oes = [ovec.RewardCollector(ovec.TimeLimit(make(i, coef), kw["max_episode_steps"])) for i in range(N)]
    ov = ovec.VecEnv(oes)
    rng = np.random.RandomState(7)
    acts = rng.randint(lo, 4, (steps, N)).astype(np.int32)
    ov.reset()
    want = []
    for t in range(steps):
        (_, olar), orew, odone, oinfos = ov.step(acts[t])
        want.append((f32bits(orew), olar.view(np.uint32).copy(), odone.copy(),
                     [oinfos[i].get("episode") for i in range(N)],
                     np.array([np.float32(oe.ret) for oe in oes], np.float32).view(np.uint32)))
    assert sum(w[2].sum() for w in want) > 50
    dev_acts = torch.from_numpy(acts).cuda()
    dw = None
    for gather in MODES:
        for host in (True, False):
            env = vn.GraphVecEnv(world, N, seed=1, gather=gather, host_outputs=host, reward_progress=coef,
                                 device_world=dw, **kw)
            dw = env.dw
            env.reset()
            for t in range(steps):
                if host:
                    (_, lar), rew, done, infos = env.step(acts[t])
                else:
                    env.step_enqueue(dev_acts[t], actions_ready=t > 0)
                    lar, rew, done = env.lar, env.reward, env.done.bool()
                    infos = vn.vec_env.LazyInfos(env, lambda: env._unpack(env._pack.cpu().numpy()), None)
                w = want[t]
                assert np.array_equal(f32bits(_host(rew)), w[0]), (gather, host, t)
                assert np.array_equal(f32bits(_host(lar)), w[1]), (gather, host, t)
                assert np.array_equal(_host(done), w[2]), (gather, host, t)
                assert [infos[i].get("episode") for i in range(N)] == w[3], (gather, host, t)
                assert np.array_equal(env.ep_return.cpu().numpy().view(np.uint32), w[4]), (gather, host, t)
            st = env.episode_stats()
            eps = [e for w in want for e in w[3] if e is not None]
            assert st["episodes"] == len(eps)
            # the statistics add episode returns per warp in float32 before the double atomics: not an exact sum
            assert math.isclose(st["return_sum"], sum(e["r"] for e in eps), rel_tol=1e-5)


# --------------------------------------------------------------------------- the hand-worked scenarios on the device
@pytest.mark.parametrize("gather", MODES)
def test_hand_worked_scenarios_in_every_launch_mode(gather):
    """The scenarios of tests/progress_reward.py (toward / away, collision, no-op, goal with auto-reset, truncation,
    unreachable start), each copied into 150 envs so the scalar kernel runs more than one block."""
    import torch
    N = 150
    for kind, scs, maze, goal, fam in (("oriented", P.ORIENTED_SCENARIOS, P.ORIENTED_MAZE, P.ORIENTED_GOAL, T.GYM_GRAPH),
                                       ("compass", P.COMPASS_SCENARIOS, P.COMPASS_MAZE, P.COMPASS_GOAL, T.SIMPLE_GRAPH)):
        scene = H.scenes.GridScene(maze, [goal], fam.oriented, (84, 84), ("rgb",))
        world = T.compile_world([scene], fam)
        for k, (limit, starts, actions, want_r, want_d) in enumerate(scs):
            start = np.tile(np.array([[scene.state_index(s) for s in starts]], np.int32), (N, 1))
            env = vn.GraphVecEnv(world, N, seed=0, max_episode_steps=limit, rewards=P.REWARDS, gather=gather,
                                 obs_layout="frame", inject=(np.zeros_like(start), start), reward_progress=P.COEF)
            env.reset()
            rets = []
            for t, a in enumerate(actions):
                (_, lar), r, d, infos = env.step(np.full(N, a, np.int32))
                assert (f32bits(r) == f32bits(want_r[t])).all(), (kind, k, t, r[0], want_r[t])
                assert (d == bool(want_d[t])).all(), (kind, k, t)
                assert bool((lar[:, -1] == (0.0 if want_d[t] else min(max(want_r[t], -1.0), 1.0))).all()), (kind, k, t)
                if want_d[t]:
                    assert all(infos[i]["episode"]["r"] == infos[0]["episode"]["r"] for i in range(N))
                    rets.append(infos[0]["episode"]["r"])
            assert rets == P.EPISODE_RETURNS[(kind, k)]
            assert torch.equal(env.stats[1:2].view(torch.float64),
                               torch.tensor([N * sum(rets)], dtype=torch.float64, device="cuda"))


# --------------------------------------------------------------------------- ties to the tables users see
def test_shaped_reward_is_base_plus_coef_times_the_optimal_actions_distance_change():
    """reward(coef) == reward(0) + coef * (d_before - d_after), the distances read from optimal_actions() / the shared
    table in torch: before the step, and for the state the action led to (info_state) under the task the step ran."""
    import torch
    scene = H.scenes.make_maze_scene((12, 12), 0.25, 8, n_goals=3, planes=("rgb",))
    world = T.compile_world([scene], T.GYM_GRAPH)
    N, coef = 700, 0.01
    kw = dict(seed=5, max_episode_steps=25, host_outputs=False, obs_layout="frame",
              env_tasks=np.tile(np.array([[0, 3]], np.int32), (N, 1)))
    base = vn.GraphVecEnv(world, N, **kw)
    env = vn.GraphVecEnv(world, N, reward_progress=coef, device_world=base.dw, **kw)
    base.reset()
    env.reset()
    _, dist = env.dw.shortest_paths()
    c = torch.tensor(coef, dtype=torch.float32, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(1)
    moved = 0
    for t in range(150):
        a = torch.randint(0, 4, (N,), device="cuda", generator=gen, dtype=torch.int32)
        _, d_prev = env.optimal_actions()
        task = env.task.clone()
        base.step(a)
        env.step(a)
        d_next = dist[task.long(), env.info_state.long()]
        delta = torch.where((d_prev < 0) | (d_next < 0), torch.zeros_like(d_prev), d_prev - d_next).float()
        term = c * delta
        assert torch.equal(env.reward.view(torch.int32), (base.reward + term).view(torch.int32)), t
        assert torch.equal(env.done, base.done) and torch.equal(env.state, base.state)
        moved += int((delta != 0).sum())
    assert moved > N * 30


def test_sharding_is_invisible():
    """Two shards of 24 envs give the rewards, ep_return and last_action_reward of one 48-env process."""
    import torch
    scene = H.scenes.make_maze_scene((10, 10), 0.25, 0, n_goals=2, planes=("rgb",))
    world = T.compile_world([scene], T.GYM_GRAPH)
    kw = dict(seed=11, max_episode_steps=15, reward_progress=0.01, obs_layout="frame")
    whole = vn.GraphVecEnv(world, 48, **kw)
    parts = [vn.GraphVecEnv(world, 48, rank=r, world_size=2, device_world=whole.dw, **kw) for r in range(2)]
    whole.reset()
    [p.reset() for p in parts]
    rng = np.random.RandomState(1)
    for _ in range(60):
        a = rng.randint(0, 4, 48)
        (_, lar), r, d, _ = whole.step(a)
        outs = [p.step(a[p.env_lo:p.env_lo + p.num_envs]) for p in parts]
        assert np.array_equal(f32bits(r), f32bits(np.concatenate([o[1] for o in outs])))
        assert np.array_equal(d, np.concatenate([o[2] for o in outs]))
        assert torch.equal(lar, torch.cat([o[0][1] for o in outs]))
        assert torch.equal(whole.ep_return, torch.cat([p.ep_return for p in parts]))


def test_rollout_rows_returns_replay_and_cuda_graphs_carry_the_shaped_reward():
    """RolloutBuffer rows written by the step kernel, its n-step returns and a replay ring hold the shaped reward; a
    CUDA graph of the steps (capture_steps) replays the eager steps bit for bit."""
    import torch
    scene = H.scenes.make_maze_scene((10, 10), 0.25, 2, n_goals=2, planes=("rgb",))
    world = T.compile_world([scene], T.GYM_GRAPH)
    N, S, coef = 64, 16, 0.01
    kw = dict(seed=6, max_episode_steps=7, host_outputs=False, obs_layout="frame", reward_progress=coef)
    eager = vn.GraphVecEnv(world, N, **kw)
    rolled = vn.GraphVecEnv(world, N, device_world=eager.dw, **kw)
    base = vn.GraphVecEnv(world, N, device_world=eager.dw, **dict(kw, reward_progress=0.0))
    graphed = vn.GraphVecEnv(world, N, device_world=eager.dw, **kw)
    for e in (eager, rolled, base, graphed):
        e.reset()
    acts = torch.randint(0, 4, (S, N), device="cuda", dtype=torch.int32)
    buf = R.RolloutBuffer(rolled.dw, N, S)
    buf.start(rolled)
    ring = R.ReplayRing(eager.dw, N, capacity=S)
    ring.start(eager)
    g_rew = torch.zeros(S, N, device="cuda")
    g_done = torch.zeros(S, N, dtype=torch.uint8, device="cuda")
    rewards, base_rewards = [], []
    for t in range(S):
        eager.step_enqueue(acts[t])
        ring.insert(eager, acts[t])
        rewards.append(eager.reward.clone())
        base.step_enqueue(acts[t])
        base_rewards.append(base.reward.clone())
        buf.step(rolled, acts[t], actions_ready=t > 0)
    rewards = torch.stack(rewards)
    assert torch.equal(buf.rewards, rewards) and torch.equal(ring.reward, rewards)
    assert not torch.equal(rewards, torch.stack(base_rewards))
    last = torch.randn(N, device="cuda")
    assert torch.equal(buf.returns(last, 0.99), R.nstep_returns(rewards.t(), buf.dones.t(), last, 0.99))

    def record(t):
        g_rew[t].copy_(graphed.reward)
        g_done[t].copy_(graphed.done)

    cap = graphed.capture_steps(acts, after_step=record)
    cap.replay()
    torch.cuda.synchronize()
    assert torch.equal(g_rew, rewards) and torch.equal(g_done, buf.dones)
    assert torch.equal(graphed.ep_return, eager.ep_return) and torch.equal(graphed.lar, eager.lar)


# --------------------------------------------------------------------------- bounds, arguments, surfaces
def test_outputs_and_the_distance_table_stay_inside_their_buffers():
    """Canaries: the distance table and every output and state array the kernels write are re-pointed into the middle
    of guarded allocations; every launch mode steps with the rule on and frequent resets; the guard bytes and the
    (read-only) table must be untouched."""
    import torch
    G = 4096
    scene = H.scenes.make_thor_scene(120, (14, 18), seed=5, n_goals=3, planes=("rgb", "depth"))
    world = T.compile_world([scene], T.GYM_GRAPH)
    lay = world.layout
    for N, gather in ((23, "fused"), (23, "bulk"), (777, "bulk"), (777, "ldg"), (777, "persistent"), (5, "persistent")):
        guards = []

        def guarded(t):
            raw = torch.full((t.numel() * t.element_size() + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
            inner = raw[G:G + t.numel() * t.element_size()].view(t.dtype).view(t.shape)
            inner.copy_(t)
            guards.append(raw)
            return inner

        env = vn.GraphVecEnv(world, N, seed=3, max_episode_steps=5, host_outputs=False, obs_layout="rgbd_goal",
                             gather=gather, reward_progress=0.3)
        table = guarded(env.dw.shortest_paths()[1])
        env.dw.tables.task_dist = table.data_ptr()
        before = table.clone()
        for i, p in enumerate(lay.planes):
            if p in env.obs_buf:
                env.obs_buf[p] = guarded(env.obs_buf[p])
                env._c_out.obs[i] = env.obs_buf[p].data_ptr()
            if p in env.goal_buf:
                env.goal_buf[p] = guarded(env.goal_buf[p])
                env._c_out.goal_obs[i] = env.goal_buf[p].data_ptr()
        env._pack = guarded(env._pack)
        n = N
        for name, lo, hi, dt in (("reward", 0, 4, torch.float32), ("episode_return", 4, 8, torch.float32),
                                 ("episode_length", 8, 12, torch.int32), ("info_state", 12, 16, torch.int32)):
            setattr(env, name, env._pack[lo * n:hi * n].view(dt))
        env.done, env.truncated, env.win, env.did_reset = (env._pack[k * n:(k + 1) * n] for k in range(16, 20))
        o = env._c_out
        o.reward, o.episode_return, o.episode_length = env.reward.data_ptr(), env.episode_return.data_ptr(), \
            env.episode_length.data_ptr()
        o.info_state, o.done, o.truncated = env.info_state.data_ptr(), env.done.data_ptr(), env.truncated.data_ptr()
        o.win, o.did_reset = env.win.data_ptr(), env.did_reset.data_ptr()
        env.lar = guarded(env.lar)
        o.last_action_reward = env.lar.data_ptr()
        env.stats = guarded(env.stats)
        o.stats = env.stats.data_ptr()
        env.obs_state = guarded(env.obs_state)
        o.obs_state = env.obs_state.data_ptr()
        env._gather_desc = guarded(env._gather_desc)
        o.gather_desc = env._gather_desc.data_ptr()
        for name in ("state", "goal", "task", "elapsed", "epoch", "ep_return", "ep_length"):
            setattr(env, name, guarded(getattr(env, name)))
            setattr(env._c_envs, name, getattr(env, name).data_ptr())
        env._obs_cache = None
        rows = [guarded(torch.zeros(N, dtype=dt, device="cuda"))
                for dt in (torch.int32, torch.float32, torch.uint8, torch.int32, torch.int32)]
        env.reset()
        acts = torch.randint(0, 4, (40, N), device="cuda", dtype=torch.int32)
        for t in range(40):
            env.step_enqueue(acts[t], actions_ready=(t % 2 == 1 and gather == "bulk"), record=rows)
        torch.cuda.synchronize()
        for raw in guards:
            assert bool((raw[:G] == 0xA5).all()) and bool((raw[-G:] == 0xA5).all()), (N, gather)
        assert torch.equal(table, before)
        assert torch.equal(rows[1], env.reward) and env.episode_stats()["resets"] > N
        env.dw.tables.task_dist = env.dw.shortest_paths()[1].data_ptr()


def test_python_surface():
    """Non-finite coefficients are refused, the setter takes effect from the next step, the coefficient is used as
    float32, the single-env class passes the keyword on and has the setter, and state_dict does not carry it."""
    import torch
    sc = H.scenes.GridScene(P.ORIENTED_MAZE, [P.ORIENTED_GOAL], True, (84, 84), ("rgb",))
    world = T.compile_world([sc], T.GYM_GRAPH)
    for bad in (float("nan"), float("inf")):
        with pytest.raises(ValueError):
            vn.GraphVecEnv(world, 4, obs_layout="frame", reward_progress=bad)
    env = vn.GraphVecEnv(world, 4, obs_layout="frame", reward_progress=0.01)
    assert env.reward_progress == float(np.float32(0.01))
    with pytest.raises(ValueError):
        env.set_reward_progress(float("-inf"))
    assert "reward_progress" not in env.state_dict()
    # the first steps of the hand-worked oriented scenario, switching the rule on after the first step
    limit, starts, actions, want_r, _ = P.ORIENTED_SCENARIOS[0]
    start = np.array([[sc.state_index(s) for s in starts]], np.int32)
    one = vn.single_env.GraphEnv(world, max_episode_steps=limit, rewards=P.REWARDS, obs_layout="frame",
                                 inject=(np.zeros_like(start), start))
    one.reset()
    assert one.step(actions[0])[1] == P.REWARDS[1]
    one.set_reward_progress(P.COEF)
    for t in range(1, 8):
        assert one.step(actions[t])[1] == want_r[t], t
    vec = vn.single_env.GraphEnv(world, max_episode_steps=limit, rewards=P.REWARDS, reward_progress=P.COEF,
                                 obs_layout="frame", inject=(np.zeros_like(start), start))
    vec.reset()
    assert [vec.step(a)[1] for a in actions[:8]] == want_r[:8]
    assert torch.cuda.is_available()
