"""GPU tests of the fixed episode list (GraphVecEnv.set_episodes, vn_episodes_t, evaluation.evaluate_episodes) in every
launch mode: without a list nothing changes, with one the step matches the oracle restatement of tests/episode_list.py
bit for bit, the results do not depend on batch size or sharding, known policies score what they must, and every
listed episode is recorded exactly once, inside its buffers."""
import importlib
import math

import numpy as np
import pytest

import episode_list as EL
import helpers as H
from oracle import envs as oenvs
from oracle import graph_util as gu
from oracle import vec as ovec

pytestmark = pytest.mark.gpu

vn = importlib.import_module("a2cat-vn-pytorch_b200")
T = vn.tables
EV = vn.evaluation

MODES = ("ldg", "bulk", "fused", "persistent", "auto")
RESULT_KEYS = ("length", "ret", "win", "truncated", "final_state")


def f32bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def _host(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _world(kind):
    """(scenes, world, rewards, lowest action) of the three families the list is tested on."""
    if kind == "oriented":           # one scene, three tasks, collisions, rotations
        scs = [H.scenes.make_maze_scene((9, 11), 0.3, 21, n_goals=3, planes=("rgb",))]
        return scs, T.compile_world(scs, T.GYM_GRAPH), (1.0, -0.01, -0.1), 0
    if kind == "multi_scene":        # MultipleGraphEnv: two un-oriented scenes, no-op actions
        scs = [H.scenes.make_maze_scene((8, 8), 0.3, 30 + k, n_goals=1, oriented=False, planes=("rgb",), scene_id=k)
               for k in range(2)]
        return scs, T.compile_world(scs, T.SIMPLE_GRAPH), (1.0, -0.01, -0.1), -1
    # thor_cached: h5 action order, -0.0 step reward, a collision overrides the goal reward
    scs = [H.scenes.make_maze_scene((8, 9), 0.25, 40, n_goals=1, planes=("rgb",))]
    return scs, T.compile_world(scs, T.THOR_CACHED, tasks=[(0, 3), (0, 29), (0, 50)]), (1.0, 0.0, 0.0), 0


def _mixed_list(world, n, seed):
    """n (task, start) pairs from every reachable candidate of every task, shuffled so that tasks interleave."""
    task, start = EV.episode_set(world, None, seed=seed)
    pick = np.random.RandomState(seed).permutation(len(task))[:n]
    return task[pick], start[pick]


# --------------------------------------------------------------------------- no list changes nothing
@pytest.mark.parametrize("host_outputs", [True, False])
@pytest.mark.parametrize("gather", MODES)
def test_no_list_is_bit_identical(gather, host_outputs):
    """An env that never had a list, one whose list was installed and removed again, and one with an EMPTY list
    installed give the same rewards (-0.0 of the thor-cached rules included), dones, last_action_reward, states,
    ep_return, statistics, episode infos and observation bytes."""
    import torch
    for kind in ("oriented", "thor_cached"):
        _, world, rewards, _ = _world(kind)
        N, nt = 37, len(world.tasks)
        kw = dict(seed=3, max_episode_steps=9, gather=gather, host_outputs=host_outputs, rewards=rewards,
                  env_tasks=np.tile(np.array([[0, nt]], np.int32), (N, 1)), obs_layout="frame")
        plain = vn.GraphVecEnv(world, N, **kw)
        cleared = vn.GraphVecEnv(world, N, device_world=plain.dw, **kw)
        cleared.set_episodes(*_mixed_list(world, 50, 0))
        cleared.set_episodes(None)
        empty = vn.GraphVecEnv(world, N, device_world=plain.dw, **kw)
        empty.set_episodes(np.zeros(0, np.int32), np.zeros(0, np.int32))
        envs = (plain, cleared, empty)
        for e in envs:
            e.reset()
        rng = np.random.RandomState(0)
        zero_sign = 0
        for t in range(60):
            a = rng.randint(0, 4, N).astype(np.int32)
            outs = [e.step(a) for e in envs]
            (obs0, lar0), r0, d0, i0 = outs[0]
            zero_sign += int(np.signbit(_host(r0)[_host(r0) == 0]).sum())
            for (obs, lar), r, d, infos in outs[1:]:
                assert np.array_equal(f32bits(_host(r)), f32bits(_host(r0))), (kind, t)
                assert np.array_equal(_host(d), _host(d0)) and torch.equal(lar, lar0), (kind, t)
                assert torch.equal(obs, obs0), (kind, t)
                assert [infos[i].get("episode") for i in range(N)] == [i0[i].get("episode") for i in range(N)], t
            for e in envs[1:]:
                assert torch.equal(e.ep_return.view(torch.int32), plain.ep_return.view(torch.int32))
                assert torch.equal(e.state, plain.state) and torch.equal(e.stats, plain.stats)
                assert torch.equal(e.epoch, plain.epoch) and torch.equal(e.task, plain.task)
        assert (zero_sign > 0) == (kind == "thor_cached")
        assert empty.episodes_recorded == 0 and bool((empty._episodes["cursor"] == -1).all())


# --------------------------------------------------------------------------- against the oracle restatement
PATHS = ("ldg", "bulk", "pipelined", "fused", "persistent", "host", "graph")


def _oracle_run(kind, coef, N, steps, seed, limit):
    scs, world, rewards, lo = _world(kind)
    task, start = _mixed_list(world, 3 * N, seed)
    make = EL.oracle_case(kind, world, scs, seed, limit, rewards, coef)
    results = {}
    stacks = [make(g, task, start, N, results) for g in range(N)]
    ov = ovec.VecEnv([s for s, _ in stacks])
    ov.reset()
    acts = np.random.RandomState(seed + 1).randint(lo, 4, (steps, N)).astype(np.int32)
    want = []
    for t in range(steps):
        _, r, d, _ = ov.step(acts[t])
        want.append((f32bits(r), d.copy(), np.array([s.state_of(b) for s, b in stacks], np.int32)))
    assert sorted(results) == list(range(len(task)))          # every listed episode ended within the run
    kw = dict(seed=seed, max_episode_steps=limit, rewards=rewards, obs_layout="frame", reward_progress=coef,
              env_tasks=np.tile(np.array([[0, len(world.tasks)]], np.int32), (N, 1)))
    return world, kw, task, start, acts, want, results


def _check_step(w, r, d, state, obs_state, where):
    assert np.array_equal(f32bits(_host(r)), w[0]), where
    assert np.array_equal(_host(d).astype(bool), w[1]), where
    assert np.array_equal(_host(state), w[2]), where
    assert np.array_equal(_host(obs_state), w[2]), where      # auto-reset: the observation shows the state


@pytest.mark.parametrize("kind,coef", [("oriented", 0.0), ("multi_scene", 0.0), ("thor_cached", 0.0),
                                       ("oriented", 0.25)])
def test_matches_the_oracle_bit_for_bit(kind, coef):
    """300 steps of random actions (no-ops included on SIMPLE_GRAPH) with a list of 3 episodes per env on every launch
    path - split ldg / bulk, pipelined, fused, persistent, the host-facing step(numpy) and a capture_steps graph replay:
    rewards (float bits), dones, states, observation bytes and every recorded result equal the restatement's, before
    and after the envs fall back to their Philox resets."""
    import torch
    N, steps = 24, 300
    world, kw, task, start, acts, want, results = _oracle_run(kind, coef, N, steps, seed=9, limit=11)
    E = len(task)
    dev_acts = torch.from_numpy(acts).cuda()
    dw = None
    for path in PATHS:
        gather = {"pipelined": "bulk", "host": "auto", "graph": "auto"}.get(path, path)
        env = vn.GraphVecEnv(world, N, gather=gather, host_outputs=(path == "host"), device_world=dw, **kw)
        dw = env.dw
        rgb = dw.plane_view("rgb")
        env.set_episodes(task, start)
        env.reset()
        if path == "graph":
            rec = [torch.zeros(steps, N, dtype=dt, device="cuda") for dt in (torch.float32, torch.uint8, torch.int32,
                                                                             torch.int32)]

            def after(t):
                for buf, src in zip(rec, (env.reward, env.done, env.state, env.obs_state)):
                    buf[t].copy_(src)
            cap = env.capture_steps(dev_acts, after_step=after)
            assert env.episodes_recorded == 0
            cap.replay()
            torch.cuda.synchronize()
            for t in range(steps):
                _check_step(want[t], rec[0][t], rec[1][t], rec[2][t], rec[3][t], (path, t))
        else:
            for t in range(steps):
                if path == "host":
                    _, r, d, _ = env.step(acts[t])
                else:
                    env.step_enqueue(dev_acts[t], actions_ready=(path == "pipelined" and t > 0))
                    r, d = env.reward, env.done
                _check_step(want[t], r, d, env.state, env.obs_state, (path, t))
                if t % 50 == 0 or t == steps - 1:
                    o = env.obs_buf["rgb"]
                    assert torch.equal(o, rgb[env.obs_state.long()]), (path, t)
        o = env.obs_buf["rgb"]
        assert torch.equal(o, rgb[torch.from_numpy(want[-1][2]).long().cuda()]), path
        assert env.episodes_recorded == E, path
        res = {k: v.cpu().numpy() for k, v in env.episode_results().items()}
        for j in range(E):
            w = results[j]
            got = (int(res["length"][j]), f32bits(res["ret"][j]), bool(res["win"][j]), bool(res["truncated"][j]),
                   int(res["final_state"][j]))
            assert got == (w["length"], f32bits(w["ret"]), w["win"], w["truncated"], w["final_state"]), (path, j)
        assert bool((env._episodes["cursor"] == -1).all()), path


@pytest.mark.parametrize("gather", MODES)
def test_hand_worked_case_on_the_device(gather):
    """The hand-worked case of tests/episode_list.py (3 envs, 7 episodes, TimeLimit 2, always forward) gives the
    hand-computed results, each env leaves its list on the step the restatement does, and the Philox resets that follow
    put the envs where the restatement puts them."""
    import torch
    scene = H.scenes.GridScene(EL.HAND_MAZE, [EL.HAND_GOAL], True, (84, 84), ("rgb",))
    world = T.compile_world([scene], T.GYM_GRAPH)
    osc = oenvs.OracleScene(scene)
    cands = [gu.initial_state_candidates(scene.maze, osc.graph, osc.optimal_actions, EL.HAND_GOAL)]
    starts = np.array([scene.state_index(s) for s in EL.HAND_STARTS], np.int32)
    results, stacks = {}, []
    for g in range(3):
        base = oenvs.GymGraphEnv(osc, goals=[EL.HAND_GOAL], rewards=EL.HAND_REWARDS)
        base.reset_source = ovec.PhiloxResetSource(5, g, cands, lambda t: None, False)
        stack = ovec.RewardCollector(ovec.TimeLimit(base, EL.HAND_LIMIT))
        stacks.append(EL.EpisodeList(stack, base, np.zeros(7, np.int32), starts, g, 3, results, scene.state_tuple,
                                     lambda e: scene.state_index(e.state)))
    ov = ovec.VecEnv(stacks)
    env = vn.GraphVecEnv(world, 3, seed=5, max_episode_steps=EL.HAND_LIMIT, rewards=EL.HAND_REWARDS, gather=gather,
                         obs_layout="frame")
    env.set_episodes(np.zeros(7, np.int32), starts)
    env.reset()
    ov.reset()
    for t in range(1, 13):
        _, r, d, _ = env.step(np.zeros(3, np.int32))
        _, orr, od, _ = ov.step([0, 0, 0])
        assert np.array_equal(f32bits(r), f32bits(orr)) and np.array_equal(d, od), (gather, t)
        assert env.state.cpu().tolist() == [scene.state_index(s.base.state) for s in stacks], (gather, t)
        cur = env._episodes["cursor"].cpu().tolist()
        assert cur == [s.cursor for s in stacks], (gather, t)
    assert env.episodes_recorded == 7
    res = {k: v.cpu().numpy() for k, v in env.episode_results().items()}
    for j, (length, ret, win, trunc, final) in enumerate(EL.HAND_RESULTS):
        assert (res["length"][j], res["win"][j], res["truncated"][j]) == (length, win, trunc), (gather, j)
        assert f32bits(res["ret"][j]) == f32bits(ret) and res["final_state"][j] == scene.state_index(final), j
    assert torch.equal(env.epoch.cpu(), torch.tensor([s.ordinary.epoch for s in stacks], dtype=torch.int32))


# --------------------------------------------------------------------------- batch-size and shard invariance
def _hash_policy(env):
    """A deterministic function of (state, goal): the shortest-path action, replaced by a hashed one in about a third
    of the (state, goal) pairs - so some episodes win and some run into the TimeLimit."""
    import torch

    def policy(obs):
        act, _ = env.optimal_actions()
        h = (env.state.long() * 0x9E3779B1 + env.goal.long() * 0x85EBCA77 + 0x165667B1) & 0xFFFFFFFF
        h = h ^ (h >> 15)
        return torch.where(h % 3 == 0, (h >> 4) % 4, act.long()).to(torch.int32)
    return policy


def _invariance_world():
    scene = H.scenes.make_maze_scene((12, 12), 0.25, 8, n_goals=3, planes=("rgb",))
    world = T.compile_world([scene], T.GYM_GRAPH)
    task, start = _mixed_list(world, 150, 4)
    return world, task, start


def _per_episode(res):
    p = res["per_episode"]
    return {k: (f32bits(p[k]) if k == "reward" else np.asarray(p[k])) for k in p}


def test_results_do_not_depend_on_batch_size_or_launch_mode():
    """The same list under the same (state, goal) policy gives identical result arrays for 1, 5, 64 and 777 envs, each
    with the fused, persistent and bulk launches."""
    world, task, start = _invariance_world()
    ref, dw = None, None
    for N in (1, 5, 64, 777):
        for gather in ("fused", "persistent", "bulk"):
            env = vn.GraphVecEnv(world, N, seed=N, max_episode_steps=40, obs_layout="frame", host_outputs=False,
                                 gather=gather, device_world=dw)
            dw = env.dw
            res = EV.evaluate_episodes(env, _hash_policy(env), task, start, check_every=16)
            assert res["complete"] and res["episodes"] == len(task), (N, gather)
            got = _per_episode(res)
            if ref is None:
                ref = got
                assert 0 < res["success_rate"] < 1 and res["truncated_rate"] > 0
            for k in ref:
                assert np.array_equal(got[k], ref[k]), (N, gather, k)
            assert env._episodes is None          # the list is removed again


def test_two_shards_equal_one_process():
    """Two shards of a 64-env job each score the episodes their envs own; together they are the one-process result."""
    world, task, start = _invariance_world()
    kw = dict(seed=2, max_episode_steps=40, obs_layout="frame", host_outputs=False)
    whole = vn.GraphVecEnv(world, 64, **kw)
    one = _per_episode(EV.evaluate_episodes(whole, _hash_policy(whole), task, start))
    parts = []
    for r in range(2):
        env = vn.GraphVecEnv(world, 64, rank=r, world_size=2, device_world=whole.dw, **kw)
        res = EV.evaluate_episodes(env, _hash_policy(env), task, start)
        assert res["complete"]
        parts.append(_per_episode(res))
    assert not set(parts[0]["index"].tolist()) & set(parts[1]["index"].tolist())
    order = np.argsort(np.concatenate([p["index"] for p in parts]))
    for k in one:
        assert np.array_equal(np.concatenate([p[k] for p in parts])[order], one[k]), k


# --------------------------------------------------------------------------- known answers
@pytest.mark.parametrize("kind", ["oriented", "thor_cached"])
def test_shortest_path_policy_scores_spl_one_on_every_candidate_start(kind):
    import torch
    _, world, rewards, _ = _world(kind)
    task, start = EV.episode_set(world, None, seed=0)
    env = vn.GraphVecEnv(world, 256, seed=1, max_episode_steps=300, rewards=rewards, obs_layout="frame",
                         host_outputs=False)
    res = EV.evaluate_episodes(env, lambda obs: env.optimal_actions()[0], task, start)
    p = res["per_episode"]
    assert res["complete"] and res["episodes"] == len(task)
    assert res["success_rate"] == 1.0 and res["spl"] == 1.0 and res["truncated_rate"] == 0.0
    assert res["distance_to_goal"] == 0.0
    assert (p["win"] == 1).all() and (p["length"] == p["distance"]).all() and (p["spl"] == 1.0).all()
    _, dist = env.dw.shortest_paths()
    assert np.array_equal(p["distance"], dist[torch.from_numpy(task).long(), torch.from_numpy(start).long()].cpu().numpy())


def test_random_policy_summary_equals_a_torch_recomputation():
    import torch
    world, task, start = _invariance_world()
    env = vn.GraphVecEnv(world, 100, seed=3, max_episode_steps=5, obs_layout="frame", host_outputs=False)
    gen = torch.Generator(device="cuda").manual_seed(0)
    res = EV.evaluate_episodes(env, lambda obs: torch.randint(0, 4, (100,), device="cuda", dtype=torch.int32,
                                                              generator=gen), task, start, check_every=3)
    p = {k: torch.from_numpy(np.asarray(v)) for k, v in res["per_episode"].items()}
    assert res["complete"] and bool(((p["win"].int() + p["truncated"].int()) == 1).all())
    assert bool((p["length"] <= 5).all()) and 0 < res["success_rate"] < 1
    win, length, l = p["win"].double(), p["length"].double(), p["distance"].double()
    want = dict(success_rate=win.mean(), spl=(win * l / torch.maximum(length, l)).mean(), episode_length=length.mean(),
                reward=p["reward"].double().mean(), truncated_rate=p["truncated"].double().mean(),
                distance_to_goal=p["final_distance"].double().mean())
    for k, v in want.items():
        assert math.isclose(res[k], float(v), rel_tol=1e-12, abs_tol=1e-15), k
    assert res["steps"] % 3 == 0 and res["steps"] >= int(p["length"].max())


# --------------------------------------------------------------------------- exactly once, inside the buffers
def test_every_episode_is_recorded_exactly_once_inside_its_buffers():
    """Canaries round the cursor and every result array; every launch mode runs the list to its end and 150 steps
    beyond: the counter ends at E and stays there, and the guard bytes are untouched."""
    import torch
    G = 4096
    scene = H.scenes.make_thor_scene(120, (14, 18), seed=5, n_goals=3, planes=("rgb", "depth"))
    world = T.compile_world([scene], T.GYM_GRAPH)
    task, start = _mixed_list(world, 150, 1)
    for N, gather in ((23, "fused"), (23, "bulk"), (777, "bulk"), (777, "ldg"), (777, "persistent"), (5, "persistent"),
                      (23, "host")):
        env = vn.GraphVecEnv(world, N, seed=3, max_episode_steps=5, host_outputs=(gather == "host"),
                             obs_layout="rgbd_goal", gather="auto" if gather == "host" else gather)
        env.set_episodes(task, start)
        e = env._episodes
        guards = []
        for k in ("cursor",) + RESULT_KEYS + ("count",):
            t = e[k]
            raw = torch.full((t.numel() * t.element_size() + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
            inner = raw[G:G + t.numel() * t.element_size()].view(t.dtype)
            inner.copy_(t)
            guards.append(raw)
            e[k] = inner
            setattr(e["c"], k, inner.data_ptr())
        env.reset()
        rng = np.random.RandomState(0)
        acts = torch.randint(0, 4, (300, N), device="cuda", dtype=torch.int32)
        counts = []
        for t in range(300):
            if gather == "host":
                env.step(rng.randint(0, 4, N).astype(np.int32))
            else:
                env.step_enqueue(acts[t], actions_ready=(t % 2 == 1 and gather == "bulk"))
            if t % 50 == 49:
                counts.append(env.episodes_recorded)
        torch.cuda.synchronize()
        owned = len(env.episodes_owned)
        assert owned == len(task) and counts[-1] == owned and counts[-3:] == [owned] * 3, (N, gather, counts)
        res = env.episode_results()
        assert bool((res["length"] >= 1).all()) and bool((res["length"] <= 5).all()), (N, gather)
        assert bool(((res["win"].int() + res["truncated"].int()) == 1).all()), (N, gather)
        for raw in guards:
            assert bool((raw[:G] == 0xA5).all()) and bool((raw[-G:] == 0xA5).all()), (N, gather)


# --------------------------------------------------------------------------- the Python surface
def test_python_surface():
    """Host-side checks of set_episodes, the masked-reset refusal, the shard's owned ids, state_dict without the list,
    and a reset that starts the list again."""
    import torch
    scs, world, rewards, _ = _world("multi_scene")
    env = vn.GraphVecEnv(world, 8, obs_layout="frame", rewards=rewards)
    _, dist = env.dw.shortest_paths()
    b1 = int(world.scene_base[1])
    good = int(torch.nonzero(dist[1, b1:] >= 1)[0, 0]) + b1
    with pytest.raises(ValueError, match="task indices"):
        env.set_episodes([2], [good])
    with pytest.raises(ValueError, match="start states"):
        env.set_episodes([1], [world.n_states])
    with pytest.raises(ValueError, match="not in the scene"):
        env.set_episodes([0], [good])
    with pytest.raises(ValueError, match="cannot reach"):
        env.set_episodes([1], [int(world.task_goal[1])])                 # distance 0: the goal itself
    with pytest.raises(ValueError, match="same length"):
        env.set_episodes([1, 1], [good])
    hand = H.scenes.GridScene(EL.HAND_MAZE, [EL.HAND_GOAL], True, (84, 84), ("rgb",))
    hw = T.compile_world([hand], T.GYM_GRAPH)
    henv = vn.GraphVecEnv(hw, 2, obs_layout="frame")
    with pytest.raises(ValueError, match="cannot reach"):
        henv.set_episodes([0], [hand.state_index((3, 0, 1))])            # a cell no path joins to the goal
    with pytest.raises(ValueError, match="auto_reset"):
        vn.GraphVecEnv(world, 4, obs_layout="frame", auto_reset=False).set_episodes([1], [good])
    inj = np.zeros((4, 3), np.int32), np.full((4, 3), good, np.int32)
    with pytest.raises(ValueError, match="inject"):
        vn.GraphVecEnv(world, 4, obs_layout="frame", inject=inj).set_episodes([1], [good])
    with pytest.raises(RuntimeError):
        env.episode_results()
    assert env.episodes_owned is None and env.episodes_recorded == 0

    task = np.array([1] * 20, np.int32)
    start = np.array([good] * 20, np.int32)
    env.set_episodes(torch.from_numpy(task).cuda(), torch.from_numpy(start))
    with pytest.raises(ValueError, match="mask"):
        env.reset(mask=np.ones(8, bool))
    env.reset()
    assert env._episodes["cursor"].cpu().tolist() == list(range(8))
    assert env.task.cpu().tolist() == [1] * 8 and env.state.cpu().tolist() == [good] * 8
    assert "episodes" not in " ".join(env.state_dict())
    for _ in range(40):
        env.step(np.full(8, -1, np.int32))                               # no-ops: nothing ends before the TimeLimit
    env.reset()                                                          # the list starts again, results zeroed
    assert env.episodes_recorded == 0 and env._episodes["cursor"].cpu().tolist() == list(range(8))
    assert bool((env.episode_results()["length"] == -1).all())
    shards = [vn.GraphVecEnv(world, 7, rank=r, world_size=2, obs_layout="frame", device_world=env.dw) for r in range(2)]
    for s in shards:
        s.set_episodes(task, start)
    assert shards[0].episodes_owned.tolist() == [j for j in range(20) if j % 7 < 4]
    assert shards[1].episodes_owned.tolist() == [j for j in range(20) if j % 7 >= 4]
    shards[1].reset()
    assert shards[1]._episodes["cursor"].cpu().tolist() == [4, 5, 6]
