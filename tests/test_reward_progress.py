"""CPU tests of the geodesic-progress reward (GraphVecEnv(reward_progress=...), vn_rules_t.reward_progress): the
hand-worked scenarios of tests/progress_reward.py through its oracle restatement, the restatement's distances against
the table the step kernel reads (tables.optimal_policy_table), and the C ABI: struct layout, version, argument checks."""
import ctypes as C
import importlib

import numpy as np
import pytest

import helpers as H
import progress_reward as P
from oracle import envs as oenvs
from oracle import vec as ovec

vn = importlib.import_module("a2cat-vn-pytorch_b200")
T = vn.tables
L = vn.lib

EINVAL = -1


def oracle_env(kind, scenario, coef=P.COEF):
    """One oracle env of a hand-worked scenario: ProgressReward innermost, then TimeLimit and RewardCollector."""
    limit, starts, _, _, _ = scenario
    if kind == "oriented":
        scene = H.scenes.GridScene(P.ORIENTED_MAZE, [P.ORIENTED_GOAL], True, (84, 84), ("rgb",))
        e = oenvs.GymGraphEnv(oenvs.OracleScene(scene), rewards=P.REWARDS)
        graph = P.oriented_graph(P.ORIENTED_MAZE)
    else:
        scene = H.scenes.GridScene(P.COMPASS_MAZE, [P.COMPASS_GOAL], False, (84, 84), ("rgb",))
        e = oenvs.SimpleGraphEnv(oenvs.OracleScene(scene), goal=P.COMPASS_GOAL, rewards=P.REWARDS)
        graph = P.compass_graph(P.COMPASS_MAZE)
    e.reset_source = H.StreamSource(np.zeros(len(starts), np.int32), np.array(starts), len(starts))
    return ovec.RewardCollector(ovec.TimeLimit(P.ProgressReward(e, coef, graph), limit))


CASES = [("oriented", k) for k in range(len(P.ORIENTED_SCENARIOS))] + \
        [("compass", k) for k in range(len(P.COMPASS_SCENARIOS))]


def scenario_of(kind, k):
    return (P.ORIENTED_SCENARIOS if kind == "oriented" else P.COMPASS_SCENARIOS)[k]


@pytest.mark.parametrize("kind,k", CASES)
def test_hand_worked_rewards_through_the_oracle(kind, k):
    """Toward / away from the goal, collision, no-op, goal with auto-reset, time-limit truncation and an unreachable
    start: the restated rule gives the rewards worked out by hand, and the episode returns and last_action_reward
    carry them."""
    sc = scenario_of(kind, k)
    _, _, actions, want_r, want_d = sc
    vec = ovec.VecEnv([oracle_env(kind, sc)])
    vec.reset()
    returns = []
    for t, a in enumerate(actions):
        (_, lar), r, d, infos = vec.step([a])
        assert np.float32(r[0]).view(np.uint32) == np.float32(want_r[t]).view(np.uint32), (t, r[0], want_r[t])
        assert bool(d[0]) == bool(want_d[t]), t
        # UnrealEnvBaseWrapper: clip(shaped reward) unless the env just reset
        assert lar[0, -1] == (0.0 if d[0] else np.clip(want_r[t], -1, 1)), t
        if d[0]:
            returns.append(infos[0]["episode"]["r"])
    assert returns == P.EPISODE_RETURNS[(kind, k)]


def _graph_of(scene):
    return P.oriented_graph(scene.maze) if scene.oriented else P.compass_graph(scene.maze)


@pytest.mark.parametrize("oriented,seed", [(True, 0), (True, 7), (False, 3), (False, 11)])
def test_oracle_distances_equal_the_kernel_table(oriented, seed):
    """The restatement's BFS over the oracle's transition rule and tables.optimal_policy_table (what
    DeviceWorld.shortest_paths uploads and the step kernel reads) give the same distance for every state and task,
    -1 included, on random mazes with several goals and a multi-scene world."""
    fam = T.GYM_GRAPH if oriented else T.SIMPLE_GRAPH
    planes = ("rgb",)
    scs = [H.scenes.make_maze_scene((9, 7), 0.3, seed + k, n_goals=3, oriented=oriented, planes=planes, scene_id=k)
           for k in range(2)]
    world = T.compile_world(scs, fam)
    assert len(world.tasks) == 6
    for ti, task in enumerate(world.tasks):
        sc = scs[task.scene]
        dist, _ = T.optimal_policy_table(world, ti)
        want = P.distances_to(_graph_of(sc), [tuple(task.goal)])
        got = {sc.state_tuple(s): int(dist[s]) for s in range(sc.n_states)}
        assert got == {st: want.get(st, -1) for st in got}, ti
    hand = [(T.GYM_GRAPH, True, P.ORIENTED_MAZE, P.ORIENTED_GOAL), (T.SIMPLE_GRAPH, False, P.COMPASS_MAZE, P.COMPASS_GOAL)]
    for f, o, maze, goal in hand:
        sc = H.scenes.GridScene(maze, [goal], o, (84, 84), planes)
        dist, _ = T.optimal_policy_table(T.compile_world([sc], f), 0)
        want = P.distances_to(_graph_of(sc), [goal])
        assert [int(v) for v in dist] == [want.get(sc.state_tuple(s), -1) for s in range(sc.n_states)]
        assert (dist < 0).sum() == (8 if o else 2)      # the component no path joins to the goal


def test_abi_layout_of_the_new_fields():
    """ABI 7: vn_rules_t keeps its 40 bytes (the former reserved int32 is the float coefficient) and vn_tables_t ends
    with the distance-table pointer; the library agrees with the ctypes mirrors."""
    lib = L.load()
    assert L.ABI_VERSION == 7 and lib.vn_abi_version() == 7
    mirrors = (L.Store, L.Tables, L.Envs, L.Rules, L.Inject, L.StepOut, L.Replay, L.FloatLeaf, L.HostCall, L.U8Frames)
    for which, m in enumerate(mirrors):
        assert lib.vn_abi_struct_size(which) == C.sizeof(m), m.__name__
    assert C.sizeof(L.Rules) == 40
    assert L.Rules.reward_progress.offset == 28 and L.Rules.reward_progress.size == 4
    assert L.Rules.seed.offset == 32
    assert L.Tables.task_dist.offset == 48 and C.sizeof(L.Tables) == 56
    r = L.Rules()
    r.reward_progress = 0.01
    assert r.reward_progress == float(np.float32(0.01))


def _scalar_call(coef, task_dist):
    """vn_env_step_scalar with descriptors whose device pointers are never dereferenced: the calls below are all
    rejected while the arguments are checked, before anything is enqueued."""
    lib = L.load()
    fake = 1 << 20
    tab = L.Tables(fake, fake, fake, fake, fake, 16, 2, task_dist)
    envs = L.Envs(8, 0, *([fake] * 9))
    rules = L.Rules(1.0, 0.0, 0.0, 10, 0, 0, 4, coef, 0)
    out = L.StepOut()
    out.obs_state = fake
    rc = lib.vn_env_step_scalar(C.byref(tab), C.byref(envs), C.byref(rules), None, fake, C.byref(out), None)
    return rc, lib.vn_last_error().decode()


@pytest.mark.parametrize("coef", [0.01, -2.0, 1e-30])
def test_nonzero_coefficient_needs_the_distance_table(coef):
    rc, msg = _scalar_call(coef, None)
    assert rc == EINVAL
    assert "reward_progress" in msg and "task_dist" in msg, msg


@pytest.mark.parametrize("coef", [float("inf"), float("-inf"), float("nan")])
def test_non_finite_coefficient_is_rejected(coef):
    rc, msg = _scalar_call(coef, 1 << 20)
    assert rc == EINVAL
    assert "reward_progress" in msg and "not finite" in msg, msg
