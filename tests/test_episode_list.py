"""CPU tests of the fixed episode list (GraphVecEnv.set_episodes, vn_episodes_t, evaluation.evaluate_episodes /
episode_set): the hand-worked case through the oracle restatement of tests/episode_list.py, the C ABI (struct layout,
version, argument checks) and the episode sets."""
import ctypes as C
import importlib
import types

import numpy as np
import pytest

import episode_list as EL
import helpers as H
from oracle import envs as oenvs
from oracle import graph_util as gu
from oracle import vec as ovec

vn = importlib.import_module("a2cat-vn-pytorch_b200")
T = vn.tables
L = vn.lib
EV = vn.evaluation

EINVAL = -1


def _hand_batch(seed=5):
    """The hand-worked case of tests/episode_list.py: 3 oracle envs with the list deal on top of the Philox stream."""
    scene = H.scenes.GridScene(EL.HAND_MAZE, [EL.HAND_GOAL], True, (84, 84), ("rgb",))
    osc = oenvs.OracleScene(scene)
    cands = [gu.initial_state_candidates(scene.maze, osc.graph, osc.optimal_actions, EL.HAND_GOAL)]
    starts = [scene.state_index(s) for s in EL.HAND_STARTS]
    task = np.zeros(len(starts), np.int32)
    results, envs = {}, []
    for g in range(3):
        base = oenvs.GymGraphEnv(osc, goals=[EL.HAND_GOAL], rewards=EL.HAND_REWARDS)
        base.reset_source = ovec.PhiloxResetSource(seed, g, cands, lambda t: None, False)
        stack = ovec.RewardCollector(ovec.TimeLimit(base, EL.HAND_LIMIT))
        envs.append(EL.EpisodeList(stack, base, task, starts, g, 3, results, scene.state_tuple,
                                   lambda e: scene.state_index(e.state)))
    return scene, osc, cands, envs, results


def test_hand_worked_deal_results_and_fallback():
    """3 envs, 7 episodes, always forward: a one-step win, a win on the limit step (truncated = 0), collisions and a
    walk cut off by the TimeLimit; each env runs its own ids in order, every result is written once, and after its list
    each env draws from the Philox stream at the epoch its resets reached."""
    scene, osc, cands, envs, results = _hand_batch()
    vec = ovec.VecEnv(envs)
    vec.reset()
    order = []
    for t in range(1, 9):
        before = dict(results)
        _, _, done, infos = vec.step([0, 0, 0])
        order += sorted(set(results) - set(before))
        for g, e in enumerate(envs):
            if t == EL.HAND_LAST_STEP[g]:
                # the auto-reset after its last listed episode is the env's first Philox draw, at the epoch its
                # resets (listed ones included) reached
                assert done[g] and e.cursor == -1, (t, g)
                assert e.ordinary.epoch == EL.HAND_EPOCH_AFTER[g] + 1, g
                ref = ovec.PhiloxResetSource(5, g, cands, lambda t: None, False)
                ref.epoch = EL.HAND_EPOCH_AFTER[g]
                assert tuple(e.base.state) == ref()[1], g
    assert order == [0, 1, 2, 3, 5, 4, 6]
    assert sorted(results) == list(range(7))
    for j, (length, ret, win, trunc, final) in enumerate(EL.HAND_RESULTS):
        r = results[j]
        assert (r["length"], r["win"], r["truncated"]) == (length, bool(win), bool(trunc)), j
        assert np.float32(r["ret"]).view(np.uint32) == np.float32(ret).view(np.uint32), j
        assert r["final_state"] == scene.state_index(final), j
    # many more steps: no listed episode starts again and no result is written again
    snap = {k: dict(v) for k, v in results.items()}
    for _ in range(50):
        vec.step([0, 0, 0])
    assert results == snap and all(e.cursor == -1 for e in envs)
    # an explicit reset starts the list again from each env's global id
    vec.reset()
    assert [e.cursor for e in envs] == [0, 1, 2]


def test_abi_layout_of_the_episode_list():
    """ABI 7 unchanged in number: vn_envs_t ends with the vn_episodes_t pointer (vn_step_out_t keeps its 296 bytes),
    vn_episodes_t is struct 10 and the library agrees with the ctypes mirrors."""
    lib = L.load()
    assert L.ABI_VERSION == 7 and lib.vn_abi_version() == 7
    mirrors = (L.Store, L.Tables, L.Envs, L.Rules, L.Inject, L.StepOut, L.Replay, L.FloatLeaf, L.HostCall, L.U8Frames,
               L.Episodes)
    for which, m in enumerate(mirrors):
        assert lib.vn_abi_struct_size(which) == C.sizeof(m), m.__name__
    assert lib.vn_abi_struct_size(11) == -1
    assert C.sizeof(L.Episodes) == 80 and lib.vn_abi_struct_size(10) == 80
    assert L.Envs.episodes.offset == 80 and C.sizeof(L.Envs) == 88 and C.sizeof(L.StepOut) == 296
    want = dict(task=0, start=8, n_episodes=16, stride=20, cursor=24, length=32, ret=40, win=48, truncated=56,
                final_state=64, count=72)
    assert {k: getattr(L.Episodes, k).offset for k in want} == want


FAKE = 1 << 20


def _call(ep, reset=False, mask=None, inject=None, flags=L.RULE_AUTO_RESET, n_envs=8, env_id_base=0):
    """vn_env_step_scalar / vn_env_reset with descriptors whose device pointers are never dereferenced: the calls below
    are all rejected while the arguments are checked, before anything is enqueued."""
    lib = L.load()
    tab = L.Tables(FAKE, FAKE, FAKE, FAKE, FAKE, 16, 2, None)
    envs = L.Envs(n_envs, env_id_base, *([FAKE] * 9))
    envs.episodes = C.cast(C.pointer(ep), C.c_void_p)
    rules = L.Rules(1.0, 0.0, 0.0, 10, 0, flags, 4, 0.0, 0)
    out = L.StepOut()
    out.obs_state = FAKE
    inj = C.byref(inject) if inject is not None else None
    if reset:
        store = L.Store(FAKE, 128, 16, 1)
        store.plane_bytes[0] = 16
        rc = lib.vn_env_reset(C.byref(store), C.byref(tab), C.byref(envs), C.byref(rules), inj, mask, C.byref(out),
                              L.GATHER_BULK, None)
    else:
        rc = lib.vn_env_step_scalar(C.byref(tab), C.byref(envs), C.byref(rules), inj, FAKE, C.byref(out), None)
    return rc, lib.vn_last_error().decode()


def _episodes(n=5, stride=8, **null):
    p = {k: (None if k in null else FAKE) for k in ("task", "start", "cursor", "length", "ret", "win", "truncated",
                                                    "final_state", "count")}
    return L.Episodes(p["task"], p["start"], n, stride, p["cursor"], p["length"], p["ret"], p["win"], p["truncated"],
                      p["final_state"], p["count"])


def test_rejections():
    """Every combination the list cannot run with is VN_EINVAL with a message naming it."""
    cases = [
        (dict(inject=L.Inject(FAKE, FAKE, 4, 0)), "injected reset stream"),
        (dict(flags=0), "VN_RULE_AUTO_RESET"),
        (dict(reset=True, mask=FAKE), "masked reset"),
        (dict(n_envs=9), "stride=8"),
        (dict(n_envs=4, env_id_base=6), "stride=8"),
    ]
    for kw, words in cases:
        rc, msg = _call(_episodes(), **kw)
        assert rc == EINVAL and "episodes" in msg and words in msg, (kw, msg)
    for field in ("task", "start", "length", "ret", "win", "truncated", "final_state"):
        rc, msg = _call(_episodes(**{field: 1}))
        assert rc == EINVAL and "null list or result pointer" in msg, (field, msg)
    for field in ("cursor", "count"):
        rc, msg = _call(_episodes(n=0, **{field: 1}))
        assert rc == EINVAL and "cursor and count" in msg, (field, msg)
    rc, msg = _call(_episodes(n=-1))
    assert rc == EINVAL and "n_episodes=-1" in msg, msg


def _worlds():
    scene = H.scenes.make_maze_scene((9, 11), 0.3, 21, n_goals=3, planes=("rgb",))
    thor = H.scenes.make_maze_scene((8, 9), 0.25, 40, n_goals=1, planes=("rgb",))
    two = [H.scenes.make_maze_scene((8, 8), 0.3, 30 + k, n_goals=1, oriented=False, planes=("rgb",), scene_id=k)
           for k in range(2)]
    return [T.compile_world([scene], T.GYM_GRAPH), T.compile_world([thor], T.THOR_CACHED, tasks=[(0, 3), (0, 29)]),
            T.compile_world(two, T.SIMPLE_GRAPH)]


@pytest.mark.parametrize("complexity", [None, 0.3])
def test_episode_set_is_reproducible_inside_the_prefix_and_reachable(complexity):
    for world in _worlds():
        task, start = EV.episode_set(world, 7, seed=3, complexity=complexity)
        t2, s2 = EV.episode_set(world, 7, seed=3, complexity=complexity)
        assert task.dtype == np.int32 and start.dtype == np.int32
        assert np.array_equal(task, t2) and np.array_equal(start, s2)
        t3, s3 = EV.episode_set(world, 7, seed=4, complexity=complexity)
        assert not np.array_equal(s3, start)
        pre = world.prefixes(complexity)
        for ti, t in enumerate(world.tasks):
            mine = start[task == ti] - int(world.scene_base[t.scene])
            dist, _ = T.optimal_policy_table(world, ti)
            pool = [s for s in t.cand_state[:pre[ti]] if dist[s] >= 1]
            assert len(mine) == min(7, len(pool)) and len(set(mine.tolist())) == len(mine), ti
            assert set(mine.tolist()) <= set(int(s) for s in pool), ti
            assert (dist[mine] >= 1).all(), ti
        # per_task=None: every reachable candidate once
        ta, sa = EV.episode_set(world, None, seed=0, complexity=complexity)
        for ti, t in enumerate(world.tasks):
            dist, _ = T.optimal_policy_table(world, ti)
            want = sorted(int(s) for s in t.cand_state[:pre[ti]] if dist[s] >= 1)
            assert sorted((sa[ta == ti] - int(world.scene_base[t.scene])).tolist()) == want, ti


def test_episode_set_drops_the_thor_cached_unreachable_candidates():
    """thor-cached candidate lists keep unreachable cells at rotation difference 2 ("distance" 1, tables.build_task);
    the set drops them."""
    thor = H.scenes.GridScene(EL.HAND_MAZE, [], True, (84, 84), ("rgb",))     # (2,0), (3,0): cut off from the goal
    world = T.compile_world([thor], T.THOR_CACHED, tasks=[(0, thor.state_index(EL.HAND_GOAL))])
    dist, _ = T.optimal_policy_table(world, 0)
    cands = world.tasks[0].cand_state
    assert (dist[cands] < 1).any()
    _, start = EV.episode_set(world, None, seed=0)
    assert len(start) == int((dist[cands] >= 1).sum()) and (dist[start] >= 1).all()


def test_evaluate_episodes_needs_a_way_to_end_episodes():
    env = types.SimpleNamespace(max_episode_steps=0)
    with pytest.raises(ValueError, match="TimeLimit"):
        EV.evaluate_episodes(env, None, [0], [1])
