"""Test-side restatement of the fixed episode list (``GraphVecEnv.set_episodes``, ``vn_episodes_t``) and the cases its
tests share.

The reference has no episode list, so the oracle classes under oracle/ stay as they are.  ``EpisodeList`` wraps one of
them OUTERMOST - above RewardCollector and TimeLimit, so it sees what the VecEnv worker sees - and replaces the base
env's reset source with the deal: the env with global id ``g`` runs listed episodes ``g, g + stride, g + 2 * stride,
...`` (while they exist), each started by the reset that follows the previous one's end, then falls back to its
ordinary source.  The ordinary source is the oracle's own restatement of the device's Philox stream
(oracle/vec.PhiloxResetSource), whose epoch - like the device's - also counts the listed resets.  When a listed episode
ends, the wrapper records its length and return (RewardCollector's ``info['episode']``), win, truncation
(``info['TimeLimit.truncated'] is True``) and final state."""
import numpy as np

from oracle import envs as oenvs
from oracle import graph_util as gu
from oracle import vec as ovec


class EpisodeList:
    """``env`` = the oracle stack of one env (RewardCollector(TimeLimit(...))), ``base`` = the env class at its bottom,
    whose ``reset_source`` is replaced.  ``results`` is a dict shared by all envs of a batch: listed episode id ->
    dict(length, ret, win, truncated, final_state).  ``start_of(global state)`` gives what the base env's reset source
    returns as a start, ``state_of(base)`` the base env's current GLOBAL state."""

    def __init__(self, env, base, task, start, g, stride, results, start_of, state_of):
        self.env, self.base = env, base
        self.task, self.start = np.asarray(task), np.asarray(start)
        self.g, self.stride, self.results = int(g), int(stride), results
        self.start_of, self.state_of = start_of, state_of
        self.ordinary = base.reset_source
        base.reset_source = self._draw
        self.cursor = -1
        self._ended = False       # the next reset is the auto-reset after an episode end (else: the list restarts)

    def __getattr__(self, name):
        return getattr(self.env, name)

    def _draw(self):
        j = self.g if not self._ended else (self.cursor + self.stride if self.cursor >= 0 else -1)
        self.cursor = j if 0 <= j < len(self.task) else -1
        if self.cursor < 0:
            return self.ordinary()
        if hasattr(self.ordinary, "epoch"):
            self.ordinary.epoch += 1      # every reset advances the env's epoch, listed or not
        return int(self.task[j]), self.start_of(int(self.start[j]))

    def reset(self):
        obs = self.env.reset()
        self._ended = False
        return obs

    def step(self, action):
        obs, reward, done, info = self.env.step(action)
        if done:
            if self.cursor >= 0:
                trunc = info.get("TimeLimit.truncated") is True
                self.results[self.cursor] = dict(length=int(info["episode"]["l"]), ret=np.float32(info["episode"]["r"]),
                                                 win=not trunc, truncated=trunc, final_state=int(self.state_of(self.base)))
            self._ended = True
        return obs, reward, done, info


# --------------------------------------------------------------------------- the hand-worked case
# The oriented 4 x 4 maze of tests/progress_reward.py (a corridor (0,0) .. (0,3), (1,3) .. (3,3); goal (2,3) facing
# r = 0), TimeLimit 2, rewards (goal, step, collision) = (1.0, -0.125, -0.5), every env always moves forward (action 0).
# From (1,3,0) the goal is one step away; from (0,3,0) two - reached ON the limit step, so TimeLimit reports
# truncated = False (code 2) and the episode is a win; from (3,3,0) forward runs off the grid (two collisions); from
# (0,0,1) the env walks (0,1,1), (0,2,1) and is cut off.  3 envs, 7 episodes: env 0 runs 0, 3, 6, env 1 runs 1, 4,
# env 2 runs 2, 5.
HAND_MAZE = np.array([[1, 1, 1, 1],
                      [0, 0, 0, 1],
                      [1, 0, 0, 1],
                      [1, 0, 0, 1]], bool)
HAND_GOAL = (2, 3, 0)
HAND_REWARDS = (1.0, -0.125, -0.5)
HAND_LIMIT = 2
HAND_STARTS = [(1, 3, 0), (0, 3, 0), (3, 3, 0), (0, 0, 1), (3, 3, 0), (1, 3, 0), (0, 3, 0)]
# listed episode -> (length, return, win, truncated, final state)
HAND_RESULTS = [(1, 1.0, 1, 0, (2, 3, 0)),
                (2, 0.875, 1, 0, (2, 3, 0)),
                (2, -1.0, 0, 1, (3, 3, 0)),
                (2, -0.25, 0, 1, (0, 2, 1)),
                (2, -1.0, 0, 1, (3, 3, 0)),
                (1, 1.0, 1, 0, (2, 3, 0)),
                (2, 0.875, 1, 0, (2, 3, 0))]
# step (1-based) on which each env ends its last listed episode; its resets so far (the epoch of its first Philox draw)
HAND_LAST_STEP = [5, 4, 3]
HAND_EPOCH_AFTER = [3, 2, 2]


# --------------------------------------------------------------------------- oracle stacks of the parity cases
def oracle_case(kind, world, scenes, seed, limit, rewards, coef=0.0):
    """make(g, task, start, results) -> (EpisodeList stack of the env with global id g, base env): the oracle env class
    of ``kind`` driven by the device's Philox stream (env_tasks (0, n_tasks) for every env, no curriculum), with the
    list deal on top and, for coef != 0, the geodesic-progress restatement innermost."""
    import progress_reward as P
    nt = len(world.tasks)
    base_of = lambda t: int(world.scene_base[world.tasks[t].scene])
    if kind == "oriented":
        scene = scenes[0]
        osc = oenvs.OracleScene(scene)
        goals = list(scene.goals)
        cands = [gu.initial_state_candidates(scene.maze, osc.graph, osc.optimal_actions, gl) for gl in goals]
        graph = P.oriented_graph(scene.maze)

        def base_env(g):
            e = oenvs.GymGraphEnv(osc, goals=goals, rewards=rewards)
            e.reset_source = ovec.PhiloxResetSource(seed, g, cands, lambda t: None, False)
            return e, (P.ProgressReward(e, coef, graph) if coef else e)
        start_of = lambda s: world.state_tuple(s)
        state_of = lambda e: scene.state_index(e.state)
    elif kind == "multi_scene":
        oscs = [oenvs.OracleScene(s) for s in scenes]
        cands = [gu.initial_position_candidates(s.maze, o.graph, tuple(s.goals[0])) for s, o in zip(scenes, oscs)]
        graphs = [P.compass_graph(s.maze) for s in scenes]

        def base_env(g):
            e = oenvs.MultipleGraphEnv(oscs, rewards=rewards)
            e.reset_source = ovec.PhiloxResetSource(seed, g, cands, lambda t: None, True)
            return e, (P.ProgressReward(e, coef, graphs, scene_of=lambda e: e.graph_number) if coef else e)
        start_of = lambda s: world.state_tuple(s)
        state_of = lambda e: scenes[e.graph_number].state_index(e.state) + int(world.scene_base[e.graph_number])
    else:
        scene = scenes[0]
        dist, _ = gu.compute_shortest_path_data(scene.maze)
        _, h5graph, spd = gu.h5_tables(scene.maze, dist)
        goals = [int(t.goal_state) for t in world.tasks]
        cands = [(list(np.nonzero(spd[:, g] > 0)[0]), spd[np.nonzero(spd[:, g] > 0)[0], g]) for g in goals]
        graph = (list(range(scene.n_states)), lambda s: [int(n) for n in h5graph[s] if n != -1])

        def base_env(g):
            e = oenvs.ThorCachedEnv(h5graph, np.zeros((scene.n_states, 1), np.uint8), spd, tasks=goals)
            e.reset_source = ovec.PhiloxResetSource(seed, g, cands, lambda t: None, False)
            return e, (P.ProgressReward(e, coef, graph, goal_of=lambda e: e._current_goal_idx,
                                        state_of=lambda e: e._current_state_idx) if coef else e)
        start_of = lambda s: s - base_of(0)
        state_of = lambda e: e._current_state_idx
    assert all(len(c[0]) for c in cands) and nt == len(cands)

    def make(g, task, start, stride, results):
        base, inner = base_env(g)
        stack = ovec.RewardCollector(ovec.TimeLimit(inner, limit))
        return EpisodeList(stack, base, task, start, g, stride, results, start_of, state_of), base
    return make
