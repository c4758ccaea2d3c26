"""Test-side restatement of the geodesic-progress reward (``GraphVecEnv(reward_progress=...)``,
``vn_rules_t.reward_progress``) and the hand-worked scenarios its tests share.

The reference has no such reward, so the oracle classes under oracle/ - pinned to the reference by the goldens - stay as
they are.  ``ProgressReward`` wraps one of them INNERMOST, below TimeLimit, RewardCollector and the VecEnv's
last_action_reward, so every consumer of the reward sees the shaped value, as every output of the device step does.  Its
distances come from a breadth-first search over the oracle env's own transition rule (oracle/graph_util.py), not from
the product's tables, and it adds the term in the fp32 operation order of the kernel:
``float32(base) + float32(coef) * float32(d_prev - d_next)``, two roundings, no fused multiply-add."""
from collections import deque

import numpy as np

from oracle import graph_util as gu


def oriented_graph(maze):
    """State graph of the oriented envs (graph/util.py:15-25): (x, y, r) -> the states its four actions lead to;
    an action into a wall has no edge."""
    states = [p + (r,) for p in gu.enumerate_positions(maze) for r in range(4)]
    return states, lambda s: [n for n in (gu.step(s, a) for a in range(4)) if gu.is_valid_state(maze, n)]


def compass_graph(maze):
    """State graph of SimpleGraphEnv (graph/env.py:117-133): a cell -> its free 4-neighbours."""
    def succ(s):
        out = []
        for a in range(4):
            c = gu.direction_to_change(a)
            n = (s[0] + c[0], s[1] + c[1])
            if gu.is_valid_state(maze, n):
                out.append(n)
        return out
    return list(gu.enumerate_positions(maze)), succ


def distances_to(graph, goals):
    """{state: fewest actions to reach any of ``goals``}; a state that is missing cannot reach them."""
    states, succ = graph
    rev = {}
    for s in states:
        for n in succ(s):
            if n != s:
                rev.setdefault(n, []).append(s)
    dist = {g: 0 for g in goals}
    q = deque(goals)
    while q:
        d = q.popleft()
        for s in rev.get(d, ()):
            if s not in dist:
                dist[s] = dist[d] + 1
                q.append(s)
    return dist


class ProgressReward:
    """reward = base + coef * (d(state before the step) - d(state after it)), 0 where either distance is unknown; ``d``
    counts actions to the goal of the env's current episode (``goal_of(env)``) on ``graph`` - or on ``graph[scene_of(env)]``
    for an env that changes scene on reset (MultipleGraphEnv)."""

    def __init__(self, env, coef, graph, goal_of=lambda e: tuple(e.goal), state_of=lambda e: e.state,
                 scene_of=None):
        self.env, self.coef = env, np.float32(coef)
        self._graph, self._goal_of, self._state_of, self._scene_of = graph, goal_of, state_of, scene_of
        self._dist = {}

    def __getattr__(self, name):
        return getattr(self.env, name)

    def distance(self, state):
        k = (self._scene_of(self.env) if self._scene_of else None, self._goal_of(self.env))
        if k not in self._dist:
            self._dist[k] = distances_to(self._graph[k[0]] if self._scene_of else self._graph, [k[1]])
        return self._dist[k].get(state, -1)

    def reset(self):
        return self.env.reset()

    def step(self, action):
        if self.coef == 0:          # off: the base reward untouched, -0.0 included
            return self.env.step(action)
        d_prev = self.distance(self._state_of(self.env))
        obs, reward, done, info = self.env.step(action)
        d_next = self.distance(self._state_of(self.env))
        delta = 0 if d_prev < 0 or d_next < 0 else d_prev - d_next
        return obs, float(np.float32(reward) + self.coef * np.float32(delta)), done, info


# --------------------------------------------------------------------------- hand-worked scenarios
# Rewards (goal, step, collision) and coefficient are dyadic, so every expected reward below is exact in float32.
REWARDS = (1.0, -0.125, -0.5)
COEF = 0.25

# Oriented 4 x 4 maze (gym_graph actions 0 forward, 1 rotate +, 2 back, 3 rotate -; direction r moves by
# (1,0) (0,1) (-1,0) (0,-1)): a corridor (0,0) .. (0,3), (1,3) .. (3,3) and the cells (2,0), (3,0), which no path joins
# to it.  Goal (2,3) facing r = 0.  Distances used below: (0,0,1) 6, (0,1,1) 5, (0,2,1) 4, (0,2,0) 5, (0,3,1) 3,
# (0,3,0) 2, (1,3,0) 1, (3,3,0) 1, (3,3,1) 2; every state of (2,0), (3,0) is unreachable (-1).
ORIENTED_MAZE = np.array([[1, 1, 1, 1],
                          [0, 0, 0, 1],
                          [1, 0, 0, 1],
                          [1, 0, 0, 1]], bool)
ORIENTED_GOAL = (2, 3, 0)
ORIENTED_SCENARIOS = [
    # (max_episode_steps, reset starts, actions, expected rewards, dones)
    (20, [(0, 1, 1), (3, 3, 0), (0, 0, 1)],
     [0, 2, 0, 0, 0, 3, 0, 0, 1, 3, 2],
     # toward 5->4, away 4->5, toward, toward 4->3, collision (state kept), turn 3->2, 2->1, goal 1->0 = 1 + 0.25,
     # new episode from (3,3,0): turn away 1->2, back 2->1, goal from behind
     [0.125, -0.375, 0.125, 0.125, -0.5, 0.125, 0.125, 1.25, -0.375, 0.125, 1.25],
     [0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 1]),
    (3, [(3, 0, 2), (0, 2, 1), (0, 0, 1), (3, 0, 2)],
     [0, 0, 2, 0, 2, 3, 0, 0, 0, 1, 1],
     # unreachable start: move, collision, move (no shaping), truncated; from (0,2,1): toward 4->3, away 3->4,
     # turn away 4->5 on the truncating step (the terminal state counts, not the next start); from (0,0,1): 6->5 uses
     # the new start's distance, 5->4, 4->3 truncated; unreachable start again
     [-0.125, -0.5, -0.125, 0.125, -0.375, -0.375, 0.125, 0.125, 0.125, -0.125, -0.125],
     [0, 0, 1, 0, 0, 1, 0, 0, 1, 0, 0]),
]

# Un-oriented 4 x 4 maze (SimpleGraphEnv compass actions 0 (1,0), 1 (0,1), 2 (-1,0), 3 (0,-1); -1 = no-op with reward
# 0.0).  Goal (2,2).  Distances: (0,1) 5, (0,0) 4, (1,0) 3, (2,0) 2, (2,1) 1, (3,2) 1; (0,3), (1,3) are unreachable.
COMPASS_MAZE = np.array([[1, 1, 0, 1],
                         [1, 0, 0, 1],
                         [1, 1, 1, 0],
                         [0, 0, 1, 0]], bool)
COMPASS_GOAL = (2, 2)
COMPASS_SCENARIOS = [
    (5, [(0, 1), (2, 0), (0, 3)],
     [3, 1, -1, 0, 3, 1, 1, 0, -1, 1, 2],
     # toward 5->4, away 4->5, no-op, collision, toward 5->4 truncated; from (2,0): 2->1, goal; unreachable start:
     # move, no-op, collision (off the grid), move
     [0.125, -0.375, 0.0, -0.5, 0.125, 0.125, 1.25, -0.125, 0.0, -0.5, -0.125],
     [0, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0]),
]

# info['episode']['r'] of every finished episode, in order, per scenario
EPISODE_RETURNS = {
    ("oriented", 0): [1.0, 1.0],
    ("oriented", 1): [-0.75, -0.625, 0.375],
    ("compass", 0): [-0.625, 1.375],
}
