"""Single-environment surface of the reference classes (gym.Env duck type) over the CUDA path.

``reset() -> obs``, ``step(a) -> (obs, reward, done, info)`` WITHOUT auto-reset (the reference envs
never reset themselves: gym_graph/graph.py:67-79, cached.py:74-99), ``set_complexity(c)``,
``unwrapped``, ``render(mode='rgbarray')``, fields ``state`` and ``goal`` as reference tuples
(gym_graph/graph.py:39-54,81-93).  It is a 1-env ``GraphVecEnv`` with ``auto_reset=False``; useful for
evaluation loops and for the keyboard / browser tools, not for throughput.
"""
import numpy as np

from .vec_env import GraphVecEnv


class GraphEnv:
    metadata = {"render.modes": ["rgbarray"]}

    def __init__(self, world, *, task_range=None, max_episode_steps=None, numpy_obs=True, **kwargs):
        """task_range: (lo, count) into world.tasks this env draws its goal from on reset (default all).
        max_episode_steps: None reproduces the bare class (no TimeLimit); gym.make adds 100 / 900."""
        tasks = np.array([[0, len(world.tasks)] if task_range is None else list(task_range)], np.int32)
        kwargs.setdefault("unreal_wrapper", False)
        kwargs.setdefault("episode_info", False)      # the bare classes have no RewardCollector
        self._vec = GraphVecEnv(world, 1, env_tasks=tasks, auto_reset=False, max_episode_steps=max_episode_steps or 0,
                                **kwargs)
        self.numpy_obs = numpy_obs
        self.observation_space = self._vec.observation_space
        self.action_space = self._vec.action_space
        self.world = world

    @property
    def unwrapped(self):
        return self

    def _one(self, obs):
        conv = (lambda t: t[0].cpu().numpy()) if self.numpy_obs else (lambda t: t[0])
        if isinstance(obs, tuple):
            return tuple(self._one_leaf(o, conv) for o in obs)
        if isinstance(obs, dict):
            return {k: conv(v) for k, v in obs.items()}
        return conv(obs)

    @staticmethod
    def _one_leaf(o, conv):
        return tuple(conv(x) for x in o) if isinstance(o, tuple) else conv(o)

    def set_complexity(self, complexity=None):
        self._vec.set_complexity(complexity)

    def set_reward_progress(self, coef):
        """GraphVecEnv.set_reward_progress (also the ``reward_progress`` keyword of the constructor)."""
        self._vec.set_reward_progress(coef)

    def reset(self):
        return self._one(self._vec.reset())

    def step(self, action):
        obs, r, d, infos = self._vec.step(np.array([-1 if action is None else int(action)], np.int32))
        return self._one(obs), float(r[0]), bool(d[0]), infos[0]

    @property
    def state(self):
        return self._vec.states()[0]

    @property
    def goal(self):
        return self.world.state_tuple(int(self._vec.goal.cpu()[0]))

    def render(self, mode="rgbarray"):
        if mode != "rgbarray":
            raise Exception("Render mode %s is not supported" % mode)     # gym_graph/graph.py:93
        from .vec_env import gather_plane
        return gather_plane(self._vec.dw, "rgb", self._vec.obs_state)[0].cpu().numpy()

    def close(self):
        self._vec.close()
