"""Drop-in vectorised environment: the reference's gym ``Env`` / baselines-style ``VecEnv`` surface
over the CUDA hot path.

Reference surface kept (SURVEY.md section 8(b)):
  * ``reset() -> obs``; ``step(actions) -> (obs, rewards, dones, infos)``; ``step_async`` /
    ``step_wait``; ``close()``; ``num_envs``; ``observation_space``; ``action_space.n == 4``
    (deep_rl SubprocVecEnv as used at experiments/thor_cached_auxiliary.py:58-71);
  * ``call_unwrapped('set_complexity', c)`` and ``set_hardness`` (thor_cached_auxiliary.py:68-70);
  * observation layouts: ``((rgb, goal_rgb, depth, seg, goal_seg), last_action_reward)``
    (gym_graph/graph.py:117-120 + UnrealEnvBaseWrapper), a bare frame (gym_graph/graph.py:56-58),
    ``(obs, goal)`` (gym_ai2thor/envs/cached.py:53-57) or ``{'image','goal'}`` (gym_thor_cached.py:89-92);
  * ``info`` keys ``state``, ``win`` (gym_graph/graph.py:72-79), ``episode`` (RewardCollector),
    ``TimeLimit.truncated`` (gym TimeLimit).

What changes: observations are ``uint8`` CUDA tensors (views of persistent batch buffers that the
next ``step`` overwrites) instead of pickled float32 numpy arrays; the goal leaves are rewritten only
for envs that reset; all envs advance in two kernel launches (one for small batches), and the row of an env whose state did not
change is not copied again.
"""
import ctypes as C
import weakref

import numpy as np
import torch

from . import lib as L
from . import spaces
from .store import DeviceWorld
from .tables import World, Family

try:        # raw handle of torch's current stream without building a torch.cuda.Stream object (0.2 us instead of 2 us)
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:      # pragma: no cover - older / newer torch without the private helper
    def _raw_stream(index):
        return torch.cuda.current_stream(index).cuda_stream

#: named observation layouts -> leaves.  A leaf is a store plane ("rgb", "depth", "segmentation") or the
#: same plane of the goal state ("goal_rgb", "goal_segmentation").
OBS_LAYOUTS = {
    # GoalGymGraphAuxiliaryEnv.observe, environments/gym_graph/graph.py:117-120
    "aux5": ("rgb", "goal_rgb", "depth", "segmentation", "goal_segmentation"),
    # OrientedGraphEnv.observe, environments/gym_graph/graph.py:56-58 (also graph/env.py envs)
    "frame": "rgb",
    # THORDiscreteCachedEnv, environments/gym_ai2thor/envs/cached.py:53-57
    "pair": ("rgb", "goal_rgb"),
    # THORCachedEnv.process, environments/gym_thor_cached.py:89-92
    "dict": {"image": "rgb", "goal": "goal_rgb"},
    # ThorGridWorld.render of the third-person variant, graph/thor_graph.py:15-36 (modes rgb, depth, segmentation)
    "thor6": ("rgb", "depth", "segmentation", "tp_rgb", "tp_depth", "tp_segmentation"),
    # BASELINE.json configs[1]: "84x84 RGB+depth+goal"
    "rgbd_goal": ("rgb", "goal_rgb", "depth"),
}


def resolve_layout(layout):
    if isinstance(layout, str):
        if layout not in OBS_LAYOUTS:
            raise ValueError("obs_layout must be one of %s or a tuple / dict of leaves" % (sorted(OBS_LAYOUTS),))
        return OBS_LAYOUTS[layout]
    return layout


def build_spaces(store_layout, obs_layout, scaled_float=False, unreal_wrapper=True, n_actions=4):
    """(observation_space, action_space) of a GraphVecEnv - no device needed.  What the reference's trainer reads:
    ``observation_space.spaces[0].spaces[0].shape[0]`` = channels of the first leaf after TransposeImage and
    ``action_space.n`` (experiments/thor_cached_auxiliary.py:55).  uint8 leaves are HWC as the raw env emits them
    (gym_graph/graph.py:26-31,99-104); with scaled_float they are float32 CHW in [0, 1], the spaces the wrapper stack
    TransposeImage + ScaledFloatFrame leaves behind (:61-62); unreal_wrapper appends the last_action_reward Box (:63)."""
    lay = store_layout
    h, w = lay.frame_hw
    leaves = resolve_layout(obs_layout)

    def frame(leaf):
        p = leaf[5:] if leaf.startswith("goal_") else leaf
        c = lay.channels[lay.planes.index(p)]
        if scaled_float:
            return spaces.Box(0.0, 1.0, (c, h, w), np.float32)
        return spaces.Box(0, 255, (h, w, c), np.uint8)

    if isinstance(leaves, dict):
        inner = spaces.Dict({k: frame(v) for k, v in leaves.items()})
    elif isinstance(leaves, tuple):
        inner = spaces.Tuple(tuple(frame(v) for v in leaves))
    else:
        inner = frame(leaves)
    obs = spaces.Tuple((inner, spaces.Box(0.0, 1.0, (n_actions + 1,), np.float32))) if unreal_wrapper else inner
    return obs, spaces.Discrete(n_actions)


def shard_range(num_envs_total, rank=0, world_size=1):
    """Envs [lo, hi) owned by ``rank``: contiguous, sizes differ by at most one."""
    base, rem = divmod(num_envs_total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class LazyInfos:
    """``infos`` of one step.  Behaves like the tuple of dicts the reference VecEnv returns, built from
    the packed per-env info arrays only when an element is read (host_outputs=False: the arrays are
    fetched from the device on first access and are valid until the next step)."""

    def __init__(self, env, arrays, noop, in_place=False):
        self._env, self._a, self._noop = env, arrays, noop
        self._in_place = in_place      # `arrays` is a pinned host pack of the env, read in place (no copy was taken)

    def __len__(self):
        return self._env.num_envs

    def _snapshot(self):
        """The env is about to reuse the pinned host pack this object still reads in place: take a private copy."""
        if self._in_place:
            if isinstance(self._a, np.ndarray):
                self._a = self._a.copy()
            elif isinstance(self._a, dict):
                self._a = {k: v.copy() for k, v in self._a.items()}
            self._in_place = False

    def _host(self):
        if callable(self._a):
            self._a = self._a()
        if isinstance(self._a, np.ndarray):          # the raw host pack: split it on first use
            self._a = self._env._unpack(self._a)
        if torch.is_tensor(self._noop):
            self._noop = self._noop.cpu().numpy()
        return self._a

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        h = self._host()
        env = self._env
        info = {}
        graph_family = env.family.name != "thor_cached"        # cached.py:99 returns an empty dict
        if graph_family and not (env.family.noop_action and self._noop is not None and self._noop[i]):
            info["state"] = env.world.state_tuple(int(h["info_state"][i]))     # gym_graph/graph.py:72-79
        if graph_family and h["win"][i]:
            info["win"] = True
        if h["truncated"][i]:                                   # gym TimeLimit: key exists only at the limit
            info["TimeLimit.truncated"] = bool(h["truncated"][i] == 1)
        if env.episode_info and h["done"][i]:                   # RewardCollector
            info["episode"] = dict(r=float(h["episode_return"][i]), l=int(h["episode_length"][i]))
        return info

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class CapturedSteps:
    """What ``GraphVecEnv.capture_steps`` returns: ``replay()`` launches the captured CUDA graph (``.graph`` is the
    ``torch.cuda.CUDAGraph``) and tells the env that the next eager step follows a replay."""

    def __init__(self, env, graph):
        self.env, self.graph = env, graph

    def replay(self):
        self.graph.replay()
        self.env._serial_next = True


class GraphVecEnv:
    def __init__(self, world, num_envs, *, device="cuda", seed=0, max_episode_steps=900, rewards=(1.0, 0.0, 0.0),
                 obs_layout="aux5", unreal_wrapper=True, env_tasks=None, auto_reset=True, rank=0, world_size=1,
                 gather="auto", inject=None, host_outputs=True, device_world=None, scaled_float=False,
                 episode_info=True, skip_unchanged=True, numpy_obs=False, reward_progress=0.0):
        """
        world            tables.World (compiled scenes) - or pass a ready ``device_world``
        num_envs         TOTAL number of envs of the job; this process owns shard_range(num_envs, rank, world_size)
        env_tasks        per GLOBAL env (lo, count) range into world.tasks the env draws its task from on reset
                         (default: tasks dealt round-robin, one per env - see _default_env_tasks)
        inject           optional (task [n_local, R] int32, start [n_local, R] int32 GLOBAL states) reset stream
        host_outputs     rewards / dones as numpy (reference behaviour) or as CUDA tensors
        scaled_float     observation leaves as float32 CHW in [0, 1] - what TransposeImage + ScaledFloatFrame
                         (experiments/thor_cached_auxiliary.py:61-62) hand to the model - in persistent batches filled
                         by one fused gather/convert kernel per leaf straight from the store (no uint8 batch is
                         written; rows that did not change / goal rows of envs that did not reset are skipped)
        gather           "auto" | "ldg" | "bulk" | "fused" | "persistent" (include/vn_b200.h VN_GATHER_*); "auto" runs the
                         whole step as ONE fused launch for batches of one wave of CTAs; beyond that "persistent" is one
                         launch of a persistent grid (CTAs own envs: lanes step them, lane 0 copies their records) and
                         "bulk" / "ldg" are scalar kernel + gather kernel
        numpy_obs        return the observation leaves (and last_action_reward) as numpy arrays, like the reference's
                         SubprocVecEnv, for a trainer that cannot take CUDA tensors: one device-to-host copy of the whole
                         batch per step (PCIe-bound).  True: views of two alternating sets of pinned buffers, valid
                         until the step after next; "copy": private arrays (one more host copy of the batch)
        skip_unchanged   the observation leaves are views of persistent batch buffers owned by this object, so the
                         row of an env whose state did not change (collision, no-op) is not copied again
                         (VN_STEP_SKIP_UNCHANGED).  Pass False if the returned observation tensors are modified in
                         place between steps.
        reward_progress  dense geodesic-progress reward, NOT part of the reference (see set_reward_progress); 0 = off
        """
        self.dw = device_world if device_world is not None else DeviceWorld(world, device)
        self.world: World = self.dw.world
        self.family: Family = self.world.family
        self.lib = self.dw.lib
        self.device = self.dw.device
        self.rank, self.world_size = rank, world_size
        self.num_envs_total = num_envs
        lo, hi = shard_range(num_envs, rank, world_size)
        self.env_lo, self.num_envs = lo, hi - lo
        n = self.num_envs
        self.max_episode_steps = int(max_episode_steps or 0)
        self.obs_layout = obs_layout
        self.unreal_wrapper = unreal_wrapper
        self.host_outputs = host_outputs
        self.scaled_float = scaled_float
        self.numpy_obs = numpy_obs
        self._host_stage = {}
        self.episode_info = episode_info     # RewardCollector's info['episode'] (create_envs wraps with it, :60)
        self.n_actions = 4
        self.gather = {"auto": L.GATHER_AUTO, "ldg": L.GATHER_LDG, "bulk": L.GATHER_BULK,
                       "fused": L.GATHER_FUSED, "persistent": L.GATHER_PERSISTENT}[gather]
        self._step_flags = L.STEP_SKIP_UNCHANGED if skip_unchanged else 0
        lay = self.world.layout
        self.leaves = resolve_layout(obs_layout)
        names = self.leaves.values() if isinstance(self.leaves, dict) else \
            (self.leaves if isinstance(self.leaves, tuple) else (self.leaves,))
        self.obs_planes = tuple(dict.fromkeys(x for x in names if not x.startswith("goal_")))
        self.goal_planes = tuple(dict.fromkeys(x[5:] for x in names if x.startswith("goal_")))
        for p in self.obs_planes + self.goal_planes:
            if p not in lay.planes:
                raise ValueError("obs_layout %r needs plane %r in the store (has %s)" % (obs_layout, p, lay.planes))

        tasks = self._default_env_tasks(num_envs) if env_tasks is None else np.asarray(env_tasks, np.int32)
        if tasks.shape != (num_envs, 2):
            raise ValueError("env_tasks must be [num_envs, 2] (lo, count)")
        if (tasks[:, 1] < 1).any() or (tasks[:, 0] < 0).any() or (tasks.sum(1) > len(self.world.tasks)).any():
            raise ValueError("env_tasks ranges fall outside the task table")
        tasks = tasks[lo:hi]

        h, w = lay.frame_hw
        with torch.cuda.device(self.device):
            i32 = lambda: torch.zeros(n, dtype=torch.int32, device=self.device)
            self.state, self.goal, self.task, self.elapsed, self.ep_length = i32(), i32(), i32(), i32(), i32()
            self.epoch = i32()      # uint32 on the device side, same bits
            self.ep_return = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.task_lo = torch.from_numpy(np.ascontiguousarray(tasks[:, 0])).to(self.device)
            self.task_cnt = torch.from_numpy(np.ascontiguousarray(tasks[:, 1])).to(self.device)
            # per-env scalars the host reads every step, packed so ONE D2H copy returns them:
            # reward f32 | episode_return f32 | episode_length i32 | info_state i32 | done | truncated | win | did_reset
            self._pack = torch.zeros(n * 20, dtype=torch.uint8, device=self.device)
            self.reward = self._pack[:4 * n].view(torch.float32)
            self.episode_return = self._pack[4 * n:8 * n].view(torch.float32)
            self.episode_length = self._pack[8 * n:12 * n].view(torch.int32)
            self.info_state = self._pack[12 * n:16 * n].view(torch.int32)
            self.done = self._pack[16 * n:17 * n]
            self.truncated = self._pack[17 * n:18 * n]
            self.win = self._pack[18 * n:19 * n]
            self.did_reset = self._pack[19 * n:20 * n]
            self.lar = torch.zeros((n, self.n_actions + 1), dtype=torch.float32, device=self.device)
            self.obs_state = i32()
            self.stats = torch.zeros(L.VN_N_STATS, dtype=torch.int64, device=self.device)
            self.actions_dev = i32()
            self._sched = torch.zeros(4, dtype=torch.int32, device=self.device)     # scheduler / completion counters
            self._gather_desc = torch.zeros((2, max(n, 1), 2), dtype=torch.int32, device=self.device)
            if scaled_float:
                # float mode: no uint8 batch at all - persistent float32 CHW batches, one per leaf, converted straight
                # from the store after every step (only rows that changed; goal leaves only for envs that reset)
                self.obs_buf, self.goal_buf = {}, {}
                chw = lambda p: (n, lay.channels[lay.planes.index(p)], h, w)
                self.float_buf = {("goal_" + p if g else p): torch.zeros(chw(p), dtype=torch.float32, device=self.device)
                                  for g, ps in ((False, self.obs_planes), (True, self.goal_planes)) for p in ps}
            else:
                self.obs_buf = {p: lay.batch(p, n, self.device) for p in self.obs_planes}
                self.goal_buf = {p: lay.batch(p, n, self.device) for p in self.goal_planes}
                self.float_buf = {}
            # two host packs used alternately: rewards / dones are copied out of the pinned block every step, the rest
            # (what `infos` is built from) is read in place, lazily, and stays valid until the step after next
            self._pack_hosts = [torch.zeros(n * 20, dtype=torch.uint8).pin_memory() for _ in range(2)]
            self._pack_host = self._pack_hosts[0]
            self._actions_host = torch.zeros(n, dtype=torch.int32).pin_memory()
        self._inject_keep = None
        self._c_inject = None
        if inject is not None:
            self.set_inject(*inject)

        self._c_envs = L.Envs(n, lo, *(t.data_ptr() for t in (self.state, self.goal, self.task, self.elapsed,
                                                              self.epoch, self.ep_return, self.ep_length,
                                                              self.task_lo, self.task_cnt)))
        fam = self.family
        flags = 0
        flags |= L.RULE_COLLISION_SKIPS_GOAL if fam.collision_skips_goal else 0
        flags |= L.RULE_NEG_STEP_REWARD if fam.neg_step_reward else 0
        flags |= L.RULE_COLLISION_OVERRIDES if fam.collision_overrides else 0
        flags |= L.RULE_TERM_PREV_OBS if fam.term_prev_obs else 0
        flags |= L.RULE_TWO_LEVEL if fam.two_level_sampling else 0
        flags |= L.RULE_NOOP_ACTION if fam.noop_action else 0
        flags |= L.RULE_AUTO_RESET if auto_reset else 0
        self._c_rules = L.Rules(float(rewards[0]), float(rewards[1]), float(rewards[2]), self.max_episode_steps,
                                fam.goal_compare, flags, self.n_actions, 0.0, C.c_uint64(seed & (2 ** 64 - 1)))
        self.reward_progress = 0.0
        self.set_reward_progress(reward_progress)
        out = L.StepOut()
        for i, p in enumerate(lay.planes):
            out.obs[i] = self.obs_buf[p].data_ptr() if p in self.obs_buf else None
            out.goal_obs[i] = self.goal_buf[p].data_ptr() if p in self.goal_buf else None
        out.reward, out.done, out.truncated = self.reward.data_ptr(), self.done.data_ptr(), self.truncated.data_ptr()
        out.win, out.did_reset = self.win.data_ptr(), self.did_reset.data_ptr()
        out.last_action_reward = self.lar.data_ptr()
        out.episode_return, out.episode_length = self.episode_return.data_ptr(), self.episode_length.data_ptr()
        out.info_state, out.obs_state, out.stats = self.info_state.data_ptr(), self.obs_state.data_ptr(), self.stats.data_ptr()
        out.sched = self._sched.data_ptr()
        out.gather_desc = self._gather_desc.data_ptr()
        self._c_out = out
        # same outputs + the mapped pinned host mirror of the per-env scalars (host-actions path)
        out_h = L.StepOut()
        C.memmove(C.byref(out_h), C.byref(out), C.sizeof(L.StepOut))
        out_h.host_pack = self._pack_host.data_ptr()
        # one sequence word per thread block of the scalar kernel, published once that block's scalars are on the host
        self._seq_words = self.lib.vn_env_host_seq_words(C.byref(self.dw.store), C.byref(self._c_envs), C.byref(out_h),
                                                         self.gather)
        if self._seq_words <= 0:
            L.check(self._seq_words)
        self._seq_host = torch.zeros(self._seq_words, dtype=torch.int32).pin_memory()
        out_h.host_seq = self._seq_host.data_ptr()
        self._c_out_host = out_h
        self._seq = 0
        self._actions_ptr, self._actions_dev_ptr = self._actions_host.data_ptr(), self.actions_dev.data_ptr()
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        # constant arguments of the per-step C calls, converted once
        self._ref = dict(store=C.byref(self.dw.store), tables=C.byref(self.dw.tables), envs=C.byref(self._c_envs),
                         rules=C.byref(self._c_rules), out=C.byref(self._c_out), out_host=C.byref(self._c_out_host))

        self.observation_space, self.action_space = build_spaces(lay, obs_layout, scaled_float, unreal_wrapper,
                                                                 self.n_actions)
        self.set_hardness = self.set_complexity     # experiments/thor_cached_auxiliary.py:68
        self._float_leaves = None
        if self.float_buf and (h * w) % 4 == 0 and len(self.float_buf) <= 6 and \
                all(b.shape[1] in (1, 3) for b in self.float_buf.values()):
            self._float_leaves = (L.FloatLeaf * len(self.float_buf))(*[
                L.FloatLeaf(lay.planes.index(name[5:] if name.startswith("goal_") else name),
                            1 if name.startswith("goal_") else 0, buf.shape[1], 0, buf.data_ptr())
                for name, buf in self.float_buf.items()])
            # the conversion is part of every reset / step call (vn_step_out_t.float_leaves): no extra C call per step
            for o in (self._c_out, self._c_out_host):
                o.float_leaves = C.cast(self._float_leaves, C.c_void_p)
                o.n_float_leaves, o.float_h, o.float_w = len(self._float_leaves), h, w
        self._pending = False
        self._modes, self._prev_mode = {}, None
        self._hc = None
        self._h2d_done = None
        self._serial_next = False
        self._obs_cache = None
        self.closed = False
        self._launches0 = self.lib.vn_launch_count()
        self._calls = 0          # parity of the double-buffered gather descriptors
        # host path: pinned staging seen as numpy views; the scalar kernel publishes a sequence word once its
        # results have landed on the host (the gather is still running when step() returns)
        self._actions_np = self._actions_host.numpy()
        self._pack_nps = [t.numpy() for t in self._pack_hosts]
        self._pack_ptrs = [t.data_ptr() for t in self._pack_hosts]
        self._pack_np = self._pack_nps[0]
        self._infos_refs = [None, None]        # weak references to the LazyInfos reading each pack in place
        self._slot = 0

    @property
    def kernel_launches(self):
        """Kernels the library enqueued since this object was built (process-wide counter, vn_launch_count)."""
        return int(self.lib.vn_launch_count() - self._launches0)

    # ------------------------------------------------------------------ construction helpers
    def _default_env_tasks(self, num_envs):
        """Reference create_envs builds one env per (scene, goal) task (thor_cached_auxiliary.py:66);
        with more envs than tasks the tasks are dealt round-robin, each env owning ONE task.  Families
        whose env samples its task on reset (MultipleGraphEnv, THORCachedEnv task lists) should pass
        ``env_tasks`` explicitly."""
        t = len(self.world.tasks)
        lo = np.arange(num_envs, dtype=np.int32) % t
        return np.stack([lo, np.ones(num_envs, np.int32)], 1)

    def set_inject(self, task, start):
        """Injected reset stream for parity runs: [n_local, R] task offsets (relative to the env's task
        range) and GLOBAL start states; reset k of env i consumes column k."""
        task = torch.as_tensor(np.ascontiguousarray(task, dtype=np.int32)).to(self.device)
        start = torch.as_tensor(np.ascontiguousarray(start, dtype=np.int32)).to(self.device)
        assert task.shape == start.shape and task.shape[0] == self.num_envs
        self._inject_keep = (task, start)
        self._c_inject = L.Inject(task.data_ptr(), start.data_ptr(), task.shape[1], 0)

    # ------------------------------------------------------------------ reference surface
    def _stream(self):
        return _raw_stream(self._dev_index)

    def _call(self, fn, *args):
        """One C-ABI call with this env's device current (the guard is skipped when it already is)."""
        if torch.cuda.current_device() == self._dev_index:
            L.check(fn(*args))
        else:
            with torch.cuda.device(self.device):
                L.check(fn(*args))

    def _leaf(self, name):
        if self.scaled_float:
            return self.float_buf[name]
        return self.goal_buf[name[5:]] if name.startswith("goal_") else self.obs_buf[name]

    def _obs(self):
        if self._obs_cache is None:     # the leaves are persistent batch buffers: build the structure once
            self._obs_cache = self._build_obs()
        return self._obs_cache

    def _obs_out(self):
        """What reset() / step() hand back: the persistent CUDA batches, or (numpy_obs) fresh host copies of them."""
        obs = self._obs()
        if not self.numpy_obs:
            return obs
        leaves = []

        def walk(x):
            if isinstance(x, tuple):
                return tuple(walk(v) for v in x)
            if isinstance(x, dict):
                return {k: walk(v) for k, v in x.items()}
            leaves.append(x)
            return len(leaves) - 1

        shape = walk(obs)
        # two sets of pinned staging buffers used alternately: the arrays handed back are views of pinned memory (no
        # second host copy of a 100+ MB batch, no page faults on fresh allocations) and stay valid until the step after
        # next.  numpy_obs="copy" returns private copies instead, like SubprocVecEnv's np.stack.
        self._stage_slot = getattr(self, "_stage_slot", 0) ^ 1
        staged = []
        for i, t in enumerate(leaves):
            key = (self._stage_slot, i)
            buf = self._host_stage.get(key)
            if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
                buf = self._host_stage[key] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
            buf.copy_(t, non_blocking=True)
            staged.append(buf)
        torch.cuda.current_stream(self.device).synchronize()
        host = [b.numpy().copy() if self.numpy_obs == "copy" else b.numpy() for b in staged]

        def build(x):
            if isinstance(x, tuple):
                return tuple(build(v) for v in x)
            if isinstance(x, dict):
                return {k: build(v) for k, v in x.items()}
            return host[x]

        return build(shape)

    def _convert_float_leaves(self, all_rows=False):
        """Float mode: TransposeImage + ScaledFloatFrame (thor_cached_auxiliary.py:61-62) of the step just enqueued,
        reading the step's gather descriptors (record or -1 = row unchanged; goal record or -1 = no reset): rows that
        did not change are not converted again.  Normally the step call itself enqueues the one-launch conversion
        (vn_step_out_t.float_leaves); this method serves odd geometries (one launch per leaf) and full refreshes."""
        if self.num_envs == 0:
            return
        if not all_rows and self._float_leaves is not None:
            return      # already enqueued by the reset / step call
        lay = self.world.layout
        h, w = lay.frame_hw
        desc = self._gather_desc[self._calls & 1]
        stream = self._stream()
        for name, buf in self.float_buf.items():
            goal = name.startswith("goal_")
            pi = lay.planes.index(name[5:] if goal else name)
            if all_rows:
                idx, stride = (self.goal if goal else self.obs_state).data_ptr(), 1
            else:
                idx, stride = desc.data_ptr() + (4 if goal else 0), 2
            self._call(self.lib.vn_gather_plane_f32_chw_rows, self._ref["store"], pi, idx, stride, self.num_envs, h, w,
                       lay.channels[pi], buf.data_ptr(), stream)

    def _build_obs(self):
        lv = self.leaves
        if isinstance(lv, dict):
            inner = {k: self._leaf(v) for k, v in lv.items()}
        elif isinstance(lv, tuple):
            inner = tuple(self._leaf(v) for v in lv)
        else:
            inner = self._leaf(lv)
        return (inner, self.lar) if self.unreal_wrapper else inner

    def reset(self, mask=None):
        """(Re)starts every env (or the masked ones) and returns the stacked observation."""
        self._check_open()
        m = None
        if mask is not None:
            m = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8)
        self._tick(self._c_out, 0)
        r = self._ref
        self._call(self.lib.vn_env_reset, r["store"], r["tables"], r["envs"], r["rules"],
                   C.byref(self._c_inject) if self._c_inject is not None else None,
                   L.ptr(m), r["out"], self.gather, self._stream())
        if self.scaled_float:
            self._convert_float_leaves()
        return self._obs_out()

    def _mode_of(self, out, flags):
        """How the library runs a call with these flags on this output block (0 two kernels / 1 fused / 2 persistent),
        asked once per (block, pipelined or not) - under VN_GATHER_AUTO the answer depends on both."""
        key = (id(out), bool(flags & L.STEP_ACTIONS_READY))
        m = self._modes.get(key)
        if m is None:
            saved = out.flags
            out.flags = flags
            m = self.lib.vn_env_step_mode(C.byref(self.dw.store), C.byref(self._c_envs), C.byref(out), self.gather)
            out.flags = saved
            if m < 0:
                L.check(m)
            self._modes[key] = m
        return m

    def _tick(self, out, flags):
        self._calls += 1
        out.parity = self._calls & 1
        if flags & L.STEP_ACTIONS_READY and (self._serial_next or self._prev_mode != L.MODE_SPLIT):
            # A pipelined step's scalar kernel overlaps the launch before it.  That is only sound when that launch is the
            # gather half of this env batch's previous two-kernel step; after a reset, a one-launch step (which WRITES the
            # env state this step reads) or a graph replay (whose descriptor parity is not the host's) it waits instead.
            flags |= L.STEP_NO_OVERLAP
        self._serial_next = False
        out.flags = flags
        self._prev_mode = self._mode_of(out, flags)

    def step_async(self, actions, actions_ready=False):
        """``actions_ready=True`` promises that the action buffer was complete before the previous step's
        gather was enqueued (pre-computed action streams, CUDA-graph replays): the scalar kernel of this step
        then overlaps the previous gather (include/vn_b200.h VN_STEP_ACTIONS_READY)."""
        self._check_open()
        if self._pending:
            # the staging buffers (pinned actions, host pack) of the step in flight would be overwritten
            raise RuntimeError("step_async() called again before step_wait()")
        inj = C.byref(self._c_inject) if self._c_inject is not None else None
        if self.host_outputs and not (torch.is_tensor(actions) and actions.is_cuda):
            # reference-facing path: host actions in, host scalars out - ONE C call enqueues
            # scalar kernel (reads / writes mapped pinned memory) and gather kernel
            a = np.asarray(actions.cpu() if torch.is_tensor(actions) else actions).reshape(-1)
            if a.size != self.num_envs:
                raise ValueError("expected %d actions, got %d" % (self.num_envs, a.size))
            self._actions_np[:] = a
            self._last_actions = self._actions_np
            # host actions were written just now, after the scalars of the previous step arrived: the previous
            # scalar kernel has finished reading them, and the gather never produces them
            self._tick(self._c_out_host, L.STEP_ACTIONS_READY | self._step_flags)
            self._seq = (self._seq % 0x7FFFFFFF) + 1
            self._c_out_host.seq = self._seq
            self._next_pack()
            r = self._ref
            self._call(self.lib.vn_env_step_host, r["store"], r["tables"], r["envs"], r["rules"], inj,
                       self._actions_host.data_ptr(), self.actions_dev.data_ptr(), r["out_host"], None,
                       self.gather, self._stream())
            if self.scaled_float:
                self._convert_float_leaves()
            self._pending = "host"
            return
        if torch.is_tensor(actions) and actions.is_cuda:
            a = actions if actions.dtype == torch.int32 else actions.to(torch.int32)
            a = a.contiguous()
        else:
            src = actions if torch.is_tensor(actions) else torch.as_tensor(np.asarray(actions))
            # one pinned staging buffer: the asynchronous H2D copy of the PREVIOUS step must have read it before it
            # is rewritten (step_wait does not synchronise when host_outputs is False)
            if self._h2d_done is not None:
                self._h2d_done.synchronize()
            self._actions_host.copy_(src.reshape(-1).to(torch.int32))
            self.actions_dev.copy_(self._actions_host, non_blocking=True)
            if self._h2d_done is None:
                self._h2d_done = torch.cuda.Event()
            self._h2d_done.record(torch.cuda.current_stream(self.device))
            a = self.actions_dev
        if a.numel() != self.num_envs:
            raise ValueError("expected %d actions, got %d" % (self.num_envs, a.numel()))
        self._last_actions = a
        self._tick(self._c_out, (L.STEP_ACTIONS_READY if actions_ready else 0) | self._step_flags)
        r = self._ref
        self._call(self.lib.vn_env_step, r["store"], r["tables"], r["envs"], r["rules"], inj, a.data_ptr(), r["out"],
                   self.gather, self._stream())
        if self.scaled_float:
            self._convert_float_leaves()
        self._pending = "device"

    def step_enqueue(self, actions, actions_ready=False, record=None):
        """Device-resident loops: enqueue one vectorised step for CUDA int32 ``actions`` and return at once.
        Nothing is copied to the host; ``env.reward`` / ``env.done`` / the observation buffers hold the
        results in stream order.  See step_async for ``actions_ready``.  ``record`` = (actions, rewards, dones,
        next_states, next_goals) CUDA tensors of ``num_envs`` elements (int32, float32, uint8, int32, int32; any may
        be None) that the step kernel fills as well - a rollout storage row written without copy kernels
        (``RolloutBuffer.step``)."""
        if record is not None:
            o = self._c_out
            o.rec_action, o.rec_reward, o.rec_done, o.rec_state, o.rec_goal = (L.ptr(t) for t in record)
            try:
                self.step_async(actions, actions_ready)
            finally:
                o.rec_action = o.rec_reward = o.rec_done = o.rec_state = o.rec_goal = None
        else:
            self.step_async(actions, actions_ready)
        self._pending = False

    def capture_steps(self, actions, after_step=None):
        """Captures ``len(actions)`` consecutive device-resident steps into ONE CUDA graph and returns a
        ``CapturedSteps`` (``.replay()`` runs them).  For launch-bound batches: 16 envs step in 7.7 us per step from a
        graph instead of 19 us from Python.  ``actions`` is a CUDA int32 ``[T, N]`` tensor whose CONTENT may
        be rewritten between replays; ``after_step(t)`` runs inside the capture after step ``t`` (e.g.
        ``rollout_buffer.insert``).  The env state is left exactly as it was before the call."""
        if not (torch.is_tensor(actions) and actions.is_cuda and actions.dtype == torch.int32 and actions.dim() == 2):
            raise ValueError("capture_steps needs a CUDA int32 [T, N] action tensor")
        saved = self.state_dict()
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):                 # warm-up outside the capture (lazy CUDA / torch initialisation)
            self.step_enqueue(actions[0])
            if after_step is not None:
                after_step(0)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        self._restore(saved)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for t in range(actions.shape[0]):
                # The action tensor is complete before the graph is launched -> pipelined mode is safe from the
                # second step on.  The FIRST step runs in serial mode: whatever preceded the replay (another replay
                # - whose last step has the same descriptor parity when T is odd -, an eager step) may still be
                # gathering from the descriptor half this step writes.
                self.step_enqueue(actions[t], actions_ready=(t > 0))
                if after_step is not None:
                    after_step(t)
        self._restore(saved)
        return CapturedSteps(self, graph)

    def _restore(self, d):
        for k in ("state", "goal", "task", "elapsed", "epoch", "ep_return", "ep_length", "stats"):
            getattr(self, k).copy_(d[k].to(self.device))
        self.gather_current()
        torch.cuda.synchronize(self.device)

    def _next_pack(self):
        """Points the step about to be enqueued at the other pinned host pack.  An `infos` object of two steps ago that
        is still alive and still reads that pack in place gets its private copy first."""
        s = self._slot = self._slot ^ 1
        self._release_pack(s)
        self._c_out_host.host_pack = self._pack_ptrs[s]
        self._pack_np = self._pack_nps[s]

    def _release_pack(self, s):
        """Pinned host pack `s` is about to be overwritten: an `infos` object still reading it in place copies it first."""
        ref = self._infos_refs[s]
        if ref is not None:
            old = ref()
            if old is not None:
                old._snapshot()
            self._infos_refs[s] = None

    def _host_results(self, reward, done, noop):
        """(rewards, dones, infos) of the host-facing step whose scalars have just arrived in the current pack."""
        infos = LazyInfos(self, self._pack_np, noop, in_place=True)
        self._infos_refs[self._slot] = weakref.ref(infos)
        return reward, done, infos

    def _unpack(self, host):
        n = self.num_envs
        return dict(reward=host[:4 * n].view(np.float32), episode_return=host[4 * n:8 * n].view(np.float32),
                    episode_length=host[8 * n:12 * n].view(np.int32), info_state=host[12 * n:16 * n].view(np.int32),
                    done=host[16 * n:17 * n], truncated=host[17 * n:18 * n], win=host[18 * n:19 * n],
                    did_reset=host[19 * n:20 * n])

    def step_wait(self):
        if not self._pending:
            raise RuntimeError("step_wait() without step_async()")
        mode, self._pending = self._pending, False
        noop = (self._last_actions < 0) if self.family.noop_action else None
        if mode == "host":
            # wait for the scalars only (the kernel publishes a sequence word in pinned memory once they have all
            # landed); the gather of this step is still in flight - or not even started - on the stream
            n = self.num_envs
            if n:
                L.check(self.lib.vn_host_wait_seq(self._seq_host.data_ptr(), self._seq_words, self._seq, self._stream(),
                                                  60_000_000))
            h = self._pack_np
            return (self._obs_out(),) + self._host_results(h[:4 * n].view(np.float32).copy(),
                                                           h[16 * n:17 * n].view(np.bool_).copy(), noop)
        if self.host_outputs:
            self._release_pack(0)
            self._pack_hosts[0].copy_(self._pack, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            h = self._unpack(self._pack_nps[0].copy())
            return self._obs_out(), h["reward"], h["done"].view(np.bool_), LazyInfos(self, h, noop)
        fetch = lambda: self._unpack(self._pack.cpu().numpy())
        return self._obs_out(), self.reward, self.done.bool(), LazyInfos(self, fetch, noop)

    def _bind_host_call(self):
        """The constant arguments of the host-facing step bound once (vn_host_call_t): the per-step call converts
        four arguments instead of fifteen."""
        hc = L.HostCall()
        hc.store = C.cast(C.pointer(self.dw.store), C.c_void_p)
        hc.tables = C.cast(C.pointer(self.dw.tables), C.c_void_p)
        hc.envs = C.cast(C.pointer(self._c_envs), C.c_void_p)
        hc.rules = C.cast(C.pointer(self._c_rules), C.c_void_p)
        hc.inject = C.cast(C.pointer(self._c_inject), C.c_void_p) if self._c_inject is not None else None
        hc.host_actions, hc.dev_actions_copy = self._actions_ptr, self._actions_dev_ptr
        hc.out = C.cast(C.pointer(self._c_out_host), C.c_void_p)
        hc.seq_words, hc.gather_variant, hc.timeout_us = self._seq_words, self.gather, 60_000_000
        self._hc, self._hc_ptr = hc, C.addressof(hc)
        self._hc_inject = self._c_inject
        self._hc_fn = self.lib.vn_env_step_host_call

    def step(self, actions):
        if self.host_outputs and type(actions) is np.ndarray and not self._pending and not self.closed \
                and actions.size == self.num_envs and self.num_envs and \
                (not self.scaled_float or self._float_leaves is not None):
            # the reference-facing call, numpy in / numpy out, as ONE C call: stage the actions, enqueue the kernels,
            # spin until the scalars are in pinned memory, copy rewards / dones out (vn_env_step_host_call)
            n = self.num_envs
            np.copyto(self._actions_np, actions if actions.ndim == 1 else actions.reshape(-1), casting="same_kind")
            if self._hc is None or self._hc_inject is not self._c_inject:
                self._bind_host_call()
            out = self._c_out_host
            self._calls += 1
            out.parity = self._calls & 1
            if self._serial_next or self._prev_mode != L.MODE_SPLIT:    # see _tick
                out.flags = L.STEP_ACTIONS_READY | L.STEP_NO_OVERLAP | self._step_flags
                self._serial_next = False
                self._prev_mode = self._mode_of(out, out.flags)
            else:
                out.flags = L.STEP_ACTIONS_READY | self._step_flags     # previous and this step: two kernels (host caller)
            self._seq = out.seq = (self._seq % 0x7FFFFFFF) + 1
            self._next_pack()
            res = np.empty(5 * n, np.uint8)         # rewards (4n bytes) + dones (n bytes) in one allocation
            ptr = res.__array_interface__["data"][0]
            if torch.cuda.current_device() == self._dev_index:
                rc = self._hc_fn(self._hc_ptr, ptr, ptr + 4 * n, _raw_stream(self._dev_index))
            else:
                with torch.cuda.device(self.device):
                    rc = self._hc_fn(self._hc_ptr, ptr, ptr + 4 * n, _raw_stream(self._dev_index))
            if rc:
                L.check(rc)
            noop = (self._actions_np < 0) if self.family.noop_action else None
            infos = LazyInfos(self, self._pack_np, noop, True)
            self._infos_refs[self._slot] = weakref.ref(infos)
            return self._obs_out(), res[:4 * n].view(np.float32), res[4 * n:].view(np.bool_), infos
        self.step_async(actions)
        return self.step_wait()

    def close(self):
        if not self.closed and torch.cuda.is_available():
            # kernels in flight may still write the mapped pinned buffers this object owns
            torch.cuda.synchronize(self.device)
        self.closed = True

    def _check_open(self):
        if self.closed:
            raise RuntimeError("environment is closed")

    @property
    def unwrapped(self):
        return self

    def call_unwrapped(self, name, *args, **kwargs):
        """deep_rl SubprocVecEnv.call_unwrapped: calls a method on every (unwrapped) env; here the
        batch is one object, so the result list repeats the single return value."""
        r = getattr(self, name)(*args, **kwargs)
        return [r] * self.num_envs

    def set_complexity(self, complexity=None):
        self.dw.set_complexity(complexity)

    def set_reward_progress(self, coef):
        """Dense geodesic-progress reward from the next step on (call between steps, like set_hardness): every step adds
        ``coef * (d(s_t, g) - d(s_t+1, g))`` to the reward, ``d`` the number of actions on the shortest path to the env's
        current goal (the distances optimal_actions() returns), ``s_t+1`` the state the action led to before any auto-reset,
        and 0 where either distance is -1 (unreachable).  The step kernel adds it in float32, ``coef`` rounded to float32,
        so rewards, episode returns, statistics, last_action_reward and rollout rows all carry the shaped reward.  The
        reference has no such term; 0 (the default) gives the reference's rewards bit for bit.  A non-zero coefficient
        builds the distance table (DeviceWorld.shortest_paths) on first use.  A CUDA graph captured earlier
        (capture_steps) keeps the coefficient it was captured with."""
        coef = float(coef)
        if not np.isfinite(coef):
            raise ValueError("reward_progress must be finite, got %r" % coef)
        if coef != 0.0:
            self.dw.shortest_paths()
        self._c_rules.reward_progress = coef
        self.reward_progress = float(np.float32(coef))

    # ------------------------------------------------------------------ extras
    def states(self):
        """Current states as reference tuples (x, y[, r]) - host copy."""
        return [self.world.state_tuple(int(s)) for s in self.state.cpu().numpy()]

    def episode_stats(self, reduce=False, reset=False):
        """Running device-side episode statistics.  ``reduce=True`` sums them over all ranks with ONE
        all-reduce of 8 numbers (NCCL) - the only collective anywhere near this path."""
        v = self.stats.clone()
        vals = v.cpu().numpy().copy()
        out = np.zeros(L.VN_N_STATS, np.float64)
        for i, name in enumerate(L.STAT_NAMES):
            out[i] = vals[i:i + 1].view(np.float64)[0] if name == "return_sum" else float(vals[i])
        if reduce and self.world_size > 1:
            out = reduce_stats(out, self.device)
        if reset:
            self.stats.zero_()
        return dict(zip(L.STAT_NAMES, out.tolist()))

    def optimal_actions(self):
        """Evaluation service (SURVEY.md section 8(f) rank 4): for every env the first action of a shortest
        action sequence to its current goal, and the remaining distance, from per-task tables computed once
        on the host (tables.optimal_policy_table) and kept on the device (DeviceWorld.shortest_paths, shared with the
        geodesic-progress reward).  Returns (actions, dist) int32 [N]."""
        act, dst = self.dw.shortest_paths()
        t, s = self.task.long(), self.state.long()
        return act[t, s], dst[t, s]

    def state_dict(self):
        keys = ("state", "goal", "task", "elapsed", "epoch", "ep_return", "ep_length", "stats")
        d = {k: getattr(self, k).cpu().clone() for k in keys}
        d["complexity"] = self.dw.complexity
        return d

    def load_state_dict(self, d):
        for k in ("state", "goal", "task", "elapsed", "epoch", "ep_return", "ep_length", "stats"):
            getattr(self, k).copy_(d[k].to(self.device))
        self.set_complexity(d.get("complexity"))
        # refresh observation / goal batches for the restored states
        self.gather_current()

    def gather_current(self):
        """Re-gathers observation and goal planes for the current states (after load_state_dict)."""
        for p, buf in self.obs_buf.items():
            gather_plane(self.dw, p, self.state, out=buf, variant=self.gather)
        for p, buf in self.goal_buf.items():
            gather_plane(self.dw, p, self.goal, out=buf, variant=self.gather)
        self.obs_state.copy_(self.state)       # the rows now hold the frames of `state` (skip_unchanged compares to it)
        if self.scaled_float:
            self._convert_float_leaves(all_rows=True)
        return self._obs()


def gather_plane(dw: DeviceWorld, plane, idx, out=None, variant=L.GATHER_AUTO):
    """out[i] = frame ``plane`` of state idx[i]: the batched ``ThorGridWorld.render``
    (graph/multi_graph_no_tp.py:12-25) for an arbitrary index list (replay sampling etc.)."""
    pi = dw.plane_index(plane)
    lay = dw.world.layout
    h, w = lay.frame_hw
    idx = idx.to(device=dw.device, dtype=torch.int32).contiguous()
    n = idx.numel()
    if out is None:
        out = lay.batch(plane, n, dw.device)
    elif n > 1 and out.stride(0) != lay.plane_bytes[pi]:
        raise ValueError("gather_plane: rows of `out` must be %d bytes apart (StoreLayout.batch)" % lay.plane_bytes[pi])
    with torch.cuda.device(dw.device):
        L.check(dw.lib.vn_gather_plane(C.byref(dw.store), pi, idx.data_ptr(), n, out.data_ptr(), variant,
                                       torch.cuda.current_stream(dw.device).cuda_stream))
    return out


def reduce_stats(vec, device=None, group=None):
    """Sum of the 8-number statistics vector over all ranks.  NCCL when the process group is NCCL
    (tensor on ``device``), gloo otherwise (CPU tensor)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return vec
    backend = dist.get_backend(group)
    t = torch.as_tensor(np.asarray(vec, np.float64))
    if backend == "nccl":
        t = t.to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()
