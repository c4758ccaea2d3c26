"""Rollout buffer and return / auxiliary-target builders on the device.

Host-side mirror of what the reference gets from deep_rl (un-vendored) and from
experiments/ai2_auxiliary/trainer.py: every function takes / returns CUDA tensors and calls one
C-ABI entry point of libvn_b200.so.  Batch-major ``[B, T, ...]`` like the reference tensors.

The rollout buffer stores STATE INDICES, not frames: a 128-step rollout of 8,192 envs is 4 MB of
int32 instead of 22 GB of uint8 frames, and the target builders re-gather the frames they need from
the HBM store (which mostly sits in the 126 MB L2).
"""
import ctypes as C

import torch

from . import lib as L
from .store import DeviceWorld


def _call(device, fn, *args, stream_of=None):
    """Calls library entry point ``fn`` with ``device`` current and, as its stream argument, the current stream of the
    device ``stream_of`` lives on (default: ``device``); raises VnError when the call fails."""
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device if stream_of is None else stream_of.device).cuda_stream
        L.check(getattr(L.load(), fn)(*args, stream))


def _strided2d(x, dtype):
    """A 2-D tensor as the kernels take it: any element strides (a ``.t()`` view of time-major rollout storage is
    read in place, no transpose kernel), the given dtype (bool is read as uint8 in place)."""
    if x.dtype == torch.bool and dtype == torch.uint8:
        x = x.view(torch.uint8)
    if x.dtype != dtype:
        x = x.to(dtype)
    if x.dim() != 2:
        raise ValueError("expected a 2-D [B, T] tensor, got %s" % (tuple(x.shape),))
    return x


def nstep_returns(rewards, dones, last_values, gamma, time_major=False, method="serial", out=None):
    """A2C n-step returns (deep_rl RolloutStorage.batch; SURVEY.md D4).
    rewards float32, dones uint8/bool: [B, T] with ANY strides (``storage.t()`` views are read in place); last_values
    [B].  Returns a contiguous [B, T] tensor.  ``time_major=True``: the arguments are [T, B] and so is the result.
    method="serial" (default): thread per env, the reference's loop order, bit-identical to it.
    method="scan": warp per env, 32 steps per pass composed with shuffles - for few envs and long rollouts; equal
    within ~1e-6 relative (float re-association), not bit for bit."""
    fn = {"serial": "vn_nstep_returns", "scan": "vn_nstep_returns_scan"}[method]
    rewards, dones = _strided2d(rewards, torch.float32), _strided2d(dones, torch.uint8)
    if time_major:
        rewards, dones = rewards.t(), dones.t()
    if dones.stride() != rewards.stride():
        rewards, dones = rewards.contiguous(), dones.contiguous()
    last_values = last_values.contiguous().float()
    n, t = rewards.shape
    if out is None:
        out = torch.empty((t, n) if time_major else (n, t), dtype=torch.float32, device=rewards.device)
    if n == 0:
        return out
    ob = out.t() if time_major else out
    _call(rewards.device, fn, rewards.data_ptr(), dones.data_ptr(), last_values.data_ptr(), float(gamma), n, t,
          rewards.stride(0), rewards.stride(1), out.data_ptr(), ob.stride(0), ob.stride(1), stream_of=rewards)
    return out


def discounted_backup(rewards, dones, bootstrap, gamma):
    """rewards [B, T, ...]; dones [B, T] (any strides); bootstrap [B, ...] -> R_t = r_t + gamma (1 - done_t) R_{t+1}."""
    b, t = rewards.shape[:2]
    d = rewards.shape[2:].numel()
    rewards = rewards.contiguous().float()
    dones = _strided2d(dones, torch.uint8)
    bootstrap = bootstrap.contiguous().float()
    out = torch.empty_like(rewards)
    if b == 0:
        return out
    _call(rewards.device, "vn_discounted_backup", rewards.data_ptr(), dones.data_ptr(), dones.stride(0), dones.stride(1),
          bootstrap.data_ptr(), float(gamma), b, t, d, out.data_ptr(), stream_of=rewards)
    return out


def _geom(dw, plane, cell, output_size):
    lay = dw.world.layout
    pi = dw.plane_index(plane)
    h, w = lay.frame_hw
    c = lay.channels[pi]
    if output_size is None:
        output_size = (h // cell, w // cell)
    return pi, h, w, c, int(output_size[0]), int(output_size[1])


def _on_device(dw, states):
    if states.device != dw.device or states.dtype != torch.int32:
        states = states.to(device=dw.device, dtype=torch.int32)
    return states


def _states2d(dw, states):
    states = _on_device(dw, states)
    if states.dim() != 2:
        raise ValueError("states must be [B, T+1]")
    return states


def _pixel_control_direct(dw, states, cell_size, output_size, plane):
    pi, h, w, c, oh, ow = _geom(dw, plane, cell_size, output_size)
    b, t1 = states.shape
    out = torch.empty((b, t1 - 1, 1, oh, ow), dtype=torch.float32, device=dw.device)
    if b == 0:
        return out
    _call(dw.device, "vn_pixel_control", C.byref(dw.store), pi, states.data_ptr(), b, t1 - 1, states.stride(0),
          states.stride(1), h, w, c, cell_size, oh, ow, out.data_ptr(), stream_of=states)
    return out


def _aux_direct(dw, states, plane, cell_size, output_size):
    pi, h, w, c, oh, ow = _geom(dw, plane, cell_size, output_size)
    states = states.contiguous()
    out = torch.empty(tuple(states.shape) + (c, oh, ow), dtype=torch.float32, device=dw.device)
    if states.numel() == 0:
        return out
    _call(dw.device, "vn_aux_target", C.byref(dw.store), pi, states.data_ptr(), states.numel(), h, w, c, cell_size, oh,
          ow, out.data_ptr(), stream_of=states)
    return out


class TargetTables:
    """Per-world table that turns the pixel-control builders into row gathers.  On a cached graph the target is a
    pure function of state indices, so it is evaluated once (with the direct kernel) and kept resident in HBM - the
    same move as caching the frames themselves:

      pc[s * 4 + a]  = pixel-control reward of the transition s -> adj[s][a]     [4 S, oh * ow] f32

    C2 (6,000 states, 20x20): 38 MB.  The auxiliary targets have tables of their own (_aux_table).
    """

    def __init__(self, dw: DeviceWorld, cell_size=4, output_size=None, plane="rgb"):
        self.dw, self.cell, self.plane = dw, cell_size, plane
        _, h, w, _, oh, ow = _geom(dw, plane, cell_size, output_size)
        self.out_hw = (oh, ow)
        S = dw.world.n_states
        adj = dw.adj.view(S, 4)
        me = torch.arange(S, dtype=torch.int32, device=dw.device)
        nxt = torch.where(adj >= 0, adj, me[:, None])                       # collisions: s -> s (never looked up)
        self.pc = torch.empty((4 * S, oh * ow), dtype=torch.float32, device=dw.device)
        step = 1 << 16                                                       # bounded scratch while building
        pairs = torch.stack([me.repeat_interleave(4), nxt.reshape(-1)], 1).contiguous()
        for lo in range(0, 4 * S, step):
            self.pc[lo:lo + step] = _pixel_control_direct(dw, pairs[lo:lo + step], cell_size, (oh, ow), plane).view(-1, oh * ow)
        self._scratch = {}

    def scratch(self, n, chained=False):
        """(rows, miss_pos, miss_count) int32 scratch for n transitions, reused between calls on the same stream.
        The chained call (vn_pixel_control_returns_from_states) owns its own set: its miss_count starts at zero and is
        re-armed by the call's last kernel, while vn_transition_rows on its own zeroes the counter it is given."""
        key = (n, chained)
        if key not in self._scratch:
            dev = self.dw.device
            self._scratch[key] = (torch.empty(n, dtype=torch.int32, device=dev),
                                  torch.empty(n, dtype=torch.int32, device=dev),
                                  torch.zeros(1, dtype=torch.int32, device=dev))
        return self._scratch[key]

    def miss_rows(self, max_miss):
        """float32 [max_miss, oh * ow] side buffer of the chained call (the rewards of the transitions the table cannot
        serve), reused between calls."""
        key = ("miss", max_miss)
        if key not in self._scratch:
            self._scratch[key] = torch.empty((max_miss, self.pc.shape[1]), dtype=torch.float32, device=self.dw.device)
        return self._scratch[key]

    def nbytes(self):
        return self.pc.numel() * 4


def target_tables(dw: DeviceWorld, cell_size=4, output_size=None, plane="rgb") -> TargetTables:
    """Cached per (world, plane, cell, output size)."""
    _, _, _, _, oh, ow = _geom(dw, plane, cell_size, output_size)
    cache = dw.__dict__.setdefault("_target_tables", {})
    key = (plane, cell_size, oh, ow)
    if key not in cache:
        cache[key] = TargetTables(dw, cell_size, (oh, ow), plane)
    return cache[key]


def _aux_table(dw: DeviceWorld, plane, cell_size, out_hw):
    """aux[s] = avg_pool(crop(plane(s) / 255)), float32 [S, C, oh, ow], built with the direct kernel on first use and
    cached per (world, plane, cell, output size).  C2 (6,000 states, 20x20): 10 MB (depth), 29 MB (segmentation)."""
    cache = dw.__dict__.setdefault("_aux_tables", {})
    key = (plane, cell_size) + tuple(out_hw)
    if key not in cache:
        me = torch.arange(dw.world.n_states, dtype=torch.int32, device=dw.device)
        cache[key] = _aux_direct(dw, me, plane, cell_size, out_hw).contiguous()
    return cache[key]


def pixel_control_reward(dw: DeviceWorld, states, cell_size=4, output_size=None, plane="rgb", method="table"):
    """deep_rl.a2c_unreal.util.pixel_control_reward (SURVEY.md D5) computed from state indices.
    states: int32 [B, T+1] (any strides) GLOBAL state of every observation of the sequence -> float32 [B, T, 1, h, w].

    method="table" (default): rows of the per-world transition table (TargetTables) are gathered; the few
    transitions the table cannot serve (resets) are computed directly by a list kernel in the same pass.
    method="direct": every transition is computed from the two frames.  Both give identical bits."""
    pi, h, w, c, oh, ow = _geom(dw, plane, cell_size, output_size)
    states = _states2d(dw, states)
    if method == "direct" or (oh * ow) % 4 or states.shape[0] == 0:
        return _pixel_control_direct(dw, states, cell_size, (oh, ow), plane)
    tab = target_tables(dw, cell_size, (oh, ow), plane)
    b, t1 = states.shape
    t = t1 - 1
    out = torch.empty((b, t, 1, oh, ow), dtype=torch.float32, device=dw.device)
    rows, miss_pos, miss_count = tab.scratch(b * t)
    sn, st = states.stride()
    rsn, rst = t, 1          # batch-major row scratch (the lookup kernel orders its threads for coalesced state reads)
    _call(dw.device, "vn_transition_rows", dw.adj.data_ptr(), states.data_ptr(), b, t, sn, st, rows.data_ptr(), rsn, rst,
          miss_pos.data_ptr(), miss_count.data_ptr(), stream_of=states)
    _call(dw.device, "vn_gather_rows", tab.pc.data_ptr(), oh * ow * 4, rows.data_ptr(), b * t, t, rsn, rst, out.data_ptr(),
          stream_of=states)
    _call(dw.device, "vn_pixel_control_list", C.byref(dw.store), pi, states.data_ptr(), b, t, sn, st, h, w, c, cell_size,
          oh, ow, miss_pos.data_ptr(), miss_count.data_ptr(), b * t, 0, out.data_ptr(), stream_of=states)
    return out


def pixel_control_returns(dw: DeviceWorld, states, dones, bootstrap, gamma, cell_size=4, output_size=None, plane="rgb",
                          with_reward=False, max_miss=None):
    """Pixel-control rewards AND their discounted back-up (UNREAL: gamma_pc = 0.9, bootstrap = max_a Q_aux(s_T);
    SURVEY.md D5) in one pass over the per-world transition table: equal, bit for bit, to
    ``discounted_backup(pixel_control_reward(states), dones, bootstrap, gamma)`` without ever writing the rewards.

    states int32 [B, T+1], dones uint8/bool [B, T] (any strides: ``storage.t()`` views are read in place), bootstrap
    float32 [B, h*w] (or [B, h, w]).  Returns float32 [B, T, h*w] (and the rewards [B, T, h*w] with with_reward).
    max_miss bounds the side buffer for the transitions the table cannot serve (episode resets; default: all B*T).  When
    more transitions than that miss the table, the ones past the bound (which ones is up to the device) get no reward:
    their rows of the rewards are NaN, and so are the returns of their env at their step and every earlier one.  All
    other elements are what an unbounded call gives."""
    pi, h, w, c, oh, ow = _geom(dw, plane, cell_size, output_size)
    cells = oh * ow
    if cells % 4:
        r = pixel_control_reward(dw, states, cell_size, (oh, ow), plane).view(states.shape[0], -1, cells)
        ret = discounted_backup(r, dones, bootstrap.reshape(states.shape[0], cells), gamma)
        return (ret, r) if with_reward else ret
    states = _states2d(dw, states)
    dones = _strided2d(dones, torch.uint8)
    b, t1 = states.shape
    t = t1 - 1
    out = torch.empty((b, t, cells), dtype=torch.float32, device=dw.device)
    rew = torch.empty((b, t, cells), dtype=torch.float32, device=dw.device) if with_reward else None
    if b == 0:
        return (out, rew) if with_reward else out
    tab = target_tables(dw, cell_size, (oh, ow), plane)
    bootstrap = bootstrap.reshape(b, cells).contiguous().float()
    rows, miss_pos, miss_count = tab.scratch(b * t, chained=True)
    max_miss = max(b * t if max_miss is None else int(max_miss), 1)
    side = tab.miss_rows(max_miss)
    sn, st = states.stride()
    # one C call, three chained kernels: transition rows -> misses computed directly -> gather + back-up
    _call(dw.device, "vn_pixel_control_returns_from_states", C.byref(dw.store), pi, dw.adj.data_ptr(), tab.pc.data_ptr(),
          states.data_ptr(), sn, st, dones.data_ptr(), dones.stride(0), dones.stride(1), bootstrap.data_ptr(),
          float(gamma), b, t, h, w, c, cell_size, oh, ow, rows.data_ptr(), miss_pos.data_ptr(), miss_count.data_ptr(),
          side.data_ptr(), max_miss, out.data_ptr(), L.ptr(rew), stream_of=states)
    return (out, rew) if with_reward else out


def auxiliary_target(dw: DeviceWorld, states, plane, cell_size=4, output_size=None, method="table"):
    """compute_auxiliary_target (experiments/ai2_auxiliary/trainer.py:9-15) from state indices.
    states int32 [B, T] (any strides) -> float32 [B, T, C, h, w].  method="table": one row gather from the per-world
    pooled-plane table; method="direct": pooled from the frame."""
    pi, h, w, c, oh, ow = _geom(dw, plane, cell_size, output_size)
    states = _on_device(dw, states)
    if method == "direct" or (c * oh * ow) % 4 or states.numel() == 0:
        return _aux_direct(dw, states, plane, cell_size, (oh, ow))
    shape = tuple(states.shape)
    if states.dim() != 2:
        states = states.contiguous().view(-1, 1)
    tab = _aux_table(dw, plane, cell_size, (oh, ow))
    out = torch.empty(shape + (c, oh, ow), dtype=torch.float32, device=dw.device)
    _call(dw.device, "vn_gather_rows", tab.data_ptr(), c * oh * ow * 4, states.data_ptr(), states.numel(),
          states.shape[1], states.stride(0), states.stride(1), out.data_ptr(), stream_of=states)
    return out


def auxiliary_targets(dw, states, goal_states, cell_size=4, output_size=None, method="table"):
    """compute_auxiliary_targets (trainer.py:17-19): targets for observation leaves 2.. of the aux5
    tuple = (depth, segmentation, goal_segmentation)."""
    return (auxiliary_target(dw, states, "depth", cell_size, output_size, method),
            auxiliary_target(dw, states, "segmentation", cell_size, output_size, method),
            auxiliary_target(dw, goal_states, "segmentation", cell_size, output_size, method))


def policy_input(dw: DeviceWorld, states, plane="rgb"):
    """TransposeImage + ScaledFloatFrame fused with the gather: float32 [..., C, H, W] in [0, 1]."""
    pi, h, w, c, _, _ = _geom(dw, plane, 1, None)
    states = states.to(device=dw.device, dtype=torch.int32).contiguous()
    out = torch.empty(tuple(states.shape) + (c, h, w), dtype=torch.float32, device=dw.device)
    if states.numel() == 0:
        return out
    _call(dw.device, "vn_gather_plane_f32_chw", C.byref(dw.store), pi, states.data_ptr(), states.numel(), h, w, c,
          out.data_ptr(), stream_of=states)
    return out


def reward_prediction_labels(rewards, with_lists=True, sync=True, buffers=None):
    """UNREAL reward-prediction classes (0 zero / 1 positive / 2 negative) and the ascending lists of
    zero / non-zero reward positions (row-major positions of the [B, T] argument, whatever its strides) that the
    50/50 sampler draws from (SURVEY.md D6).
    Returns (labels int8 [B, T] contiguous, zero_idx int32, nonzero_idx int32).  sync=True: the lists are trimmed
    to their lengths (one 8-byte D2H read for the two counts).  sync=False: nothing waits for the device - the
    lists come back at full length together with a device tensor ``counts`` = (#zero, #non-zero) as a 4th value."""
    r = rewards if rewards.dtype == torch.float32 else rewards.float()
    flat = r.dim() != 2
    if flat:
        r = r.contiguous().view(-1, 1).t()        # [1, n]: positions in storage order
    n = r.numel()
    if buffers is not None:          # (labels, zero, nonzero, counts, scratch) owned by the caller, reused call after call
        labels, zero, nonzero, counts, scratch = buffers
    else:
        labels = torch.empty(tuple(rewards.shape), dtype=torch.int8, device=r.device)
        scratch = torch.empty((n + 1023) // 1024 + 1, dtype=torch.int32, device=r.device)
        counts = torch.empty(2, dtype=torch.int32, device=r.device)     # always written by the scan kernel
        zero = torch.empty(n, dtype=torch.int32, device=r.device) if with_lists else None
        nonzero = torch.empty(n, dtype=torch.int32, device=r.device) if with_lists else None
    if n > 0:
        _call(r.device, "vn_rp_labels", r.data_ptr(), n, r.shape[1], r.stride(0), r.stride(1), labels.data_ptr(),
              L.ptr(zero), L.ptr(nonzero), counts.data_ptr(), scratch.data_ptr(), stream_of=r)
    else:
        counts.zero_()
    if buffers is not None:
        return labels, zero, nonzero, counts
    if not with_lists:
        return labels, None, None
    if not sync:
        return labels, zero, nonzero, counts
    cz, cn = counts.tolist() if n > 0 else (0, 0)
    return labels, zero[:cz], nonzero[:cn]


class RolloutBuffer:
    """Device-resident rollout of T steps x B envs: int32 states / goals, float32 rewards, uint8 dones,
    int32 actions; time-major storage (each env step appends one contiguous row).  The builders read the storage in
    place through ``.t()`` views (explicit strides at the C ABI) and write batch-major ``[B, T, ...]`` results like the
    reference tensors: no transpose or copy kernel between the step and the loss."""

    def __init__(self, dw: DeviceWorld, num_envs, num_steps):
        self.dw, self.B, self.T = dw, num_envs, num_steps
        dev = dw.device
        self.states = torch.zeros((num_steps + 1, num_envs), dtype=torch.int32, device=dev)
        self.goals = torch.zeros((num_steps + 1, num_envs), dtype=torch.int32, device=dev)
        self.rewards = torch.zeros((num_steps, num_envs), dtype=torch.float32, device=dev)
        self.dones = torch.zeros((num_steps, num_envs), dtype=torch.uint8, device=dev)
        self.actions = torch.zeros((num_steps, num_envs), dtype=torch.int32, device=dev)
        self.t = 0

    def start(self, env):
        """Records the observation the rollout starts from (after reset() or the previous rollout)."""
        self.states[0].copy_(env.obs_state)      # contiguous same-dtype rows: cudaMemcpyAsync, not a kernel
        self.goals[0].copy_(env.goal)
        self.t = 0

    def insert(self, env, actions):
        """Call after env.step(actions): appends (action, reward, done) and the NEXT observation's state."""
        t = self.t
        self.actions[t].copy_(actions.to(torch.int32) if torch.is_tensor(actions) else torch.as_tensor(actions))
        self.rewards[t].copy_(env.reward)
        self.dones[t].copy_(env.done)
        self.states[t + 1].copy_(env.obs_state)
        self.goals[t + 1].copy_(env.goal)
        self.t = t + 1

    def step(self, env, actions, actions_ready=False):
        """``env.step_enqueue(actions)`` + ``insert`` in one: the step kernel writes (action, reward, done, next
        state, next goal) straight into row ``t`` of this buffer (vn_step_out_t.rec_*), no copy kernels."""
        t = self.t
        if not (torch.is_tensor(actions) and actions.is_cuda and actions.dtype == torch.int32):
            raise ValueError("RolloutBuffer.step needs CUDA int32 actions")
        env.step_enqueue(actions, actions_ready,
                         record=(self.actions[t], self.rewards[t], self.dones[t], self.states[t + 1], self.goals[t + 1]))
        self.t = t + 1

    def returns(self, last_values, gamma):
        """[B, T] n-step returns."""
        return nstep_returns(self.rewards.t(), self.dones.t(), last_values, gamma)

    def pixel_control(self, cell_size=4, output_size=None):
        return pixel_control_reward(self.dw, self.states.t(), cell_size, output_size)

    def pixel_control_returns(self, bootstrap, gamma, cell_size=4, output_size=None, with_reward=False, max_miss=None):
        """[B, T, h*w] discounted pixel-control returns (rewards + back-up in one pass, see pixel_control_returns)."""
        return pixel_control_returns(self.dw, self.states.t(), self.dones.t(), bootstrap, gamma, cell_size, output_size,
                                     with_reward=with_reward, max_miss=max_miss)

    def auxiliary_targets(self, cell_size=4, output_size=None):
        return auxiliary_targets(self.dw, self.states[:-1].t(), self.goals[:-1].t(), cell_size, output_size)

    def targets(self, last_values, gamma, pc_bootstrap, pc_gamma, cell_size=4, output_size=None, overlap=False):
        """Everything the A2C / UNREAL losses need from one rollout: (n-step returns [B, T], pixel-control returns
        [B, T, h*w], reward-prediction (labels, zero list, non-zero list, counts)) - seven kernels of this library, no
        host synchronisation, no torch kernel.

        overlap=True runs the small builders (returns, RP labels: launch-bound kernels) on a side stream while the
        pixel-control chain - the only bandwidth-sized one - runs on the current stream, joined by events before this
        returns.  Their outputs then live in buffers OWNED by this object and are overwritten by the next call (tensors
        allocated under one stream and consumed under another would defeat torch's caching allocator)."""
        if not overlap:
            return (self.returns(last_values, gamma),
                    self.pixel_control_returns(pc_bootstrap, pc_gamma, cell_size, output_size),
                    self.reward_prediction())
        dev = self.dw.device
        if getattr(self, "_ov", None) is None:
            n = self.B * self.T
            i32 = lambda k: torch.empty(k, dtype=torch.int32, device=dev)
            self._ov = dict(side=torch.cuda.Stream(dev), fork=torch.cuda.Event(), join=torch.cuda.Event(),
                            ret=torch.empty((self.B, self.T), dtype=torch.float32, device=dev),
                            rp=(torch.empty((self.B, self.T), dtype=torch.int8, device=dev), i32(n), i32(n), i32(2),
                                i32((n + 1023) // 1024 + 1)))
        ov = self._ov
        cur = torch.cuda.current_stream(dev)
        ov["fork"].record(cur)
        ov["side"].wait_event(ov["fork"])
        with torch.cuda.stream(ov["side"]):
            ret = nstep_returns(self.rewards.t(), self.dones.t(), last_values, gamma, out=ov["ret"])
            rp = reward_prediction_labels(self.rewards.t(), sync=False, buffers=ov["rp"])
            ov["join"].record(ov["side"])
        pcr = self.pixel_control_returns(pc_bootstrap, pc_gamma, cell_size, output_size)
        cur.wait_event(ov["join"])
        return ret, pcr, rp

    def reward_prediction(self, sync=False):
        """(labels [B, T], zero positions, non-zero positions, counts) - see reward_prediction_labels; sync=False
        (default here) keeps the whole data pass free of host synchronisation."""
        return reward_prediction_labels(self.rewards.t(), sync=sync)


class ReplayRing:
    """Device-side UNREAL experience replay (SURVEY.md D6 / section 8(f) rank 1; deep_rl's replay behind
    ``self.replay.sample_sequence()`` at experiments/ai2_auxiliary/trainer.py:29).  PARITY UNPINNED: deep_rl
    is not vendored; the sampling rule is documented in include/vn_b200.h (vn_replay_sample) and restated
    in oracle/rollout.py.

    Holds state indices (24 bytes per env step), never frames; ``frames()`` / ``policy_input`` re-gather what
    a loss needs from the HBM store.  The reference keeps ~2,000 frames in total (500 per env)."""

    def __init__(self, dw: DeviceWorld, num_envs, capacity=500, seed=0, env_id_base=0):
        self.dw, self.N, self.cap, self.seed, self.env_id_base = dw, num_envs, capacity, seed, env_id_base
        dev = dw.device
        z = lambda dt: torch.zeros((capacity, num_envs), dtype=dt, device=dev)
        self.before, self.after, self.goal, self.action = z(torch.int32), z(torch.int32), z(torch.int32), z(torch.int32)
        self.goal_before = z(torch.int32)      # goal of the BEFORE observation (differs from `goal` across an auto-reset)
        self.reward, self.done = z(torch.float32), z(torch.uint8)
        self.head, self.count, self.calls = 0, 0, 0
        self._prev = self._prev_goal = None

    def start(self, env):
        """Remember the observation the next inserted step starts from (after reset())."""
        self._prev = env.obs_state.clone()
        self._prev_goal = env.goal.clone()

    def insert(self, env, actions):
        """Call after env.step(actions)."""
        if self._prev is None:
            raise RuntimeError("ReplayRing.start(env) must be called after env.reset()")
        h = self.head
        self.before[h].copy_(self._prev)
        self.goal_before[h].copy_(self._prev_goal)
        self.after[h].copy_(env.obs_state)
        self.goal[h].copy_(env.goal)
        self.action[h].copy_(actions.to(torch.int32) if torch.is_tensor(actions) else torch.as_tensor(actions))
        self.reward[h].copy_(env.reward)
        self.done[h].copy_(env.done)
        self._prev.copy_(env.obs_state)
        self._prev_goal.copy_(env.goal)
        self.head = (h + 1) % self.cap
        self.count = min(self.count + 1, self.cap)

    def extend(self, buf):
        """Appends the ``buf.t`` steps of a RolloutBuffer in bulk (same result as ``insert`` after every step of that
        rollout): at most two copies per array and rollout instead of seven copy kernels per step."""
        T = buf.t
        if T == 0:
            return
        if T > self.cap:
            raise ValueError("rollout of %d steps does not fit a replay ring of %d" % (T, self.cap))
        src = dict(before=buf.states[:T], after=buf.states[1:T + 1], goal=buf.goals[1:T + 1], goal_before=buf.goals[:T],
                   action=buf.actions[:T], reward=buf.rewards[:T], done=buf.dones[:T])
        h = self.head
        first = min(T, self.cap - h)
        for name, rows in src.items():
            dst = getattr(self, name)
            dst[h:h + first].copy_(rows[:first])
            if first < T:
                dst[:T - first].copy_(rows[first:])
        if self._prev is None:
            self._prev, self._prev_goal = buf.states[T].clone(), buf.goals[T].clone()
        else:
            self._prev.copy_(buf.states[T])
            self._prev_goal.copy_(buf.goals[T])
        self.head = (h + T) % self.cap
        self.count = min(self.count + T, self.cap)

    def _sample(self, length, mode):
        Lw = 4 if mode == 1 else length
        dev, n = self.dw.device, self.N
        out = dict(states=torch.zeros((n, Lw + 1), dtype=torch.int32, device=dev),
                   goals=torch.zeros((n, Lw + 1), dtype=torch.int32, device=dev),
                   actions=torch.zeros((n, Lw), dtype=torch.int32, device=dev),
                   rewards=torch.zeros((n, Lw), dtype=torch.float32, device=dev),
                   dones=torch.zeros((n, Lw), dtype=torch.uint8, device=dev),
                   start=torch.full((n,), -1, dtype=torch.int32, device=dev))
        if mode == 1:
            out["label"] = torch.zeros(n, dtype=torch.int8, device=dev)
        ring = L.Replay(self.before.data_ptr(), self.after.data_ptr(), self.goal.data_ptr(), self.goal_before.data_ptr(),
                        self.action.data_ptr(),
                        self.reward.data_ptr(), self.done.data_ptr(), n, self.cap, self.head, self.count)
        _call(dev, "vn_replay_sample", C.byref(ring), Lw, mode, C.c_uint64(self.seed), self.calls, self.env_id_base,
              out["states"].data_ptr(), out["goals"].data_ptr(), out["actions"].data_ptr(), out["rewards"].data_ptr(),
              out["dones"].data_ptr(), out["start"].data_ptr(), L.ptr(out.get("label")))
        self.calls += 1
        return out

    def sample_sequence(self, length):
        """One window of ``length`` transitions per env (uniform over the env's valid windows): dict of
        states / goals [N, length+1], actions / rewards / dones [N, length], start [N] (-1 = none yet)."""
        return self._sample(length, 0)

    def sample_rp_sequence(self):
        """Reward-prediction sample per env: 3 history observations (states[:, :3]), the class of the reward
        that followed (label: 0 zero / 1 positive / 2 negative), zero / non-zero drawn 50/50."""
        return self._sample(4, 1)

    def frames(self, sample, plane="rgb", scaled_float=False, goal=False):
        """Gathers the observation (or goal) frames of a sample: uint8 [N, L+1, H, W, C] or float32 CHW."""
        from .vec_env import gather_plane
        idx = sample["goals" if goal else "states"]
        if scaled_float:
            return policy_input(self.dw, idx, plane)
        out = gather_plane(self.dw, plane, idx.reshape(-1))
        return out.reshape(tuple(idx.shape) + tuple(out.shape[1:]))     # a view unless the rows are padded
