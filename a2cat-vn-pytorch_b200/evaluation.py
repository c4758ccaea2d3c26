"""Evaluation services (SURVEY.md section 8(f) rank 4): what ``trainer.test()`` (test-train.py:26) needs from the
environment side - evaluation roll-outs of a policy with success rate, episode length and SPL - and the hardness
schedule the reference sketches (``scene_complexity = LinearSchedule(0.3, 1.0, 200000)``,
experiments/thor_cached_auxiliary.py:45).  Everything stays on the device; only the final numbers are read back.

SPL (success weighted by path length): mean over episodes of ``success * l / max(p, l)`` with ``l`` the
fewest actions from the episode's start state to its goal on the STATE graph (tables.optimal_policy_table) and
``p`` the number of actions the agent took.

Two ways to evaluate: ``evaluate`` counts the first episodes to finish on the env's own random resets (quick, but biased
toward short episodes and dependent on ``num_envs``); ``evaluate_episodes`` runs a fixed list of (task, start) episodes
exactly once each - the benchmark protocol - and ``episode_set`` draws such a list reproducibly.
"""
import numpy as np
import torch


class LinearSchedule:
    """deep_rl.common.schedules.LinearSchedule as used by the experiments (thor_cached_auxiliary.py:38,45):
    linear from ``initial`` to ``final`` over ``steps`` time steps, then constant."""

    def __init__(self, initial, final, steps):
        self.initial, self.final, self.steps = float(initial), float(final), float(steps)

    def __call__(self, time_step):
        f = min(max(time_step / self.steps, 0.0), 1.0) if self.steps > 0 else 1.0
        return self.initial + (self.final - self.initial) * f


def apply_hardness_schedule(env, schedule, time_step):
    """``env.set_hardness(schedule(time_step))``; returns the value set."""
    h = schedule(time_step)
    env.set_hardness(h)
    return h


@torch.no_grad()
def evaluate(env, policy, episodes, max_steps=None):
    """Runs ``policy(obs) -> int32 CUDA actions [N]`` on ``env`` (a GraphVecEnv with ``host_outputs=False``) until
    ``episodes`` episodes have finished (the first ``episodes`` to finish are counted, like a validation run over a
    vectorised env).  Returns dict(episodes, success_rate, episode_length, reward, spl, truncated_rate, steps)."""
    if env.host_outputs:
        raise ValueError("evaluate() drives the device-resident interface: build the env with host_outputs=False")
    dev = env.device
    n = env.num_envs
    obs = env.reset()
    _, start = env.optimal_actions()
    start = start.clone().float()
    acc = torch.zeros(6, dtype=torch.float64, device=dev)      # episodes, successes, length, return, spl, truncated
    budget = torch.tensor(float(episodes), dtype=torch.float64, device=dev)
    steps = 0
    limit = max_steps if max_steps is not None else 1 << 62
    while steps < limit:
        obs, reward, done, _ = env.step(policy(obs))
        steps += 1
        # count finished episodes in env order until the budget is used up
        take = done & (torch.cumsum(done.to(torch.float64), 0) <= (budget - acc[0]))
        if bool(take.any()) or steps % 64 == 0:
            t = take.to(torch.float64)
            win = env.win.to(torch.float64) * t
            length = env.episode_length.to(torch.float64)
            acc[0] += t.sum()
            acc[1] += win.sum()
            acc[2] += (length * t).sum()
            acc[3] += (env.episode_return.to(torch.float64) * t).sum()
            acc[4] += (win * start.double() / torch.maximum(length, start.double()).clamp_min(1.0)).sum()
            acc[5] += ((env.truncated == 1).to(torch.float64) * t).sum()
            if float(acc[0]) >= episodes:
                break
        _, dist = env.optimal_actions()                         # envs that reset start a new episode here
        start = torch.where(done, dist.float(), start)
    e = max(float(acc[0]), 1.0)
    vals = acc.cpu().tolist()
    return dict(episodes=int(vals[0]), success_rate=vals[1] / e, episode_length=vals[2] / e, reward=vals[3] / e,
                spl=vals[4] / e, truncated_rate=vals[5] / e, steps=steps)


def episode_set(world, per_task, seed, complexity=None):
    """A reproducible evaluation list ``(task, start)`` (int32 numpy ``[E]``, GLOBAL indices) for
    ``evaluate_episodes`` / ``GraphVecEnv.set_episodes``: for every task, ``per_task`` start states drawn without
    replacement (all of them when ``per_task`` is None or exceeds the pool) from the task's candidate starts within the
    curriculum prefix at ``complexity`` (tables.curriculum_prefix; None = every candidate), in draw order, tasks in
    order.  Candidates that cannot reach the goal are dropped first (thor-cached lists unreachable cells at "distance"
    1, tables.build_task).  Task ``t`` draws from ``numpy.random.default_rng([seed, t])``, so its starts do not depend
    on the other tasks."""
    from .tables import optimal_policy_table
    pre = world.prefixes(complexity)
    tasks, starts = [], []
    for ti, t in enumerate(world.tasks):
        dist, _ = optimal_policy_table(world, ti)
        cand = np.asarray(t.cand_state[:int(pre[ti])], np.int64)
        cand = cand[dist[cand] >= 1]
        k = len(cand) if per_task is None else min(int(per_task), len(cand))
        pick = np.random.default_rng([int(seed), ti]).choice(len(cand), k, replace=False)
        tasks.append(np.full(k, ti, np.int32))
        starts.append((cand[pick] + int(world.scene_base[t.scene])).astype(np.int32))
    return np.concatenate(tasks), np.concatenate(starts)


@torch.no_grad()
def evaluate_episodes(env, policy, task, start, check_every=64, max_steps=None):
    """Runs ``policy(obs) -> actions [N]`` (CUDA int32 tensor, or anything ``env.step`` takes) on ``env`` over a fixed
    list of episodes, each (``task[j]``, ``start[j]``) exactly once (GraphVecEnv.set_episodes: episode ``j`` runs on the
    env with global id ``j % num_envs_total``), and scores them.  Unlike ``evaluate`` - the first episodes to finish on
    random resets, a sample biased toward short episodes that changes with ``num_envs`` - every listed episode counts,
    however long it runs, so the numbers are unbiased and the same for any batch size or shard count.  The step kernel
    records each result on the device; the host reads one counter every ``check_every`` steps.  Each rank scores the
    episodes its envs own (``env.episodes_owned``); the list is removed again before returning.

    Stops when all of this shard's episodes have ended or after ``max_steps`` steps; with neither a TimeLimit
    (``max_episode_steps > 0``) nor ``max_steps`` an episode might never end, so that is refused.  Returns a dict: the
    summary over the recorded episodes - ``episodes``, ``success_rate``, ``spl`` (mean of ``win * l / max(p, l)``,
    ``l`` = shortest-path distance of the start, ``p`` = actions taken), ``episode_length``, ``reward``,
    ``truncated_rate``, ``distance_to_goal`` (mean shortest-path distance of the final state), ``steps``,
    ``complete`` - and ``per_episode``: numpy arrays over ``env.episodes_owned`` (``index``, ``task``, ``start``,
    ``length`` (-1 = not finished), ``reward``, ``win``, ``truncated``, ``final_state``, ``distance``,
    ``final_distance``, ``spl``)."""
    if env.max_episode_steps <= 0 and max_steps is None:
        raise ValueError("evaluate_episodes needs a TimeLimit (max_episode_steps > 0) or max_steps: without one an "
                         "episode might never end")
    if check_every < 1:
        raise ValueError("check_every must be >= 1")
    env.set_episodes(task, start)
    try:
        owned = env.episodes_owned
        obs = env.reset()
        steps = 0
        while env.episodes_recorded < len(owned) and (max_steps is None or steps < max_steps):
            k = check_every if max_steps is None else min(check_every, max_steps - steps)
            for _ in range(k):
                obs = env.step(policy(obs))[0]
            steps += k
        res = {k: v.cpu().numpy() for k, v in env.episode_results().items()}
    finally:
        env.set_episodes(None)
    _, dist = env.dw.shortest_paths()
    t = torch.from_numpy(res["task"][owned].astype(np.int64)).to(env.device)
    l = dist[t, torch.from_numpy(res["start"][owned].astype(np.int64)).to(env.device)].cpu().numpy()
    fs = res["final_state"][owned].astype(np.int64)
    fd = dist[t, torch.from_numpy(np.maximum(fs, 0)).to(env.device)].cpu().numpy()
    length = res["length"][owned]
    done = length >= 0
    fd = np.where(done, fd, -1)
    win = res["win"][owned].astype(np.float64)
    spl = np.where(done, win * l / np.maximum(np.maximum(length, l), 1), 0.0)
    per = dict(index=owned, task=res["task"][owned], start=res["start"][owned], length=length,
               reward=res["ret"][owned], win=res["win"][owned], truncated=res["truncated"][owned],
               final_state=res["final_state"][owned], distance=l, final_distance=fd, spl=spl)
    m = int(done.sum())
    mean = (lambda x: float(np.mean(x[done])) if m else float("nan"))
    return dict(episodes=m, success_rate=mean(win), spl=mean(spl), episode_length=mean(length.astype(np.float64)),
                reward=mean(per["reward"].astype(np.float64)), truncated_rate=mean(per["truncated"].astype(np.float64)),
                distance_to_goal=mean(fd.astype(np.float64)), steps=steps, complete=m == len(owned), per_episode=per)
