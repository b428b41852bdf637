"""TEST INFRASTRUCTURE: SB3's ``evaluate_policy`` restated, and the same bookkeeping over recorded transitions.

PARITY UNPINNED, like the other SB3 restatements (stable-baselines3 is not installed here).  The code restated is
``stable_baselines3.common.evaluation.evaluate_policy`` (published behaviour; the reference calls SB3 through
``PPO.predict`` only, train.py / test.py), for an env that is ``VecMonitor(DummyVecEnv([DroneGymEnv] * N))``:

* ``env.reset()`` once; env ``i`` records ``target_i = (n_eval_episodes + i) // N`` episodes;
* all envs step together while any env is below its target; an env past its target keeps stepping (and auto-resetting)
  but records nothing;
* on ``done`` of an env below target, VecMonitor's ``info["episode"]`` -- the float32 running return and the int
  length -- is appended, so the lists are ordered by step of completion, then by env index;
* ``mean`` / ``std`` are ``np.mean`` / ``np.std`` (population) of the returns; ``reward_threshold`` asserts
  ``mean > threshold``; ``return_episode_rewards`` returns the two lists.

``evaluate_policy`` below is that loop, literally, over any VecEnv-shaped object (``VecMonitorOracle(DummyVecEnvOracle(
...))`` in the tests).  ``episodes_from_transitions`` is the same bookkeeping over a record of float32 rewards and done
flags ``[T, N]`` -- what the GPU evaluation is checked against, after a rollout of the same envs.
"""
from __future__ import annotations

import dataclasses

import numpy as np

from . import drone_oracle as do


def evaluate_policy(policy, env, n_eval_episodes: int = 10, reward_threshold=None, return_episode_rewards: bool = False):
    """SB3's loop; ``policy(obs [N,D]) -> actions [N,4]`` (the action the env receives, already clipped)."""
    n_envs = env.num_envs
    episode_rewards, episode_lengths = [], []
    episode_counts = np.zeros(n_envs, dtype="int")
    episode_count_targets = np.array([(n_eval_episodes + i) // n_envs for i in range(n_envs)], dtype="int")
    observations = env.reset()
    while (episode_counts < episode_count_targets).any():
        actions = policy(observations)
        new_observations, rewards, dones, infos = env.step(actions)
        for i in range(n_envs):
            if episode_counts[i] < episode_count_targets[i]:
                if dones[i] and "episode" in infos[i]:
                    episode_rewards.append(infos[i]["episode"]["r"])
                    episode_lengths.append(infos[i]["episode"]["l"])
                    episode_counts[i] += 1
        observations = new_observations
    mean_reward, std_reward = np.mean(episode_rewards), np.std(episode_rewards)
    if reward_threshold is not None:
        assert mean_reward > reward_threshold, f"Mean reward below threshold: {mean_reward:.2f} < {reward_threshold:.2f}"
    if return_episode_rewards:
        return episode_rewards, episode_lengths
    return mean_reward, std_reward


def episodes_from_transitions(reward, done, n_eval_episodes: int):
    """The same bookkeeping over recorded transitions: ``reward`` float32 [T, N], ``done`` bool [T, N] of N envs stepped in
    lockstep from a reset.  Returns (returns, lengths, T_needed): the episode lists in SB3's order and the number of steps
    after which every env had reached its target (ValueError if the record is too short)."""
    reward, done = np.asarray(reward, np.float32), np.asarray(done, bool)
    T, n = reward.shape
    targets = np.array([(n_eval_episodes + i) // n for i in range(n)])
    counts = np.zeros(n, int)
    ret = np.zeros(n, np.float32)            # VecMonitor keeps a float32 running return
    length = np.zeros(n, int)
    returns, lengths = [], []
    for t in range(T):
        if not (counts < targets).any():
            return returns, lengths, t
        ret += reward[t]
        length += 1
        for i in np.flatnonzero(done[t]):
            if counts[i] < targets[i]:
                returns.append(float(ret[i]))
                lengths.append(int(length[i]))
                counts[i] += 1
            ret[i], length[i] = 0.0, 0
    if (counts < targets).any():
        raise ValueError("the record ends before every env reached its target")
    return returns, lengths, T


def shard_targets(n_eval_episodes: int, env_index0: int, n_global: int, n: int):
    """the targets of the n envs of one shard: env i is env ``env_index0 + i`` of the ``n_global`` evaluation envs"""
    return (int(n_eval_episodes) + int(env_index0) + np.arange(n, dtype=np.int64)) // int(n_global)


def launch_sequence(reward, done, targets, launches, max_eps: int, ep_ret0=None, ep_len0=None):
    """The launch contract of ``dronecu_evaluate_policy`` (csrc/ppo_eval.cuh) restated over a record: ``reward`` float32
    [T, n] and ``done`` bool [T, n] of the n envs stepped from the evaluation's first step, ``targets`` [n],
    ``launches`` a list of (limit, catch_up), ``ep_ret0`` / ``ep_len0`` the running return and length of every env at
    the first step (default 0: a fresh reset).

    One launch steps env i from ``steps[i]`` while ``steps[i] < limit`` and (catch-up or ``count[i] < target[i]``);
    step c adds reward[c] to the float32 running return and 1 to the length, and on done[c] records (return, length) in
    slot ``count[i]`` if ``count[i] < target[i]`` (then ``count[i] += 1``) and zeroes both.  A probe adds to ``pending``
    the envs still below target; a catch-up leaves it alone.

    Returns ``(after, ep_return, ep_length, written)``: ``after`` one dict of ``steps``, ``count`` and ``pending`` (None
    for a catch-up) per launch; ``ep_return`` float32 / ``ep_length`` int [n, max_eps] with ``written`` [n, max_eps] bool
    the slots the launches wrote.  ValueError if a launch needs a step past the end of the record."""
    reward, done = np.asarray(reward, np.float32), np.asarray(done, bool)
    T, n = reward.shape
    targets = np.asarray(targets, np.int64)
    ret = np.zeros(n, np.float32) if ep_ret0 is None else np.asarray(ep_ret0, np.float32).copy()
    length = np.zeros(n, np.int64) if ep_len0 is None else np.asarray(ep_len0, np.int64).copy()
    steps, count = np.zeros(n, np.int64), np.zeros(n, np.int64)
    ep_return, ep_length = np.zeros((n, max_eps), np.float32), np.zeros((n, max_eps), np.int64)
    written = np.zeros((n, max_eps), bool)
    after = []
    for limit, catch_up in launches:
        lo = int(steps.min()) if n else 0
        for c in range(lo, max(lo, int(limit))):
            going = bool(catch_up) | (count < targets)
            if not (going & (steps >= c)).any():
                break
            live = going & (steps == c)
            if not live.any():
                continue
            if c >= T:
                raise ValueError(f"launch to step {limit} needs step {c}, past the end of the record ({T} steps)")
            ret[live] = (ret[live] + reward[c, live]).astype(np.float32)
            length[live] += 1
            end = live & done[c]
            rec = np.flatnonzero(end & (count < targets))
            ep_return[rec, count[rec]] = ret[rec]
            ep_length[rec, count[rec]] = length[rec]
            written[rec, count[rec]] = True
            count[rec] += 1
            ret[end], length[end] = 0.0, 0
            steps[live] += 1
        after.append({"steps": steps.copy(), "count": count.copy(),
                      "pending": None if catch_up else int((count < targets).sum())})
    return after, ep_return, ep_length, written


def episode_lists(count, ep_return, ep_length, env_index0: int = 0, ep_len0=None):
    """The rows of a shard's slots as ``evaluation.evaluate_policy`` forms them: (step of completion, global env index,
    return, length) of every recorded episode, env by env.  ``ep_len0``: the running lengths at the first step (default
    0); slots past ``count`` are not read."""
    count = np.asarray(count, np.int64)
    n, max_eps = np.shape(ep_length)
    len0 = np.zeros(n, np.int64) if ep_len0 is None else np.asarray(ep_len0, np.int64)
    env = np.repeat(np.arange(n), count)
    j = np.arange(env.size) - np.repeat(np.cumsum(count) - count, count)
    ln = np.where(np.arange(max_eps) < count[:, None], np.asarray(ep_length, np.int64), 0)
    done_at = np.cumsum(ln, axis=1)[env, j] - len0[env]
    return (done_at.tolist(), (env + int(env_index0)).tolist(), np.asarray(ep_return, np.float32)[env, j].tolist(),
            ln[env, j].tolist())


def sb3_order(*shard_rows):
    """SB3's lists from the rows of every shard: by step of completion, then by global env index"""
    rows = [[x for r in shard_rows for x in r[k]] for k in range(4)]
    order = np.lexsort((np.asarray(rows[1], np.int64), np.asarray(rows[0], np.int64)))
    return [rows[2][j] for j in order], [int(rows[3][j]) for j in order]


class OracleDroneGymEnv:
    """One float64 oracle env with the legacy gym API of ``DroneGymEnv`` (no auto-reset: DummyVecEnv resets it), global id
    ``env_id`` of the Philox streams.  The constructor resets once, as ``DroneGymEnv.__init__`` does."""

    def __init__(self, seed: int = 0, env_id: int = 0):
        self.env = do.BatchedDroneOracle(1, dataclasses.replace(do.SINGLE, auto_reset=False), seed=seed, env_offset=env_id)

    def reset(self):
        return self.env.reset()[0]

    def step(self, action):
        obs, rew, done, _ = self.env.step(np.asarray(action, np.float64).reshape(1, 4))
        return obs[0], float(rew[0]), bool(done[0]), {}
