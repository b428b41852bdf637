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
