"""TEST INFRASTRUCTURE: the oracle PPO loops (oracle/ppo_loop.py, oracle/normalize_oracle.py) with SB3's time-limit
bootstrap, as ``collect_rollouts`` runs it on a Gymnasium env (``handle_timeout_termination``; DESIGN.md section 11):

    for idx, done in enumerate(dones):
        if done and infos[idx].get("terminal_observation") is not None and infos[idx].get("TimeLimit.truncated", False):
            terminal_value = self.policy.predict_values(terminal_obs)[0]
            rewards[idx] += self.gamma * terminal_value

``TimeLimit.truncated`` is the oracle env's ``info["truncated"]`` (time limit and no crash), the terminal observation its
``info["terminal_obs"]``.  The loops themselves are not changed: the subclasses hook the env step (and, normalised, the
VecNormalize step) of one instance.  gamma is the loops' 0.99, the gamma of their GAE.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import ppo_oracle as po
from oracle.normalize_oracle import NormalizedPPOLoopOracle
from oracle.ppo_loop import PPOLoopOracle

GAMMA = 0.99


def terminal_values(theta, info, dtype, normalize=None) -> list:
    """[(env index, V(terminal observation))] for the envs whose step ended by the time limit alone; V as SB3's
    ``policy.predict_values(terminal_obs)[0]``, a tensor of shape [1].  ``normalize``: VecNormalize.step_wait's
    normalisation of the terminal observation."""
    out = []
    with torch.no_grad():
        for idx in np.flatnonzero(info["truncated"]):
            term = info["terminal_obs"][idx:idx + 1]
            if normalize is not None:
                term = normalize(term)
            out.append((int(idx), po.forward(theta, torch.from_numpy(np.asarray(term)).to(dtype))[1]))
    return out


def bootstrap_truncated(rewards: np.ndarray, values: list, gamma: float = GAMMA) -> None:
    """SB3's line, literally: ``rewards[idx] += self.gamma * terminal_value`` (numpy rewards, Python float gamma, torch
    value), in place."""
    for idx, terminal_value in values:
        rewards[idx] += gamma * terminal_value


class TimeoutPPOLoopOracle(PPOLoopOracle):
    """PPOLoopOracle whose float32 step rewards (DummyVecEnv's buffer) carry the bootstrap of truncated steps."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        step = self.env.step

        def step_bootstrapped(action):
            obs, rew, done, info = step(action)
            r32 = rew.astype(np.float32)
            bootstrap_truncated(r32, terminal_values(self.theta, info, self.dtype))
            return obs, r32.astype(np.float64), done, info     # exact: the loop casts it back to float32
        self.env.step = step_bootstrapped


class TimeoutNormalizedPPOLoopOracle(NormalizedPPOLoopOracle):
    """NormalizedPPOLoopOracle with the bootstrap added to the NORMALISED reward (SB3's collect_rollouts runs on what
    VecNormalize returns), the terminal observation normalised with the statistics of its step (VecNormalize.step_wait;
    here the rollout's frozen ones).  The returns and the statistics see the raw rewards."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        step, apply, pending = self.env.step, self.norm.apply, []

        def step_recorded(action):
            res = step(action)
            pending.append(terminal_values(self.theta, res[3], self.dtype, self.norm.normalize))
            return res

        def apply_bootstrapped(obs, rew, done):
            obs_n, rew_n = apply(obs, rew, done)
            for t, values in enumerate(pending):
                bootstrap_truncated(rew_n[t], values)
            pending.clear()
            return obs_n, rew_n
        self.env.step = step_recorded
        self.norm.apply = apply_bootstrapped
