"""TEST INFRASTRUCTURE: SB3's ``VecNormalize`` / ``RunningMeanStd`` restated in float64 numpy (PARITY UNPINNED, like the
rest of the PPO oracle: stable-baselines3 is not installed here), plus the frozen-per-rollout application the GPU path
uses (drone_rl_b200/normalize.py): rollout i is normalised with the statistics after rollout i-1, then its raw
observations and discounted returns update them in one ``update_from_moments``.

SB3 (common/running_mean_std.py, common/vec_env/vec_normalize.py):
    RunningMeanStd(epsilon=1e-4): mean 0, var 1, count epsilon
    update(x): batch_mean = mean(x, 0), batch_var = var(x, 0) (population), batch_count = len(x) -> update_from_moments
    update_from_moments: delta = bm - m; tot = c + bc; m += delta * bc / tot;
                         var = (var * c + bv * bc + delta^2 * c * bc / tot) / tot; c = tot
    normalize_obs: clip((obs - mean) / sqrt(var + eps), -clip_obs, clip_obs), eps 1e-8, clip_obs 10
    reward: returns = returns * gamma + r; ret_rms.update(returns); r / sqrt(ret_var + eps) clipped at clip_reward 10;
            returns[dones] = 0
"""
from __future__ import annotations

import numpy as np
import torch

from . import drone_oracle as do
from . import ppo_oracle as po
from .ppo_loop import PPOLoopOracle


class RunningMeanStd:
    def __init__(self, shape=(), epsilon: float = 1e-4):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = float(epsilon)

    def update(self, x: np.ndarray):
        x = np.asarray(x, np.float64)
        self.update_from_moments(x.mean(axis=0), x.var(axis=0), x.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot
        m_2 = self.var * self.count + batch_var * batch_count + np.square(delta) * self.count * batch_count / tot
        self.mean, self.var, self.count = new_mean, m_2 / tot, tot


def shifted_moments(x: np.ndarray, c) -> tuple:
    """(batch mean, population variance, count) of the rows of x from the sums of (x - c) and (x - c)^2 -- what the pass
    accumulates (c = the running mean, so that features far from zero do not cancel)."""
    d = np.asarray(x, np.float64) - c
    n = d.shape[0]
    s1, s2 = d.sum(axis=0), np.square(d).sum(axis=0)
    delta = s1 / n
    return c + delta, np.maximum(s2 / n - delta * delta, 0.0), n


def normalize_obs(obs, rms: RunningMeanStd, clip_obs: float = 10.0, epsilon: float = 1e-8) -> np.ndarray:
    return np.clip((np.asarray(obs, np.float64) - rms.mean) / np.sqrt(rms.var + epsilon), -clip_obs, clip_obs)


def normalize_obs_f32(obs, rms: RunningMeanStd, clip_obs: float = 10.0, epsilon: float = 1e-8) -> np.ndarray:
    """The float32 form the kernels evaluate: mean_f = f32(mean), rstd_f = f32(1 / sqrt(var + eps)), then a float32
    subtract, a float32 multiply (no FMA) and the clip."""
    mean_f = rms.mean.astype(np.float32)
    rstd_f = (1.0 / np.sqrt(rms.var + epsilon)).astype(np.float32)
    y = (np.asarray(obs, np.float32) - mean_f).astype(np.float32) * rstd_f
    return np.clip(y.astype(np.float32), np.float32(-clip_obs), np.float32(clip_obs))


class FrozenVecNormalize:
    """VecNormalize with the statistics frozen per rollout.  ``apply(obs, rew, done)`` takes one rollout's RAW [K,n,15]
    observations (the rows the policy acted on), [K,n] rewards and dones; returns the normalised observations and rewards
    (float64) computed with the statistics before the call, and -- when ``training`` -- then updates the statistics."""

    def __init__(self, n_envs: int, gamma: float = 0.99, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, epsilon: float = 1e-8):
        self.obs_rms, self.ret_rms = RunningMeanStd((15,)), RunningMeanStd(())
        self.returns = np.zeros(n_envs, np.float64)
        self.gamma, self.norm_obs, self.norm_reward = gamma, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.epsilon = clip_obs, clip_reward, epsilon
        self.training = True

    def normalize(self, obs) -> np.ndarray:
        return normalize_obs(obs, self.obs_rms, self.clip_obs, self.epsilon) if self.norm_obs else np.asarray(obs, np.float64)

    def apply(self, obs, rew, done):
        obs, rew, done = np.asarray(obs, np.float64), np.asarray(rew, np.float64), np.asarray(done, bool)
        K = obs.shape[0]
        obs_n = self.normalize(obs)
        rew_n = rew.copy()
        if self.norm_reward:
            scale = np.sqrt(self.ret_rms.var + self.epsilon)
            rets = np.empty_like(rew)
            for k in range(K):
                if self.training:
                    self.returns = self.returns * self.gamma + rew[k]
                rets[k] = self.returns
                self.returns[done[k]] = 0.0
            rew_n = np.clip(rew / scale, -self.clip_reward, self.clip_reward)
            if self.training:
                self.ret_rms.update(rets.reshape(-1))
        if self.training and self.norm_obs:
            self.obs_rms.update(obs.reshape(-1, obs.shape[-1]))
        return obs_n, rew_n


class NormalizedPPOLoopOracle(PPOLoopOracle):
    """``PPOLoopOracle`` (oracle/ppo_loop.py) with the normalisation step of the GPU path: the policy sees observations
    normalised with the statistics of the previous rollout, the buffer holds normalised observations and rewards, and the
    rollout's raw rows / returns update the statistics afterwards.  The plain loop (what bench.py's CPU legs run) is not
    changed: this is a subclass."""

    def __init__(self, *args, normalize: FrozenVecNormalize, **kw):
        super().__init__(*args, **kw)
        self.norm = normalize

    def collect_rollouts(self):
        norm, K, n = self.norm, self.K, self.n
        obs_b = torch.empty(K, n, po.OBS, dtype=self.dtype)
        act_b = torch.empty(K, n, po.ACT, dtype=self.dtype)
        logp_b = torch.empty(K, n, dtype=self.dtype)
        val_b = torch.empty(K, n, dtype=self.dtype)
        rew_b = np.empty((K, n), np.float64)
        done_b = np.empty((K, n), bool)
        raw_b = np.empty((K, n, po.OBS), np.float64)
        with torch.no_grad():
            for t in range(K):
                raw_b[t] = self.obs
                o = torch.from_numpy(norm.normalize(self.obs)).to(self.dtype)
                mean, value, log_std = po.forward(self.theta, o)
                a = mean + torch.exp(log_std) * torch.randn(mean.shape, generator=self.gen, dtype=self.dtype)
                logp = po.log_prob(mean, log_std, a)
                clipped = np.clip(a.numpy().astype(np.float32), 0.0, do.MOTOR_MAX)
                self.obs, rew, done, info = self.env.step(clipped.astype(np.float64))
                obs_b[t], act_b[t], logp_b[t], val_b[t] = o, a, logp, value
                rew_b[t] = rew.astype(np.float32)
                done_b[t] = done
                for i in np.flatnonzero(done):
                    self.ep_returns.append(float(info["episode_r"][i]))
                    self.ep_lengths.append(int(info["episode_l"][i]))
            _, last_value, _ = po.forward(self.theta, torch.from_numpy(norm.normalize(self.obs)).to(self.dtype))
            _, rew_n = norm.apply(raw_b, rew_b, done_b)
            adv, ret = po.gae(torch.from_numpy(rew_n).to(self.dtype), val_b, torch.from_numpy(done_b), last_value)
        self.num_timesteps += K * n
        self.buf = tuple(x.reshape(K * n, *x.shape[2:]) for x in (obs_b, act_b, logp_b, adv, ret))
