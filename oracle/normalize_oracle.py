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


def normalize_reward_f32(rew, ret_var, clip_reward: float = 10.0, epsilon: float = 1e-8) -> np.ndarray:
    """The pass's reward: float32(clip(float64(r) / sqrt(ret_var + eps), +-clip_reward)).  Double sqrt and / are correctly
    rounded, so the kernel and numpy agree bit for bit; np.clip keeps NaN."""
    q = np.asarray(rew, np.float32).astype(np.float64) / np.sqrt(np.float64(ret_var) + np.float64(epsilon))
    return np.clip(q, -clip_reward, clip_reward).astype(np.float32)


REDUCE_GROUPS = 30      # obs_norm_reduce_kernel: 1024 threads // 34 columns


def reduce_partials(partials) -> np.ndarray:
    """obs_norm_reduce_kernel's fixed order restated: group g sums the records p = g, g + 30, ... in that order (from 0.0),
    then the 30 group sums are added in order.  Plain float64 additions: bit-identical to the kernel."""
    p = np.asarray(partials, np.float64)
    groups = np.zeros((REDUCE_GROUPS, p.shape[1]))
    for q0 in range(0, p.shape[0], REDUCE_GROUPS):
        blk = p[q0:q0 + REDUCE_GROUPS]
        groups[:blk.shape[0]] = groups[:blk.shape[0]] + blk
    out = np.zeros(p.shape[1])
    for g in range(REDUCE_GROUPS):
        out = out + groups[g]
    return out


U64 = 2.0 ** -53


def gamma_n(k) -> float:
    """Higham's gamma_k = k u / (1 - k u): the relative error bound of k float64 roundings in a row."""
    return k * U64 / (1.0 - k * U64)


def combine_bound(mean, var, count, s1, s2, cb):
    """Bound on |kernel - SB3 update_from_moments| for the (mean, var) after merging one batch given by its shifted sums
    s1 = sum(x - mean), s2 = sum((x - mean)^2) over cb values.  SB3's side receives batch_mean = mean + s1 / cb and
    batch_var = s2 / cb - (s1 / cb)^2; the kernel uses delta = s1 / cb directly and nvcc may contract its products and sums
    into FMAs.  Both evaluations are within the forward error of the exact result, so the bound is twice that:
        delta:  |e_d| <= u (|mean| + 3 |delta|)                (SB3's batch_mean - mean round trip; the kernel's is u |delta|)
        delta^2:      <= 2 |delta| e_d + 3 u delta^2
        mean'   = mean + delta cb / tot:      gamma_4 (|mean| + |delta|) + e_d
        var'    = (T1 + T2 + T3) / tot, T1 = var count, T2 = var_b cb, T3 = delta^2 count cb / tot:
                  [gamma_6 (T1 + T2 + T3 + s2) + (cb + count cb / tot) e_d2] / tot
    Returns (bound on mean', bound on var'), elementwise."""
    mean, var, s1, s2 = (np.asarray(a, np.float64) for a in (mean, var, s1, s2))
    delta = s1 / cb
    var_b = np.maximum(s2 / cb - delta * delta, 0.0)
    tot = count + cb
    e_d = U64 * (np.abs(mean) + 3 * np.abs(delta))
    e_d2 = 2 * np.abs(delta) * e_d + 3 * U64 * delta * delta
    b_mean = gamma_n(4) * (np.abs(mean) + np.abs(delta)) + e_d
    t1, t2, t3 = var * count, var_b * cb, delta * delta * count * cb / tot
    b_var = (gamma_n(6) * (t1 + t2 + t3 + s2) + (cb + count * cb / tot) * e_d2) / tot
    return 2 * b_mean, 2 * b_var


def combine_sb3(rms: RunningMeanStd, s1, s2, cb):
    """SB3 update_from_moments fed with the batch moments of the shifted sums (shift = rms.mean)."""
    delta = np.asarray(s1, np.float64) / cb
    rms.update_from_moments(rms.mean + delta, np.maximum(np.asarray(s2, np.float64) / cb - delta * delta, 0.0), cb)


def two_pass_moments(x):
    """(batch mean, population variance) of the rows of x in two passes, as np.mean / np.var take them, but summed in
    extended precision along a contiguous axis (numpy's pairwise summation): np.mean(axis=0) of a C-ordered [N, F] array
    adds the N rows one after another, an error of N float64 roundings that would swamp the kernel's.  What is left is
    the final rounding to float64 plus ~(log2 N + 20) roundings of the extended type (ref_depth)."""
    x = np.asarray(x, np.float64)
    n = x.shape[0]
    xt = np.ascontiguousarray(x.reshape(n, -1).T).astype(np.longdouble)
    m = xt.sum(axis=1) / n
    v = np.square(xt - m[:, None]).sum(axis=1) / n
    shape = x.shape[1:]
    return m.astype(np.float64).reshape(shape), v.astype(np.float64).reshape(shape)


def ref_depth(cb) -> float:
    """two_pass_moments' own error in float64 roundings (the pairwise blocks of 128, then log2 levels, in long double)"""
    return 1 + (np.log2(max(cb, 2.0)) + 20) * float(np.finfo(np.longdouble).eps) / (2 * U64)


def one_pass_bound(mean, var, count, s2, cb, depth: int):
    """Bound on |kernel - SB3 update_from_moments(two_pass_moments(data))| for the (mean, var) after one rollout: the
    kernel's batch moments come from one pass of shifted sums.  Each of the cb shifted values d = x - c carries one
    rounding; s1 and s2 are sums of depth = K + 5 + 8 + ceil(P / 30) + 30 additions deep at most (each env's K steps, the
    warp shuffle tree, the 8-warp fold, then the reduce's P / 30 records per group and its 30 groups), so
        |e_s2| <= gamma_{depth + 3} s2,  |e_s1| <= gamma_{depth + 1} sum|d| <= gamma_{depth + 1} sqrt(cb s2)
    and the shifted one-pass formula var_b = s2 / cb - delta^2 inherits
        |e_var_b| <= gamma_{depth + 4} (s2 / cb) + 2 |delta| |e_delta| <= gamma_{depth + 4} (2 s2 / cb + delta^2)
    (Cauchy-Schwarz: sum|d| / cb <= sqrt(s2 / cb); 2 a b <= a^2 + b^2).  This is relative to the spread about the shift,
    not to var_b: with the initial statistics (shift 0) and features far from zero it is the cancellation of the one-pass
    formula, |e_var_b| ~ gamma (s2 / cb + delta^2).  The reference's batch mean is rounded to float64 and SB3 subtracts
    the running mean from it (the |mean| term of e_delta); its own summation error adds ref_depth(cb) roundings.
    Propagated through the combine (var_b enters with weight cb / tot, delta^2 with count cb / tot^2, delta with
    cb / tot), plus the combine's own rounding (combine_bound), with |delta| <= sqrt(s2 / cb) throughout.  Returns
    (bound on mean', bound on var')."""
    mean, var, s2 = (np.asarray(a, np.float64) for a in (mean, var, s2))
    g = gamma_n(depth + 4 + ref_depth(cb))
    d_max = np.sqrt(s2 / cb)                            # |delta| <= sqrt(s2 / cb): the batch mean lies inside the spread
    e_delta = g * (d_max + np.abs(mean))
    e_d2 = (2 * d_max + e_delta) * e_delta              # |(delta + e)^2 - delta^2|: a constant column has s2 = 0, but
    e_var_b = g * (2 * s2 / cb + d_max * d_max) + e_d2  # its float64 batch mean minus the shift need not be 0
    tot = count + cb
    c_mean, c_var = combine_bound(mean, var, count, d_max * cb, s2, cb)
    return (e_delta * cb / tot + c_mean,
            (e_var_b * cb + e_d2 * count * cb / tot) / tot + c_var)


def pass_depth(K: int, n: int) -> int:
    """The deepest chain of additions behind one moment: K steps, 5 shuffle levels, the 8-warp fold, the reduce."""
    P = -(-n // 256)
    return K + 5 + 8 + -(-P // REDUCE_GROUPS) + REDUCE_GROUPS


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
