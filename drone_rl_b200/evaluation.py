"""Policy evaluation on the GPU: SB3's ``evaluate_policy`` and ``EvalCallback`` over one actor-only kernel
(csrc/ppo_eval.cuh, DESIGN.md section 10).

``evaluate_policy(model, env, ...)`` computes what SB3's function returns for ``env = VecMonitor(DummyVecEnv([DroneGymEnv]
* N))`` (restated in oracle/eval_oracle.py): one reset, env g of the N evaluation envs records ``(n_eval_episodes + g) //
N`` episodes, all envs step in lockstep until every env has its episodes, and the lists come in SB3's order (by step of
completion, then by env index).  The steps run inside the kernel: a few probe launches of ``PROBE_CHUNK`` steps, each
followed by one 4-byte readback (how many envs are still below target), then one catch-up launch that brings every env to
the same step count T.  SB3's per-step ``callback`` and ``render`` have nothing to run on and are refused.

The model's training env, parameters, optimiser state and normalisation statistics are not touched; with ``norm_obs`` the
policy sees observations normalised by the model's current (frozen) record, as SB3's ``sync_envs_normalization`` and
``training=False`` give.  Returns are raw rewards, also under ``norm_reward``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np
import torch

from . import _lib
from .core import _ptr, _stream_ptr

PROBE_CHUNK = 1024        # steps per probe launch (five episodes of the default 200-step limit)


def _dist():
    d = torch.distributed
    if d.is_available() and d.is_initialized():
        return d, d.get_rank(), d.get_world_size()
    return None, 0, 1


def evaluate_policy(model, env, n_eval_episodes: int = 10, deterministic: bool = True, render: bool = False,
                    callback=None, reward_threshold: Optional[float] = None, return_episode_rewards: bool = False):
    """SB3 ``evaluate_policy``: ``(mean_reward, std_reward)``, or the lists ``(episode_rewards, episode_lengths)`` with
    ``return_episode_rewards``.  ``env`` is a ``DroneBatch`` or anything with ``.batch`` (e.g. ``DroneVecEnv``).  Under
    ``torch.distributed`` every rank passes its own shard (the same number of envs on every rank); the targets count over
    all ranks' envs, and every rank returns the gathered lists."""
    if render:
        raise ValueError("evaluate_policy: render is not supported (the steps run inside one kernel)")
    if callback is not None:
        raise ValueError("evaluate_policy: a per-step callback is not supported (the steps run inside one kernel)")
    if int(n_eval_episodes) < 1:
        raise ValueError("evaluate_policy: n_eval_episodes must be at least 1")
    batch = getattr(env, "batch", env)
    if batch.obs_dim != 15 or not batch.config.auto_reset:
        raise ValueError("evaluate_policy needs the DroneGymEnv spec (15-dim obs) with auto-reset")
    n_eval_episodes = int(n_eval_episodes)
    lib, dev, n = batch.lib, batch.device, batch.n
    dist, rank, world = _dist()
    if dist is not None:
        sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([n], dtype=torch.int64, device=dev))
        if any(int(s) != n for s in sizes):
            raise ValueError(f"evaluate_policy: every rank needs the same number of eval envs, got {[int(s) for s in sizes]}")
    n_global, index0 = world * n, rank * n
    max_eps = -(-n_eval_episodes // n_global)

    batch.reset()                                          # SB3: observations = env.reset()
    steps = torch.zeros(n, dtype=torch.int32, device=dev)
    count = torch.zeros(n, dtype=torch.int32, device=dev)
    ep_ret = torch.zeros(n, max_eps, dtype=torch.float32, device=dev)
    ep_len = torch.zeros(n, max_eps, dtype=torch.int32, device=dev)
    pending = torch.zeros(1, dtype=torch.int32, device=dev)
    a = _lib.EvalArgs()
    a.t0, a.deterministic, a.max_eps = batch.global_step, int(bool(deterministic)), max_eps
    a.env_index0, a.n_global, a.n_eval_episodes = index0, n_global, n_eval_episodes
    a.d_steps, a.d_count, a.d_ep_return, a.d_ep_length, a.d_pending = (t.data_ptr() for t in (steps, count, ep_ret, ep_len, pending))
    nz = getattr(model, "normalizer", None)
    affine = nz.affine_ptr() if nz is not None else None
    tc = int(model.rollout_precision == "tf32" and n > model.tc_min_envs)
    st = _stream_ptr(dev)

    def launch(limit: int, catch_up: bool):
        a.limit, a.catch_up = limit, int(catch_up)
        _lib.check(lib.dronecu_evaluate_policy(batch._h, _ptr(model.params), affine, tc, C.byref(a), st), "dronecu_evaluate_policy")

    limit = 0
    while True:                                            # probe: each env runs to its target or the end of the chunk
        limit += PROBE_CHUNK
        pending.zero_()
        launch(limit, False)
        if dist is not None:
            dist.all_reduce(pending)
        if int(pending.item()) == 0:
            break
    T = steps.max()
    if dist is not None:
        dist.all_reduce(T, op=dist.ReduceOp.MAX)
    T = int(T.item())
    launch(T, True)                                         # catch-up: every env to step T
    batch.global_step = a.t0 + T

    # the recorded episodes of an env are its first count_i after the reset: episode j ended at step sum(len[:j + 1])
    cnt, r, ln = count.cpu().numpy(), ep_ret.cpu().numpy(), ep_len.cpu().numpy()
    env = np.repeat(np.arange(n), cnt)
    j = np.arange(env.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    done_at = np.cumsum(np.where(np.arange(max_eps) < cnt[:, None], ln, 0), axis=1)[env, j]
    rows = (done_at.astype(np.int64), env.astype(np.int64) + index0, r[env, j], ln[env, j])
    if dist is not None:
        every = [None] * world
        dist.all_gather_object(every, rows)
        rows = tuple(np.concatenate(part) for part in zip(*every))
    order = np.lexsort((rows[1], rows[0]))                  # by step of completion, then by global env index
    episode_rewards, episode_lengths = rows[2][order].tolist(), rows[3][order].tolist()
    mean_reward, std_reward = np.mean(episode_rewards), np.std(episode_rewards)
    if reward_threshold is not None:
        assert mean_reward > reward_threshold, f"Mean reward below threshold: {mean_reward:.2f} < {reward_threshold:.2f}"
    if return_episode_rewards:
        return episode_rewards, episode_lengths
    return mean_reward, std_reward


class EvalCallback:
    """SB3 ``EvalCallback`` as a ``PPO.learn(callback=...)`` callable.  It evaluates after every iteration that crossed a
    multiple of ``eval_freq`` vec-env steps (one vec-env step = one step of every env of a rank).  This is the one departure
    from SB3, which evaluates in the middle of the rollout with the parameters before the update: here the evaluation
    sees the parameters after the iteration's update.

    Per evaluation: ``eval/mean_reward`` and ``eval/mean_ep_length`` go into ``model.logger_values``; with ``log_path`` the
    lists are appended to ``log_path/evaluations.npz`` (SB3's keys ``timesteps``, ``results``, ``ep_lengths``); on a new best
    mean reward, with ``best_model_save_path``, ``best_model.zip`` is saved (``model.save`` on every rank, as train.py
    saves)."""

    def __init__(self, eval_env, n_eval_episodes: int = 5, eval_freq: int = 10000, deterministic: bool = True,
                 log_path: Optional[str] = None, best_model_save_path: Optional[str] = None, verbose: int = 1):
        self.eval_env, self.n_eval_episodes, self.eval_freq = eval_env, int(n_eval_episodes), int(eval_freq)
        self.deterministic, self.verbose = deterministic, verbose
        self.log_path = None if log_path is None else os.path.join(log_path, "evaluations.npz")
        self.best_model_save_path = best_model_save_path
        self.best_mean_reward, self.last_mean_reward = -np.inf, -np.inf
        self.evaluations_timesteps, self.evaluations_results, self.evaluations_length = [], [], []
        self.n_calls = 0                  # vec-env steps seen

    def __call__(self, model) -> bool:
        before = self.n_calls
        self.n_calls += model.n_steps
        if self.eval_freq <= 0 or self.n_calls // self.eval_freq == before // self.eval_freq:
            return True
        rewards, lengths = evaluate_policy(model, self.eval_env, self.n_eval_episodes, self.deterministic,
                                           return_episode_rewards=True)
        mean_reward, std_reward = float(np.mean(rewards)), float(np.std(rewards))
        mean_len, std_len = float(np.mean(lengths)), float(np.std(lengths))
        self.last_mean_reward = mean_reward
        rank = getattr(model, "rank", 0)
        if self.log_path is not None:
            self.evaluations_timesteps.append(model.num_timesteps)
            self.evaluations_results.append(rewards)
            self.evaluations_length.append(lengths)
            if rank == 0:
                np.savez(self.log_path, timesteps=self.evaluations_timesteps, results=self.evaluations_results,
                         ep_lengths=self.evaluations_length)
        if self.verbose >= 1 and rank == 0:
            print(f"Eval num_timesteps={model.num_timesteps}, episode_reward={mean_reward:.2f} +/- {std_reward:.2f}")
            print(f"Episode length: {mean_len:.2f} +/- {std_len:.2f}", flush=True)
        model.logger_values.update({"eval/mean_reward": mean_reward, "eval/mean_ep_length": mean_len})
        if mean_reward > self.best_mean_reward:
            if self.verbose >= 1 and rank == 0:
                print("New best mean reward!", flush=True)
            if self.best_model_save_path is not None:
                model.save(os.path.join(self.best_model_save_path, "best_model"))
            self.best_mean_reward = mean_reward
        return True
