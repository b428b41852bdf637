"""Observation and reward normalisation of the GPU rollout: SB3's ``VecNormalize(norm_obs, norm_reward)`` where the rollout
lives, in the rollout kernels and one pass over the rollout buffer (csrc/obs_norm.cuh, include/dronecu.h).

One deliberate departure from SB3: the running statistics are frozen for the length of a rollout launch.  SB3 updates
``obs_rms`` / ``ret_rms`` after every env step; inside a fused K-step kernel that would need a grid-wide reduction per step.
Here rollout i normalises with the statistics as they stood after rollout i-1 and the moments of rollout i are merged in
one update afterwards (the first rollout runs with the initial statistics: mean 0, var 1, i.e. identity clipped at +-10).

All state lives on the device (the statistics, the float32 affine record the kernels read, the per-env discounted returns,
the CTA partial records); :class:`ObsNormalizer` hides the record layouts from ``PPO``.
"""
from __future__ import annotations

import ctypes as C
from types import SimpleNamespace
from typing import Callable, Optional

import numpy as np
import torch

from . import _lib
from .core import _ptr, _stream_ptr

OBS = 15


class ObsNormalizer:
    def __init__(self, n_envs: int, device: torch.device, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, epsilon: float = 1e-8, gamma: float = 0.99):
        self.lib = _lib.load()
        self.n, self.device = n_envs, device
        self.norm_obs, self.norm_reward = bool(norm_obs), bool(norm_reward)
        self.clip_obs, self.clip_reward, self.epsilon, self.gamma = float(clip_obs), float(clip_reward), float(epsilon), float(gamma)
        self.training = True
        d = dict(device=device)
        self.stats = torch.zeros(_lib.NORM_STATS, dtype=torch.float64, **d)
        self.affine = torch.zeros(_lib.NORM_AFFINE, dtype=torch.float32, **d)
        self.returns = torch.zeros(n_envs, dtype=torch.float64, **d)
        self.n_partials = (n_envs + _lib.NORM_BLOCK - 1) // _lib.NORM_BLOCK
        self.partials = torch.empty(self.n_partials, _lib.NORM_MOMENTS, dtype=torch.float64, **d)
        self.moments = torch.zeros(_lib.NORM_MOMENTS, dtype=torch.float64, **d)
        self.reset_statistics()

    # -- layout of the [34] stats block ------------------------------------------------------------
    def reset_statistics(self):
        """SB3 RunningMeanStd(epsilon=1e-4): mean 0, var 1, count 1e-4, for the observations and the returns."""
        s = torch.zeros(_lib.NORM_STATS, dtype=torch.float64)
        s[OBS:2 * OBS] = 1.0
        s[2 * OBS] = 1e-4
        s[2 * OBS + 2], s[2 * OBS + 3] = 1.0, 1e-4
        self.stats.copy_(s)
        self._combine(None)

    def _combine(self, moments: Optional[torch.Tensor]):
        _lib.check(self.lib.dronecu_norm_combine(self.device.index, _ptr(self.stats), _ptr(moments), self.epsilon, self.clip_obs,
                                                 _ptr(self.affine), _stream_ptr(self.device)), "dronecu_norm_combine")

    @property
    def obs_rms(self):
        s = self.stats.cpu().numpy()
        return SimpleNamespace(mean=s[:OBS].copy(), var=s[OBS:2 * OBS].copy(), count=float(s[2 * OBS]))

    @property
    def ret_rms(self):
        s = self.stats.cpu().numpy()
        return SimpleNamespace(mean=np.float64(s[2 * OBS + 1]), var=np.float64(s[2 * OBS + 2]), count=float(s[2 * OBS + 3]))

    def affine_ptr(self):
        """What the rollout kernels read: the affine record, or None (observations are not normalised)."""
        return _ptr(self.affine) if self.norm_obs else None

    # -- per rollout -----------------------------------------------------------------------------------
    def process_rollout(self, obs_store: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, K: int,
                        allreduce: Optional[Callable[[torch.Tensor], None]] = None, side_env: int = -1,
                        side_obs: Optional[torch.Tensor] = None) -> int:
        """After the rollout launch: rewrite the buffer normalised (observations, rewards), then -- when training -- merge
        the rollout's moments into the statistics and derive the next affine record.  ``allreduce`` sums the moment record
        over the ranks (data parallel).  ``side_obs`` [K,15] receives env ``side_env``'s raw rows.  Returns the number of
        launches issued."""
        a = _lib.NormPassArgs()
        if self.norm_obs:
            a.d_obs, a.obs_stride, a.d_affine = obs_store.data_ptr(), obs_store.shape[-1], self.affine.data_ptr()
        elif side_obs is not None:           # the buffer holds raw rows anyway
            side_obs.copy_(obs_store[:, side_env, :OBS])
        if self.norm_reward:
            a.d_reward, a.d_done, a.d_returns = reward.data_ptr(), done.data_ptr(), self.returns.data_ptr()
        a.K, a.n, a.d_stats = K, self.n, self.stats.data_ptr()
        a.gamma, a.epsilon, a.clip_reward = self.gamma, self.epsilon, self.clip_reward
        a.update = int(self.training)
        a.side_env = side_env if (side_obs is not None and self.norm_obs) else -1
        a.d_side_obs = side_obs.data_ptr() if (side_obs is not None and self.norm_obs) else None
        a.d_partials = self.partials.data_ptr()
        st, dev = _stream_ptr(self.device), self.device.index
        _lib.check(self.lib.dronecu_norm_pass(dev, C.byref(a), st), "dronecu_norm_pass")
        if not self.training:
            return 1
        _lib.check(self.lib.dronecu_norm_reduce(dev, _ptr(self.partials), self.n_partials, _ptr(self.moments), st),
                   "dronecu_norm_reduce")
        if allreduce is not None:
            allreduce(self.moments)
        self._combine(self.moments)
        return 3

    def normalize_obs(self, obs: torch.Tensor) -> torch.Tensor:
        """[B,15] observations -> normalised copy on the device (the statistics are not updated)."""
        x = obs.to(self.device, torch.float32).reshape(-1, OBS).contiguous().clone()
        if not self.norm_obs or x.shape[0] == 0:
            return x
        a = _lib.NormPassArgs()
        a.d_obs, a.obs_stride, a.K, a.n, a.d_affine = x.data_ptr(), OBS, 1, x.shape[0], self.affine.data_ptr()
        a.side_env = -1
        _lib.check(self.lib.dronecu_norm_pass(self.device.index, C.byref(a), _stream_ptr(self.device)), "dronecu_norm_pass")
        return x

    # -- checkpoints ------------------------------------------------------------------------------------
    def settings(self) -> dict:
        return {"norm_obs": self.norm_obs, "norm_reward": self.norm_reward, "clip_obs": self.clip_obs,
                "clip_reward": self.clip_reward, "norm_epsilon": self.epsilon}

    def state_dict(self) -> dict:
        """The replicated part: settings and running statistics (the per-env returns go with the env shard)."""
        return {**self.settings(), "stats": self.stats.cpu().clone()}

    def load_state_dict(self, sd: dict):
        self.stats.copy_(sd["stats"].to(self.device, torch.float64))
        self._combine(None)
