"""PPO on the GPU: the rollout + update hot path of ``PPO("MlpPolicy", env)`` (reference
train.py:36-43, :63-68) with SB3's defaults, computed by the CUDA kernels behind the C ABI.

Host side only orchestrates: ONE launch collects ``n_steps`` env steps for every env with the policy
evaluated in-kernel (``dronecu_rollout_policy``), one computes GAE, and each minibatch is
adv-stats -> grad -> [exchange over peer memory] -> clip+Adam.  torch supplies device memory and
``torch.distributed``; no torch op touches the numerics.

Data parallel (``torch.distributed`` initialised, one process per GPU): every rank owns a contiguous
shard of global env ids and its own rollout buffers; per optimiser step the flat sum-form gradient (10,705
float32 incl. statistics) is summed over the ranks and per epoch the advantage sums of its minibatches, so
the update equals the single-GPU update over the union of the shards (SURVEY.md section 8e).  The exchange is
``dp_backend="peer"`` (default): one kernel per optimiser step pushes the gradient into mailboxes in every
peer's HBM over NVLink, waits on flags, sums in fixed rank order and runs clip + Adam (csrc/ppo_dp.cuh) -- no
NCCL call on the data path, and the epoch stays one CUDA graph; ``"nccl"``: torch.distributed.all_reduce
between the reduce and apply kernels (the round-1 path, kept for comparison).  torch.distributed is used for the
set-up (exchange of IPC handles, barriers) either way.

PARITY: the primitives SB3 composes are pinned to torch's own (tests/test_ppo_oracle_torch_pin.py); the composition
(SB3 itself) is not in the reference tree and not installable -- unpinned; tests compare against oracle/ppo_oracle.py.
"""
from __future__ import annotations

import ctypes as C
import math
import sys
import time
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import GRAD_LEN, POLICY_PARAMS, PolicyOut, PPOConfig
from .core import DroneBatch, EnvConfig, _ptr, _stream_ptr

_SHAPES = [("pi.W1", (64, 15)), ("pi.b1", (64,)), ("pi.W2", (64, 64)), ("pi.b2", (64,)), ("pi.W3", (4, 64)),
           ("pi.b3", (4,)), ("vf.W1", (64, 15)), ("vf.b1", (64,)), ("vf.W2", (64, 64)), ("vf.b2", (64,)),
           ("vf.W3", (1, 64)), ("vf.b3", (1,)), ("log_std", (4,))]
# names of the same tensors in an SB3 ActorCriticPolicy state_dict (for zip import / export)
SB3_NAMES = {"pi.W1": "mlp_extractor.policy_net.0.weight", "pi.b1": "mlp_extractor.policy_net.0.bias",
             "pi.W2": "mlp_extractor.policy_net.2.weight", "pi.b2": "mlp_extractor.policy_net.2.bias",
             "pi.W3": "action_net.weight", "pi.b3": "action_net.bias",
             "vf.W1": "mlp_extractor.value_net.0.weight", "vf.b1": "mlp_extractor.value_net.0.bias",
             "vf.W2": "mlp_extractor.value_net.2.weight", "vf.b2": "mlp_extractor.value_net.2.bias",
             "vf.W3": "value_net.weight", "vf.b3": "value_net.bias", "log_std": "log_std"}


def init_policy_params(seed: int = 0) -> torch.Tensor:
    """The initial parameters of SB3's ``ActorCriticPolicy`` for ``PPO("MlpPolicy", env, seed=seed)`` (reference
    train.py:36-43), built from torch's own ``nn.Linear`` / ``nn.init.orthogonal_``: modules constructed in SB3's order
    under ``torch.manual_seed(seed)`` (policy tower, value tower, action head, value head), then orthogonal weights
    (gain sqrt2 towers, 0.01 action head, 1 value head), zero biases, log_std = 0.  The global torch RNG is left
    untouched.  Flat float32 CPU vector [10697]."""
    nn = torch.nn
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        pi = nn.Sequential(nn.Linear(15, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        vf = nn.Sequential(nn.Linear(15, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        action_net, value_net = nn.Linear(64, 4), nn.Linear(64, 1)
        with torch.no_grad():
            for layer, gain in ((pi[0], math.sqrt(2)), (pi[2], math.sqrt(2)), (vf[0], math.sqrt(2)), (vf[2], math.sqrt(2)),
                                (action_net, 0.01), (value_net, 1.0)):
                nn.init.orthogonal_(layer.weight, gain=gain)
                layer.bias.fill_(0.0)
    tensors = {"pi.W1": pi[0].weight, "pi.b1": pi[0].bias, "pi.W2": pi[2].weight, "pi.b2": pi[2].bias,
               "pi.W3": action_net.weight, "pi.b3": action_net.bias,
               "vf.W1": vf[0].weight, "vf.b1": vf[0].bias, "vf.W2": vf[2].weight, "vf.b2": vf[2].bias,
               "vf.W3": value_net.weight, "vf.b3": value_net.bias, "log_std": torch.zeros(4)}
    return torch.cat([tensors[name].detach().reshape(-1) for name, _ in _SHAPES]).to(torch.float32)


def unpack_params(flat: torch.Tensor) -> dict:
    out, off = {}, 0
    for name, shape in _SHAPES:
        n = int(np.prod(shape))
        out[name] = flat[off:off + n].reshape(shape)
        off += n
    return out


class RolloutBuffers:
    """Device-resident rollout buffers [K, n, ...] (SB3 RolloutBuffer).  ``obs`` is always the [K, n, 15] view; with
    ``padded_obs`` the storage behind it (``obs_store``) has 64-byte rows [K, n, 16] whose 16th value the rollout kernel
    writes as 1.0 -- four aligned 16-byte chunks per row for the update kernel's gathers."""

    def __init__(self, K, n, device, padded_obs: bool = False):
        f = dict(dtype=torch.float32, device=device)
        self.obs_stride = 16 if padded_obs else 15
        self.obs_store = torch.empty(K, n, self.obs_stride, **f)
        self.obs = self.obs_store[..., :15]
        self.actions = torch.empty(K, n, 4, **f)
        self.logp = torch.empty(K, n, **f)
        self.value = torch.empty(K, n, **f)
        self.reward = torch.empty(K, n, **f)
        self.done = torch.empty(K, n, dtype=torch.uint8, device=device)
        self.last_value = torch.empty(n, **f)
        self.adv = torch.empty(K, n, **f)
        self.ret = torch.empty(K, n, **f)


class PPO:
    """SB3-shaped trainer: ``PPO(env).learn(total_timesteps)``, ``predict``, ``save`` / ``load``.

    ``env`` is a ``DroneBatch`` (or anything with a ``.batch`` DroneBatch, e.g. ``DroneVecEnv``), or an
    int = number of envs to create.  Defaults are SB3's (n_steps 2048, batch_size 64, n_epochs 10,
    gamma 0.99, gae_lambda 0.95, clip 0.2, ent 0, vf 0.5, max_grad_norm 0.5, lr 3e-4, Adam eps 1e-5).
    ``batch_size`` counts samples PER RANK.

    ``norm_obs`` / ``norm_reward``: SB3's ``VecNormalize`` (clip_obs, clip_reward, norm_epsilon as there; gamma is PPO's),
    computed inside the rollout (normalize.py).  The running statistics are frozen for the length of one rollout and merged
    after it (SB3 updates them after every env step).  The rollout buffer then holds normalised observations and rewards, as
    SB3's does under VecNormalize; episode statistics stay in raw reward.  ``obs_rms`` / ``ret_rms`` / ``training`` /
    ``normalize_obs`` mirror the VecNormalize attributes, and ``predict`` normalises its input with the model's statistics
    (under SB3 the wrapped env does that).
    """

    tc_min_envs = 1024       # rollout_precision "tf32": tensor-core rollout kernel above this many envs per rank

    def __init__(self, env=1, n_steps: int = 2048, batch_size: int = 64, n_epochs: int = 10, gamma: float = 0.99,
                 gae_lambda: float = 0.95, clip_range: float = 0.2, ent_coef: float = 0.0, vf_coef: float = 0.5,
                 max_grad_norm: float = 0.5, learning_rate: float = 3e-4, normalize_advantage: bool = True,
                 seed: int = 0, device: int = 0, verbose: int = 0, policy_seed: Optional[int] = None,
                 rollout_precision: str = "fp32", update_precision: str = "fp32", cuda_graph: Optional[bool] = None,
                 dp_backend: str = "peer", padded_obs: Optional[bool] = None, norm_obs: bool = False,
                 norm_reward: bool = False, clip_obs: float = 10.0, clip_reward: float = 10.0, norm_epsilon: float = 1e-8):
        self.lib = _lib.load()
        self.rank, self.world = 0, 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.rank, self.world = torch.distributed.get_rank(), torch.distributed.get_world_size()
        if isinstance(env, int):
            env = DroneBatch(env, EnvConfig.single(), device=device, seed=seed, env_offset=self.rank * env)
        self.batch: DroneBatch = getattr(env, "batch", env)
        if self.batch.obs_dim != 15 or not self.batch.config.auto_reset:
            raise ValueError("PPO needs the DroneGymEnv spec (15-dim obs) with auto-reset")
        self.device = self.batch.device
        self.n_envs, self.n_steps, self.batch_size, self.n_epochs = self.batch.n, n_steps, batch_size, n_epochs
        self.gamma, self.gae_lambda, self.normalize_advantage = gamma, gae_lambda, normalize_advantage
        self.verbose, self.seed = verbose, seed
        if rollout_precision not in ("fp32", "tf32"):
            raise ValueError("rollout_precision must be 'fp32' (CUDA cores, parity path) or 'tf32' (tcgen05 tensor cores)")
        if update_precision not in ("fp32", "tf32", "bf16"):
            raise ValueError("update_precision must be 'fp32' (CUDA cores, parity path), 'tf32' (tcgen05, all products tf32) or "
                             "'bf16' (tcgen05, weight-gradient products with bf16 operands, three tiles per SM)")
        self.rollout_precision, self.update_precision = rollout_precision, update_precision
        cfg = PPOConfig()
        self.lib.dronecu_ppo_config_default(C.byref(cfg))
        cfg.learning_rate, cfg.clip_range, cfg.ent_coef = learning_rate, clip_range, ent_coef
        cfg.vf_coef, cfg.max_grad_norm = vf_coef, max_grad_norm
        self.cfg = cfg
        h = C.c_void_p()
        _lib.check(self.lib.dronecu_ppo_create(C.byref(cfg), self.device.index, C.byref(h)), "dronecu_ppo_create")
        self._h = h
        self.params = init_policy_params(seed if policy_seed is None else policy_seed).to(self.device)
        # 64-byte observation rows in the rollout buffer: default for the bf16 update kernel (its gathers and X staging are
        # vectorised for them); every kernel accepts either layout
        self.padded_obs = (update_precision == "bf16") if padded_obs is None else bool(padded_obs)
        self.buf = RolloutBuffers(n_steps, self.n_envs, self.device, self.padded_obs)
        self._grad = torch.zeros(GRAD_LEN, dtype=torch.float32, device=self.device)
        self._adv_stats = torch.zeros(3, dtype=torch.float64, device=self.device)
        self._info = torch.zeros(9, dtype=torch.float32, device=self.device)
        self._info_sum = torch.zeros(10, dtype=torch.float32, device=self.device)     # sums over the minibatches of one train()
        _lib.check(self.lib.dronecu_ppo_set_info_accumulator(self._h, _ptr(self._info_sum)))
        self._ev = torch.zeros(8, dtype=torch.float64, device=self.device)            # explained-variance moments
        if dp_backend not in ("peer", "nccl"):
            raise ValueError("dp_backend must be 'peer' (one exchange + clip + Adam kernel over NVLink peer memory) or 'nccl'")
        self.dp_backend = dp_backend if self.world > 1 else None
        if self.world > 1:
            self._dp_setup()
        self._gen = torch.Generator(device=self.device).manual_seed(seed + 1)
        self.normalizer = None
        if norm_obs or norm_reward:
            from .normalize import ObsNormalizer
            self.normalizer = ObsNormalizer(self.n_envs, self.device, norm_obs, norm_reward, clip_obs, clip_reward, norm_epsilon,
                                            gamma)
        self.side_env, self.side_obs = -1, None     # set_raw_obs_tap(): raw rows of one env per rollout
        self.num_timesteps, self.n_updates = 0, 0
        self._perm, self._epochs_done = None, 0
        self.grad_events = None                   # set to [] to collect (start, end, samples) events per gradient launch
        # One epoch's minibatch sequence (adv-stats -> grad -> reduce -> [exchange +] clip+Adam, x minibatches) as ONE CUDA
        # graph: with SB3's defaults (batch 64) an epoch is hundreds of 10-microsecond kernels and the host launch rate is
        # the bound.  Default: on for small minibatches, and always for data-parallel training over peer memory (the
        # exchange is a kernel; only the "nccl" backend keeps its all-reduces outside graphs).
        self.cuda_graph = cuda_graph
        self._graph, self._graph_key, self._graph_launches = None, None, 0
        self._ep_stats = None
        self._max_mb = 8 * torch.cuda.get_device_properties(self.device).multi_processor_count
        self.logger_values: dict = {}
        self.launches = 0
        self.batch.reset()          # SB3 _setup_learn: env.reset()  (ep_num 1 -> 2)

    # -- lifetime ------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "dp_backend", None) == "peer" and torch.distributed.is_initialized():
                torch.cuda.synchronize(self.device)
                torch.distributed.barrier()       # no peer may still be writing into this rank's mailbox when it is freed
            self.lib.dronecu_ppo_destroy(self._h)
            self._h = None

    # -- data-parallel set-up -------------------------------------------------------------------------
    def _dp_setup(self):
        """Every rank must hold the same number of transitions and minibatches (all ranks issue the same number of
        exchanges); with the peer backend, allocate this rank's mailbox and map the peers' (CUDA IPC)."""
        dist = torch.distributed
        mine = torch.tensor([self.n_envs * self.n_steps, self.batch_size], dtype=torch.int64, device=self.device)
        every = [torch.zeros_like(mine) for _ in range(self.world)]
        dist.all_gather(every, mine)
        if any(not torch.equal(e, mine) for e in every):
            raise ValueError("data-parallel PPO: every rank needs the same n_envs * n_steps and batch_size, got "
                             f"{[e.tolist() for e in every]}")
        if self.dp_backend != "peer":
            return
        if self.world > _lib.DP_MAX_WORLD:
            raise ValueError(f"dp_backend='peer' supports at most {_lib.DP_MAX_WORLD} ranks (one NVLink domain)")
        # peers must be reachable through CUDA IPC + peer access (the GPUs of one NVLink box); if any rank cannot map its
        # peers (another node, IPC disabled in a container) EVERY rank falls back to the NCCL backend, together
        ok, why = 1, ""
        try:
            handle = (C.c_ubyte * _lib.IPC_HANDLE_BYTES)()
            _lib.check(self.lib.dronecu_ppo_dp_alloc(self._h, self.rank, self.world, handle, None), "dronecu_ppo_dp_alloc")
            h = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device=self.device)
        except _lib.DronecuError as e:
            ok, why, h = 0, str(e), torch.zeros(_lib.IPC_HANDLE_BYTES, dtype=torch.uint8, device=self.device)
        allh = [torch.zeros_like(h) for _ in range(self.world)]
        dist.all_gather(allh, h)
        if ok:
            try:
                blob = b"".join(bytes(t.cpu().tolist()) for t in allh)
                buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
                _lib.check(self.lib.dronecu_ppo_dp_connect(self._h, self.world, buf, None), "dronecu_ppo_dp_connect")
            except _lib.DronecuError as e:
                ok, why = 0, str(e)
        flag = torch.tensor([ok], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        torch.cuda.synchronize(self.device)
        dist.barrier()                             # every mailbox is zeroed and mapped before the first push
        if int(flag.item()) == 0:
            if self.rank == 0 or why:
                print(f"[drone_rl_b200] rank {self.rank}: peer-memory exchange unavailable ({why or 'another rank failed'}); "
                      "using dp_backend='nccl'", file=sys.stderr, flush=True)
            self.dp_backend = "nccl"

    def _allreduce_f64(self, t: torch.Tensor):
        """In-place sum over the ranks of a small float64 device tensor (advantage / episode statistics)."""
        if self.world == 1:
            return
        if self.dp_backend == "peer" and t.numel() <= 5376:
            _lib.check(self.lib.dronecu_ppo_dp_allreduce_f64(self._h, _ptr(t), t.numel(), _stream_ptr(self.device)),
                       "dronecu_ppo_dp_allreduce_f64")
            self.launches += 1
        else:
            torch.distributed.all_reduce(t)

    def dp_check(self):
        """Raise if a peer-memory exchange timed out (a rank fell out of step or died)."""
        if self.dp_backend == "peer":
            st, n = C.c_int(), C.c_int64()
            _lib.check(self.lib.dronecu_ppo_dp_status(self._h, C.byref(st), C.byref(n)))
            if st.value:
                raise _lib.DronecuError(f"rank {self.rank}: a data-parallel exchange timed out after {n.value} exchanges")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- normalisation (SB3 VecNormalize attributes) ------------------------------------------------------
    @property
    def obs_rms(self):
        """Running mean / var / count of the observations (numpy, float64), or None without normalisation."""
        return None if self.normalizer is None else self.normalizer.obs_rms

    @property
    def ret_rms(self):
        return None if self.normalizer is None else self.normalizer.ret_rms

    @property
    def training(self) -> bool:
        """False (evaluation): the rollout keeps normalising but leaves the statistics unchanged and does not advance the
        per-env returns; as in SB3, a return is still zeroed where its episode ends."""
        return True if self.normalizer is None else self.normalizer.training

    @training.setter
    def training(self, value: bool):
        if self.normalizer is not None:
            self.normalizer.training = bool(value)

    def normalize_obs(self, obs) -> torch.Tensor:
        """Observations [.., 15] normalised with the current statistics (a device copy; unchanged without norm_obs)."""
        x = torch.as_tensor(np.asarray(obs, dtype=np.float32) if not torch.is_tensor(obs) else obs)
        if self.normalizer is None:
            return x.to(self.device, torch.float32).reshape(-1, 15)
        return self.normalizer.normalize_obs(x)

    def set_raw_obs_tap(self, env_index: int):
        """Keep the RAW observation rows of env ``env_index`` of every rollout in ``self.side_obs`` [n_steps, 15] (the
        rollout buffer holds normalised rows when norm_obs is on)."""
        self.side_env = int(env_index)
        self.side_obs = torch.empty(self.n_steps, 15, dtype=torch.float32, device=self.device)

    # -- rollout ------------------------------------------------------------------------------------
    def collect_rollouts(self, deterministic: bool = False):
        """One launch: n_steps env steps for every env, policy evaluated in-kernel; then GAE.  With normalisation: the
        rollout's towers see normalised observations, then one pass rewrites the buffer normalised, the moments are
        reduced [and summed over the ranks] and merged into the statistics (training only), then GAE."""
        b, K, n = self.buf, self.n_steps, self.n_envs
        out = PolicyOut(b.obs_store.data_ptr(), b.actions.data_ptr(), b.logp.data_ptr(), b.value.data_ptr(),
                        b.reward.data_ptr(), b.done.data_ptr(), b.last_value.data_ptr(), None, int(self.padded_obs), 0)
        st = _stream_ptr(self.device)
        # tensor cores pay from ~1k envs (a tile is 128 envs; below that the float32 warp-per-env kernel is both faster and exact)
        use_tc = self.rollout_precision == "tf32" and self.n_envs > self.tc_min_envs
        nz = self.normalizer
        if nz is None:
            fn = self.lib.dronecu_rollout_policy_tc if use_tc else self.lib.dronecu_rollout_policy
            _lib.check(fn(self.batch._h, K, _ptr(self.params), int(deterministic), C.byref(out), st), "dronecu_rollout_policy")
        else:
            _lib.check(self.lib.dronecu_rollout_policy_norm(self.batch._h, K, _ptr(self.params), int(deterministic), C.byref(out),
                                                            nz.affine_ptr(), int(use_tc), st), "dronecu_rollout_policy_norm")
            self.launches += nz.process_rollout(b.obs_store, b.reward, b.done, K, self._allreduce_f64 if self.world > 1 else None,
                                                self.side_env, self.side_obs)
        if nz is None and self.side_obs is not None:
            self.side_obs.copy_(b.obs[:, self.side_env])
        _lib.check(self.lib.dronecu_gae(self.device.index, K, n, _ptr(b.reward), _ptr(b.value), _ptr(b.done),
                                        _ptr(b.last_value), self.gamma, self.gae_lambda, _ptr(b.adv), _ptr(b.ret), st),
                   "dronecu_gae")
        self.launches += 2
        self.num_timesteps += K * n * self.world

    # -- update -------------------------------------------------------------------------------------
    def _minibatch(self, index: Optional[torch.Tensor], first: int, m: int, stats: Optional[torch.Tensor] = None):
        """One optimiser step.  `stats`: this minibatch's (already all-reduced) [sum, sumsq, count] of the advantages
        (train() computes them for the whole epoch at once); None: computed here."""
        b, st = self.buf, _stream_ptr(self.device)
        stats_ptr = None
        if self.normalize_advantage and stats is not None:
            stats_ptr = _ptr(stats)
        elif self.normalize_advantage:
            self._adv_stats.zero_()
            _lib.check(self.lib.dronecu_ppo_adv_stats(self._h, _ptr(b.adv), _ptr(index), first, m,
                                                      _ptr(self._adv_stats), st), "dronecu_ppo_adv_stats")
            self._allreduce_f64(self._adv_stats)
            stats_ptr = _ptr(self._adv_stats)
            self.launches += 2
        if self.grad_events is not None:          # bench.py: CUDA events around the gradient launches
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), m)
            ev[0].record()
        self.launch_grad(index, first, m, stats_ptr, self._grad)
        if self.grad_events is not None:
            ev[1].record()
            self.grad_events.append(ev)
        if self.dp_backend == "peer":
            # ONE kernel: push to the peers' mailboxes over NVLink, wait, fixed-order sum, clip + Adam (csrc/ppo_dp.cuh)
            _lib.check(self.lib.dronecu_ppo_apply_dp(self._h, _ptr(self.params), _ptr(self._grad), _ptr(self._info), st),
                       "dronecu_ppo_apply_dp")
        else:
            if self.world > 1:
                torch.distributed.all_reduce(self._grad)      # NCCL: 42.8 KB
            # every rank holds m samples of this minibatch (checked in _dp_setup)
            _lib.check(self.lib.dronecu_ppo_apply(self._h, _ptr(self.params), _ptr(self._grad),
                                                  1.0 / (m * self.world), _ptr(self._info), st), "dronecu_ppo_apply")
        # gradient kernel, its fixed-order reduce, apply; the bf16 kernel writes the gradient itself when one CTA per tower covers
        # the minibatch (up to 3 tiles of 128 samples: capi_ppo.cu), which saves the reduce launch
        self.launches += 2 if (self.update_precision == "bf16" and m <= 384) else 3
        self.n_updates += 1

    def launch_grad(self, index: Optional[torch.Tensor], first: int, m: int, stats_ptr, grad: torch.Tensor,
                    precision: Optional[str] = None):
        """One launch of the minibatch-gradient kernel (+ its fixed-order reduce) over this model's rollout buffers: rows
        ``index[0:m]`` (or ``first .. first+m``), advantage statistics from ``stats_ptr`` (a ctypes pointer to [sum, sumsq,
        count] or None: no normalisation), result in ``grad`` [GRAD_LEN]."""
        b = self.buf
        mode = {"fp32": 0, "tf32": 1, "bf16": 2}[precision or self.update_precision]
        _lib.check(self.lib.dronecu_ppo_grad_strided(self._h, mode, b.obs_stride, _ptr(self.params), _ptr(b.obs_store), _ptr(b.actions),
                                                     _ptr(b.logp), _ptr(b.adv), _ptr(b.ret), _ptr(index), first, m, 0.0, 1.0,
                                                     stats_ptr, _ptr(grad), _stream_ptr(self.device)), "dronecu_ppo_grad")

    def _epoch_graph(self, perm: torch.Tensor, B: int, ep_stats: Optional[torch.Tensor] = None):
        """Replay (capture on first use) the CUDA graph of one epoch over the index buffer `perm`."""
        key = (perm.data_ptr(), B, self.batch_size, self.normalize_advantage, self.update_precision,
               None if ep_stats is None else ep_stats.data_ptr())
        if self._graph is None or self._graph_key != key:
            torch.cuda.synchronize(self.device)
            l0, u0 = self.launches, self.n_updates
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for k, start in enumerate(range(0, B, self.batch_size)):
                    m = min(self.batch_size, B - start)
                    self._minibatch(perm[start:start + m], 0, m, None if ep_stats is None else ep_stats[k])
            # capture does not execute: undo the bookkeeping of the capture pass, remember it per replay
            self._graph_launches, self._graph_updates = self.launches - l0, self.n_updates - u0
            self.launches, self.n_updates = l0, u0
            self._graph, self._graph_key = g, key
        self._graph.replay()
        self.launches += self._graph_launches
        self.n_updates += self._graph_updates

    def train(self):
        """SB3 PPO.train(): n_epochs passes over the buffer in random minibatches of batch_size."""
        B = self.n_steps * self.n_envs
        if self._perm is None or self._perm.numel() != B:
            self._perm = torch.empty(B, dtype=torch.int32, device=self.device)
        perm = self._perm
        self._info_sum.zero_()
        n_mb = (B + self.batch_size - 1) // self.batch_size
        for _ in range(self.n_epochs):
            # SB3: np.random.permutation(B) per epoch, minibatch b = slice b of it.  Here a keyed bijection evaluated on the device
            # (no sort of B keys); with up to 64 minibatches per epoch it is read as "row r belongs to minibatch f(r) // batch" and
            # every minibatch lists its rows in ascending order (a counting sort by minibatch id): the same uniformly random
            # partition, and the update kernels sweep the rollout buffer forwards instead of gathering random rows
            if n_mb <= 64:
                _lib.check(self.lib.dronecu_minibatch_partition(self._h, B, self.batch_size, self.seed + 1, self._epochs_done,
                                                                _ptr(perm), _stream_ptr(self.device)), "dronecu_minibatch_partition")
                self.launches += 3
            else:
                _lib.check(self.lib.dronecu_minibatch_permutation(self.device.index, B, self.seed + 1, self._epochs_done,
                                                                  _ptr(perm), _stream_ptr(self.device)), "dronecu_minibatch_permutation")
                self.launches += 1
            self._epochs_done += 1
            # advantage statistics of EVERY minibatch of the epoch: two launches and (data parallel) one all-reduce per epoch
            ep_stats = None
            if self.normalize_advantage and n_mb <= self._max_mb:
                if self._ep_stats is None or self._ep_stats.shape[0] != n_mb:
                    self._ep_stats = torch.zeros(n_mb, 3, dtype=torch.float64, device=self.device)
                ep_stats = self._ep_stats
                _lib.check(self.lib.dronecu_ppo_adv_stats_epoch(self._h, _ptr(self.buf.adv), _ptr(perm), B, self.batch_size,
                                                                _ptr(ep_stats), _stream_ptr(self.device)), "dronecu_ppo_adv_stats_epoch")
                self.launches += 2
                self._allreduce_f64(ep_stats)
            use_graph = self.cuda_graph if self.cuda_graph is not None else (
                (self.batch_size <= 16384 and B // self.batch_size >= 4) or self.dp_backend == "peer")
            if use_graph and self.dp_backend != "nccl" and self.grad_events is None:
                self._epoch_graph(perm, B, ep_stats)
                continue
            for k, start in enumerate(range(0, B, self.batch_size)):
                m = min(self.batch_size, B - start)
                self._minibatch(perm[start:start + m], 0, m, None if ep_stats is None else ep_stats[k])
        # SB3 logs the MEAN over all minibatches of all epochs (policy_gradient_loss, value_loss, approx_kl, clip_fraction,
        # entropy_loss), the LAST minibatch's total loss, and the explained variance of the value estimates over the buffer
        ev = self._explained_variance()
        acc = torch.cat([self._info_sum, self._info]).cpu().numpy()
        sums, last = acc[:10], acc[10:]
        n_upd = max(float(sums[9]), 1.0)
        log_std = self.params[-4:]
        entropy_loss = -float((0.5 + 0.5 * math.log(2.0 * math.pi) + log_std).sum())
        self.logger_values.update({"train/policy_gradient_loss": float(sums[0] / n_upd), "train/value_loss": float(sums[1] / n_upd),
                                   "train/approx_kl": float(sums[2] / n_upd), "train/clip_fraction": float(sums[3] / n_upd),
                                   "train/entropy_loss": entropy_loss,
                                   "train/loss": float(last[0] + self.cfg.ent_coef * entropy_loss + self.cfg.vf_coef * last[1]),
                                   "train/grad_norm": float(sums[8] / n_upd), "train/explained_variance": ev,
                                   "train/n_updates": self.n_updates, "train/clip_range": float(self.cfg.clip_range),
                                   "train/learning_rate": float(self.cfg.learning_rate),
                                   "train/std": float(torch.exp(log_std).mean())})
        self.dp_check()

    def _explained_variance(self) -> float:
        """SB3's ``explained_variance(values, returns)`` over the whole rollout buffer (all ranks): 1 - Var[ret - value] /
        Var[ret] -- logging only, from moments summed on the device."""
        y, d = self.buf.ret.reshape(-1), (self.buf.ret - self.buf.value).reshape(-1)
        (vy, my), (vd, md) = torch.var_mean(y, unbiased=False), torch.var_mean(d, unbiased=False)
        n = float(y.numel())
        m = torch.stack([my, vy + my * my, md, vd + md * md]).double() * n          # sums and sums of squares
        self._ev[0] = n
        self._ev[1:5] = m
        self._allreduce_f64(self._ev)
        n, sy, syy, sd, sdd = self._ev[:5].tolist()
        var_y, var_d = syy / n - (sy / n) ** 2, sdd / n - (sd / n) ** 2
        return float("nan") if var_y == 0 else 1.0 - var_d / var_y

    def learn(self, total_timesteps: int, log_interval: int = 1, callback=None, reset_num_timesteps: bool = True):
        """SB3 ``learn``: collect / train until ``total_timesteps`` MORE transitions have been gathered.  As in SB3,
        ``reset_num_timesteps=True`` (the default) restarts the counter, so ``PPO.load("dd.zip", env).learn(2e6)``
        (reference train.py:22-30, :63-68) trains for another 2e6 steps; ``False`` continues the counter (and the
        logging x-axis) of the loaded model and trains ``total_timesteps`` on top of it."""
        start = 0 if reset_num_timesteps else self.num_timesteps
        if reset_num_timesteps:
            self.num_timesteps = 0
        total_timesteps = start + int(total_timesteps)
        t0, it = time.time(), 0
        while self.num_timesteps < total_timesteps:
            self.collect_rollouts()
            st = self.batch.episode_stats(reset=True)
            if self.world > 1:
                v = self._ev[5:8]
                v.copy_(torch.tensor([st["return_sum"], float(st["length_sum"]), float(st["episodes"])], dtype=torch.float64))
                torch.distributed.all_reduce(v)
                st["ep_rew_mean"] = float(v[0] / v[2]) if v[2] > 0 else float("nan")
                st["ep_len_mean"] = float(v[1] / v[2]) if v[2] > 0 else float("nan")
            self.train()
            it += 1
            self.logger_values.update({"rollout/ep_rew_mean": st["ep_rew_mean"], "rollout/ep_len_mean": st["ep_len_mean"],
                                       "time/iterations": it, "time/total_timesteps": self.num_timesteps,
                                       "time/fps": int((self.num_timesteps - start) / max(time.time() - t0, 1e-9)),
                                       "time/time_elapsed": int(time.time() - t0)})
            if callback is not None and callback(self) is False:
                break
            if self.verbose and self.rank == 0 and it % log_interval == 0:
                print(" | ".join(f"{k}={v:.4g}" if isinstance(v, float) else f"{k}={v}"
                                 for k, v in self.logger_values.items()), flush=True)
        return self

    # -- inference ----------------------------------------------------------------------------------
    def policy_forward(self, obs: torch.Tensor, precision: str = "fp32", debug: bool = False):
        """(mean [B,4], value [B]) for device observations [B,15].  precision "tf32" runs the tcgen05
        kernel; with debug=True it also returns the layer-1 / layer-2 pre-activations [B,128] each."""
        obs = obs.to(self.device, torch.float32).contiguous()
        B = obs.shape[0]
        mean = torch.empty(B, 4, dtype=torch.float32, device=self.device)
        value = torch.empty(B, dtype=torch.float32, device=self.device)
        if precision == "tf32":
            d1 = torch.zeros(B, 128, dtype=torch.float32, device=self.device) if debug else None
            d2 = torch.zeros(B, 128, dtype=torch.float32, device=self.device) if debug else None
            _lib.check(self.lib.dronecu_policy_forward_tc(self.device.index, B, _ptr(self.params), _ptr(obs), _ptr(mean),
                                                          _ptr(value), _ptr(d1), _ptr(d2), _stream_ptr(self.device)),
                       "dronecu_policy_forward_tc")
            return (mean, value, d1, d2) if debug else (mean, value)
        _lib.check(self.lib.dronecu_policy_forward(self.device.index, B, _ptr(self.params), _ptr(obs), _ptr(mean),
                                                   _ptr(value), _stream_ptr(self.device)), "dronecu_policy_forward")
        return mean, value

    def predict(self, observation, state=None, episode_start=None, deterministic: bool = False):
        """SB3 ``predict``: numpy obs [15] or [n,15] -> (clipped action, None)  (train.py:48, test.py:14)."""
        obs = np.asarray(observation, dtype=np.float32)
        single = obs.ndim == 1
        x = torch.from_numpy(obs.reshape(-1, 15))
        if self.normalizer is not None:        # the model owns the VecNormalize statistics (SB3: the wrapped env applies them)
            x = self.normalizer.normalize_obs(x)
        mean, _ = self.policy_forward(x)
        if not deterministic:
            std = torch.exp(self.params[-4:])
            mean = mean + std * torch.randn(mean.shape, device=self.device, generator=self._gen)
        act = torch.clamp(mean, 0.0, self.batch.config.motor_max).cpu().numpy()
        return (act[0] if single else act), None

    # -- checkpoint (policy + Adam + env curriculum / RNG state; the reference loses the env state) ------
    def state_dict(self) -> dict:
        mom = torch.empty(2 * POLICY_PARAMS, dtype=torch.float32, device=self.device)
        step = C.c_int64()
        _lib.check(self.lib.dronecu_ppo_get_state(self._h, _ptr(mom), C.byref(step), _stream_ptr(self.device)))
        torch.cuda.synchronize(self.device)
        return {"params": self.params.cpu(), "adam": mom.cpu(), "adam_step": step.value,
                "num_timesteps": self.num_timesteps, "n_updates": self.n_updates, "epochs_done": self._epochs_done,
                "env_state": self.batch.get_state(), "env_global_step": self.batch.global_step,
                "env_offset": int(self.batch.env_offset), "world": self.world,
                "sb3_policy": {SB3_NAMES[k]: v.clone() for k, v in unpack_params(self.params.cpu()).items()},
                **({} if self.normalizer is None else {"normalizer": self.normalizer.state_dict(),
                                                       "norm_returns": self.normalizer.returns.cpu().clone()})}

    def load_state_dict(self, sd: dict, load_env: bool = True):
        self.params.copy_(sd["params"].to(self.device))
        _lib.check(self.lib.dronecu_ppo_set_state(self._h, _ptr(sd["adam"].to(self.device)), int(sd["adam_step"]),
                                                  _stream_ptr(self.device)))
        torch.cuda.synchronize(self.device)
        self.num_timesteps, self.n_updates = sd["num_timesteps"], sd["n_updates"]
        self._epochs_done = int(sd.get("epochs_done", 0))
        # the env / curriculum / RNG state belongs to ONE shard of global env ids: restore it only onto the same shard
        # (a data-parallel run writes one archive per rank: see save()); otherwise the envs start fresh
        self.env_state_restored = False
        if (load_env and "env_state" in sd and sd["env_state"]["pos"].shape[0] == self.n_envs
                and int(sd.get("env_offset", self.batch.env_offset)) == int(self.batch.env_offset)
                and int(sd.get("world", self.world)) == self.world):
            self.batch.set_state(**sd["env_state"])
            self.batch.global_step = sd.get("env_global_step", self.batch.global_step)
            self.env_state_restored = True
            if self.normalizer is not None and "norm_returns" in sd:      # per-env returns: same shard only
                self.normalizer.returns.copy_(sd["norm_returns"].to(self.device))
        if self.normalizer is not None and "normalizer" in sd:
            self.normalizer.load_state_dict(sd["normalizer"])

    def save(self, path: str):
        """SB3 ``model.save(path)`` (train.py:70): no suffix -> ``path + ".zip"``, an archive in SB3's layout
        (sb3_zip.py) that also carries the env / curriculum / RNG state; ``.pt`` -> a plain torch checkpoint."""
        if path.endswith(".pt"):
            torch.save(self.state_dict(), path)
            return
        from . import sb3_zip
        sd = self.state_dict()
        if self.world > 1 and self.rank > 0:
            # data parallel: policy and Adam state are replicas (rank 0's archive holds them); the env / curriculum /
            # Philox state differs per shard -> every other rank writes its shard next to the archive
            base = path[:-4] if path.endswith(".zip") else path
            torch.save({k: sd[k] for k in ("env_state", "env_global_step", "env_offset", "world", "norm_returns") if k in sd},
                       f"{base}.env.rank{self.rank}.pt")
            return
        hyper = {"n_steps": self.n_steps, "batch_size": self.batch_size, "n_epochs": self.n_epochs, "gamma": self.gamma,
                 "gae_lambda": self.gae_lambda, "learning_rate": float(self.cfg.learning_rate),
                 "clip_range": float(self.cfg.clip_range), "ent_coef": float(self.cfg.ent_coef),
                 "vf_coef": float(self.cfg.vf_coef), "max_grad_norm": float(self.cfg.max_grad_norm),
                 "n_envs": self.n_envs, "num_timesteps": self.num_timesteps, "_n_updates": self.n_updates, "seed": self.seed}
        extra = {k: sd[k] for k in ("num_timesteps", "n_updates", "epochs_done", "env_state", "env_global_step", "env_offset", "world",
                                    "normalizer", "norm_returns") if k in sd}
        sb3_zip.export_zip(path if path.endswith(".zip") else path + ".zip", sd["params"], sd["adam"], sd["adam_step"],
                           hyper, extra)

    @staticmethod
    def _norm_settings(sd: dict, kw: dict) -> dict:
        """A checkpoint trained with normalisation turns it on (with its clip / epsilon) unless the caller says otherwise."""
        saved = sd.get("normalizer")
        return kw if not saved else {**{k: saved[k] for k in ("norm_obs", "norm_reward", "clip_obs", "clip_reward", "norm_epsilon")}, **kw}

    @classmethod
    def load(cls, path: str, env=1, **kw):
        """SB3 ``PPO.load(path, env, **overrides)`` (train.py:22-30, test.py:7): a ``.zip`` written by this class or by
        stable-baselines3 itself (policy + Adam state; hyper-parameters stored in the archive are defaults that
        keyword arguments override), or a ``.pt`` checkpoint."""
        import os
        if not path.endswith((".pt", ".zip")) and os.path.isfile(path + ".zip"):
            path = path + ".zip"
        if path.endswith(".pt"):
            sd = torch.load(path, weights_only=False)
            model = cls(env, **cls._norm_settings(sd, kw))
            model.load_state_dict(sd)
            return model
        from . import sb3_zip
        z = sb3_zip.import_zip(path)
        for k in ("n_steps", "batch_size", "n_epochs", "gamma", "gae_lambda", "learning_rate", "clip_range", "ent_coef",
                  "vf_coef", "max_grad_norm"):
            if k in z["hyper"] and k not in kw and isinstance(z["hyper"][k], (int, float)):
                kw[k] = z["hyper"][k]
        model = cls(env, **cls._norm_settings(z["extra"] or {}, kw))
        sd = {"params": z["params"], "adam": z["adam"] if z["adam"] is not None else torch.zeros(2 * POLICY_PARAMS),
              "adam_step": z["adam_step"], "num_timesteps": int(z["hyper"].get("num_timesteps", 0) or 0),
              "n_updates": int(z["hyper"].get("_n_updates", 0) or 0)}
        if z["extra"]:
            sd.update(z["extra"])
        if model.world > 1 and model.rank > 0:          # this rank's env shard, written by save() next to the archive
            side = f"{path[:-4]}.env.rank{model.rank}.pt"
            sd.pop("env_state", None)
            sd.pop("norm_returns", None)
            if os.path.isfile(side):
                sd.update(torch.load(side, weights_only=False))
        model.load_state_dict(sd)
        return model
