"""TEST INFRASTRUCTURE: plain-torch (CPU, float64 or float32) restatement of SB3's PPO maths.

PARITY UNPINNED.  The reference only *calls* stable-baselines3 (train.py:36-43 ``PPO("MlpPolicy",
env, device="cpu")`` with every default; train.py:25-29 resumes with n_steps=2048, batch_size=64,
learning_rate=3e-4 -- the defaults again).  SB3 itself is a PyPI dependency, un-pinned
(environment.yaml:16), absent from /root/reference and not installed here, and the reference has
no test or fixture for anything it computes.  This file restates SB3's *published* algorithm
(SURVEY.md appendix C lists the semantics relied on); the CUDA path is compared against it only.

Restated pieces
  * MlpPolicy: separate pi / vf towers Linear(15,64)-Tanh-Linear(64,64)-Tanh, heads Linear(64,4) /
    Linear(64,1), state-independent log_std (init 0), orthogonal init (gain sqrt2 / 0.01 / 1).
  * DiagGaussian sample / log_prob / entropy; actions clipped to the Box only for the env.
  * GAE(gamma=0.99, lambda=0.95) with SB3's episode_start convention, no bootstrap on time-outs
    (the reference env never sets "TimeLimit.truncated").
  * the clipped-surrogate loss with per-minibatch advantage normalisation (std + 1e-8, unbiased
    std as torch.std; skipped for a minibatch of one sample, as SB3's ``len(advantages) > 1``),
    value MSE x 0.5, entropy x 0, global-norm clip 0.5, Adam(3e-4, eps 1e-5).

Flat parameter layout (shared with drone_rl_b200/csrc/ppo_common.cuh), float32, 10697 values:
    pi.W1[64,15] pi.b1[64] pi.W2[64,64] pi.b2[64] pi.W3[4,64] pi.b3[4]
    vf.W1[64,15] vf.b1[64] vf.W2[64,64] vf.b2[64] vf.W3[1,64] vf.b3[1]  log_std[4]
(weights in torch.nn.Linear's [out, in] row-major order).
"""
from __future__ import annotations

import math

import numpy as np
import torch

OBS, HID, ACT = 15, 64, 4
SHAPES = [("pi.W1", (HID, OBS)), ("pi.b1", (HID,)), ("pi.W2", (HID, HID)), ("pi.b2", (HID,)),
          ("pi.W3", (ACT, HID)), ("pi.b3", (ACT,)),
          ("vf.W1", (HID, OBS)), ("vf.b1", (HID,)), ("vf.W2", (HID, HID)), ("vf.b2", (HID,)),
          ("vf.W3", (1, HID)), ("vf.b3", (1,)), ("log_std", (ACT,))]
N_PARAMS = sum(int(np.prod(s)) for _, s in SHAPES)
assert N_PARAMS == 10697
LOG_2PI = math.log(2.0 * math.pi)


def offsets():
    off, out = 0, {}
    for name, shape in SHAPES:
        n = int(np.prod(shape))
        out[name] = (off, shape)
        off += n
    return out


# SB3 builds the modules in this order (MlpExtractor: policy_net then value_net; then action_net, value_net) and
# re-initialises them in the order of ActorCriticPolicy._build's module_gains dict.
_BUILD_ORDER = ["pi.W1", "pi.W2", "vf.W1", "vf.W2", "pi.W3", "vf.W3"]
_INIT_ORDER = [("pi.W1", math.sqrt(2)), ("pi.W2", math.sqrt(2)), ("vf.W1", math.sqrt(2)), ("vf.W2", math.sqrt(2)),
               ("pi.W3", 0.01), ("vf.W3", 1.0)]


def orthogonal(rows: int, cols: int, gain: float, g: torch.Generator) -> torch.Tensor:
    """torch.nn.init.orthogonal_ restated on a float32 [rows, cols] weight (pinned against torch's own in
    tests/test_ppo_oracle_torch_pin.py): N(0,1) draws in the weight's own shape, transposed when rows < cols,
    reduced QR, Q's columns signed by diag(R), transposed back, scaled by the gain."""
    a = torch.empty(rows, cols, dtype=torch.float32).normal_(0, 1, generator=g)
    if rows < cols:
        a = a.t()
    q, r = torch.linalg.qr(a)
    q = q * torch.sign(torch.diag(r, 0))
    if rows < cols:
        q = q.t()
    return q * gain


def init_params(seed: int = 0, dtype=torch.float32) -> torch.Tensor:
    """What ``PPO("MlpPolicy", env, seed=seed)`` (reference train.py:36-43) holds after construction, restated:
    SB3 seeds torch's global generator, builds the six nn.Linear (each draws its default kaiming-uniform weight and
    uniform bias -- consumed here so that the stream position matches), then ActorCriticPolicy re-initialises them
    orthogonally (gain sqrt(2) towers, 0.01 action head, 1.0 value head) with zero biases; log_std = 0.
    Returns the flat vector."""
    g = torch.Generator().manual_seed(seed)
    offs = offsets()
    for name in _BUILD_ORDER:                       # nn.Linear.reset_parameters: weight then bias
        rows, cols = offs[name][1]
        torch.empty(rows, cols, dtype=torch.float32).uniform_(-1, 1, generator=g)
        torch.empty(rows, dtype=torch.float32).uniform_(-1, 1, generator=g)
    flat = torch.zeros(N_PARAMS, dtype=torch.float32)
    for name, gain in _INIT_ORDER:
        off, (rows, cols) = offs[name]
        flat[off:off + rows * cols] = orthogonal(rows, cols, gain, g).reshape(-1)
    return flat.to(dtype)


def unpack(flat: torch.Tensor):
    return {name: flat[off:off + int(np.prod(shape))].reshape(shape) for name, (off, shape) in offsets().items()}


def forward(flat: torch.Tensor, obs: torch.Tensor):
    """-> (mean [B,4], value [B], log_std [4])."""
    p = unpack(flat)
    h = torch.tanh(obs @ p["pi.W1"].t() + p["pi.b1"])
    h = torch.tanh(h @ p["pi.W2"].t() + p["pi.b2"])
    mean = h @ p["pi.W3"].t() + p["pi.b3"]
    v = torch.tanh(obs @ p["vf.W1"].t() + p["vf.b1"])
    v = torch.tanh(v @ p["vf.W2"].t() + p["vf.b2"])
    value = (v @ p["vf.W3"].t() + p["vf.b3"]).squeeze(-1)
    return mean, value, p["log_std"]


def log_prob(mean, log_std, actions):
    std = torch.exp(log_std)
    return (-((actions - mean) ** 2) / (2 * std ** 2) - log_std - 0.5 * LOG_2PI).sum(-1)


def entropy(log_std, batch):
    return (0.5 + 0.5 * LOG_2PI + log_std).sum().expand(batch)


def gae(rewards, values, dones, last_values, gamma=0.99, lam=0.95):
    """rewards/values/dones [K,n] (dones[t] = episode ended AT step t), last_values [n].
    SB3's compute_returns_and_advantage with episode_starts[t+1] == dones[t] and
    the final `dones` == dones[K-1].  Returns (advantages, returns)."""
    K = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    last = torch.zeros_like(last_values)
    for t in reversed(range(K)):
        nnt = 1.0 - dones[t].to(rewards.dtype)
        nv = last_values if t == K - 1 else values[t + 1]
        delta = rewards[t] + gamma * nv * nnt - values[t]
        last = delta + gamma * lam * nnt * last
        adv[t] = last
    return adv, adv + values


def ppo_loss(flat, obs, actions, old_logp, adv, returns, clip=0.2, vf_coef=0.5, ent_coef=0.0,
             normalize=True, adv_mean=None, adv_std=None):
    """SB3 PPO.train() loss for one minibatch.  adv_mean/adv_std override the per-minibatch
    statistics (used for the data-parallel path, where they are global over the ranks).  Without them a
    minibatch of one sample keeps its raw advantage: SB3 normalises only ``if len(advantages) > 1``."""
    mean, value, log_std = forward(flat, obs)
    logp = log_prob(mean, log_std, actions)
    if normalize and (adv_mean is not None or adv.numel() > 1):
        m = adv.mean() if adv_mean is None else adv_mean
        s = adv.std() if adv_std is None else adv_std          # torch.std: unbiased, as SB3
        adv = (adv - m) / (s + 1e-8)
    ratio = torch.exp(logp - old_logp)
    pg1 = adv * ratio
    pg2 = adv * torch.clamp(ratio, 1 - clip, 1 + clip)
    policy_loss = -torch.min(pg1, pg2).mean()
    value_loss = torch.nn.functional.mse_loss(returns, value)
    ent_loss = -entropy(log_std, obs.shape[0]).mean()
    loss = policy_loss + ent_coef * ent_loss + vf_coef * value_loss
    with torch.no_grad():
        log_ratio = logp - old_logp
        stats = {"policy_gradient_loss": float(policy_loss), "value_loss": float(value_loss),
                 "entropy_loss": float(ent_loss), "loss": float(loss),
                 "approx_kl": float(((torch.exp(log_ratio) - 1) - log_ratio).mean()),
                 "clip_fraction": float(((ratio - 1).abs() > clip).float().mean())}
    return loss, stats


class AdamState:
    def __init__(self, n, dtype):
        self.m = torch.zeros(n, dtype=dtype)
        self.v = torch.zeros(n, dtype=dtype)
        self.t = 0


def clip_and_adam(flat, grad, st: AdamState, lr=3e-4, b1=0.9, b2=0.999, eps=1e-5, max_norm=0.5):
    """torch.nn.utils.clip_grad_norm_(max_norm) followed by torch.optim.Adam.step()."""
    total = grad.norm(2)
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    g = grad * coef
    st.t += 1
    st.m = b1 * st.m + (1 - b1) * g
    st.v = b2 * st.v + (1 - b2) * g * g
    bc1, bc2 = 1 - b1 ** st.t, 1 - b2 ** st.t
    denom = st.v.sqrt() / math.sqrt(bc2) + eps
    return flat - (lr / bc1) * st.m / denom, float(total)


def minibatch_update(flat, st, batch, lr=3e-4, max_norm=0.5, **kw):
    """One optimiser step on one minibatch; returns (new flat params, stats, gradient).  ``lr`` and ``max_norm``
    go to clip_and_adam, every other keyword to ppo_loss."""
    p = flat.clone().requires_grad_(True)
    loss, stats = ppo_loss(p, *batch, **kw)
    (g,) = torch.autograd.grad(loss, p)
    new, gnorm = clip_and_adam(flat, g, st, lr=lr, max_norm=max_norm)
    stats["grad_norm"] = gnorm
    return new.detach(), stats, g.detach()
