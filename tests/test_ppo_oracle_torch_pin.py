"""Pins for the PPO oracle (oracle/ppo_oracle.py) against torch's OWN primitives.

stable-baselines3 is not installable here, so the composition (SB3's PPO.train / collect_rollouts) stays a
restatement ("composition unpinned").  Everything SB3 composes, however, is torch code that IS installed:
``nn.Linear`` / ``nn.Tanh`` / ``nn.init.orthogonal_`` (ActorCriticPolicy, reference call site train.py:36-43),
``torch.distributions.Normal`` (DiagGaussianDistribution), ``F.mse_loss``, ``nn.utils.clip_grad_norm_`` and
``torch.optim.Adam(lr=3e-4, eps=1e-5)`` (PPO.train, reference train.py:63-68).  These tests hold the oracle's
hand-written pieces to those, so that "PPO: primitives pinned to torch, composition unpinned".
"""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
nn = torch.nn

from oracle import ppo_oracle as po  # noqa: E402


class TorchMlpPolicy(nn.Module):
    """SB3's ActorCriticPolicy for MlpPolicy on Box(15) -> Box(4), written with torch modules only: modules are
    created in SB3's order (MlpExtractor.policy_net, .value_net, action_net + log_std, value_net) and re-initialised
    in the order of ``module_gains`` (mlp_extractor sqrt2, action_net 0.01, value_net 1)."""

    def __init__(self):
        super().__init__()
        self.policy_net = nn.Sequential(nn.Linear(15, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        self.value_tower = nn.Sequential(nn.Linear(15, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        self.action_net = nn.Linear(64, 4)
        self.log_std = nn.Parameter(torch.zeros(4))
        self.value_net = nn.Linear(64, 1)

        def ortho(gain):
            def f(m):
                if isinstance(m, nn.Linear):
                    nn.init.orthogonal_(m.weight, gain=gain)
                    m.bias.data.fill_(0.0)
            return f
        self.policy_net.apply(ortho(math.sqrt(2)))
        self.value_tower.apply(ortho(math.sqrt(2)))
        self.action_net.apply(ortho(0.01))
        self.value_net.apply(ortho(1.0))

    def named(self):
        return {"pi.W1": self.policy_net[0].weight, "pi.b1": self.policy_net[0].bias,
                "pi.W2": self.policy_net[2].weight, "pi.b2": self.policy_net[2].bias,
                "pi.W3": self.action_net.weight, "pi.b3": self.action_net.bias,
                "vf.W1": self.value_tower[0].weight, "vf.b1": self.value_tower[0].bias,
                "vf.W2": self.value_tower[2].weight, "vf.b2": self.value_tower[2].bias,
                "vf.W3": self.value_net.weight, "vf.b3": self.value_net.bias, "log_std": self.log_std}

    def flat(self):
        t = self.named()
        return torch.cat([t[name].detach().reshape(-1) for name, _ in po.SHAPES])

    def flat_grad(self):
        t = self.named()
        return torch.cat([t[name].grad.reshape(-1) for name, _ in po.SHAPES])

    def load_flat(self, flat):
        with torch.no_grad():
            for name, p in self.named().items():
                off, shape = po.offsets()[name]
                p.copy_(flat[off:off + p.numel()].reshape(shape))

    def evaluate_actions(self, obs, actions):
        """SB3 ActorCriticPolicy.evaluate_actions: (values, log_prob, entropy) through torch.distributions.Normal."""
        dist = torch.distributions.Normal(self.action_net(self.policy_net(obs)), torch.ones(4) * self.log_std.exp())
        return self.value_net(self.value_tower(obs)).flatten(), dist.log_prob(actions).sum(1), dist.entropy().sum(1)


def sb3_loss(policy, obs, actions, old_logp, adv, returns, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """The body of SB3's PPO.train() minibatch loop, line for line in torch ops."""
    values, log_prob, entropy = policy.evaluate_actions(obs, actions)
    if len(adv) > 1:                                   # SB3: `if self.normalize_advantage and len(advantages) > 1`
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    ratio = torch.exp(log_prob - old_logp)
    policy_loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    value_loss = torch.nn.functional.mse_loss(returns, values)
    entropy_loss = -torch.mean(entropy)
    return policy_loss + ent_coef * entropy_loss + vf_coef * value_loss


def _batch(B, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(B, 15, generator=g, dtype=dtype) * 2
    actions = torch.randn(B, 4, generator=g, dtype=dtype)
    old_logp = -4.0 + 0.5 * torch.randn(B, generator=g, dtype=dtype)
    adv = torch.randn(B, generator=g, dtype=dtype) * 3 + 0.5
    ret = torch.randn(B, generator=g, dtype=dtype)
    return obs, actions, old_logp, adv, ret


@pytest.mark.parametrize("seed", [0, 1, 12345])
def test_init_is_torch_orthogonal_in_sb3_order(seed):
    """oracle.init_params == nn.Linear construction + nn.init.orthogonal_ under torch.manual_seed(seed), bit for bit;
    the product's init (torch modules) is the same vector."""
    torch.manual_seed(seed)
    ref = TorchMlpPolicy().flat()
    got = po.init_params(seed)
    assert torch.equal(got, ref)
    p = po.unpack(got)
    for name, gain in po._INIT_ORDER:                 # (semi-)orthogonality with the stated gain
        w = p[name].double()
        gram = w @ w.t() if w.shape[0] <= w.shape[1] else w.t() @ w
        assert torch.allclose(gram, torch.eye(gram.shape[0], dtype=torch.float64) * gain ** 2, atol=1e-5)
    from drone_rl_b200.ppo import init_policy_params       # host logic: importable without the CUDA library
    state = torch.get_rng_state()
    assert torch.equal(init_policy_params(seed), ref)
    assert torch.equal(torch.get_rng_state(), state), "product init must not disturb the global RNG"


@pytest.mark.parametrize("rows,cols,gain", [(64, 15, math.sqrt(2)), (4, 64, 0.01), (1, 64, 1.0), (64, 64, math.sqrt(2))])
def test_orthogonal_restatement_equals_torch(rows, cols, gain):
    g1, g2 = torch.Generator().manual_seed(5), torch.Generator().manual_seed(5)
    w = torch.empty(rows, cols)
    nn.init.orthogonal_(w, gain=gain, generator=g1)
    assert torch.equal(po.orthogonal(rows, cols, gain, g2), w)


def test_forward_logprob_entropy_equal_torch_modules():
    torch.manual_seed(3)
    pol = TorchMlpPolicy()
    with torch.no_grad():
        pol.log_std.copy_(torch.tensor([-0.3, 0.0, 0.2, 0.7]))
        for p in pol.parameters():                      # move off the orthogonal init (non-zero biases)
            p.add_(0.05 * torch.randn(p.shape))
    flat = pol.flat()
    obs, actions, *_ = _batch(257, 1)
    mean, value, log_std = po.forward(flat, obs)
    v_ref, lp_ref, ent_ref = pol.evaluate_actions(obs, actions)
    assert torch.allclose(value, v_ref, rtol=1e-6, atol=1e-6)
    assert torch.allclose(mean, pol.action_net(pol.policy_net(obs)), rtol=1e-6, atol=1e-6)
    assert torch.allclose(po.log_prob(mean, log_std, actions), lp_ref, rtol=1e-5, atol=1e-5)
    assert torch.allclose(po.entropy(log_std, obs.shape[0]), ent_ref, rtol=1e-6, atol=1e-6)
    # float64: the formulas themselves, to rounding
    mean64, _, ls64 = po.forward(flat.double(), obs.double())
    d = torch.distributions.Normal(mean64, ls64.exp())
    assert torch.allclose(po.log_prob(mean64, ls64, actions.double()), d.log_prob(actions.double()).sum(1), rtol=1e-13, atol=1e-13)
    assert torch.allclose(po.entropy(ls64, 257), d.entropy().sum(1), rtol=1e-14)


@pytest.mark.parametrize("B", [64, 1000])
def test_loss_and_gradient_equal_torch_autograd_over_modules(B):
    """oracle.ppo_loss (flat vector) == the SB3 loss written over nn.Modules; gradients agree per parameter."""
    torch.manual_seed(11)
    pol = TorchMlpPolicy().double()
    with torch.no_grad():
        for p in pol.parameters():
            p.add_(0.1 * torch.randn(p.shape, dtype=torch.float64))
    batch = _batch(B, 2, torch.float64)
    loss_ref = sb3_loss(pol, *batch)
    loss_ref.backward()
    flat = pol.flat().clone().requires_grad_(True)
    loss, stats = po.ppo_loss(flat, *batch)
    (g,) = torch.autograd.grad(loss, flat)
    assert abs(float(loss.detach()) - float(loss_ref.detach())) <= 1e-12 * max(1.0, abs(float(loss_ref.detach())))
    assert torch.allclose(g, pol.flat_grad(), rtol=1e-10, atol=1e-13)
    assert abs(stats["value_loss"] - float(torch.nn.functional.mse_loss(batch[4], pol.evaluate_actions(batch[0], batch[1])[0]))) < 1e-12


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_clip_and_adam_equal_torch_optim_over_25_steps(dtype):
    """oracle.clip_and_adam == nn.utils.clip_grad_norm_(0.5) + torch.optim.Adam(lr=3e-4, eps=1e-5), 25 steps with
    gradient norms on both sides of the clip threshold."""
    g = torch.Generator().manual_seed(4)
    theta0 = torch.randn(po.N_PARAMS, generator=g, dtype=dtype) * 0.1
    p = nn.Parameter(theta0.clone())
    opt = torch.optim.Adam([p], lr=3e-4, eps=1e-5)
    st, theta = po.AdamState(po.N_PARAMS, dtype), theta0.clone()
    clipped = 0
    for k in range(25):
        scale = 10.0 ** ((k % 5) - 4)                  # |g| from ~1e-2 (unclipped) to ~1e2 (clipped)
        grad = torch.randn(po.N_PARAMS, generator=g, dtype=dtype) * scale
        p.grad = grad.clone()
        total_ref = nn.utils.clip_grad_norm_([p], 0.5)
        opt.step()
        theta, total = po.clip_and_adam(theta, grad, st)
        clipped += total > 0.5
        assert abs(total - float(total_ref)) <= 1e-6 * float(total_ref)
        tol = 1e-12 if dtype == torch.float64 else 2e-7
        assert torch.allclose(theta, p.detach(), rtol=0, atol=tol), f"step {k}: {float((theta - p.detach()).abs().max())}"
    assert 0 < clipped < 25


def test_size_one_minibatch_keeps_the_raw_advantage():
    """A minibatch of one sample (the ragged tail of n_envs * n_steps = 1 mod batch_size) is not normalised: SB3 skips it,
    where torch.std of one element would be NaN.  Loss and gradient equal SB3's rule and the unnormalised loss; with global
    statistics passed in (data parallel) the one sample is normalised with them."""
    torch.manual_seed(13)
    pol = TorchMlpPolicy().double()
    with torch.no_grad():
        for p in pol.parameters():
            p.add_(0.1 * torch.randn(p.shape, dtype=torch.float64))
    batch = _batch(1, 7, torch.float64)
    assert abs(float(batch[3][0])) > 0.1                # a raw advantage far from 0, where normalising would zero it
    loss_ref = sb3_loss(pol, *batch)
    loss_ref.backward()
    flat = pol.flat().clone().requires_grad_(True)
    loss, stats = po.ppo_loss(flat, *batch)
    (g,) = torch.autograd.grad(loss, flat)
    assert torch.isfinite(g).all()
    assert abs(float(loss.detach()) - float(loss_ref.detach())) <= 1e-12 * max(1.0, abs(float(loss_ref.detach())))
    assert torch.allclose(g, pol.flat_grad(), rtol=1e-10, atol=1e-13)
    loss_raw, _ = po.ppo_loss(flat, *batch, normalize=False)
    assert float(loss.detach()) == float(loss_raw.detach())
    pi = po.offsets()["pi.W3"][0]
    assert float(g[pi:pi + 256].abs().max()) > 0          # the policy head moves (normalising one sample would zero it)
    mu, sd = torch.tensor(0.25, dtype=torch.float64), torch.tensor(2.0, dtype=torch.float64)
    loss_g, _ = po.ppo_loss(flat, *batch, adv_mean=mu, adv_std=sd)
    loss_n, _ = po.ppo_loss(flat, *batch[:3], (batch[3] - mu) / (sd + 1e-8), batch[4], normalize=False)
    assert float(loss_g.detach()) == float(loss_n.detach())


def test_minibatch_update_passes_lr_and_max_norm():
    """oracle.minibatch_update with non-default learning rate and clip norm == clip_grad_norm_(max_norm) + Adam(lr) over
    nn.Modules, on both sides of the clip threshold."""
    torch.manual_seed(22)
    pol = TorchMlpPolicy().double()
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3, eps=1e-5)
    theta, st = pol.flat().clone(), po.AdamState(po.N_PARAMS, torch.float64)
    clipped = 0
    for k in range(6):
        batch = _batch(64, 200 + k, torch.float64)
        opt.zero_grad()
        sb3_loss(pol, *batch).backward()
        total = nn.utils.clip_grad_norm_(pol.parameters(), 2.0)
        clipped += float(total) > 2.0
        opt.step()
        theta, stats, _ = po.minibatch_update(theta, st, batch, lr=1e-3, max_norm=2.0)
        assert abs(stats["grad_norm"] - float(total)) <= 1e-12 * float(total)
        assert torch.allclose(theta, pol.flat(), rtol=0, atol=1e-12), f"step {k}"
    assert 0 < clipped < 6


def test_minibatch_updates_equal_torch_training_loop():
    """20 optimiser steps of oracle.minibatch_update == the same 20 steps of (SB3 loss over nn.Modules -> backward ->
    clip_grad_norm_ -> Adam.step): the composition of the pinned pieces, float64."""
    torch.manual_seed(21)
    pol = TorchMlpPolicy().double()
    opt = torch.optim.Adam(pol.parameters(), lr=3e-4, eps=1e-5)
    theta, st = pol.flat().clone(), po.AdamState(po.N_PARAMS, torch.float64)
    for k in range(20):
        batch = _batch(64, 100 + k, torch.float64)
        opt.zero_grad()
        sb3_loss(pol, *batch).backward()
        nn.utils.clip_grad_norm_(pol.parameters(), 0.5)
        opt.step()
        theta, stats, _ = po.minibatch_update(theta, st, batch)
        assert torch.allclose(theta, pol.flat(), rtol=0, atol=1e-12), f"step {k}"


def test_gae_equals_the_definition():
    """oracle.gae == the defining sum  A_t = sum_l (gamma lambda)^l delta_{t+l}  cut at episode ends, and SB3's
    buffer convention (episode_starts[t+1] = dones[t]; the value after the last step bootstraps unless done)."""
    rng = np.random.default_rng(0)
    K, n, gamma, lam = 37, 9, 0.99, 0.95
    rew, val = rng.normal(size=(K, n)), rng.normal(size=(K, n))
    done = rng.random((K, n)) < 0.15
    last = rng.normal(size=n)
    adv, ret = po.gae(torch.from_numpy(rew), torch.from_numpy(val), torch.from_numpy(done), torch.from_numpy(last), gamma, lam)
    ref = np.zeros((K, n))
    for i in range(n):
        for t in range(K):
            acc, w = 0.0, 1.0
            for l in range(t, K):
                nv = (last[i] if l == K - 1 else val[l + 1, i]) * (0.0 if done[l, i] else 1.0)
                acc += w * (rew[l, i] + gamma * nv - val[l, i])
                if done[l, i]:
                    break
                w *= gamma * lam
            ref[t, i] = acc
    assert np.allclose(adv.numpy(), ref, rtol=1e-12, atol=1e-12)
    assert np.allclose(ret.numpy(), ref + val, rtol=1e-12, atol=1e-12)
