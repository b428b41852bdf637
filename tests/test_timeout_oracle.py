"""The time-limit bootstrap (SB3 handle_timeout_termination) on the CPU: SB3's literal expression
``rewards[idx] += self.gamma * terminal_value`` pinned against the float32 expression the GPU kernel evaluates, the oracle
loops with the bootstrap (tests/timeout_oracle.py) against that literal expression, and the new C ABI declared and bound.

Pinned here (numpy + torch, as SB3 runs them):
  plain rewards (DummyVecEnv's float32 array)         f32(r + f32(f32(gamma) * V))
  normalised rewards (VecNormalize's float64 array)   the same: torch adds the float64 element as a wrapped scalar, i.e.
                                                      rounded to float32, and returns a float32 tensor.  So the GPU, which
                                                      holds the normalised reward already rounded to float32, matches SB3
                                                      exactly; against a float64 add rounded once it is within one ulp
                                                      of max(|q|, |result|).
"""
import os
import re
from dataclasses import replace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import drone_oracle as do  # noqa: E402
from oracle import normalize_oracle as no  # noqa: E402
from oracle import ppo_oracle as po  # noqa: E402
from oracle.ppo_loop import PPOLoopOracle  # noqa: E402
from tests.timeout_oracle import GAMMA, TimeoutNormalizedPPOLoopOracle, TimeoutPPOLoopOracle  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMAS = (0.99, 0.95, 0.999, 0.9)


def _values(rng, m):
    """float32 values over many binades, both signs, a few exact zeros"""
    v = (rng.standard_normal(m) * np.exp2(rng.integers(-12, 8, m))).astype(np.float32)
    v[::97] = 0.0
    return v


def kernel_expr(r, v, gamma):
    """what timeout_bootstrap_kernel computes: __fadd_rn(r, __fmul_rn(f32(gamma), v))"""
    return (np.float32(r) + (np.float32(gamma) * np.asarray(v, np.float32)).astype(np.float32)).astype(np.float32)


def _sb3(rewards, v, gamma):
    """SB3 collect_rollouts, literally, on every index: terminal_value as predict_values(...)[0], a float32 tensor [1]"""
    for idx in range(len(rewards)):
        terminal_value = torch.tensor([[v[idx]]], dtype=torch.float32)[0]
        rewards[idx] += gamma * terminal_value
    return rewards


@pytest.mark.parametrize("gamma", GAMMAS)
def test_sb3_expression_on_float32_rewards(gamma):
    rng = np.random.default_rng(int(gamma * 1000))
    r, v = _values(rng, 4000), _values(rng, 4000)
    got = _sb3(r.copy(), v, gamma)
    assert got.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), kernel_expr(r, v, gamma).view(np.uint32))
    # the pin discriminates: a float64 product rounded once differs on some values
    alt = (r.astype(np.float64) + np.float32(gamma * v.astype(np.float64))).astype(np.float32)
    assert not np.array_equal(got, alt) or gamma == 0.9


@pytest.mark.parametrize("gamma", GAMMAS)
def test_sb3_expression_on_normalised_rewards(gamma):
    """VecNormalize hands back float64 rewards; the buffer stores float32.  The GPU holds f32(q) (the pass rounds the
    normalised reward) and adds in float32."""
    rng = np.random.default_rng(7 + int(gamma * 1000))
    q = rng.standard_normal(4000) * np.exp2(rng.integers(-6, 3, 4000))
    v = _values(rng, 4000)
    got = _sb3(q.copy(), v, gamma).astype(np.float32)                 # RolloutBuffer.add stores float32
    gpu = kernel_expr(q.astype(np.float32), v, gamma)
    assert np.array_equal(got.view(np.uint32), gpu.view(np.uint32))
    # the model "add in float64, round once" is within one float32 ulp of the larger of |q| and the result (q rounded to
    # float32 first: half an ulp of q, then the rounding of the sum)
    f64 = (q + (np.float32(gamma) * v).astype(np.float32).astype(np.float64)).astype(np.float32)
    ulp = np.spacing(np.maximum.reduce([np.abs(q.astype(np.float32)), np.abs(gpu), np.abs(f64)]))
    assert np.all(np.abs(gpu.astype(np.float64) - f64) <= ulp)


def test_non_finite_value_gives_nan_reward():
    r = np.array([1.0, -2.0, 0.5], np.float32)
    v = np.array([np.nan, np.inf, -np.inf], np.float32)
    got = _sb3(r.copy(), v, 0.99)
    assert np.isnan(got[0]) and np.isposinf(got[1]) and np.isneginf(got[2])
    assert np.array_equal(got, kernel_expr(r, v, 0.99), equal_nan=True)


# ---------------------------------------------------------------------------------------------------------------------
# the oracle loops
# ---------------------------------------------------------------------------------------------------------------------
SPEC7 = replace(do.SINGLE, max_steps=7)


def _tap(loop):
    """record the (obs, info) of every env step of an oracle loop"""
    seen, step = [], loop.env.step

    def spy(action):
        res = step(action)
        seen.append(res)
        return res
    loop.env.step = spy
    return seen


def _hover(loop):
    """a policy that keeps the drones up long enough to reach the 7-step limit: bias the thrust"""
    p = po.unpack(loop.theta)
    p["pi.b3"][:] = 2.5
    p["pi.W3"][:] = 0.0


@pytest.fixture
def gae_rewards(monkeypatch):
    """the reward tensor every oracle rollout hands to GAE"""
    seen, gae = [], po.gae

    def spy(rewards, *a, **k):
        seen.append(rewards.clone())
        return gae(rewards, *a, **k)
    monkeypatch.setattr(po, "gae", spy)
    return seen


@pytest.mark.parametrize("n_envs", [1, 5])
def test_plain_loop_adds_sb3_bootstrap_on_truncated_steps(n_envs, gae_rewards):
    K, gamma = 20, GAMMA
    off = PPOLoopOracle(n_envs, K, K * n_envs, 1, spec=SPEC7)
    on = TimeoutPPOLoopOracle(n_envs, K, K * n_envs, 1, spec=SPEC7)
    for loop in (off, on):
        _hover(loop)
    seen = _tap(on)
    off.collect_rollouts()
    on.collect_rollouts()
    r_off, r_on = (r.numpy() for r in gae_rewards)
    # same trajectory: the bootstrap changes rewards only
    assert torch.equal(on.buf[0], off.buf[0]) and torch.equal(on.buf[1], off.buf[1])
    ref = r_off.copy()
    n_trunc = 0
    for t, (_, _, _, info) in enumerate(seen):
        for idx in np.flatnonzero(info["truncated"]):
            terminal_value = po.forward(on.theta, torch.from_numpy(info["terminal_obs"][idx:idx + 1]).to(torch.float32))[1]
            ref[t][idx] += gamma * terminal_value                          # SB3's line
            n_trunc += 1
        assert not (info["truncated"] & info["terminated"]).any()
    assert n_trunc >= 2 * n_envs, "the 7-step limit must be reached"
    assert np.array_equal(r_on, ref)
    trunc = np.stack([s[3]["truncated"] for s in seen])
    assert np.array_equal(r_on != r_off, trunc)


def test_normalised_loop_bootstraps_the_normalised_reward(gae_rewards):
    n, K, gamma = 3, 16, GAMMA

    def make(flag):
        cls = TimeoutNormalizedPPOLoopOracle if flag else no.NormalizedPPOLoopOracle
        loop = cls(n, K, K * n, 1, spec=SPEC7, normalize=no.FrozenVecNormalize(n, gamma=gamma, clip_obs=5.0))
        _hover(loop)
        loop.norm.obs_rms.mean[:], loop.norm.obs_rms.var[:] = 0.5, 4.0        # statistics that are not the identity
        loop.norm.ret_rms.var = 9.0
        return loop
    off, on = make(False), make(True)
    seen = _tap(on)
    rms0 = no.RunningMeanStd((15,))
    rms0.mean[:], rms0.var[:] = 0.5, 4.0
    off.collect_rollouts()
    on.collect_rollouts()
    # the statistics and the per-env returns see raw rewards: identical with and without the bootstrap
    assert np.array_equal(on.norm.returns, off.norm.returns)
    assert on.norm.ret_rms.var == off.norm.ret_rms.var and np.array_equal(on.norm.obs_rms.var, off.norm.obs_rms.var)
    r_off, r_on = (r.numpy().astype(np.float64) for r in gae_rewards)
    q = r_off.copy()                               # the normalised rewards, float64 as VecNormalize returns them
    n_trunc = 0
    for t, (_, _, _, info) in enumerate(seen):
        for idx in np.flatnonzero(info["truncated"]):
            row = no.normalize_obs(info["terminal_obs"][idx:idx + 1], rms0, 5.0)   # VecNormalize.step_wait
            q[t][idx] += gamma * po.forward(on.theta, torch.from_numpy(row).to(torch.float32))[1]
            n_trunc += 1
    assert n_trunc >= n
    assert np.array_equal(r_on, q.astype(np.float32).astype(np.float64))


# ---------------------------------------------------------------------------------------------------------------------
# the C ABI
# ---------------------------------------------------------------------------------------------------------------------
def test_new_abi_is_declared_and_bound():
    from drone_rl_b200 import _lib
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dronecu.h")).read(), flags=re.S)
    for name in ("dronecu_rollout_policy_timeouts", "dronecu_bootstrap_timeouts"):
        assert re.search(rf"\bint {name}\s*\(", txt), name
        assert name in _lib.declared_symbols()
    m = re.search(r"typedef struct dronecu_timeout_buf \{(.*?)\} dronecu_timeout_buf;", txt, flags=re.S)
    fields = re.findall(r"(\w+);", m.group(1))
    assert fields == [f for f, _ in _lib.TimeoutBuf._fields_]
    args = _lib._SIGNATURES["dronecu_rollout_policy_timeouts"][1]
    assert len(args) == 9 and args[7]._type_ is _lib.TimeoutBuf
    assert _lib._SIGNATURES["dronecu_bootstrap_timeouts"][1][5] is __import__("ctypes").c_float
