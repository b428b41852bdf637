"""The oracle's env constants as a record (oracle/drone_oracle.Params): the defaults are EnvConfig's, VecMonitor zeroes
its accumulators on every done, and oracle/verify.check_rollout checks a record against the constants it is given."""
import dataclasses

import numpy as np
import pytest

from oracle import drone_oracle as do
from oracle import philox, verify

NON_DEFAULT = do.Params(inertia=(0.004, 0.006, 0.011), mass=1.3, gravity=9.7, dt=0.015, arm_length=0.4, k_yaw=0.013,
                        r_max=30.0, z_floor=0.25, bonus=0.5, bonus_radius=0.3, reward_scale=0.02, max_steps=23,
                        curriculum_period=3, curriculum_step=0.07, start_z=1.5, target_z=2.0,
                        fixed_start=(0.25, -0.5, 1.0), fixed_target=(1.0, -2.0, 5.0))


def test_params_defaults_are_env_config_defaults():
    torch = pytest.importorskip("torch")  # noqa: F841  (drone_rl_b200.core imports it)
    from drone_rl_b200.core import EnvConfig
    assert do.Params.from_config(EnvConfig.single()) == do.Params.of(do.SINGLE) == do.DEFAULT
    assert do.Params.from_config(EnvConfig.vector()) == do.Params.of(do.VECTOR)
    assert do.DEFAULT.motor_max == do.MOTOR_MAX


def test_curriculum_eps_accumulates_in_order():
    """0.1, 0.2, 0.30000000000000004 ... at any period and step, one float64 addition per bump (drone.py:68-70)"""
    for period, step in ((2000, 0.1), (3, 0.07), (1, 0.1)):
        ep = np.array([0, period - 1, period, 3 * period, 3 * period + 1, 20 * period, 7 * period])
        eps = [0.0]
        for _ in range(20):
            eps.append(eps[-1] + step)
        want = np.array([eps[e // period] for e in ep])
        assert np.array_equal(do.curriculum_eps(ep, period, step), want)
    assert do.curriculum_eps(np.array([6000]))[0] == 0.30000000000000004
    assert do._accumulate(0.0, 0.1, 10_000_001, chunk=1 << 20) == do._accumulate(0.0, 0.1, 10_000_001, chunk=1 << 23)


@pytest.mark.parametrize("auto_reset", [False, True])
def test_vecmonitor_zeroes_on_every_done(auto_reset):
    """VecMonitor ends an episode on every done, whether or not the env resets: without auto-reset an env past its time
    limit is done on every later step, each an episode of length 1 whose return is that step's reward."""
    p = dataclasses.replace(NON_DEFAULT, max_steps=3, auto_reset=auto_reset, r_max=1e9, z_floor=-1e9)
    o = do.BatchedDroneOracle(2, p, seed=1)
    hover = np.full((2, 4), p.mass * p.gravity / 4, np.float32)
    lengths, returns, rewards = [], [], []
    for _ in range(6):
        _, rew, done, info = o.step(hover)
        rewards.append(rew.astype(np.float32))
        if done.any():
            assert done.all()
            lengths.append(int(info["episode_l"][0]))
            returns.append(info["episode_r"][0])
    if auto_reset:
        assert lengths == [3, 3]
    else:
        assert lengths == [3, 1, 1, 1]
        assert returns[0] == np.float32(np.float32(rewards[0][0] + rewards[1][0]) + rewards[2][0])
        assert returns[1:] == [r[0] for r in rewards[3:]]
        assert (o.ep_length == 0).all() and (o.ep_return == 0).all() and (o.step_count == 6).all()


def _record(p, n, K, seed, rng):
    """A float32 record of the oracle under p (no auto-reset), with the initial targets; the state is rounded to float32
    after every step, as the record is (the float64 trajectory itself drifts off it near the pitch singularity)"""
    o = do.BatchedDroneOracle(n, p, seed=seed)
    obs0 = o.reset()
    target0 = o.target.astype(np.float32)
    acts = rng.uniform(0, p.motor_max, (K, n, 4)).astype(np.float32)
    nxt, rew, done = [], [], []
    for k in range(K):
        ob, r, d, _ = o.step(acts[k])
        nxt.append(ob); rew.append(r.astype(np.float32)); done.append(d)
        for name in ("pos", "vel", "euler", "omega"):
            setattr(o, name, getattr(o, name).astype(np.float32).astype(np.float64))
    return obs0, acts, np.stack(nxt), np.stack(rew), np.stack(done), target0


@pytest.mark.parametrize("D,R", [(15, True), (15, False), (12, True), (12, False)])
def test_check_rollout_pins_the_constants(D, R):
    """check_rollout accepts the oracle's own record under non-default constants and rejects it under the mistakes a
    parameter digest can make: the roll and pitch inertia swapped, the mass in place of its inverse, the step changed."""
    p = dataclasses.replace(NON_DEFAULT, obs_dim=D, randomized=R, auto_reset=False)
    rng = np.random.default_rng(D + R)
    obs0, acts, nxt, rew, done, target0 = _record(p, 48, 30, 5, rng)
    assert done.any() and not done.all()
    kw = dict(seed=5, ep_num0=2, target0=target0)
    rep = verify.check_rollout(obs0, acts, nxt, rew, done, spec=p, **kw)
    assert rep["worst_err_over_bound"] < 0.5
    i = p.inertia
    for wrong in (dict(inertia=(i[1], i[0], i[2])), dict(mass=1.0 / p.mass), dict(dt=0.02)):
        with pytest.raises(AssertionError):
            verify.check_rollout(obs0, acts, nxt, rew, done, spec=dataclasses.replace(p, **wrong), **kw)


@pytest.mark.parametrize("R", [True, False])
def test_reset_rows_of_every_reset_kind(R):
    """verify.reset_rows: the fixed start / target of the record, or the Philox start at start_z with the target at
    target_z before the first curriculum bump and eps * u after it."""
    p = dataclasses.replace(NON_DEFAULT, randomized=R)
    ids = np.arange(5, dtype=np.uint64) + np.uint64(1 << 33)
    ep = np.array([1, 2, 3, 4, 9])
    rp, rt = verify.reset_rows(p, 7, ids, ep)
    if not R:
        assert (rp == np.float32(p.fixed_start)).all() and (rt == np.float32(p.fixed_target)).all()
        return
    u = philox.reset_uniforms(7, ids, ep)
    assert np.array_equal(rp[:, :2], (u[:2].T - 0.5).astype(np.float32)) and (rp[:, 2] == np.float32(p.start_z)).all()
    assert (rt[:2] == np.float32([0, 0, p.target_z])).all()
    eps = do.curriculum_eps(ep[2:], p.curriculum_period, p.curriculum_step)
    assert np.array_equal(rt[2:, 0], (eps * u[2, 2:]).astype(np.float32))
    assert np.array_equal(rt[2:, 2], (eps * u[4, 2:] + p.target_z).astype(np.float32))
