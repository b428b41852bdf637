"""CPU tests of the evaluation contract (oracle/eval_oracle.py), of the ``dronecu_eval_args`` mirror and of the growing
``progress.csv`` header."""
import csv
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import drone_oracle as do  # noqa: E402
from oracle import eval_oracle as eo  # noqa: E402
from oracle import ppo_oracle as po  # noqa: E402
from oracle.vecenv_oracle import DummyVecEnvOracle, VecMonitorOracle  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _policy(seed):
    """A fixed float64 policy (deterministic action clip(mean)), evaluated row by row so that the result of a row does not
    depend on the batch it is in.  Small thrust: the drones fall, episodes last a few dozen steps."""
    g = torch.Generator().manual_seed(seed)
    theta = po.init_params(seed, torch.float64) + 0.2 * torch.randn(po.N_PARAMS, generator=g, dtype=torch.float64)
    off = po.offsets()["pi.b3"][0]
    theta[off:off + 4] = 1.5

    def act(obs):
        rows = [po.forward(theta, torch.from_numpy(np.asarray(o, np.float64)[None]))[0][0].numpy() for o in obs]
        return np.clip(np.stack(rows), 0.0, do.MOTOR_MAX).astype(np.float32)
    return act


@pytest.mark.parametrize("n_envs,n_eval", [(3, 2), (3, 3), (3, 7), (4, 10), (1, 3)])
def test_sb3_loop_equals_transition_bookkeeping(n_envs, n_eval):
    seed = 11
    policy = _policy(3)
    venv = VecMonitorOracle(DummyVecEnvOracle([eo.OracleDroneGymEnv(seed, g) for g in range(n_envs)]))
    rewards, lengths = eo.evaluate_policy(policy, venv, n_eval, return_episode_rewards=True)
    assert len(rewards) == n_eval == len(lengths)
    # the same envs, stepped in lockstep and recorded
    env = do.BatchedDroneOracle(n_envs, do.SINGLE, seed=seed)
    env.reset()                                        # evaluate_policy's env.reset()
    obs, rec_r, rec_d = env.obs(), [], []
    targets = (n_eval + np.arange(n_envs)) // n_envs
    while (np.sum(rec_d, axis=0) < targets).any() if rec_d else True:
        obs, r, d, _ = env.step(policy(obs).astype(np.float64))
        rec_r.append(r.astype(np.float32))
        rec_d.append(d)
    for _ in range(5):                                 # a few steps past the end do not change the result
        obs, r, d, _ = env.step(policy(obs).astype(np.float64))
        rec_r.append(r.astype(np.float32))
        rec_d.append(d)
    ret, ln, T = eo.episodes_from_transitions(np.array(rec_r), np.array(rec_d), n_eval)
    assert ret == rewards and ln == lengths            # float32 returns, bit for bit
    assert T == len(rec_r) - 5 and len(set(lengths)) > 1
    mean, std = eo.evaluate_policy(policy, VecMonitorOracle(DummyVecEnvOracle([eo.OracleDroneGymEnv(seed, g)
                                                                               for g in range(n_envs)])), n_eval)
    assert mean == np.mean(rewards) and std == np.std(rewards)


def test_targets_and_order():
    # env 0 finishes at steps 2, 4, ...; env 1 at 3, 6, ...; env 2 never: targets (5 + i) // 3 = 1, 2, 2
    T, n = 12, 3
    rew = np.ones((T, n), np.float32) * np.array([1, 2, 3], np.float32)
    done = np.zeros((T, n), bool)
    done[1::2, 0] = True
    done[2::3, 1] = True
    done[5, 2] = done[9, 2] = True
    ret, ln, steps = eo.episodes_from_transitions(rew, done, 5)
    assert ln == [2, 3, 3, 6, 4] and ret == [2.0, 6.0, 6.0, 18.0, 12.0] and steps == 10
    with pytest.raises(ValueError):
        eo.episodes_from_transitions(rew[:8], done[:8], 5)
    # fewer episodes than envs: the last envs have target 0 and record nothing
    ret, ln, steps = eo.episodes_from_transitions(rew, done, 1)
    assert ln == [6] and steps == 6                    # target (1 + i) // 3 = 0, 0, 1: only env 2


class _NoReset:
    """A VecEnv whose reset() hands back the current observations: SB3's loop then starts mid-episode, with the
    monitor's running returns and lengths where an earlier stretch of steps left them.  Counts the loop's steps."""

    def __init__(self, venv, obs):
        self.venv, self.obs, self.num_envs, self.steps = venv, obs, venv.num_envs, 0

    def reset(self):
        return self.obs

    def step(self, actions):
        self.steps += 1
        return self.venv.step(actions)


@pytest.mark.parametrize("world,n,n_eval,warm", [(1, 3, 7, 0), (1, 4, 2, 0), (3, 2, 8, 0), (2, 3, 5, 0),
                                                 (3, 2, 2, 0), (1, 3, 7, 9), (3, 2, 9, 13)])
def test_launch_sequence_equals_sb3_loop(world, n, n_eval, warm):
    """SB3's literal loop over world * n oracle envs against launch_sequence over their record, shard by shard
    (targets of env_index0 = r n of n_global = world n): the lists in SB3's order and the loop's step count.  Covers
    zero targets (n_eval < world n) and, with ``warm`` steps before the evaluation, mid-episode starts."""
    seed, N = 11, world * n
    policy = _policy(3)
    venv = VecMonitorOracle(DummyVecEnvOracle([eo.OracleDroneGymEnv(seed, g) for g in range(N)]))
    obs = venv.reset()
    for _ in range(warm):
        obs, _, _, _ = venv.step(policy(obs))
    ep_ret0, ep_len0 = venv.episode_returns.copy(), venv.episode_lengths.copy()
    loop = _NoReset(venv, obs)
    rewards, lengths = eo.evaluate_policy(policy, loop, n_eval, return_episode_rewards=True)
    assert len(rewards) == n_eval
    if warm:
        assert (ep_len0 > 0).any() and (ep_ret0 != 0).any()
    # the same envs in lockstep, recorded from the evaluation's first step on (a few steps past its end)
    env = do.BatchedDroneOracle(N, do.SINGLE, seed=seed)
    o = env.reset()
    for _ in range(warm):
        o, _, _, _ = env.step(policy(o).astype(np.float64))
    rec_r, rec_d = [], []
    for _ in range(loop.steps + 5):
        o, r, d, _ = env.step(policy(o).astype(np.float64))
        rec_r.append(r.astype(np.float32))
        rec_d.append(d)
    reward, done = np.array(rec_r), np.array(rec_d)
    shards, T = [], 0
    for r in range(world):
        cols = slice(r * n, (r + 1) * n)
        targets = eo.shard_targets(n_eval, r * n, N, n)
        max_eps = -(-n_eval // N)
        after, ret, ln, written = eo.launch_sequence(reward[:, cols], done[:, cols], targets, [(10 ** 6, False)], max_eps,
                                                     ep_ret0[cols], ep_len0[cols])
        assert after[0]["pending"] == 0 and np.array_equal(after[0]["count"], targets)
        assert np.array_equal(written, np.arange(max_eps) < targets[:, None])
        shards.append(eo.episode_lists(after[0]["count"], ret, ln, r * n, ep_len0[cols]))
        T = max(T, int(after[0]["steps"].max()))
    assert eo.sb3_order(*shards) == (rewards, lengths)          # float32 returns, bit for bit
    assert T == loop.steps
    if world == 1 and not warm:
        assert eo.episodes_from_transitions(reward, done, n_eval) == (rewards, lengths, T)


def _limits(kind, rng):
    """probe limits: +1, +7 with the second probe repeating the first, or random steps of 0..40"""
    limit, k = 0, 0
    while True:
        limit += {"plus1": 1, "plus7": 7 if k != 1 else 0}.get(kind, int(rng.integers(0, 41)))
        k += 1
        yield limit


@pytest.mark.parametrize("kind", ["plus1", "plus7", "random"])
@pytest.mark.parametrize("split", [(1, 0, 9), (5, 0, 9), (9, 0, 9), (32, 0, 9), (21, 9, 27), (21, 18, 27)])
def test_any_limit_sequence_equals_one_probe(kind, split):
    """Over a synthetic record (uneven episode lengths, a mid-episode start), any probe sequence followed by the
    catch-up gives the slots, counts and final steps of a single probe; every probe's steps never exceed its limit, a
    repeated limit changes nothing, pending is the envs below target, and the catch-up brings every env to T."""
    rng = np.random.default_rng(sum(split) + len(kind))
    n_eval, index0, n_global = split
    n, T_rec = 9, 400
    reward = rng.normal(size=(T_rec, n)).astype(np.float32)
    done = rng.random((T_rec, n)) < np.linspace(0.02, 0.3, n)
    ret0 = rng.normal(size=n).astype(np.float32)
    len0 = rng.integers(0, 30, n)
    targets = eo.shard_targets(n_eval, index0, n_global, n)
    max_eps = -(-n_eval // n_global) + 2
    one, r1, l1, w1 = eo.launch_sequence(reward, done, targets, [(10 ** 6, False)], max_eps, ret0, len0)
    T = int(one[0]["steps"].max())
    assert T < T_rec and one[0]["pending"] == 0
    launches, gen = [], _limits(kind, rng)
    while True:
        launches.append((next(gen), False))
        after = eo.launch_sequence(reward, done, targets, launches, max_eps, ret0, len0)[0]
        if after[-1]["pending"] == 0:
            break
    launches.append((T, True))
    after, r2, l2, w2 = eo.launch_sequence(reward, done, targets, launches, max_eps, ret0, len0)
    for k, ((limit, catch_up), a) in enumerate(zip(launches, after)):
        assert (a["steps"] <= limit).all()
        if not catch_up:
            assert a["pending"] == int((a["count"] < targets).sum())
            if k and launches[k - 1] == (limit, False):
                assert np.array_equal(a["steps"], after[k - 1]["steps"]) and np.array_equal(a["count"], after[k - 1]["count"])
    assert after[-1]["pending"] is None and (after[-1]["steps"] == T).all()
    assert np.array_equal(after[-1]["count"], targets) and np.array_equal(after[-2]["steps"], one[0]["steps"])
    assert np.array_equal(w1, w2) and np.array_equal(r1[w1].view(np.uint32), r2[w2].view(np.uint32))
    assert np.array_equal(l1[w1], l2[w2])
    # the written slots are exactly the first target_i of every row
    assert np.array_equal(w2, np.arange(max_eps) < targets[:, None])
    with pytest.raises(ValueError):
        eo.launch_sequence(reward[:T - 1], done[:T - 1], targets, [(10 ** 6, False)], max_eps, ret0, len0)


def test_eval_args_mirror_matches_header(tmp_path):
    from drone_rl_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dronecu.h"\n'
                   'int main(){printf("%zu %zu %zu\\n", sizeof(dronecu_eval_args), offsetof(dronecu_eval_args, env_index0),'
                   ' offsetof(dronecu_eval_args, d_pending));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    size, off_idx, off_pend = (int(x) for x in subprocess.check_output([str(exe)]).split())
    assert size == C.sizeof(_lib.EvalArgs)
    assert off_idx == _lib.EvalArgs.env_index0.offset and off_pend == _lib.EvalArgs.d_pending.offset
    assert "dronecu_evaluate_policy" in _lib.declared_symbols()


def test_run_logger_header_grows_when_keys_appear(tmp_path):
    from drone_rl_b200.train import RunLogger
    lg = RunLogger(str(tmp_path), stdout=False)
    lg.dump({"rollout/ep_rew_mean": 1.5, "time/iterations": 1}, 10)
    lg.dump({"rollout/ep_rew_mean": 2.5, "time/iterations": 2, "eval/mean_reward": -3.0}, 20)
    lg.dump({"rollout/ep_rew_mean": 3.5, "time/iterations": 3}, 30)
    lg.close()
    with open(os.path.join(str(tmp_path), "progress.csv"), newline="") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["step", "rollout/ep_rew_mean", "time/iterations", "eval/mean_reward"]
    assert rows[1:] == [["10", "1.5", "1", ""], ["20", "2.5", "2", "-3.0"], ["30", "3.5", "3", ""]]
