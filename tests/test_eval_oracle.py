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
