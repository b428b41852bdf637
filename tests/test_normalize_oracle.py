"""CPU checks of the normalisation oracle (oracle/normalize_oracle.py) and of the C ABI mirror of the normalisation pass."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import normalize_oracle as no

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_running_mean_std_in_chunks_equals_whole_data(offset):
    rng = np.random.default_rng(1)
    data = offset + rng.normal(0, 1, (10_000, 15)) * np.linspace(0.1, 50, 15)
    rms = no.RunningMeanStd((15,), epsilon=0.0 + 1e-300)      # (almost) no prior: exactly the statistics of the data
    for chunk in np.array_split(data, [1, 7, 2000, 2001, 6000]):
        rms.update(chunk)
    assert _rel(rms.mean, data.mean(0)) <= 1e-12
    assert _rel(rms.var, data.var(0)) <= 1e-12
    assert rms.count == pytest.approx(10_000)


def test_shifted_moments_equal_direct_ones():
    rng = np.random.default_rng(2)
    x = 3e3 + rng.normal(0, 2.0, (4097, 15))
    for c in (x.mean(0) + 0.5, np.full(15, 3e3)):
        m, v, n = no.shifted_moments(x, c)
        assert n == 4097
        assert _rel(m, x.mean(0)) <= 1e-12 and _rel(v, x.var(0)) <= 1e-12


def test_frozen_vec_normalize_uses_previous_statistics():
    rng = np.random.default_rng(3)
    K, n = 8, 5
    vn = no.FrozenVecNormalize(n, gamma=0.9)
    obs = rng.normal(2, 3, (K, n, 15))
    rew = rng.normal(0, 0.1, (K, n))
    done = rng.random((K, n)) < 0.2
    o1, r1 = vn.apply(obs, rew, done)
    assert np.allclose(o1, np.clip(obs / np.sqrt(1 + 1e-8), -10, 10))          # first rollout: initial statistics
    assert np.allclose(r1, rew / np.sqrt(1 + 1e-8))
    ref = no.RunningMeanStd((15,))
    ref.update(obs.reshape(-1, 15))
    assert np.array_equal(vn.obs_rms.mean, ref.mean)
    # returns: ret = ret * gamma + r, zeroed after done
    ret, rets = np.zeros(n), []
    for k in range(K):
        ret = ret * 0.9 + rew[k]
        rets.append(ret.copy())
        ret[done[k]] = 0
    assert np.allclose(vn.returns, ret)
    rr = no.RunningMeanStd(())
    rr.update(np.concatenate(rets))
    assert vn.ret_rms.var == pytest.approx(rr.var, rel=1e-14)
    vn.training = False
    before = (vn.obs_rms.mean.copy(), vn.ret_rms.var, vn.returns.copy())
    vn.apply(obs, rew, done)
    assert np.array_equal(before[0], vn.obs_rms.mean) and before[1] == vn.ret_rms.var


def test_norm_pass_args_mirror_matches_header(tmp_path):
    from drone_rl_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "dronecu.h"\nint main(){printf("%zu %d %d %d %d\\n",'
                   "sizeof(dronecu_norm_pass_args),DRONECU_NORM_AFFINE,DRONECU_NORM_STATS,DRONECU_NORM_MOMENTS,"
                   "DRONECU_NORM_BLOCK);return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert sizes == [C.sizeof(_lib.NormPassArgs), _lib.NORM_AFFINE, _lib.NORM_STATS, _lib.NORM_MOMENTS, _lib.NORM_BLOCK]


def test_ppo_loop_oracle_normalisation_is_opt_in():
    import torch
    from oracle.ppo_loop import PPOLoopOracle
    a = PPOLoopOracle(n_envs=2, n_steps=16, batch_size=16, n_epochs=1, seed=4)
    b = no.NormalizedPPOLoopOracle(n_envs=2, n_steps=16, batch_size=16, n_epochs=1, seed=4, normalize=no.FrozenVecNormalize(2))
    a.collect_rollouts(); b.collect_rollouts()
    assert b.norm.obs_rms.count == pytest.approx(32 + 1e-4)
    b.train()                                          # the update runs on the normalised buffer
    # the buffer holds normalised observations (positions of up to 50 m clipped at 10)
    assert float(b.buf[0].abs().max()) <= 10.0 < float(a.buf[0].abs().max())
