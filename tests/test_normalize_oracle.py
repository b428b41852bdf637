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
    # evaluation: the returns are not advanced, but an env whose episode ended restarts from 0 (SB3 step_wait)
    assert done.any(0).any()
    assert np.array_equal(vn.returns, np.where(done.any(0), 0.0, before[2]))


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


def test_reward_formula_is_float64_then_float32_with_np_clip():
    import math
    rng = np.random.default_rng(5)
    r = np.concatenate([rng.normal(0, 0.3, 200), [np.nan, np.inf, -np.inf, 3.4028235e38, -0.0]]).astype(np.float32)
    got = no.normalize_reward_f32(r, 0.0123, clip_reward=2.0, epsilon=1e-3)
    for x, y in zip(r, got):
        q = float(x) / math.sqrt(0.0123 + 1e-3)
        want = q if math.isnan(q) else min(max(q, -2.0), 2.0)
        assert (math.isnan(want) and math.isnan(y)) or np.float32(want).tobytes() == y.tobytes()
    assert got.dtype == np.float32 and np.isnan(got[200]) and got[201] == 2 and got[202] == -2


@pytest.mark.parametrize("P", [1, 29, 30, 31, 4097])
def test_reduce_order_restates_the_kernel_loop(P):
    rng = np.random.default_rng(P)
    parts = rng.normal(0, 1, (P, 34)) * 10.0 ** rng.integers(-8, 8, (P, 34))
    got = no.reduce_partials(parts)
    for j in (0, 17, 33):               # thread (g, j): p = g, g + 30, ...; then the 30 group sums in order, from 0.0
        groups = []
        for g in range(30):
            t = 0.0
            for p in range(g, P, 30):
                t += float(parts[p, j])
            groups.append(t)
        t = 0.0
        for v in groups:
            t += v
        assert got[j] == t


def _exact_combine(mean, var, count, xs):
    """SB3 update with the batch's exact mean and population variance, in rational arithmetic"""
    from fractions import Fraction as F
    xs = [F(float(x)) for x in xs]
    cb = len(xs)
    bm = sum(xs) / cb
    bv = sum((x - bm) ** 2 for x in xs) / cb
    m, v, c = F(float(mean)), F(float(var)), F(float(count))
    d = bm - m
    tot = c + cb
    return float(m + d * cb / tot), float((v * c + bv * cb + d * d * c * cb / tot) / tot)


@pytest.mark.parametrize("shift,count", [(0.0, 1e-4), (0.9, 50.0), (0.0, 1e12), (1.0, 3.0)])
def test_combine_and_one_pass_bounds_hold(shift, count):
    """The float64 one-pass shifted evaluation (the kernel's) and SB3's combine on two_pass_moments, each within half the
    stated bound of the exact rational result; the initial statistics put the shift far from data at 7e3 +- 1."""
    rng = np.random.default_rng(int(count) % 97)
    xs = 7e3 + rng.normal(0, 1, 2000)
    mean, var = shift * 7e3, 4.0
    exact_m, exact_v = _exact_combine(mean, var, count, xs)
    d = xs - mean
    s1, s2 = 0.0, 0.0
    for v in d:                                      # sequential: depth = cb
        s1 += v
        s2 += v * v
    cb = float(len(xs))
    bm, bv = no.combine_bound(mean, var, count, s1, s2, cb)
    r = no.RunningMeanStd(())
    r.mean, r.var, r.count = np.float64(mean), np.float64(var), count
    no.combine_sb3(r, s1, s2, cb)
    om, ov = no.one_pass_bound(mean, var, count, s2, cb, depth=len(xs))
    assert abs(r.mean - exact_m) <= om / 2 + bm / 2 and abs(r.var - exact_v) <= ov / 2 + bv / 2
    r2 = no.RunningMeanStd(())
    r2.mean, r2.var, r2.count = np.float64(mean), np.float64(var), count
    r2.update_from_moments(*no.two_pass_moments(xs), cb)
    assert abs(r2.mean - exact_m) <= om / 2 and abs(r2.var - exact_v) <= ov / 2
    if shift == 0.0 and count < 1:   # the one-pass cancellation is visible, and the bound is not a relative one
        assert abs(r.var - exact_v) > 1e-15 * exact_v


def _lib_or_skip():
    from drone_rl_b200 import _lib
    try:
        return _lib, _lib.load()
    except Exception as e:          # noqa: BLE001  (no built library: the build step reports that)
        pytest.skip(f"libdronecu.so not loadable: {e}")


def test_norm_entry_points_reject_bad_arguments_without_launching():
    """Every check runs before the device is touched, so these return DRONECU_ERR_INVALID with or without a GPU."""
    _lib, lib = _lib_or_skip()
    P = lambda v: C.c_void_p(v)

    def args(**kw):
        a = _lib.NormPassArgs()
        a.d_obs, a.obs_stride, a.K, a.n, a.d_affine = 4096, 16, 4, 100, 8192
        a.d_reward, a.d_done, a.d_returns, a.d_stats = 12288, 16384, 20480, 24576
        a.update, a.d_partials, a.side_env, a.epsilon, a.clip_reward = 1, 28672, -1, 1e-8, 10.0
        for k, v in kw.items():
            setattr(a, k, v)
        return a
    bad = [dict(obs_stride=14), dict(obs_stride=16, d_obs=4100), dict(d_done=None), dict(d_stats=None),
           dict(d_returns=None), dict(d_returns=None, update=0), dict(d_partials=None), dict(n=0), dict(n=-3),
           dict(K=0), dict(K=-1), dict(d_affine=None)]
    for kw in bad:
        assert lib.dronecu_norm_pass(0, C.byref(args(**kw)), None) == -1, kw
    assert lib.dronecu_norm_pass(0, None, None) == -1
    for npart in (0, -1):
        assert lib.dronecu_norm_reduce(0, P(4096), npart, P(8192), None) == -1
    for eps, clip in ((-1e-8, 10.0), (float("nan"), 10.0), (1e-8, 0.0), (1e-8, -1.0), (1e-8, float("nan"))):
        assert lib.dronecu_norm_combine(0, P(4096), None, eps, clip, P(8192), None) == -1, (eps, clip)
