"""GPU tests of observation / reward normalisation (csrc/obs_norm.cuh, drone_rl_b200/normalize.py) against
oracle/normalize_oracle.py (SB3 VecNormalize restated in float64) and the PPO oracle.

Stated bounds:
    normalised rows vs the float32 formula (f32 subtract, f32 multiply, clip) with the same mean_f / rstd_f: bit-identical
    normalised rows vs the float64 SB3 formula on the same float32 inputs: |err| <= rstd * (3 u |x - mean| + u |mean|) * 1.01
        (u = 2^-24: rounding of mean_f, of rstd_f, of the subtraction and of the multiplication; clipping is 1-Lipschitz)
    normalised rewards (float64 then cast to float32): 1e-6 relative;  per-env returns, running statistics: 1e-12 relative;
    running means (observations and returns): 1e-12 of max(|mean|, std) -- a mean near zero is the difference of the shift and the batch offset (and
    the float64 reference mean of 4e7 values carries ~1e-16 * log2(4e7) of the spread itself), so relative to |mean| alone
    the bound would be ill-conditioned
"""
import ctypes as C
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import drone_oracle as do  # noqa: E402
from oracle import normalize_oracle as no  # noqa: E402
from oracle import philox, ppo_oracle as po, verify  # noqa: E402
from oracle.tc_bound import tc_forward_bound  # noqa: E402

U = 2.0 ** -24
OFFSETS = torch.tensor([1e3, -50, 20, 3, -2, 1, 0.5, 0, -0.3, 40, -40, 5, 0, 0, 7e3], dtype=torch.float64)
SCALES = torch.tensor([5, 10, 2, 1, 4, 0.1, 0.5, 0.2, 0.3, 1, 1, 3, 8, 0.01, 1], dtype=torch.float64)


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


def _rel_err(got, ref, floor=1e-300):
    got = torch.as_tensor(np.asarray(got.cpu() if torch.is_tensor(got) else got, np.float64))
    ref = torch.as_tensor(np.asarray(ref.cpu() if torch.is_tensor(ref) else ref, np.float64))
    if torch.is_tensor(floor):
        floor = floor.cpu().double()
    return float(((got - ref).abs() / torch.maximum(ref.abs(), torch.as_tensor(floor, dtype=torch.float64))).max())


def _set_stats(nz, mean, var, count=50.0, ret_mean=0.3, ret_var=0.04, ret_count=50.0):
    """obs_mean[15] | obs_var[15] | obs_count | ret_mean | ret_var | ret_count, then the affine record from it."""
    s = torch.cat([torch.as_tensor(mean, dtype=torch.float64), torch.as_tensor(var, dtype=torch.float64),
                   torch.tensor([count, ret_mean, ret_var, ret_count], dtype=torch.float64)])
    nz.stats.copy_(s)
    nz._combine(None)


def _rms_from_stats(s):
    s = s.cpu().double().numpy()
    o, r = no.RunningMeanStd((15,)), no.RunningMeanStd(())
    o.mean, o.var, o.count = s[:15].copy(), s[15:30].copy(), float(s[30])
    r.mean, r.var, r.count = float(s[31]), float(s[32]), float(s[33])
    return o, r


def _affine_ref(x32, nz):
    """The float32 formula evaluated by torch: separate subtract and multiply kernels (each rounded), then the clip."""
    a = nz.affine
    return torch.clamp((x32 - a[:15]) * a[15:30], -float(a[30]), float(a[30]))


@pytest.mark.parametrize("stride", [15, 16])
@pytest.mark.parametrize("K", [1, 40])
@pytest.mark.parametrize("n", [1, 127, 4097, 1 << 20])
def test_pass_vs_oracle(drl, n, K, stride):
    from drone_rl_b200.normalize import ObsNormalizer
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(n * 100 + K + stride)
    raw = (OFFSETS.cuda() + SCALES.cuda() * torch.randn(K, n, 15, generator=g, device=dev, dtype=torch.float64)).float()
    store = torch.ones(K, n, stride, device=dev)
    store[..., :15] = raw
    rew = (0.01 * torch.randn(K, n, generator=g, device=dev)).float()
    done = (torch.rand(K, n, generator=g, device=dev) < 0.05).to(torch.uint8)
    nz = ObsNormalizer(n, dev, gamma=0.97)
    # a running mean near the data (as after the first rollout), large-offset features included
    _set_stats(nz, OFFSETS + 0.3 * SCALES, (1.7 * SCALES) ** 2, ret_mean=0.02, ret_var=0.0025)
    ret0 = 0.05 * torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    nz.returns.copy_(ret0)
    stats0, aff = nz.stats.clone(), nz.affine.clone()
    side_env = n // 2
    side = torch.full((K, 15), float("nan"), device=dev)
    rew_buf = rew.clone()
    assert nz.process_rollout(store, rew_buf, done, K, side_env=side_env, side_obs=side) == 3
    torch.cuda.synchronize()
    # rows: bit-identical to the float32 formula, within the stated bound of the float64 one
    ref32 = torch.clamp((raw - aff[:15]) * aff[15:30], -float(aff[30]), float(aff[30]))
    assert torch.equal(store[..., :15], ref32)
    if stride == 16:
        assert bool((store[..., 15] == 1.0).all())
    orms, rrms = _rms_from_stats(stats0)
    mean, rstd = torch.from_numpy(orms.mean).cuda(), 1.0 / torch.sqrt(torch.from_numpy(orms.var).cuda() + 1e-8)
    ref64 = torch.clamp((raw.double() - mean) * rstd, -10, 10)
    bound = rstd * (3 * U * (raw.double() - mean).abs() + U * mean.abs()) * 1.01
    assert bool(((store[..., :15].double() - ref64).abs() <= bound).all())
    assert torch.equal(side, raw[:, side_env])
    del store, ref32, ref64, bound
    # rewards, per-env returns, running statistics
    stats1 = nz.stats.cpu()
    rets, ret = torch.empty(K, n, dtype=torch.float64, device=dev), ret0.clone()
    for k in range(K):
        ret = ret * 0.97 + rew[k].double()
        rets[k] = ret
        ret = torch.where(done[k].bool(), torch.zeros_like(ret), ret)
    assert _rel_err(nz.returns, ret, 1e-30) <= 1e-12
    rew_n = torch.clamp(rew.double() / np.sqrt(rrms.var + 1e-8), -10, 10)
    assert _rel_err(rew_buf, rew_n, 1e-30) <= 1e-6
    x = raw.double().reshape(-1, 15)
    orms.update_from_moments(x.mean(0).cpu().numpy(), x.var(0, unbiased=False).cpu().numpy(), x.shape[0])
    rr = rets.reshape(-1)
    rrms.update_from_moments(float(rr.mean()), float(rr.var(unbiased=False)), rr.numel())
    assert _rel_err(stats1[:15], orms.mean, torch.from_numpy(np.sqrt(orms.var))) <= 1e-12
    assert _rel_err(stats1[15:30], orms.var) <= 1e-12
    assert float(stats1[30]) == orms.count and float(stats1[33]) == rrms.count
    assert _rel_err(stats1[31], rrms.mean, np.sqrt(rrms.var)) <= 1e-12 and _rel_err(stats1[32], rrms.var) <= 1e-12


def test_pass_rewrites_rewards(drl):
    from drone_rl_b200.normalize import ObsNormalizer
    dev = torch.device("cuda", 0)
    K, n = 40, 4097
    g = torch.Generator(device=dev).manual_seed(9)
    rew = (0.01 * torch.randn(K, n, generator=g, device=dev)).float()
    rew[3, :5] = torch.tensor([10.0, -10.0, 3.0, 0.0, 1e-3])          # clipped at +-10 after the scale
    done = (torch.rand(K, n, generator=g, device=dev) < 0.05).to(torch.uint8)
    nz = ObsNormalizer(n, dev, norm_obs=False, norm_reward=True)
    _set_stats(nz, torch.zeros(15), torch.ones(15), ret_var=0.04)
    out = rew.clone()
    obs = torch.zeros(K, n, 16, device=dev)
    nz.process_rollout(obs, out, done, K)
    ref = torch.clamp(rew.double() / np.sqrt(0.04 + 1e-8), -10, 10)
    assert _rel_err(out, ref, 1e-30) <= 1e-6
    assert bool((obs == 0).all())                                     # norm_obs off: rows untouched
    assert float(nz.stats[30]) == 50.0                                # ... and no observation moments


def _record_model(drl, kernel, n, K, seed):
    from drone_rl_b200.ppo import PPO
    model = PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=seed, env_offset=77), n_steps=K, seed=seed, norm_obs=True)
    g = torch.Generator().manual_seed(5)
    flat = po.init_params(5, torch.float64) + 0.03 * torch.randn(po.N_PARAMS, generator=g, dtype=torch.float64)
    off = po.offsets()["pi.b3"][0]
    flat[off:off + 4] = 2.45
    off = po.offsets()["log_std"][0]
    flat[off:off + 4] = torch.tensor([-0.5, -0.2, 0.1, -1.0], dtype=torch.float64)
    model.params.copy_(flat.float().cuda())
    return model, flat.float().double()


def _rollout(model, K, affine, tc, last_obs):
    from drone_rl_b200 import _lib
    from drone_rl_b200._lib import PolicyOut
    b = model.buf
    out = PolicyOut(b.obs.data_ptr(), b.actions.data_ptr(), b.logp.data_ptr(), b.value.data_ptr(), b.reward.data_ptr(),
                    b.done.data_ptr(), b.last_value.data_ptr(), last_obs.data_ptr())
    _lib.check(model.lib.dronecu_rollout_policy_norm(model.batch._h, K, C.c_void_p(model.params.data_ptr()), 0, C.byref(out),
                                                     None if affine is None else C.c_void_p(affine.data_ptr()), int(tc), None))
    torch.cuda.synchronize()


@pytest.fixture
def rollout_kernel_mode():
    from drone_rl_b200 import _lib
    lib = _lib.load()
    yield lambda mode: _lib.check(lib.dronecu_set_rollout_kernel(mode))
    lib.dronecu_set_rollout_kernel(0)


@pytest.mark.parametrize("kernel", ["thread_per_env", "warp_per_env", "tensor_cores"])
def test_rollout_with_normalised_towers(drl, rollout_kernel_mode, kernel):
    tc = kernel == "tensor_cores"
    if not tc:
        rollout_kernel_mode({"thread_per_env": 1, "warp_per_env": 2}[kernel])
    n, K, seed = (2048 if tc else 3000), 40, 21
    model, theta = _record_model(drl, kernel, n, K, seed)
    nz = model.normalizer
    # a non-identity record: typical observation means / spreads of this task
    _set_stats(nz, torch.linspace(-3, 12, 15), torch.linspace(0.5, 30, 15) ** 2)
    b = model.buf
    last_obs = torch.empty(n, 15, device="cuda")
    t0 = model.batch.global_step
    state0 = model.batch.get_state()
    _rollout(model, K, nz.affine, tc, last_obs)
    obs = b.obs.clone()
    x_n = _affine_ref(obs, nz)
    act = b.actions.cpu().numpy()
    ids = np.arange(77, 77 + n, dtype=np.uint64)
    std = np.exp(theta[-4:].numpy())
    tol_a, tol_v, tol_lp = 2e-5, 2e-5, 1e-4
    th32 = theta.float().numpy()
    for k in range(K):
        mean, value, log_std = po.forward(theta, x_n[k].cpu().double())
        z = philox.noise_normals(seed, ids, t0 + k)
        ref_a = mean.numpy() + std * z
        lp_got = b.logp[k].cpu().numpy()
        v = b.value[k].cpu().double()
        if tc:      # the tensor-core forward within its derived bound (oracle/tc_bound.py); logp from z alone
            _, _, mb, vb = tc_forward_bound(th32, x_n[k].cpu().numpy())
            bound_a = mb + 2.0 ** -20 * std * np.abs(z) + 2.0 ** -24 * np.abs(act[k])
            assert (np.abs(act[k] - ref_a) <= bound_a).all(), f"action k={k}"
            ref_lp = -0.5 * (z * z).sum(1) - th32[-4:].astype(np.float64).sum() - 2 * np.log(2 * np.pi)
            assert (np.abs(lp_got - ref_lp) <= 2.0 ** -19 * (0.5 * (z * z).sum(1) + np.abs(th32[-4:]).sum() + 4)).all()
            assert bool(((v - value).abs() <= torch.from_numpy(vb)).all()), f"value k={k}"
            continue
        assert (np.abs(act[k] - ref_a) <= tol_a * np.maximum(np.abs(ref_a), 1)).all(), f"action k={k}"
        lp = po.log_prob(mean, log_std, torch.from_numpy(act[k]).double())
        assert np.abs(lp_got - lp.numpy()).max() < tol_lp
        assert bool(((v - value).abs() <= tol_v * value.abs().clamp(min=1)).all()), f"value k={k}"
    _, lv, _ = po.forward(theta, _affine_ref(last_obs, nz).cpu().double())
    lv_bound = (torch.from_numpy(tc_forward_bound(th32, _affine_ref(last_obs, nz).cpu().numpy())[3]) if tc
                else tol_v * lv.abs().clamp(min=1))
    assert bool(((b.last_value.cpu().double() - lv).abs() <= lv_bound).all())
    # the env transitions, on the raw rows
    o = obs.cpu().numpy()
    nxt = np.concatenate([o[1:], last_obs.cpu().numpy()[None]], 0)
    rep = verify.check_rollout(o[0], np.clip(act, 0, np.float32(7.3575)), nxt, b.reward.cpu().numpy(),
                               b.done.cpu().numpy().astype(bool), spec=do.SINGLE, seed=seed, env_ids=ids)
    assert rep["dones"] > 0
    # after the pass the buffer holds exactly what the towers saw
    nz.training = False
    nz.process_rollout(b.obs_store, b.reward, b.done, K)
    torch.cuda.synchronize()
    assert torch.equal(b.obs, x_n)
    # an identity record reproduces the plain rollout bit for bit
    ident = torch.cat([torch.zeros(15), torch.ones(15), torch.tensor([float("inf")])]).cuda()
    outs = []
    for aff in (None, ident):
        model.batch.set_state(**state0)
        model.batch.global_step = t0
        _rollout(model, K, aff, tc, last_obs)
        outs.append([t.clone() for t in (b.obs, b.actions, b.logp, b.value, b.reward, b.done, b.last_value, last_obs)])
    assert all(torch.equal(x, y) for x, y in zip(*outs))
    model.close()


def test_statistics_are_bit_reproducible(drl):
    from drone_rl_b200.ppo import PPO
    runs = []
    for _ in range(2):
        m = PPO(drl.DroneBatch(1 << 18, drl.EnvConfig.single(), seed=4), n_steps=8, seed=4, norm_obs=True, norm_reward=True,
                rollout_precision="tf32")
        for _ in range(8):
            m.collect_rollouts()
        torch.cuda.synchronize()
        runs.append((m.normalizer.stats.cpu(), m.normalizer.returns.cpu(), m.buf.obs.cpu()))
        m.close()
    assert all(torch.equal(a, b) for a, b in zip(*runs))


def _spy(model):
    """Capture the raw rollout (rows, rewards, dones) before the normalisation pass rewrites it."""
    nz, raw = model.normalizer, []
    orig = nz.process_rollout

    def spy(obs_store, reward, done, K, *a, **k):
        raw.append((obs_store[..., :15].double().cpu().numpy(), reward.double().cpu().numpy(), done.bool().cpu().numpy()))
        return orig(obs_store, reward, done, K, *a, **k)
    nz.process_rollout = spy
    return raw


def test_ppo_statistics_and_evaluation_returns_follow_the_oracle(drl, tmp_path):
    from drone_rl_b200.ppo import PPO
    n, K = 256, 32
    model = PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=2), n_steps=K, batch_size=2048, n_epochs=2, seed=2,
                norm_obs=True, norm_reward=True)
    l0 = model.launches
    raw = _spy(model)
    ora = no.FrozenVecNormalize(n, gamma=model.gamma)
    for it in range(3):
        model.collect_rollouts()
        assert model.launches - l0 == 5                 # rollout, pass, reduce, combine, GAE
        obs_n, rew_n = ora.apply(*raw[-1])
        # the buffer: float32 formula of the statistics before this rollout; rewards from the float64 formula
        assert _rel_err(model.buf.reward.cpu(), torch.from_numpy(rew_n), 1e-30) <= 1e-6
        st = model.normalizer.stats.cpu().numpy()
        assert _rel_err(st[:15], ora.obs_rms.mean, torch.from_numpy(np.sqrt(ora.obs_rms.var))) <= 1e-12
        assert _rel_err(st[15:30], ora.obs_rms.var) <= 1e-12
        assert _rel_err(st[31], ora.ret_rms.mean, np.sqrt(ora.ret_rms.var)) <= 1e-12 and _rel_err(st[32], ora.ret_rms.var) <= 1e-12
        assert st[30] == pytest.approx(ora.obs_rms.count, rel=1e-15) and st[33] == pytest.approx(ora.ret_rms.count, rel=1e-15)
        assert _rel_err(model.normalizer.returns.cpu(), torch.from_numpy(ora.returns), 1e-30) <= 1e-12
        model.train()
        l0 = model.launches
    assert model.obs_rms.count == pytest.approx(3 * n * K + 1e-4)
    # evaluation: statistics unchanged, per-env returns not advanced but zeroed where an episode ended (SB3 step_wait)
    model.training = False
    before = (model.normalizer.stats.clone(), model.normalizer.returns.clone())
    model.collect_rollouts()
    ended = model.buf.done.bool().any(0)
    assert bool(ended.any())
    assert torch.equal(before[0], model.normalizer.stats)
    assert torch.equal(model.normalizer.returns, torch.where(ended, torch.zeros_like(before[1]), before[1]))
    model.training = True
    # checkpoints: statistics, per-env returns (same shard), identical predict
    obs = np.random.default_rng(0).normal(0, 5, (64, 15)).astype(np.float32)
    ref, _ = model.predict(obs, deterministic=True)
    pt, zp = str(tmp_path / "m.pt"), str(tmp_path / "m")
    model.save(pt)
    model.save(zp)
    for path in (pt, zp + ".zip"):
        m2 = PPO.load(path, drl.DroneBatch(n, drl.EnvConfig.single(), seed=2))
        assert m2.normalizer is not None and m2.normalizer.norm_obs and m2.normalizer.norm_reward
        assert torch.equal(m2.normalizer.stats, model.normalizer.stats)
        assert torch.equal(m2.normalizer.returns, model.normalizer.returns)
        assert np.array_equal(m2.predict(obs, deterministic=True)[0], ref)
        m2.close()
        m3 = PPO.load(path, drl.DroneBatch(n // 2, drl.EnvConfig.single(), seed=2))     # another shard: fresh returns
        assert torch.equal(m3.normalizer.stats, model.normalizer.stats) and bool((m3.normalizer.returns == 0).all())
        m3.close()
    # an explicit override wins over the archive
    m4 = PPO.load(pt, drl.DroneBatch(n, drl.EnvConfig.single(), seed=2), norm_obs=False, norm_reward=False)
    assert m4.normalizer is None
    m4.close()
    model.close()


def test_predict_normalises_and_default_is_unchanged(drl):
    from drone_rl_b200.ppo import PPO
    a = PPO(drl.DroneBatch(8, drl.EnvConfig.single(), seed=1), n_steps=4, seed=1)
    b = PPO(drl.DroneBatch(8, drl.EnvConfig.single(), seed=1), n_steps=4, seed=1, norm_obs=True)
    assert a.normalizer is None and a.obs_rms is None
    _set_stats(b.normalizer, torch.linspace(-3, 12, 15), torch.linspace(0.5, 30, 15) ** 2)
    obs = np.random.default_rng(1).normal(0, 5, (16, 15)).astype(np.float32)
    x = b.normalize_obs(obs)
    assert torch.equal(x, _affine_ref(torch.from_numpy(obs).cuda(), b.normalizer))
    mean, _ = a.policy_forward(x)
    assert np.array_equal(b.predict(obs, deterministic=True)[0], torch.clamp(mean, 0, 7.3575).cpu().numpy())
    l0 = a.launches
    a.collect_rollouts()
    assert a.launches - l0 == 2
    a.close(); b.close()


def test_train_driver_with_normalisation_records_raw_positions(drl, tmp_path, monkeypatch):
    from drone_rl_b200 import train
    from drone_rl_b200.ppo import PPO
    monkeypatch.chdir(tmp_path)
    train.main(["--total-timesteps", "8192", "--n-envs", "64", "--n-steps", "64", "--batch-size", "1024", "--n-epochs", "1",
                "--norm-obs", "--norm-reward", "--quiet", "--save", "dd"])
    m = PPO.load("dd.zip", 1)
    assert m.normalizer is not None and m.obs_rms.count > 8192
    m.close()
    # the reference's test.py flow on that archive: raw DroneGymEnv observations -> model.predict normalises them
    from drone_rl_b200 import test as eval_script
    eval_script.main(["--model", "dd.zip", "--steps", "10", "--out", "n.gif"])
    assert os.path.isfile("n.gif")
    # the callback plots RAW positions: feed it a normalised model, one block per two episodes
    model = PPO(drl.DroneBatch(64, drl.EnvConfig.single(), seed=3), n_steps=256, seed=3, norm_obs=True, norm_reward=True)
    model.set_raw_obs_tap(0)
    raw = _spy(model)
    cb = train.TrajectoryCallback(str(tmp_path), record_interval=1, block_size=2)
    model.collect_rollouts()
    cb(model)
    assert cb.blocks_written >= 1
    z = np.load(os.path.join(str(tmp_path), "trajectory_block1.npz"))
    ep = z["ep_1"]
    assert np.array_equal(ep, raw[0][0][:ep.shape[0], 0, 0:3].astype(np.float32))
    model.close()


# ---------------------------------------------------------------------------------------------------------------------
# data parallel: two ranks, both exchange backends
# ---------------------------------------------------------------------------------------------------------------------
N_DP, K_DP, IT_DP = 2048, 16, 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, backend, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import drone_rl_b200 as drl
    from drone_rl_b200.ppo import PPO
    env = drl.DroneBatch(N_DP, drl.EnvConfig.single(), device=rank, seed=3, env_offset=rank * N_DP)
    model = PPO(env, n_steps=K_DP, seed=3, dp_backend=backend, norm_obs=True, norm_reward=True)
    for _ in range(IT_DP):           # fixed parameters: the union of the shards is the 1-rank rollout
        model.collect_rollouts()
    torch.cuda.synchronize()
    mine = model.normalizer.stats.clone()
    every = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(every, mine)
    out = {"identical": all(torch.equal(e, every[0]) for e in every), "stats": mine.cpu(), "backend": model.dp_backend}
    model.close()
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("backend", ["peer", "nccl"])
def test_two_rank_statistics_equal_one_rank_on_the_union(drl, backend):
    import torch.multiprocessing as mp
    from drone_rl_b200.ppo import PPO
    ctx = mp.get_context("spawn")
    q, port = ctx.Queue(), _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, backend, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert out["identical"] and out["backend"] == backend
    one = PPO(drl.DroneBatch(2 * N_DP, drl.EnvConfig.single(), seed=3), n_steps=K_DP, seed=3, norm_obs=True, norm_reward=True)
    for _ in range(IT_DP):
        one.collect_rollouts()
    st, ref = out["stats"], one.normalizer.stats.cpu()
    assert _rel_err(st[:15], ref[:15], ref[15:30].sqrt()) <= 1e-12 and _rel_err(st[31], ref[31], ref[32].sqrt()) <= 1e-12
    assert _rel_err(st[15:31], ref[15:31]) <= 1e-12 and _rel_err(st[32:], ref[32:]) <= 1e-12
    one.close()
