"""GPU tests of policy evaluation (csrc/ppo_eval.cuh, drone_rl_b200/evaluation.py).

Each evaluation kernel is checked against its rollout counterpart: two envs with the same seed, offset and clock; one is
evaluated, the other runs dronecu_rollout_policy[_tc|_norm] for the same T steps recording rewards and done flags, whose
transitions go through the SB3 bookkeeping of oracle/eval_oracle.py.  Same arithmetic on the same operands, so the
episode returns must agree bit for bit as float32, the lengths and T exactly, and both envs must end in bit-identical
states at the same clock.
"""
import ctypes as C
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import eval_oracle as eo  # noqa: E402
from oracle import ppo_oracle as po  # noqa: E402

SEED, OFFSET = 13, 5


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


@pytest.fixture
def rollout_kernel_mode():
    from drone_rl_b200 import _lib
    lib = _lib.load()
    yield lambda mode: _lib.check(lib.dronecu_set_rollout_kernel(mode))
    lib.dronecu_set_rollout_kernel(0)


def _model(drl, precision="fp32", norm=False, device=0):
    """A policy with hovering thrust (long, varied episodes) and distinct action stds."""
    from drone_rl_b200.ppo import PPO
    model = PPO(drl.DroneBatch(16, drl.EnvConfig.single(), device=device, seed=1), n_steps=8, seed=1, rollout_precision=precision,
                norm_obs=norm)
    g = torch.Generator().manual_seed(5)
    flat = po.init_params(5, torch.float64) + 0.03 * torch.randn(po.N_PARAMS, generator=g, dtype=torch.float64)
    off = po.offsets()["pi.b3"][0]
    flat[off:off + 4] = 2.45
    off = po.offsets()["log_std"][0]
    flat[off:off + 4] = torch.tensor([-0.5, -0.2, 0.1, -1.0], dtype=torch.float64)
    model.params.copy_(flat.float())
    if norm:                     # a non-identity record: typical observation means / spreads of this task
        s = torch.cat([torch.linspace(-3, 12, 15, dtype=torch.float64), torch.linspace(0.5, 30, 15, dtype=torch.float64) ** 2,
                       torch.tensor([50.0, 0.3, 0.04, 50.0], dtype=torch.float64)])
        model.normalizer.stats.copy_(s)
        model.normalizer._combine(None)
    return model


def _rollout_record(drl, model, env, T, deterministic):
    """T steps of the same-flavour rollout kernel on `env`: reward and done [T, n]."""
    from drone_rl_b200 import _lib
    n = env.n
    rew = torch.empty(T, n, device="cuda")
    done = torch.empty(T, n, dtype=torch.uint8, device="cuda")
    out = _lib.PolicyOut(None, None, None, None, rew.data_ptr(), done.data_ptr(), None, None, 0, 0)
    tc = int(model.rollout_precision == "tf32" and n > model.tc_min_envs)
    aff = model.normalizer.affine_ptr() if model.normalizer is not None else None
    _lib.check(model.lib.dronecu_rollout_policy_norm(env._h, T, C.c_void_p(model.params.data_ptr()), int(deterministic),
                                                     C.byref(out), aff, tc, None))
    torch.cuda.synchronize()
    return rew.cpu().numpy(), done.cpu().numpy().astype(bool)


def _check_against_rollout(drl, model, n, n_eval, deterministic):
    from drone_rl_b200.evaluation import evaluate_policy
    ev = drl.DroneBatch(n, drl.EnvConfig.single(), seed=SEED, env_offset=OFFSET)
    ro = drl.DroneBatch(n, drl.EnvConfig.single(), seed=SEED, env_offset=OFFSET)
    for b in (ev, ro):           # same, non-zero clock
        b.global_step = 1000
    t0 = ev.global_step
    rewards, lengths = evaluate_policy(model, ev, n_eval, deterministic=deterministic, return_episode_rewards=True)
    T = ev.global_step - t0
    assert len(rewards) == n_eval and T > 0
    ro.reset()
    rew, done = _rollout_record(drl, model, ro, T, deterministic)
    ref_r, ref_l, ref_T = eo.episodes_from_transitions(rew, done, n_eval)
    assert ref_T == T
    assert np.array_equal(np.array(rewards, np.float32), np.array(ref_r, np.float32)) and rewards == ref_r
    assert lengths == ref_l
    assert ro.global_step == ev.global_step
    sa, sb = ev.get_state(), ro.get_state()
    for k in sa:
        assert np.array_equal(sa[k].view(np.uint32) if sa[k].dtype == np.float32 else sa[k],
                              sb[k].view(np.uint32) if sb[k].dtype == np.float32 else sb[k]), k
    mean, std = evaluate_policy(model, ro, n_eval, deterministic=deterministic)
    assert np.isfinite(mean) and std >= 0
    ev.close(); ro.close()
    return rewards, lengths, T


@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("deterministic", [True, False])
@pytest.mark.parametrize("kernel", ["thread_per_env", "warp_per_env", "tensor_cores"])
def test_eval_equals_rollout(drl, rollout_kernel_mode, kernel, deterministic, norm):
    tc = kernel == "tensor_cores"
    if not tc:
        rollout_kernel_mode({"thread_per_env": 1, "warp_per_env": 2}[kernel])
    # tensor cores: 1500 envs = 11 full tiles and a partial one; 2000 episodes = targets of 1 and 2
    n, n_eval = (1500, 2000) if tc else (300, 450)
    model = _model(drl, "tf32" if tc else "fp32", norm)
    _check_against_rollout(drl, model, n, n_eval, deterministic)
    model.close()


@pytest.mark.parametrize("n,n_eval", [(1, 7), (64, 10), (64, 64), (64, 100)])
def test_eval_targets_and_chunks(drl, monkeypatch, n, n_eval):
    from drone_rl_b200 import evaluation
    monkeypatch.setattr(evaluation, "PROBE_CHUNK", 50)        # several probe launches per evaluation
    model = _model(drl)
    _, lengths, T = _check_against_rollout(drl, model, n, n_eval, True)
    assert T > 50 or n > 1
    model.close()


def test_eval_leaves_the_model_untouched(drl):
    from drone_rl_b200.evaluation import evaluate_policy
    from drone_rl_b200.ppo import PPO
    model = PPO(drl.DroneBatch(64, drl.EnvConfig.single(), seed=2), n_steps=32, batch_size=512, n_epochs=1, seed=2,
                norm_obs=True, norm_reward=True)
    model.learn(64 * 32 * 2)
    torch.cuda.synchronize()
    before = model.state_dict()
    nz = (model.normalizer.stats.clone(), model.normalizer.returns.clone(), model.normalizer.affine.clone())
    ev = drl.DroneBatch(32, drl.EnvConfig.single(), seed=3)
    evaluate_policy(model, ev, 20)
    evaluate_policy(model, ev, 20, deterministic=False)
    after = model.state_dict()
    for k in ("params", "adam", "adam_step", "env_global_step", "num_timesteps", "n_updates"):
        assert (torch.equal(before[k], after[k]) if torch.is_tensor(before[k]) else before[k] == after[k]), k
    for k in before["env_state"]:
        assert np.array_equal(before["env_state"][k], after["env_state"][k]), k
    assert all(torch.equal(x, y) for x, y in zip(nz, (model.normalizer.stats, model.normalizer.returns,
                                                      model.normalizer.affine)))
    model.close(); ev.close()


def test_eval_callback_in_learn(drl, tmp_path):
    from drone_rl_b200.evaluation import EvalCallback
    from drone_rl_b200.ppo import PPO
    n, K = 64, 32
    model = PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=4), n_steps=K, batch_size=1024, n_epochs=2, seed=4)
    ev = drl.DroneBatch(4, drl.EnvConfig.single(), seed=5)
    cb = EvalCallback(ev, n_eval_episodes=6, eval_freq=2 * K, log_path=str(tmp_path), best_model_save_path=str(tmp_path),
                      verbose=0)
    snaps = []

    def both(m):
        cb(m)
        if "eval/mean_reward" in m.logger_values:
            snaps.append((m.logger_values.pop("eval/mean_reward"), m.params.clone()))
        return True
    model.learn(n * K * 6, callback=both)
    z = np.load(os.path.join(str(tmp_path), "evaluations.npz"))
    assert z["results"].shape == (3, 6) and z["ep_lengths"].shape == (3, 6) and z["timesteps"].tolist() == [n * K * 2, n * K * 4, n * K * 6]
    assert [s[0] for s in snaps] == pytest.approx(z["results"].mean(axis=1).tolist())
    best = int(np.argmax([s[0] for s in snaps]))
    assert cb.best_mean_reward == snaps[best][0] and cb.last_mean_reward == snaps[-1][0]
    m2 = PPO.load(os.path.join(str(tmp_path), "best_model.zip"), 1)
    assert torch.equal(m2.params, snaps[best][1])
    m2.close(); model.close(); ev.close()


def test_train_driver_logs_eval_keys(drl, tmp_path, monkeypatch):
    import csv
    from drone_rl_b200 import train
    monkeypatch.chdir(tmp_path)
    train.main(["--total-timesteps", "8192", "--n-envs", "64", "--n-steps", "32", "--batch-size", "1024", "--n-epochs", "1",
                "--eval-freq", "64", "--n-eval-episodes", "3", "--n-eval-envs", "2", "--quiet", "--save", "dd"])
    run = os.path.join("tensorboard", "drone_runs_1")
    with open(os.path.join(run, "progress.csv"), newline="") as f:
        rows = list(csv.DictReader(f))
    assert len(rows) == 4
    assert [r["eval/mean_reward"] != "" for r in rows] == [False, True, False, True]
    assert all(r["eval/mean_ep_length"] != "" for r in rows[1::2])
    assert np.load(os.path.join(run, "evaluations.npz"))["results"].shape == (2, 3)
    assert os.path.isfile(os.path.join(run, "best_model.zip"))


def test_value_errors(drl):
    from drone_rl_b200.evaluation import evaluate_policy
    model = _model(drl)
    ev = drl.DroneBatch(4, drl.EnvConfig.single(), seed=1)
    for kw in ({"render": True}, {"callback": lambda *a: None}, {"n_eval_episodes": 0}):
        with pytest.raises(ValueError):
            evaluate_policy(model, ev, **{"n_eval_episodes": 4, **kw})
    for cfg in (drl.EnvConfig.vector(), drl.EnvConfig.single(auto_reset=False)):
        b = drl.DroneBatch(4, cfg)
        with pytest.raises(ValueError):
            evaluate_policy(model, b, 4)
        b.close()
    with pytest.raises(AssertionError):
        evaluate_policy(model, ev, 4, reward_threshold=1e9)
    model.close(); ev.close()


# ---------------------------------------------------------------------------------------------------------------------
# data parallel: two ranks evaluate their shards
# ---------------------------------------------------------------------------------------------------------------------
N_DP, EPS_DP = 96, 150


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    import drone_rl_b200 as drl
    from drone_rl_b200.evaluation import evaluate_policy
    model = _model(drl, device=rank)             # built before the process group: a plain single-GPU model on each rank
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ev = drl.DroneBatch(N_DP, drl.EnvConfig.single(), device=rank, seed=SEED, env_offset=rank * N_DP)
    r, l = evaluate_policy(model, ev, EPS_DP, return_episode_rewards=True)
    if rank == 0:
        q.put((r, l, ev.global_step))
    model.close(); ev.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_equal_one_rank_on_the_union(drl):
    import torch.multiprocessing as mp
    from drone_rl_b200.evaluation import evaluate_policy
    ctx = mp.get_context("spawn")
    q, port = ctx.Queue(), _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    r2, l2, t2 = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    model = _model(drl)
    one = drl.DroneBatch(2 * N_DP, drl.EnvConfig.single(), seed=SEED)
    r1, l1 = evaluate_policy(model, one, EPS_DP, return_episode_rewards=True)
    assert r1 == r2 and l1 == l2 and one.global_step == t2
    model.close(); one.close()
