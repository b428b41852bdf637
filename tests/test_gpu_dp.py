"""GPU tests of the data-parallel PPO update over peer memory (csrc/ppo_dp.cuh; north_star configs[4]).

* one GPU: the time-out path and the rejected arguments of the C ABI; ``_handles`` wires optimiser handles of one process
  as ranks (mailboxes joined with raw pointers).  The exchange kernels at every world size, inside CUDA graphs and under
  PPO.train() are pinned against float64 in tests/test_gpu_dp_parity.py;
* two GPUs (skipped on a one-GPU box; run with ``gpurun --gpus 2``): two processes under NCCL-initialised
  torch.distributed run ``PPO.collect_rollouts`` + ``PPO.train`` on their shards.  Asserted: parameters bit-identical
  across the ranks, equal to the "nccl" backend to float rounding, and equal (<= 1e-6) to ONE rank training on the union
  of the shards.
"""
import ctypes as C
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


def _handles(lib, n, device=0, timeout=5.0):
    from drone_rl_b200 import _lib
    cfg = _lib.PPOConfig()
    lib.dronecu_ppo_config_default(C.byref(cfg))
    hs, mails = [], []
    for r in range(n):
        h, mail = C.c_void_p(), C.c_void_p()
        _lib.check(lib.dronecu_ppo_create(C.byref(cfg), device, C.byref(h)))
        _lib.check(lib.dronecu_ppo_dp_alloc(h, r, n, None, C.byref(mail)))
        hs.append(h); mails.append(mail.value)
    arr = (C.c_void_p * n)(*mails)
    for h in hs:
        _lib.check(lib.dronecu_ppo_dp_connect(h, n, None, arr))
        _lib.check(lib.dronecu_ppo_dp_set_timeout(h, timeout))
    return hs


def test_peer_exchange_times_out_instead_of_hanging(drl):
    from drone_rl_b200 import _lib
    from drone_rl_b200.core import _ptr
    lib, dev = _lib.load(), torch.device("cuda", 0)
    hs = _handles(lib, 2, timeout=0.2)
    p, g = torch.zeros(_lib.POLICY_PARAMS, device=dev), torch.ones(_lib.GRAD_LEN, device=dev)
    _lib.check(lib.dronecu_ppo_apply_dp(hs[0], _ptr(p), _ptr(g), None, None))       # rank 1 never shows up
    torch.cuda.synchronize()
    st = C.c_int()
    _lib.check(lib.dronecu_ppo_dp_status(hs[0], C.byref(st), None))
    assert st.value == 1
    for h in hs:
        lib.dronecu_ppo_destroy(h)


def test_dp_entry_points_reject_bad_arguments(drl):
    from drone_rl_b200 import _lib
    lib = _lib.load()
    cfg = _lib.PPOConfig()
    lib.dronecu_ppo_config_default(C.byref(cfg))
    h = C.c_void_p()
    _lib.check(lib.dronecu_ppo_create(C.byref(cfg), 0, C.byref(h)))
    g = torch.zeros(_lib.GRAD_LEN, device="cuda")
    assert lib.dronecu_ppo_apply_dp(h, C.c_void_p(g.data_ptr()), C.c_void_p(g.data_ptr()), None, None) != 0   # not connected
    assert lib.dronecu_ppo_dp_alloc(h, 3, 2, None, None) != 0 and lib.dronecu_ppo_dp_alloc(h, 0, 17, None, None) != 0
    assert lib.dronecu_ppo_dp_connect(h, 2, None, None) != 0
    lib.dronecu_ppo_destroy(h)


# ------------------------------------------------------------------------------------------------------------------
# two GPUs, two processes
# ------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


N_ENVS, N_STEPS, EPOCHS = 4096, 16, 3


def _dp_worker(rank, world, port, backend, precision, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import drone_rl_b200 as drl
    from drone_rl_b200.ppo import PPO
    env = drl.DroneBatch(N_ENVS, drl.EnvConfig.single(), device=rank, seed=3, env_offset=rank * N_ENVS)
    # ONE minibatch per epoch = the rank's whole shard, so that the union over the ranks is the whole buffer whatever the
    # permutation: the N-rank update must equal the 1-rank update over the union
    model = PPO(env, n_steps=N_STEPS, batch_size=N_ENVS * N_STEPS, n_epochs=EPOCHS, seed=3, dp_backend=backend,
                rollout_precision="fp32", update_precision=precision)
    model.collect_rollouts()
    model.train()
    first, logs = model.params.cpu(), dict(model.logger_values)
    model.collect_rollouts()                 # second iteration: the captured epoch graph is replayed
    model.train()
    torch.cuda.synchronize()
    out = {"params_it1": first, "params": model.params.cpu(), "logs": logs, "graph": model._graph is not None}
    mine = model.params.clone()
    every = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(every, mine)
    out["identical"] = all(torch.equal(e, every[0]) for e in every)
    model.close()
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def _run_dp(backend, precision="fp32", world=2):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q, port = ctx.Queue(), _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, backend, precision, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return out


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs (gpurun --gpus 2)")
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_two_rank_training_equals_one_rank_on_the_union(drl, precision):
    from drone_rl_b200.ppo import PPO
    peer = _run_dp("peer", precision)
    assert peer["identical"], "parameter replicas drifted apart"
    assert peer["graph"], "the peer backend must keep the epoch in a CUDA graph"
    nccl = _run_dp("nccl", precision)
    assert nccl["identical"]
    # same per-rank gradients, same fixed order of the two-term sum: only the count scaling (1/(2m) vs 1/count) could differ
    assert torch.allclose(peer["params"], nccl["params"], rtol=0, atol=1e-7)
    # one rank, the union of the shards (env ids 0 .. 2n-1)
    env = drl.DroneBatch(2 * N_ENVS, drl.EnvConfig.single(), device=0, seed=3)
    model = PPO(env, n_steps=N_STEPS, batch_size=2 * N_ENVS * N_STEPS, n_epochs=EPOCHS, seed=3, rollout_precision="fp32",
                update_precision=precision)
    model.collect_rollouts()
    model.train()
    one = model.params.cpu()
    # fp32 path: the same per-sample terms, summed in a different grouping (float32 partials) -> <= 1e-6 after 3 Adam steps
    # of size ~3e-4; bf16 weight-gradient operands: the tile grouping changes the bf16-rounded products' accumulation order only
    tol = 1e-6 if precision == "fp32" else 5e-6
    err = float((peer["params_it1"] - one).abs().max())
    assert err <= tol, f"2-rank vs union: {err:.3g}"
    for k in ("train/value_loss", "train/policy_gradient_loss", "train/approx_kl", "train/explained_variance"):
        assert abs(peer["logs"][k] - model.logger_values[k]) <= 1e-4 * max(1.0, abs(model.logger_values[k])), k
    model.close()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 4, reason="needs at least four GPUs (gpurun --gpus 4 / 8)")
def test_all_ranks_hold_identical_replicas(drl):
    """Every GPU of the box as one rank: after two PPO iterations (the second replays the captured epoch graphs) the
    parameter replicas are bit-identical -- the fixed-rank-order sum of the peer exchange at world = 4 / 8."""
    world = 8 if torch.cuda.device_count() >= 8 else 4
    out = _run_dp("peer", "bf16", world=world)
    assert out["identical"] and out["graph"]
    assert torch.isfinite(out["params"]).all()


def _ckpt_worker(rank, world, port, path, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import drone_rl_b200 as drl
    from drone_rl_b200.ppo import PPO
    n = 512
    mk = lambda: drl.DroneBatch(n, drl.EnvConfig.single(), device=rank, seed=9, env_offset=rank * n)
    a = PPO(mk(), n_steps=16, batch_size=n * 16 // 2, n_epochs=1, seed=9)
    a.learn(3 * n * 16 * world)
    a.save(path)                                    # rank 0: the archive; rank 1: its env shard next to it
    dist.barrier()
    b = PPO.load(path, mk(), n_steps=16, batch_size=n * 16 // 2, n_epochs=1)
    sa, sb = a.batch.get_state(), b.batch.get_state()
    out = {"restored": bool(b.env_state_restored),
           "env_equal": all(np.array_equal(sa[k], sb[k], equal_nan=True) for k in sa),
           "params_equal": bool(torch.equal(a.params, b.params)),
           "first_pos": sa["pos"][0].tolist(), "step": (a.batch.global_step, b.batch.global_step)}
    gathered = [None] * world
    dist.all_gather_object(gathered, out)
    a.close(); b.close()
    if rank == 0:
        q.put(gathered)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs (gpurun --gpus 2)")
def test_data_parallel_checkpoint_restores_every_ranks_own_shard(drl, tmp_path):
    """ADVICE r1: rank 0's archive holds rank 0's env shard only -- on resume every rank must get ITS OWN env / curriculum / RNG
    state back (side files next to the archive), not a copy of shard 0; policy and Adam state are the replicas."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q, port, path = ctx.Queue(), _free_port(), str(tmp_path / "dp_ckpt")
    procs = [ctx.Process(target=_ckpt_worker, args=(r, 2, port, path, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert os.path.isfile(path + ".zip") and os.path.isfile(path + ".env.rank1.pt")
    for r, o in enumerate(res):
        assert o["restored"] and o["env_equal"] and o["params_equal"], (r, o)
        assert o["step"][0] == o["step"][1]
    assert res[0]["first_pos"] != res[1]["first_pos"]          # the two shards really differ
