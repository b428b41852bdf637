"""tcgen05 / TMEM path of the policy MLP (tc_mlp.cuh) against the float64 oracle and the fp32 CUDA-core
path.  Stated tolerance: tf32 products (10-bit mantissa, inputs rounded to nearest) with fp32
accumulation and tanh.approx.f32 (max rel error 2^-11):
    layer-1 pre-activations  |err| <= 2^-10 * sum_k |w_k x_k|   (each product carries two 2^-11 roundings)
    layer-2 pre-activations  |err| <= 1.5e-2 * max(1, |ref|)      (adds the layer-1 error through tanh)
    mean / value             per element within the bound of oracle/tc_bound.py
PARITY UNPINNED for the same reason as tests/test_gpu_ppo.py (SB3 is not in the reference tree)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import ppo_oracle as po  # noqa: E402
from oracle.tc_bound import tc_forward_bound  # noqa: E402


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


def _params(seed):
    g = torch.Generator().manual_seed(seed)
    return po.init_params(seed, dtype=torch.float64) + 0.1 * torch.randn(po.N_PARAMS, generator=g, dtype=torch.float64)


def _pre_activations(theta, obs):
    p = po.unpack(theta)
    z1 = torch.cat([obs @ p["pi.W1"].t() + p["pi.b1"], obs @ p["vf.W1"].t() + p["vf.b1"]], 1)
    h1 = torch.tanh(z1)
    z2 = torch.cat([h1[:, :64] @ p["pi.W2"].t() + p["pi.b2"], h1[:, 64:] @ p["vf.W2"].t() + p["vf.b2"]], 1)
    return z1, z2


@pytest.mark.parametrize("B", [128, 1000, 128 * 300 + 5])
def test_tc_forward_matches_oracle(drl, B):
    from drone_rl_b200.ppo import PPO
    model = PPO(8, n_steps=4)
    theta = _params(3)
    model.params.copy_(theta.float().cuda())
    g = torch.Generator().manual_seed(B)
    obs = (torch.randn(B, 15, generator=g) * torch.tensor([1.0] * 3 + [2.0] * 3 + [1.0] * 3 + [4.0] * 3 + [1.0] * 3)).float()
    mean, value, d1, d2 = model.policy_forward(obs.cuda(), precision="tf32", debug=True)
    torch.cuda.synchronize()
    th = theta.float().double()
    z1, z2 = _pre_activations(th, obs.double())
    rm, rv, _ = po.forward(th, obs.double())

    def check(got, ref, rel, what):
        got, ref = got.cpu().double().numpy(), ref.numpy()
        err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
        assert err.max() <= rel, f"{what}: max scaled err {err.max():.3g} at {np.unravel_index(err.argmax(), err.shape)}"
        return err.max()
    p = po.unpack(th)
    scale1 = torch.cat([obs.double().abs() @ p["pi.W1"].abs().t() + p["pi.b1"].abs(),
                        obs.double().abs() @ p["vf.W1"].abs().t() + p["vf.b1"].abs()], 1).numpy()
    err1 = np.abs(d1.cpu().double().numpy() - z1.numpy())
    assert (err1 <= 2.0 ** -10 * scale1 + 1e-6).all(), f"layer-1: worst err/bound {(err1 / (2.0 ** -10 * scale1 + 1e-6)).max():.3g}"
    e1 = (err1 / np.maximum(1.0, np.abs(z1.numpy()))).max()
    e2 = check(d2, z2, 1.5e-2, "layer-2 pre-activation")
    # mean and value: per element within the derived bound of oracle/tc_bound.py
    rm_b, rv_b, mb, vb = tc_forward_bound(theta.float().numpy(), obs.numpy())
    assert np.allclose(rm_b, rm.numpy(), rtol=1e-12, atol=1e-14) and np.allclose(rv_b, rv.numpy(), rtol=1e-12, atol=1e-14)
    em = (np.abs(mean.cpu().double().numpy() - rm_b) / mb).max()
    ev = (np.abs(value.cpu().double().numpy() - rv_b) / vb).max()
    assert em <= 1.0 and ev <= 1.0, f"worst err/bound: mean {em:.3g}, value {ev:.3g}"
    # and against the fp32 CUDA-core kernel of the same library
    m32, v32 = model.policy_forward(obs.cuda())
    assert (mean - m32).abs().max().item() < 2e-2 and (value - v32).abs().max().item() < 4e-2
    print(f"B={B}: scaled errors L1 {e1:.2e} L2 {e2:.2e}; err/bound mean {em:.2e} value {ev:.2e}")
    model.close()


# ------------------------------------------------------------------------------------------------------
# tensor-core minibatch gradient (csrc/ppo_update_tc.cuh)
# ------------------------------------------------------------------------------------------------------
def _grad(model, index, m, first=0, tc=True):
    import ctypes as C
    from drone_rl_b200 import _lib
    b = model.buf
    P = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    model._adv_stats.zero_()
    _lib.check(model.lib.dronecu_ppo_adv_stats(model._h, P(b.adv), P(index), first, m, P(model._adv_stats), None))
    fn = {True: model.lib.dronecu_ppo_grad_tc, False: model.lib.dronecu_ppo_grad, "tf32": model.lib.dronecu_ppo_grad_tc,
          "bf16": model.lib.dronecu_ppo_grad_bf16}[tc]
    _lib.check(fn(model._h, P(model.params), P(b.obs), P(b.actions), P(b.logp), P(b.adv), P(b.ret), P(index), first, m,
                  0.0, 1.0, P(model._adv_stats), P(model._grad), None))
    torch.cuda.synchronize()
    return model._grad.cpu().double().numpy().copy()


def _separated_buffers(model, seed, clip=None):
    """Like tests/test_gpu_ppo._fake_buffers, but the old log-probs sit at offsets {-0.45, -0.08, 0, 0.07,
    0.4} (+- 0.01) from the current policy's: ratios of 1.57 / 1.08 / 1 / 0.93 / 0.67 exercise both sides
    of the clip, and no sample lies within the tf32 forward error of the 0.8 / 1.2 boundaries -- the clipped
    objective's gradient is discontinuous there, so a borderline sample would make ANY reduced-precision
    forward differ from float64 by that sample's whole gradient (measured with the unseparated buffers:
    1-2 % of the samples flip, 5 % error on the policy blocks, value blocks unaffected).
    ``clip``: place the offsets around the boundaries log(1 -+ clip) of that clip range instead: 0.2 outside
    each boundary, 0.45 of the way from 0 to each boundary, and 0."""
    b = model.buf
    K, n = b.obs.shape[0], b.obs.shape[1]
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(K, n, 15, generator=g) * 2.0
    theta = model.params.cpu().double()
    mean, value, log_std = po.forward(theta, obs.double().reshape(-1, 15))
    act = mean + torch.exp(log_std) * torch.randn(K * n, 4, generator=g, dtype=torch.float64)
    table = [-0.45, -0.08, 0.0, 0.07, 0.4]
    if clip is not None:
        lo, hi = np.log1p(-clip), np.log1p(clip)
        table = [lo - 0.2, 0.45 * lo, 0.0, 0.45 * hi, hi + 0.2]
    offs = torch.tensor(table, dtype=torch.float64)[torch.randint(0, 5, (K * n,), generator=g)]
    old_logp = po.log_prob(mean, log_std, act) + offs + 0.01 * torch.randn(K * n, generator=g, dtype=torch.float64)
    adv = torch.randn(K * n, generator=g, dtype=torch.float64) * 3 + 0.5
    # a biased value function: with ret - value pure noise the reference gradient is a sqrt(m)-sized noise sum
    # while the tf32 forward error of the value adds coherently (~ m * 1e-3): the relative error would grow
    # like sqrt(m) without saying anything about the kernel
    ret = value + 0.7 + torch.randn(K * n, generator=g, dtype=torch.float64)
    b.obs.copy_(obs.cuda()); b.actions.copy_(act.float().reshape(K, n, 4).cuda())
    b.logp.copy_(old_logp.float().reshape(K, n).cuda()); b.adv.copy_(adv.float().reshape(K, n).cuda())
    b.ret.copy_(ret.float().reshape(K, n).cuda())
    torch.cuda.synchronize()
    f64 = lambda t: t.cpu().double()
    return (f64(b.obs).reshape(-1, 15), f64(b.actions).reshape(-1, 4), f64(b.logp).reshape(-1),
            f64(b.adv).reshape(-1), f64(b.ret).reshape(-1))


@pytest.mark.parametrize("mode", ["tf32", "bf16"])
@pytest.mark.parametrize("m", [3, 64, 128, 1000, 128 * 300 + 37, 128 * 2 * 148 * 3])
def test_tc_minibatch_gradient(drl, m, mode):
    """tensor-core gradient (all-tf32 kernel; kernel with bf16 weight-gradient operands) vs float64 autograd of the oracle loss (and vs the fp32 CUDA-core kernel).
    Stated tolerance: every parameter block within 1e-2 of its own largest entry (tf32 operands carry
    2^-11 relative rounding, MUFU tanh 2^-11; the sum over m samples averages part of it out), whole
    vector within 5e-3 of the largest entry; statistics as for the fp32 kernel but rtol 5e-3."""
    from tests.test_gpu_ppo import _rand_params
    from drone_rl_b200.ppo import PPO
    n, K = 1024, (m + 1023) // 1024 + 1
    model = PPO(n, n_steps=K, ent_coef=0.01)
    model.params.copy_(_rand_params(9, 0.5).float().cuda())
    obs, act, old_logp, adv, ret = _separated_buffers(model, 4)
    B = obs.shape[0]
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(1))[:m]
    g = _grad(model, idx.to(torch.int32).cuda(), m, tc=mode)
    g32 = _grad(model, idx.to(torch.int32).cuda(), m, tc=False)
    theta = model.params.cpu().double().requires_grad_(True)
    loss, stats = po.ppo_loss(theta, obs[idx], act[idx], old_logp[idx], adv[idx], ret[idx], ent_coef=0.01)
    (ref,) = torch.autograd.grad(loss, theta)
    ref = ref.numpy() * m
    scale = np.abs(ref).max()
    report, bad = [], []
    for name, (off, shape) in po.offsets().items():
        k = int(np.prod(shape))
        blk_ref, blk = ref[off:off + k], g[off:off + k]
        e = np.abs(blk - blk_ref).max() / max(np.abs(blk_ref).max(), 1e-3 * scale)
        e32 = np.abs(blk - g32[off:off + k]).max() / max(np.abs(blk_ref).max(), 1e-3 * scale)
        report.append(f"{name} {e:.2e} (vs fp32 kernel {e32:.2e})")
        if not e <= 1e-2:
            bad.append(name)
    print(f"{mode} m={m}: " + "; ".join(report))
    assert not bad, f"blocks out of tolerance: {bad}: " + "; ".join(report)
    assert np.abs(g[:po.N_PARAMS] - ref).max() <= 5e-3 * scale
    st = g[po.N_PARAMS:]
    assert st[4] == m
    np.testing.assert_allclose(st[0] / m, stats["policy_gradient_loss"], rtol=5e-3, atol=1e-4)
    np.testing.assert_allclose(st[1] / m, stats["value_loss"], rtol=5e-3)
    np.testing.assert_allclose(st[3] / m, stats["clip_fraction"], atol=2.0 / m)
    assert m < 128 or 0.2 < stats["clip_fraction"] < 0.6
    again = _grad(model, idx.to(torch.int32).cuda(), m, tc=mode)
    assert np.array_equal(g, again)                       # fixed tile order + fixed-order reduction
    model.close()


def test_tc_update_trains_like_fp32(drl):
    """A few PPO iterations with the tf32 update track the fp32 update (same seeds, same rollouts at
    iteration 0): parameters stay within 2e-3 after the first 8 optimiser steps."""
    from drone_rl_b200.ppo import PPO
    ps = []
    for prec in ("fp32", "tf32"):
        m = PPO(drl.DroneBatch(2048, drl.EnvConfig.single(), seed=3), n_steps=16, batch_size=8192, n_epochs=2, seed=3,
                update_precision=prec)
        m.collect_rollouts()
        m.train()
        torch.cuda.synchronize()
        assert torch.isfinite(m.params).all()
        ps.append(m.params.clone())
        m.close()
    assert (ps[0] - ps[1]).abs().max().item() < 2e-3


@pytest.mark.parametrize("mode", ["tf32", "bf16"])
def test_tc_gradient_is_race_free_under_repetition(drl, mode):
    """40 back-to-back launches of the tensor-core gradient over the same ragged minibatch (several tiles per
    warpgroup, a partial last tile, an idle warpgroup tail) must be bit-identical: the kernel's hand-overs
    (mbarriers, tcgen05 fences, async-proxy fences) leave no window for a stale operand."""
    from tests.test_gpu_ppo import _rand_params
    from drone_rl_b200.ppo import PPO
    m = 128 * 2 * 74 * 3 + 128 * 5 + 77
    n, K = 2048, (m + 2047) // 2048 + 1
    model = PPO(n, n_steps=K, ent_coef=0.01)
    model.params.copy_(_rand_params(11, 0.5).float().cuda())
    _separated_buffers(model, 6)
    idx = torch.randperm(n * K, generator=torch.Generator().manual_seed(2))[:m].to(torch.int32).cuda()
    first = _grad(model, idx, m, tc=mode)
    assert np.isfinite(first).all() and np.abs(first).max() > 0
    for _ in range(40):
        assert np.array_equal(_grad(model, idx, m, tc=mode), first)
    model.close()


def test_tc_gradient_is_race_free_at_the_c5_scale(drl):
    """1500 launches of the bf16 gradient kernel on ONE 8.4M-sample minibatch of a 1M-env x 32-step buffer (configs[4]) must be
    bit-identical.  At this size DRAM latency jitters the warps far more than in the small repetition test above: an aliasing
    race between the staged X tile and another warp's tanh' stash (r02) showed up here once per ~1500 launches and never at
    the small sizes (scratch/stress_determinism.py found it)."""
    import ctypes as C
    from drone_rl_b200 import _lib
    from drone_rl_b200.ppo import PPO
    n, K, mb = 1 << 20, 32, 4
    model = PPO(n, n_steps=K, batch_size=n * K // mb, rollout_precision="tf32", update_precision="bf16")
    model.collect_rollouts()
    P = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    b, B, m = model.buf, n * K, n * K // mb
    perm = torch.empty(B, dtype=torch.int32, device="cuda")
    _lib.check(model.lib.dronecu_minibatch_partition(model._h, B, m, 1, 0, P(perm), None))
    stats = torch.zeros(mb, 3, dtype=torch.float64, device="cuda")
    _lib.check(model.lib.dronecu_ppo_adv_stats_epoch(model._h, P(b.adv), P(perm), B, m, P(stats), None))
    g, ref, bad = torch.zeros(_lib.GRAD_LEN, device="cuda"), None, 0
    for i in range(1500):
        model.launch_grad(perm[:m], 0, m, P(stats[0]), g)
        if ref is None:
            ref = g.clone()
            assert bool(torch.isfinite(ref).all())
        else:
            bad += int(not torch.equal(g, ref))
    assert bad == 0, f"{bad} of 1500 launches differ"
    model.close()


def test_padded_and_packed_observation_rows_give_identical_results(drl):
    """The rollout buffer with 64-byte observation rows (the bf16 update's default) and with packed 60-byte rows hold the same
    observations, and the gradient kernel forms bit-identical gradients from either (same values staged, same MMAs)."""
    import ctypes as C
    from drone_rl_b200 import _lib
    from drone_rl_b200.ppo import PPO
    n, K = 3000, 9                                     # ragged: not a multiple of 128 / 32
    models = [PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=8), n_steps=K, batch_size=n * K // 3, n_epochs=2, seed=8,
                  rollout_precision="tf32", update_precision="bf16", padded_obs=flag) for flag in (True, False)]
    assert models[0].buf.obs_store.shape[-1] == 16 and models[1].buf.obs_store.shape[-1] == 15
    grads = []
    for mdl in models:
        mdl.collect_rollouts()
        g = torch.zeros(_lib.GRAD_LEN, device="cuda")
        idx = torch.randperm(n * K, generator=torch.Generator().manual_seed(2))[: n * K // 2].sort().values.to(torch.int32).cuda()
        mdl.launch_grad(idx, 0, idx.numel(), None, g)
        grads.append(g.clone())
        for prec in ("tf32", "fp32"):                  # the other two kernels honour the row stride as well
            g2 = torch.zeros_like(g)
            mdl.launch_grad(idx, 0, idx.numel(), None, g2, precision=prec)
            grads.append(g2.clone())
    torch.cuda.synchronize()
    assert torch.equal(models[0].buf.obs, models[1].buf.obs)
    assert (models[0].buf.obs_store[..., 15] == 1.0).all()
    for a, b in zip(grads[:3], grads[3:]):
        assert torch.equal(a, b)
    for mdl in models:
        mdl.train()
    assert torch.equal(models[0].params, models[1].params)
    for mdl in models:
        mdl.close()
