"""The PPO update step against float64 torch, at every minibatch shape it runs.

  a. the three minibatch-gradient kernels (``dronecu_ppo_grad_strided``: fp32 CUDA cores, tf32 and bf16 tensor cores) over
     a covering design of minibatch size (on both sides of every launch-shape boundary), observation row stride, row
     addressing, advantage handling and loss coefficients, and once at the production size (8,388,608 samples);
  b. clip_grad_norm_ + Adam (``dronecu_ppo_apply``) against ``torch.nn.utils.clip_grad_norm_`` + ``torch.optim.Adam``;
  c. ``PPO.train()`` teacher-forced per optimiser step: minibatch rows, advantage statistics, gradient and step;
  d. GAE (``dronecu_gae``) against ``oracle.ppo_oracle.gae``, bounded by the recursion's forward error.

The reference is float64 autograd of oracle/ppo_oracle.py on the float32 values the kernels read, with the float32 values of
the hyper-parameters the kernels receive.  Tolerances are those of tests/test_gpu_ppo.py and tests/test_gpu_tc.py:
    fp32 gradient          whole vector <= 2e-4 x max|ref|, every parameter block <= 5e-4 x its own max
    tf32 / bf16 gradient   whole vector <= 5e-3 x max|ref|, every parameter block <= 1e-2 x its own max
    parameters of a step   <= 2^-22 |ref| + 1e-9 (the float32 result is the float64 step rounded once)
"""
import ctypes as C
import math
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import philox, ppo_oracle as po  # noqa: E402
from tests.test_gpu_ppo import _rand_params  # noqa: E402
from tests.test_gpu_tc import _separated_buffers  # noqa: E402

N = po.N_PARAMS
MODES = {"fp32": 0, "tf32": 1, "bf16": 2}
TOL = {"fp32": (2e-4, 5e-4), "tf32": (5e-3, 1e-2), "bf16": (5e-3, 1e-2)}     # (whole vector, block)
STEP_REL, STEP_ABS = 2.0 ** -22, 1e-9


def P(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def f32(x):
    return float(np.float32(x))


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


@pytest.fixture(scope="module")
def lib(drl):
    from drone_rl_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def handles(lib):
    """dronecu_ppo handles keyed by their configuration (clip_range, vf_coef, ent_coef, learning_rate, max_grad_norm)."""
    from drone_rl_b200 import _lib
    made = {}

    def get(clip=0.2, vf=0.5, ent=0.0, lr=3e-4, max_norm=0.5):
        key = (clip, vf, ent, lr, max_norm)
        if key not in made:
            cfg = _lib.PPOConfig()
            lib.dronecu_ppo_config_default(C.byref(cfg))
            cfg.clip_range, cfg.vf_coef, cfg.ent_coef, cfg.learning_rate, cfg.max_grad_norm = clip, vf, ent, lr, max_norm
            h = C.c_void_p()
            _lib.check(lib.dronecu_ppo_create(C.byref(cfg), 0, C.byref(h)))
            made[key] = (h, cfg)
        return made[key]
    yield get
    torch.cuda.synchronize()
    for h, _ in made.values():
        lib.dronecu_ppo_destroy(h)


# ------------------------------------------------------------------------------------------------------------------------
# reference gradient
# ------------------------------------------------------------------------------------------------------------------------
def _normalised(adv, rows, how):
    """The advantages the kernel uses, in float64.  Statistics: SB3's (adv - mean) / (std + 1e-8) with the unbiased std,
    skipped for one sample.  The kernels subtract the float32-rounded mean, as SB3's float32 ``advantages.mean()`` does:
    with a mean of 1e3 and a std of 1e-2 that rounding alone (up to 3e-5, 3e-3 std) is larger than the fp32 tolerance."""
    a = adv[rows]
    if how == "stats":
        if a.numel() == 1:
            return a
        return (a - f32(float(a.mean()))) / (float(a.std()) + 1e-8)
    if how == "explicit":
        return (a - f32(0.3)) * f32(0.5)
    return a


def _ref_grad(theta, data, rows, adv_n, clip, vf, ent, chunk=1 << 20):
    """Sum-form float64 gradient [N] and statistic sums over ``rows`` of ``data`` (obs, act, old_logp, _, ret: float64, on
    the device), summed over chunks of ``chunk`` rows."""
    obs, act, old_logp, _, ret = data
    g = torch.zeros(N, dtype=torch.float64, device=obs.device)
    sums = dict.fromkeys(("policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction"), 0.0)
    for s in range(0, rows.numel(), chunk):
        r, a = rows[s:s + chunk], adv_n[s:s + chunk]
        p = theta.clone().requires_grad_(True)
        loss, st = po.ppo_loss(p, obs[r], act[r], old_logp[r], a, ret[r], clip=clip, vf_coef=vf, ent_coef=ent, normalize=False)
        (gc,) = torch.autograd.grad(loss, p)
        g += gc * r.numel()
        for k in sums:
            sums[k] += st[k] * r.numel()
    return g.cpu().numpy(), sums


def _grad_error(got, ref, mode):
    """Worst error over tolerance of the gradient (1.0 = at the tolerance) and a per-block report."""
    whole, blk = TOL[mode]
    scale = np.abs(ref).max()
    worst = np.abs(got[:N] - ref).max() / (whole * scale)
    report = []
    for name, (off, shape) in po.offsets().items():
        k = int(np.prod(shape))
        r = ref[off:off + k]
        e = np.abs(got[off:off + k] - r).max() / max(np.abs(r).max(), 1e-3 * scale)
        worst = max(worst, e / blk)
        report.append(f"{name} {e:.2e}")
    return worst, "; ".join(report)


def _check_stats(st, sums, m, mode):
    assert st[4] == m                                                     # the count column is exact
    if mode == "fp32":
        np.testing.assert_allclose(st[0] / m, sums["policy_gradient_loss"] / m, rtol=2e-4, atol=1e-5)
        np.testing.assert_allclose(st[1] / m, sums["value_loss"] / m, rtol=2e-4)
        np.testing.assert_allclose(st[2] / m, sums["approx_kl"] / m, rtol=2e-3, atol=1e-6)
    else:
        np.testing.assert_allclose(st[0] / m, sums["policy_gradient_loss"] / m, rtol=5e-3, atol=1e-4)
        np.testing.assert_allclose(st[1] / m, sums["value_loss"] / m, rtol=5e-3)
    np.testing.assert_allclose(st[3] / m, sums["clip_fraction"] / m, atol=2.0 / m)


def _launch(lib, h, mode, stride, params, store, buf, adv, index, first, m, mean, inv_std, stats, grad):
    from drone_rl_b200 import _lib
    _lib.check(lib.dronecu_ppo_grad_strided(h, MODES[mode], stride, P(params), P(store), P(buf.actions), P(buf.logp), P(adv),
                                            P(buf.ret), P(index), first, m, mean, inv_std, P(stats), P(grad), None),
               "dronecu_ppo_grad_strided")
    torch.cuda.synchronize()
    return grad.cpu().double().numpy()


# ------------------------------------------------------------------------------------------------------------------------
# a. gradient kernels over a covering design
# ------------------------------------------------------------------------------------------------------------------------
# 128 samples per tile; the bf16 kernel writes the gradient itself up to 3 tiles (m <= 384); 148 SMs: the tf32 kernel fills
# every CTA at 2 x 74 tiles (18944), the bf16 kernel at 3 x 74 (28416)
SIZES = [1, 2, 127, 128, 129, 383, 384, 385, 18943, 18944, 18945, 28415, 28416, 28417]
STRIDES, ROWS, ADV = (15, 16), ("gather", "ascending", "contiguous"), ("stats", "none", "explicit", "shifted")
CLIPS, VFS, ENTS = (0.1, 0.2, 0.3), (0.5, 1.0), (0.0, 0.01)
BUF_N, BUF_K, FIRST = 1024, 29, 1000                                     # 29,696 rows >= FIRST + max(SIZES)


def _cases():
    out = []
    for mi, mode in enumerate(MODES):
        for i, m in enumerate(SIZES):
            j = i + 5 * mi                                                # every axis value with every mode; modes differ
            adv = "stats" if m == 1 else ADV[j % 4]
            out.append(pytest.param(mode, m, STRIDES[j % 2], ROWS[j % 3], adv, CLIPS[(j // 2) % 3], VFS[(j // 3) % 2],
                                    ENTS[(j // 4) % 2],
                                    id=f"{mode}-m{m}-s{STRIDES[j % 2]}-{ROWS[j % 3]}-{adv}-c{CLIPS[(j // 2) % 3]}"
                                       f"-vf{VFS[(j // 3) % 2]}-ent{ENTS[(j // 4) % 2]}"))
    return out


@pytest.fixture(scope="module")
def design_buffers(drl):
    """Rollout buffers per (obs stride, clip range): _separated_buffers with the log-prob offsets placed around that clip
    range; stride 16 rows carry 1.0 in column 15 as the rollout writes them.  Plus a second advantage array with mean 1e3
    and std 1e-2 (float32 keeps ~160 levels per std there; the kernels' float64 sumsq - sum * mu must not cancel)."""
    from drone_rl_b200.ppo import RolloutBuffers
    theta = _rand_params(9, 0.5).float().cuda()
    made = {}

    def get(stride, clip):
        if (stride, clip) not in made:
            model = types.SimpleNamespace(buf=RolloutBuffers(BUF_K, BUF_N, torch.device("cuda"), stride == 16), params=theta)
            _separated_buffers(model, 4, clip=clip)
            b = model.buf
            if stride == 16:
                b.obs_store[..., 15] = 1.0
            g = torch.Generator().manual_seed(17)
            shifted = (1e3 + 1e-2 * torch.randn(BUF_K * BUF_N, generator=g, dtype=torch.float64)).float().cuda()
            f64 = lambda t: t.double().reshape(t.shape[0] * t.shape[1], *t.shape[2:])
            data = (f64(b.obs), f64(b.actions), f64(b.logp), f64(b.adv), f64(b.ret))
            made[(stride, clip)] = (b, shifted, data)
        return made[(stride, clip)]
    return theta, get


@pytest.mark.parametrize("mode,m,stride,rows,adv,clip,vf,ent", _cases())
def test_gradient_kernel_matches_float64(lib, handles, design_buffers, mode, m, stride, rows, adv, clip, vf, ent):
    """One launch of the minibatch gradient against float64 autograd of the oracle loss: the gradient within the mode's
    tolerance, the statistics columns as in tests/test_gpu_tc.py, the count exact.  With m = 1 and statistics the raw
    advantage is used, as SB3 does for a minibatch of one sample."""
    from drone_rl_b200 import _lib
    theta, get = design_buffers
    b, shifted, data = get(stride, clip)
    h, _ = handles(clip=clip, vf=vf, ent=ent)
    B = BUF_N * BUF_K
    g = torch.Generator().manual_seed(1000 + m)
    if rows == "contiguous":
        index, first, r = None, FIRST, torch.arange(FIRST, FIRST + m)
    else:
        r = torch.randperm(B, generator=g)[:m]
        if rows == "ascending":
            r = r.sort().values
        index, first = r.to(torch.int32).cuda(), 0
    r = r.cuda()
    adv_buf = shifted if adv == "shifted" else b.adv
    adv64 = adv_buf.double().reshape(-1)
    how = "stats" if adv == "shifted" else adv
    stats = None
    if how == "stats":
        a = adv64[r]
        stats = torch.stack([a.sum(), (a * a).sum(), torch.tensor(float(m), dtype=torch.float64, device="cuda")])
    mean, inv_std = (0.3, 0.5) if how == "explicit" else (0.0, 1.0)
    grad = torch.zeros(_lib.GRAD_LEN, device="cuda")
    got = _launch(lib, h, mode, stride, theta, b.obs_store, b, adv_buf, index, first, m, mean, inv_std, stats, grad)
    ref, sums = _ref_grad(theta.double(), data, r, _normalised(adv64, r, how), f32(clip), f32(vf), f32(ent))
    worst, report = _grad_error(got, ref, mode)
    print(f"{mode} m={m}: worst err/tolerance {worst:.3f}; {report}")
    assert worst <= 1.0, report
    _check_stats(got[N:], sums, m, mode)


@pytest.fixture(scope="module")
def production(drl):
    """A 1M-env x 8-step buffer (8,388,608 rows, 64-byte observation rows) generated on the device with the recipe of
    _separated_buffers, and the float64 reference over all of it as one minibatch with its statistics."""
    n, K = 1 << 20, 8
    B = n * K
    dev = torch.device("cuda")
    theta = _rand_params(9, 0.5).float().to(dev)
    g = torch.Generator(device=dev).manual_seed(5)
    buf = types.SimpleNamespace(obs_store=torch.empty(B, 16, device=dev), actions=torch.empty(B, 4, device=dev),
                                logp=torch.empty(B, device=dev), adv=torch.empty(B, device=dev), ret=torch.empty(B, device=dev))
    table = torch.tensor([-0.45, -0.08, 0.0, 0.07, 0.4], dtype=torch.float64, device=dev)
    th64 = theta.double()
    for s in range(0, B, 1 << 20):
        e = min(B, s + (1 << 20))
        obs = torch.randn(e - s, 15, generator=g, device=dev) * 2.0
        mean, value, log_std = po.forward(th64, obs.double())
        act = mean + torch.exp(log_std) * torch.randn(e - s, 4, generator=g, device=dev, dtype=torch.float64)
        offs = table[torch.randint(0, 5, (e - s,), generator=g, device=dev)]
        old = po.log_prob(mean, log_std, act) + offs + 0.01 * torch.randn(e - s, generator=g, device=dev, dtype=torch.float64)
        buf.obs_store[s:e, :15] = obs
        buf.actions[s:e] = act.float()
        buf.logp[s:e] = old.float()
        buf.adv[s:e] = (torch.randn(e - s, generator=g, device=dev, dtype=torch.float64) * 3 + 0.5).float()
        buf.ret[s:e] = (value + 0.7 + torch.randn(e - s, generator=g, device=dev, dtype=torch.float64)).float()
    buf.obs_store[:, 15] = 1.0
    data = (buf.obs_store[:, :15].double(), buf.actions.double(), buf.logp.double(), None, buf.ret.double())
    rows = torch.arange(B, device=dev)
    adv64 = buf.adv.double()
    stats = torch.stack([adv64.sum(), (adv64 * adv64).sum(), torch.tensor(float(B), dtype=torch.float64, device=dev)])
    ref, sums = _ref_grad(th64, data, rows, _normalised(adv64, rows, "stats"), f32(0.2), f32(0.5), f32(0.0))
    del data, adv64
    torch.cuda.empty_cache()
    return theta, buf, rows.to(torch.int32), stats, ref, sums, B


@pytest.mark.parametrize("mode", list(MODES))
def test_gradient_kernel_at_the_production_minibatch(lib, handles, production, mode):
    """c5's minibatch: 8,388,608 samples in ascending rows, ~886 tiles per CTA of the tensor-core kernels and ~443 per CTA of
    the fp32 kernel, every per-CTA sum in float32 before the fixed-order reduce.  Same tolerances as at the small sizes."""
    from drone_rl_b200 import _lib
    theta, buf, index, stats, ref, sums, B = production
    h, _ = handles()
    grad = torch.zeros(_lib.GRAD_LEN, device="cuda")
    got = _launch(lib, h, mode, 16, theta, buf.obs_store, buf, buf.adv, index, 0, B, 0.0, 1.0, stats, grad)
    worst, report = _grad_error(got, ref, mode)
    print(f"{mode} m={B}: worst err/tolerance {worst:.3f}; {report}")
    assert worst <= 1.0, report
    _check_stats(got[N:], sums, B, mode)


# ------------------------------------------------------------------------------------------------------------------------
# b. clip + Adam
# ------------------------------------------------------------------------------------------------------------------------
def _get_state(lib, h):
    mom, step = torch.empty(2 * N, device="cuda"), C.c_int64()
    from drone_rl_b200 import _lib
    _lib.check(lib.dronecu_ppo_get_state(h, P(mom), C.byref(step), None))
    torch.cuda.synchronize()
    return mom, step.value


def _set_state(lib, h, mom, step):
    from drone_rl_b200 import _lib
    _lib.check(lib.dronecu_ppo_set_state(h, P(mom), step, None))


def _torch_step(theta, grad_mean, mom, t, cfg):
    """clip_grad_norm_ + Adam.step() in float64 from the float32 parameters, mean gradient and moments, with the float32
    hyper-parameters of ``cfg`` and Adam's step count t before the step.  -> (params, exp_avg, exp_avg_sq, pre-clip norm)."""
    p = torch.nn.Parameter(theta.detach().double().cpu())
    p.grad = grad_mean.double().cpu()
    norm = float(torch.nn.utils.clip_grad_norm_([p], cfg.max_grad_norm))
    opt = torch.optim.Adam([p], lr=cfg.learning_rate, betas=(cfg.beta1, cfg.beta2), eps=cfg.adam_eps)
    m, v = mom[:N].double().cpu(), mom[N:].double().cpu()
    opt.state[p] = {"step": torch.tensor(float(t), dtype=torch.float64), "exp_avg": m.clone(), "exp_avg_sq": v.clone()}
    opt.step()
    st = opt.state[p]
    return p.detach(), st["exp_avg"], st["exp_avg_sq"], norm, (m, v)


def _check_step(theta_after, mom_after, ref, cfg, what, norm_gpu):
    """Parameters within 2^-22 |ref| + 1e-9 of the float64 step.  The pre-clip norm the kernel used (``norm_gpu``, its info
    column) within 2^-20 of the float64 norm: a float32 sum of 10,697 positive squares in chains of at most 11 fmas and two
    5-level trees is off by at most ~21 roundings, ~11 after the square root.  The moments within their own float32
    roundings given that norm: the clipped gradient g carries the norm's relative error plus 3 roundings (1e-6 add, divide,
    product), exp_avg = b1 m + (1 - b1) g adds 3 more, exp_avg_sq = b2 v + (1 - b2) g g doubles g's error and adds 4."""
    p, m, v, norm, (m0, v0) = ref
    got = theta_after.double().cpu()
    err = (got - p).abs()
    bound = STEP_REL * p.abs() + STEP_ABS
    assert bool((err <= bound).all()), f"{what}: params worst err/bound {float((err / bound).max()):.3g}"
    u = 2.0 ** -24
    e_norm = abs(norm_gpu - norm) / norm if norm > 0 else abs(norm_gpu)
    assert e_norm <= 2.0 ** -20, f"{what}: pre-clip norm {norm_gpu} vs {norm} (relative error {e_norm:.3g})"
    e_g = (e_norm if norm > cfg.max_grad_norm else 0.0) + 3 * u
    gm, gv = mom_after[:N].double().cpu(), mom_after[N:].double().cpu()
    mb = (e_g + 3 * u) * (cfg.beta1 * m0.abs() + (m - cfg.beta1 * m0).abs()) + 1e-30
    vb = (2 * e_g + 4 * u) * v.abs() + 1e-30
    assert bool(((gm - m).abs() <= mb).all()), f"{what}: exp_avg worst err/bound {float(((gm - m).abs() / mb).max()):.3g}"
    assert bool(((gv - v).abs() <= vb).all()), f"{what}: exp_avg_sq worst err/bound {float(((gv - v).abs() / vb).max()):.3g}"
    return float((err / bound).max())


def _random_state(seed):
    g = torch.Generator().manual_seed(seed)
    theta = (0.3 * torch.randn(N, generator=g)).cuda()
    mom = torch.cat([1e-3 * torch.randn(N, generator=g), 1e-9 + 1e-5 * torch.rand(N, generator=g)]).cuda()
    return theta, mom, g


@pytest.mark.parametrize("regime,lr,max_norm,count", [
    ("clipped", 3e-4, 0.5, 1), ("clipped", 1e-3, 2.0, 8388608), ("clipped", 1e-4, 0.25, 64),
    ("unclipped", 3e-4, 0.5, 64), ("unclipped", 1e-3, 2.0, 8388608), ("unclipped", 1e-4, 0.25, 3),
    ("zero", 3e-4, 0.5, 1), ("zero", 1e-3, 2.0, 8388608)])
def test_clip_adam_matches_torch(lib, handles, regime, lr, max_norm, count):
    """Three consecutive dronecu_ppo_apply steps, each against clip_grad_norm_ + Adam in float64 from the device's own
    parameters and moments; the info row (mean statistics, unscaled count, pre-clip norm) and its accumulator."""
    from drone_rl_b200 import _lib
    h, cfg = handles(lr=lr, max_norm=max_norm)
    theta, mom, g = _random_state(count % 1000 + len(regime))
    _set_state(lib, h, mom, 37)
    info, info_sum = torch.zeros(9, device="cuda"), torch.zeros(10, device="cuda")
    _lib.check(lib.dronecu_ppo_set_info_accumulator(h, P(info_sum)))
    inv = 1.0 / count
    scale = {"clipped": 0.1, "unclipped": 1e-3 * max_norm, "zero": 0.0}[regime]
    infos, worst = [], 0.0
    try:
        for k in range(3):
            gmean = scale * torch.randn(N, generator=g)
            stats = torch.tensor([0.3, 2.0, 0.01, 0.2, 1.0, 0.0, 0.0, 0.0]) * count
            grad = torch.cat([gmean * count, stats]).float().cuda()
            mom0, t0 = _get_state(lib, h)
            th0 = theta.clone()
            ref = _torch_step(th0, grad[:N].double() * f32(inv), mom0, t0, cfg)
            _lib.check(lib.dronecu_ppo_apply(h, P(theta), P(grad), inv, P(info), None))
            mom1, t1 = _get_state(lib, h)
            assert t1 == t0 + 1
            worst = max(worst, _check_step(theta, mom1, ref, cfg, f"{regime} step {k}", float(info[8])))
            norm = ref[3]
            assert (norm > max_norm) == (regime == "clipped") and (norm == 0) == (regime == "zero")
            got = info.cpu().double().numpy()
            want = grad[N:].cpu().double().numpy() * f32(inv)
            want[4] = count
            np.testing.assert_allclose(got[:8], want, rtol=1e-6, atol=1e-30)
            assert got[4] == count
            np.testing.assert_allclose(got[8], norm, rtol=1e-5, atol=1e-30)
            infos.append(got)
        acc = info_sum.cpu().double().numpy()
        np.testing.assert_allclose(acc[:9], np.sum(infos, 0), rtol=1e-6, atol=1e-30)
        assert acc[9] == 3
    finally:
        lib.dronecu_ppo_set_info_accumulator(h, None)
    print(f"{regime} lr={lr} max_norm={max_norm} count={count}: worst param err/bound {worst:.3f}")


@pytest.mark.parametrize("t", [0, 1, 9, 10 ** 4, 10 ** 7])
def test_adam_clock_after_set_state(lib, handles, t):
    """set_state(step=t) recomputes beta^t with pow: the next apply equals torch Adam with state["step"] = t."""
    h, cfg = handles(lr=1e-3, max_norm=2.0)
    theta, mom, g = _random_state(t % 997)
    _set_state(lib, h, mom, t)
    grad = torch.cat([1e-3 * torch.randn(N, generator=g), torch.zeros(8)]).cuda()
    mom0, t0 = _get_state(lib, h)
    assert t0 == t and torch.equal(mom0, mom)
    ref = _torch_step(theta, grad[:N].double(), mom0, t, cfg)
    from drone_rl_b200 import _lib
    info = torch.zeros(9, device="cuda")
    _lib.check(lib.dronecu_ppo_apply(h, P(theta), P(grad), 1.0, P(info), None))
    mom1, t1 = _get_state(lib, h)
    assert t1 == t + 1
    _check_step(theta, mom1, ref, cfg, f"t={t}", float(info[8]))


def test_adam_clock_running_powers_equal_pow(lib, handles):
    """3000 in-kernel steps advance beta^t as running float64 products; one more step from there equals, within float32
    rounding, the same step after set_state(3000) (pow), and torch Adam at step 3000."""
    from drone_rl_b200 import _lib
    ha, cfg = handles(lr=1e-4, max_norm=1.0)
    hb, _ = handles(lr=1e-4, max_norm=1.0, ent=0.01)              # same optimiser settings, another handle
    theta, mom, g = _random_state(3)
    _set_state(lib, ha, mom, 0)
    grads = [torch.cat([1e-3 * torch.randn(N, generator=g), torch.zeros(8)]).cuda() for _ in range(4)]
    for k in range(3000):
        _lib.check(lib.dronecu_ppo_apply(ha, P(theta), P(grads[k % 4]), 1.0, None, None))
    mom_a, t_a = _get_state(lib, ha)
    assert t_a == 3000
    _set_state(lib, hb, mom_a, 3000)
    theta_b = theta.clone()
    last = torch.cat([2e-3 * torch.randn(N, generator=g), torch.zeros(8)]).cuda()
    ref = _torch_step(theta, last[:N].double(), mom_a, 3000, cfg)
    info = torch.zeros(9, device="cuda")
    _lib.check(lib.dronecu_ppo_apply(ha, P(theta), P(last), 1.0, P(info), None))
    _lib.check(lib.dronecu_ppo_apply(hb, P(theta_b), P(last), 1.0, None, None))
    (ma, ta), (mb, tb) = _get_state(lib, ha), _get_state(lib, hb)
    assert ta == tb == 3001 and torch.equal(ma, mb)
    d = (theta.double() - theta_b.double()).abs()
    assert bool((d <= 2.0 ** -23 * theta_b.double().abs() + 1e-12).all()), f"running powers vs pow: {float(d.max()):.3g}"
    _check_step(theta, ma, ref, cfg, "step 3001", float(info[8]))


# ------------------------------------------------------------------------------------------------------------------------
# c. PPO.train(), teacher-forced per optimiser step
# ------------------------------------------------------------------------------------------------------------------------
def _adam_state(model):
    from drone_rl_b200 import _lib
    from drone_rl_b200.core import _stream_ptr
    mom, step = torch.empty(2 * N, device=model.device), C.c_int64()
    _lib.check(model.lib.dronecu_ppo_get_state(model._h, P(mom), C.byref(step), _stream_ptr(model.device)))
    return mom, step.value


def _spy_train(model, n_train, forced, own_grad=False):
    """Run train() n_train times with cuda_graph=False, recording at every optimiser step the index slice and the statistics
    row used, and at the steps k with forced(k) the parameters, moments and Adam step before and after and model._grad.
    ``own_grad``: also record model._grad right after the gradient launch, before a data-parallel exchange replaces it by
    the sum over the ranks.  Every read is ordered on the current stream, so each rank of a one-GPU data-parallel run can
    call this from its own thread; it ends with a synchronisation of that stream only."""
    records, orig, orig_grad = [], model._minibatch, model.launch_grad
    pending = {}

    def spy_grad(index, first, m, stats_ptr, grad, precision=None):
        orig_grad(index, first, m, stats_ptr, grad, precision)
        pending["own_grad"] = grad.clone()

    def spy(index, first, m, stats=None):
        k = len(records)
        r = {"index": index.clone(), "m": m, "first": first}
        if forced(k):
            r["theta"] = model.params.clone()
            r["mom"], r["t"] = _adam_state(model)
        orig(index, first, m, stats)
        r.update(pending)
        pending.clear()
        if model.normalize_advantage:
            r["stats"] = (model._adv_stats if stats is None else stats).clone()
        else:
            r["stats"] = stats
        if forced(k):
            r["grad"] = model._grad.clone()
            r["norm"] = float(model._info[8])
            r["theta_after"] = model.params.clone()
            r["mom_after"], r["t_after"] = _adam_state(model)
        records.append(r)
    model._minibatch = spy
    if own_grad:
        model.launch_grad = spy_grad
    try:
        for _ in range(n_train):
            model.train()
    finally:
        del model._minibatch
        if own_grad:
            del model.launch_grad
    torch.cuda.current_stream(model.device).synchronize()
    return records


TRAIN_CONFIGS = {
    # name: (n_envs, n_steps, batch_size, n_epochs, train() calls, data, PPO keywords, teacher-forced steps)
    "c1_shape": (1, 2048, 64, 2, 1, "rollout", {}, None),
    "size1_tail": (25, 41, 64, 2, 2, "rollout", {}, None),
    "permutation": (16, 64, 8, 1, 2, "rollout", {}, None),
    "per_minibatch_stats": (64, 160, 8, 1, 1, "rollout", {}, 61),
    "no_normalisation": (16, 64, 256, 2, 2, "rollout", {"normalize_advantage": False}, None),
    "fp32_hyper": (64, 32, 600, 2, 1, "separated", {"update_precision": "fp32"}, None),
    "tf32_hyper": (64, 32, 600, 2, 1, "separated", {"update_precision": "tf32"}, None),
    "bf16_hyper": (64, 32, 600, 2, 1, "separated", {"update_precision": "bf16"}, None),
}
HYPER = dict(clip_range=0.3, vf_coef=1.0, ent_coef=0.01, max_grad_norm=1.0, learning_rate=1e-4)


def _make(drl, name, graph):
    from drone_rl_b200.ppo import PPO
    n, K, bs, E, _, data, kw, _ = TRAIN_CONFIGS[name]
    kw = dict(kw, **HYPER) if data == "separated" else kw
    model = PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=12), n_steps=K, batch_size=bs, n_epochs=E, seed=12,
                cuda_graph=graph, **kw)
    if data == "rollout":
        model.collect_rollouts()
    else:
        _separated_buffers(model, 7, clip=model.cfg.clip_range)
        model.buf.value.zero_()
        if model.padded_obs:
            model.buf.obs_store[..., 15] = 1.0
    torch.cuda.synchronize()
    return model


@pytest.mark.parametrize("name", list(TRAIN_CONFIGS))
def test_train_is_teacher_forced_sb3(drl, name):
    """Every optimiser step of train(): rows = the slice of the epoch's partition (<= 64 minibatches) or permutation, the epoch
    counter continuing across train() calls; the statistics row = float64 sum, sum of squares and exact count of those
    advantages (None without normalisation); at the teacher-forced steps model._grad = the oracle gradient at the pre-step
    parameters and the step = float64 clip + Adam from the device's own gradient and moments.  The same run as one CUDA graph
    per epoch ends bit-identical."""
    n, K, bs, E, n_train, data, kw, every = TRAIN_CONFIGS[name]
    model = _make(drl, name, False)
    mode, cfg = model.update_precision, model.cfg
    B = n * K
    n_mb = (B + bs - 1) // bs
    if name == "per_minibatch_stats":
        assert n_mb > model._max_mb                     # advantage statistics per minibatch, not per epoch
    steps = n_train * E * n_mb
    forced = (lambda k: True) if every is None else (lambda k: k % every == 0 or k == steps - 1)
    records = _spy_train(model, n_train, forced)
    assert len(records) == steps and model.n_updates == steps
    b = model.buf
    obs = b.obs.reshape(B, 15).double().cpu()
    act, old_logp = b.actions.reshape(B, 4).double().cpu(), b.logp.reshape(B).double().cpu()
    adv, ret = b.adv.reshape(B).double().cpu(), b.ret.reshape(B).double().cpu()
    clip, vf, ent = cfg.clip_range, cfg.vf_coef, cfg.ent_coef
    sizes, worst_grad, worst_step = set(), 0.0, 0.0
    for e in range(n_train * E):
        perm = (philox.minibatch_partition(B, bs, 13, e) if n_mb <= 64 else philox.minibatch_permutation(B, 13, e))
        for k in range(n_mb):
            step = e * n_mb + k
            r = records[step]
            rows = perm[k * bs:(k + 1) * bs]
            m = len(rows)
            sizes.add(m)
            assert r["m"] == m and r["first"] == 0 and np.array_equal(r["index"].cpu().numpy(), rows), f"step {step}: rows"
            a = adv[torch.from_numpy(rows)]
            if not model.normalize_advantage:
                assert r["stats"] is None
            else:
                st = r["stats"].cpu().numpy()
                assert st[2] == m, f"step {step}: count"
                np.testing.assert_allclose(st[:2], [float(a.sum()), float((a * a).sum())], rtol=1e-12,
                                           atol=1e-12 * float(a.abs().sum() + (a * a).sum()), err_msg=f"step {step}")
            if "grad" not in r:
                continue
            idx = torch.from_numpy(rows)
            an = _normalised(adv, idx, "stats") if model.normalize_advantage else a
            theta = r["theta"].double().cpu()
            if mode != "fp32":                            # the reduced-precision forward must not straddle a clip boundary
                mean, _, log_std = po.forward(theta, obs[idx])
                lr_ = po.log_prob(mean, log_std, act[idx]) - old_logp[idx]
                gap = torch.minimum((lr_ - math.log1p(-clip)).abs(), (lr_ - math.log1p(clip)).abs()).min()
                assert float(gap) > 0.02, f"step {step}: a sample within {float(gap):.3g} of a clip boundary"
            ref, _ = _ref_grad(theta, (obs, act, old_logp, None, ret), idx, an, clip, vf, ent)
            got = r["grad"].double().cpu().numpy()
            wg, report = _grad_error(got, ref, mode)
            assert wg <= 1.0, f"step {step} (m={m}): {report}"
            assert got[N + 4] == m
            worst_grad = max(worst_grad, wg)
            assert r["t_after"] == r["t"] + 1
            sref = _torch_step(r["theta"], r["grad"][:N].double().cpu() * f32(1.0 / m), r["mom"], r["t"], cfg)
            worst_step = max(worst_step, _check_step(r["theta_after"], r["mom_after"], sref, cfg, f"step {step}",
                                                        r["norm"]))
    if name == "size1_tail":
        assert 1 in sizes
    print(f"{name}: {steps} steps, minibatch sizes {sorted(sizes)}; worst gradient err/tolerance {worst_grad:.3f}, "
          f"step err/bound {worst_step:.3f}")
    eager_params = model.params.clone()
    eager_mom, eager_t = _adam_state(model)
    torch.cuda.synchronize()
    model.close()
    graph = _make(drl, name, True)
    for _ in range(n_train):
        graph.train()
    torch.cuda.synchronize()
    assert graph._graph is not None and graph.n_updates == steps
    mom, t = _adam_state(graph)
    torch.cuda.synchronize()
    assert t == eager_t == steps
    assert torch.equal(graph.params, eager_params) and torch.equal(mom, eager_mom)
    graph.close()


# ------------------------------------------------------------------------------------------------------------------------
# d. GAE
# ------------------------------------------------------------------------------------------------------------------------
GAMMA_LAMBDA = [(0.99, 0.95), (1.0, 1.0), (0.0, 0.95), (0.9, 0.0)]
DONES = ["none", "all", "first", "last", "random"]


def _gae_cases():
    out = []
    for K in (1, 2048):
        for n in (1, 255, 257):
            for gi, gl in enumerate(GAMMA_LAMBDA):
                for di, d in enumerate(DONES):
                    if n == 257 or (gi + di + n) % 3 == 0:               # every pair at n = 257, a third of them elsewhere
                        out.append((K, n, gl, d))
    big = (1 << 20) + 3
    for gl in GAMMA_LAMBDA:
        for d in DONES:
            out.append((1, big, gl, d))
    out += [(2048, big, (0.99, 0.95), "random"), (2048, big, (1.0, 1.0), "none")]
    return [pytest.param(K, n, gl, d, id=f"K{K}-n{n}-g{gl[0]}-l{gl[1]}-{d}") for K, n, gl, d in out]


@pytest.mark.parametrize("K,n,gl,done_kind", _gae_cases())
def test_gae_within_forward_error(lib, K, n, gl, done_kind):
    """dronecu_gae against the float64 recursion of oracle.ppo_oracle.gae on the same float32 inputs (gamma and lambda as the
    float32 values the kernel receives): |err_t| <= 8 * 2^-24 * (K - t) * M_t, M_t the same recursion on |r|, |v|, |next v|
    (each step adds at most a few roundings of terms bounded by M_t, and earlier errors are damped by gamma * lambda <= 1).
    Returns: the same bound over M_t + |v_t| with one more rounding."""
    from drone_rl_b200 import _lib
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(K * 7919 + n)
    rew = torch.randn(K, n, generator=g, device=dev)
    val = torch.randn(K, n, generator=g, device=dev)
    last = torch.randn(n, generator=g, device=dev)
    done = torch.zeros(K, n, dtype=torch.uint8, device=dev)
    if done_kind == "all":
        done.fill_(1)
    elif done_kind == "first":
        done[0] = 1
    elif done_kind == "last":
        done[K - 1] = 1
    elif done_kind == "random":
        done.copy_(torch.rand(K, n, generator=g, device=dev) < 0.05)
    adv, ret = torch.empty(K, n, device=dev), torch.empty(K, n, device=dev)
    gamma, lam = f32(gl[0]), f32(gl[1])
    _lib.check(lib.dronecu_gae(0, K, n, P(rew), P(val), P(done), P(last), gamma, lam, P(adv), P(ret), None))
    torch.cuda.synchronize()
    # the recursion of po.gae in float64, evaluated row by row (the full float64 arrays would not fit at K x n = 2^31)
    work = dev if K * n > 1 << 22 else torch.device("cpu")
    rw, vl, dn = rew.to(work), val.to(work), done.to(work)
    nv, nv_abs = last.to(work).double(), last.to(work).double().abs()
    acc = torch.zeros(n, dtype=torch.float64, device=work)
    acc_abs = torch.zeros(n, dtype=torch.float64, device=work)
    worst_adv = worst_ret = 0.0
    u = 8.0 * 2.0 ** -24
    for t in reversed(range(K)):
        nnt = 1.0 - dn[t].double()
        r, v = rw[t].double(), vl[t].double()
        acc = r + gamma * nv * nnt - v + gamma * lam * nnt * acc
        acc_abs = r.abs() + gamma * nv_abs * nnt + v.abs() + gamma * lam * nnt * acc_abs
        bound = u * (K - t) * acc_abs
        e_adv = (adv[t].to(work).double() - acc).abs()
        e_ret = (ret[t].to(work).double() - (acc + v)).abs()
        worst_adv = max(worst_adv, float((e_adv / bound).max()))
        worst_ret = max(worst_ret, float((e_ret / (u * (K - t + 1) * (acc_abs + v.abs()))).max()))
        nv, nv_abs = v, v.abs()
    if K == 1 or n <= 257:                                        # the row-by-row recursion is po.gae itself
        ref_adv, _ = po.gae(rew.double().cpu(), val.double().cpu(), done.cpu().bool(), last.double().cpu(), gamma, lam)
        assert torch.allclose(ref_adv[0], acc.cpu(), rtol=1e-12, atol=1e-12)
    print(f"K={K} n={n} gamma={gl[0]} lambda={gl[1]} done={done_kind}: worst err/bound advantages {worst_adv:.3g}, "
          f"returns {worst_ret:.3g}")
    assert worst_adv <= 1.0 and worst_ret <= 1.0
