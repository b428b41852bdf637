"""Every in-kernel policy rollout kernel -- thread per env, warp per env, tensor cores (csrc/ppo_rollout.cuh,
csrc/ppo_rollout_tc.cuh) -- teacher-forced against float64 over a covering design of launch shapes, start states,
clocks, modes, normalisation, row layouts and policies.  Every level of every factor appears, and every level of
every other factor appears with every kernel.

Checked at every (step, env):
  env transition      obs / reward / done / last_obs / auto-resets through oracle/verify.check_rollout (clipped actions)
  mean and value      tensor cores and thread per env: bit-identical to policy_forward (tf32 / fp32) on the recorded
                      (normalised) rows; warp per env: within 1e-5 of it (its head sums are warp reductions);
                      policy_forward within the oracle/tc_bound.py bound (tf32) or 2e-5 * max(1, |ref|) (fp32) of
                      ppo_oracle.forward
  stochastic action   a = fmaf(std, z, mean) with z = philox.noise_normals in float64: float32 Box-Muller (logf and
                      sincospif 1 ulp, sqrtf and the products 0.5 ulp) leaves z within 2^-21 relative, expf 2 ulp,
                      the fmaf 0.5 ulp: |err| <= 2^-20 std |z| + 2^-24 |a|
  log-prob            stochastic: -|z|^2 / 2 - sum log_std - 2 ln 2 pi in float64 within 2^-19 of the magnitudes
                      (z^2 carries 2^-20, four float32 sums); deterministic: bit-equal to the kernel's float32 formula
  state after         step, ep_num, ep_len as the record implies; ep_ret bit-exact by a float32 replay of the rewards
  episode statistics  episodes, length_sum exactly; terminated against the oracle's crash decisions (borderline rows
                      are the only slack); truncated = episodes - terminated; return_sum within the float32 rounding
                      of each env's sum over its episodes
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import drone_oracle as do  # noqa: E402
from oracle import philox, ppo_oracle as po, verify  # noqa: E402
from oracle.tc_bound import tc_forward_bound  # noqa: E402

SEED = 21
MOTOR_MAX = np.float32(7.3575)
HALF_LOG_2PI = np.float32(0.91893853320467274178)
KERNELS = ("thread", "warp", "tc")
NS = (1, 31, 33, 127, 129, 1000, 1025, 2049, 4097, 8193)


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


def _policy(kind):
    """hover: the policy of tests/test_gpu_ppo.py (mean near hover thrust); wide: three times its perturbation and a
    positive log_std, so sampled actions cross both clip limits."""
    g = torch.Generator().manual_seed(5)
    flat = po.init_params(5, dtype=torch.float64) + (0.03 if kind == "hover" else 0.09) * torch.randn(
        po.N_PARAMS, generator=g, dtype=torch.float64)
    off = po.offsets()["pi.b3"][0]
    flat[off:off + 4] = 2.45 if kind == "hover" else 3.5
    off = po.offsets()["log_std"][0]
    flat[off:off + 4] = torch.tensor([-0.5, -0.2, 0.1, -1.0] if kind == "hover" else [0.5, 0.7, 0.4, 0.6], dtype=torch.float64)
    return flat.float().numpy()


def _norm_affine(n):
    """the non-identity record of tests/test_gpu_normalize.py"""
    from drone_rl_b200.normalize import ObsNormalizer
    from tests.test_gpu_normalize import _set_stats
    nz = ObsNormalizer(n, torch.device("cuda", 0))
    _set_stats(nz, torch.linspace(-3, 12, 15), torch.linspace(0.5, 30, 15) ** 2)
    return nz


def _forward(theta_dev, rows, tc):
    """policy_forward through the C entry points: rows [B, 15] float32 on the device -> (mean [B, 4], value [B])"""
    from drone_rl_b200 import _lib
    lib = _lib.load()
    rows = rows.contiguous()
    B = rows.shape[0]
    mean = torch.empty(B, 4, device="cuda")
    value = torch.empty(B, device="cuda")
    P = lambda t: C.c_void_p(t.data_ptr())
    if tc:
        _lib.check(lib.dronecu_policy_forward_tc(0, B, P(theta_dev), P(rows), P(mean), P(value), None, None, None))
    else:
        _lib.check(lib.dronecu_policy_forward(0, B, P(theta_dev), P(rows), P(mean), P(value), None))
    return mean, value


def _launch(batch, kernel, K, theta_dev, det, stride, affine, set_mode):
    from drone_rl_b200 import _lib
    from drone_rl_b200._lib import PolicyOut
    n = batch.n
    e = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device="cuda")
    r = {"obs_store": torch.full((K, n, stride), -7.0, device="cuda"), "actions": e(K, n, 4), "logp": e(K, n),
         "value": e(K, n), "reward": e(K, n), "done": e(K, n, dt=torch.uint8), "last_value": e(n), "last_obs": e(n, 15)}
    P = lambda t: t.data_ptr()
    out = PolicyOut(P(r["obs_store"]), P(r["actions"]), P(r["logp"]), P(r["value"]), P(r["reward"]), P(r["done"]),
                    P(r["last_value"]), P(r["last_obs"]), int(stride == 16), 0)
    tc = kernel == "tc"
    if not tc:
        set_mode({"thread": 1, "warp": 2}[kernel])
    th = C.c_void_p(theta_dev.data_ptr())
    lib = batch.lib
    if affine is not None:
        rc = lib.dronecu_rollout_policy_norm(batch._h, K, th, int(det), C.byref(out), C.c_void_p(affine.data_ptr()), int(tc), None)
    elif tc:
        rc = lib.dronecu_rollout_policy_tc(batch._h, K, th, int(det), C.byref(out), None)
    else:
        rc = lib.dronecu_rollout_policy(batch._h, K, th, int(det), C.byref(out), None)
    _lib.check(rc)
    torch.cuda.synchronize()
    r["obs"] = r["obs_store"][..., :15]
    return r


def _mid_episode(batch, rng):
    """late steps (timeouts within 15 steps) and episode counters just below several curriculum bumps"""
    n = batch.n
    step = rng.integers(185, 200, n).astype(np.int32)
    ep_num = rng.choice([5, 1999, 3999, 5998, 19999, 40001], n).astype(np.int32)
    ep_ret = (-rng.uniform(0, 3, n)).astype(np.float32)
    batch.set_state(step=step, ep_num=ep_num, ep_len=step, ep_ret=ep_ret)


def _expected_after(st0, done, reward):
    """(step, ep_num, ep_len, ep_ret, per-env episode returns, length_sum) implied by the record"""
    K, n = done.shape
    ep_ret = st0["ep_ret"].copy()
    rets = [[] for _ in range(n)]
    for k in range(K):
        ep_ret = (ep_ret + reward[k]).astype(np.float32)
        for i in np.flatnonzero(done[k]):
            rets[i].append(ep_ret[i])
        ep_ret[done[k]] = 0.0
    any_done = done.any(0)
    last = np.where(any_done, K - 1 - np.argmax(done[::-1], 0), -1)
    since = np.where(any_done, K - 1 - last, st0["ep_len"] + K)
    step = np.where(any_done, K - 1 - last, st0["step"] + K)
    ep_num = st0["ep_num"] + done.sum(0)
    length_sum = int(np.where(any_done, st0["ep_len"].astype(np.int64) + last + 1, 0).sum())
    return step, ep_num, since, ep_ret, rets, length_sum


def _ratio(err, bound):
    return float(np.max(err / bound)) if err.size else 0.0


def _check_record(batch, rec, theta, theta_dev, kernel, det, nz, st0, t0, cols=None):
    """Every check of the module docstring on the envs `cols` (None = all).  Returns the worst err/bound per check."""
    n = batch.n
    idx = torch.arange(n, device="cuda") if cols is None else cols
    g = lambda t: t[:, idx] if t.dim() >= 2 else t[idx]
    obs_d, act_d = g(rec["obs"]), g(rec["actions"])
    K, m = obs_d.shape[:2]
    aff = (lambda x: x) if nz is None else (lambda x: _affine_ref(x, nz))
    xn = aff(obs_d).reshape(-1, 15)
    last_xn = aff(rec["last_obs"][idx])
    tc = kernel == "tc"
    pm, pv = _forward(theta_dev, xn, tc)
    _, plv = _forward(theta_dev, last_xn, tc)
    value, last_value = g(rec["value"]).reshape(-1), rec["last_value"][idx]
    worst = {}
    # mean and value against policy_forward
    if kernel == "warp":
        worst["value_vs_forward"] = max(float((value - pv).abs().max()), float((last_value - plv).abs().max())) / 1e-5
        assert worst["value_vs_forward"] <= 1.0
        if det:
            worst["mean_vs_forward"] = float((act_d.reshape(-1, 4) - pm).abs().max()) / 1e-5
            assert worst["mean_vs_forward"] <= 1.0
    else:
        assert torch.equal(value, pv) and torch.equal(last_value, plv), "value differs from policy_forward"
        if det:
            assert torch.equal(act_d.reshape(-1, 4), pm), "deterministic action differs from policy_forward"
    # policy_forward against the oracle
    x64 = xn.cpu().numpy()
    pm_h, pv_h = pm.cpu().double().numpy(), pv.cpu().double().numpy()
    if tc:
        m_ref, v_ref, mb, vb = tc_forward_bound(theta, x64)
        _, lv_ref, _, lvb = tc_forward_bound(theta, last_xn.cpu().numpy())
    else:
        th64 = torch.from_numpy(theta).double()
        m_ref, v_ref, _ = (t.numpy() for t in po.forward(th64, torch.from_numpy(x64).double()))
        _, lv_ref, _ = (t.numpy() for t in po.forward(th64, last_xn.cpu().double()))
        mb, vb, lvb = 2e-5 * np.maximum(1, np.abs(m_ref)), 2e-5 * np.maximum(1, np.abs(v_ref)), 2e-5 * np.maximum(1, np.abs(lv_ref))
    worst["forward_vs_oracle"] = max(_ratio(np.abs(pm_h - m_ref), mb), _ratio(np.abs(pv_h - v_ref), vb),
                                     _ratio(np.abs(plv.cpu().double().numpy() - lv_ref), lvb))
    if kernel != "tc":      # the fp32 kernels' own record against the oracle as well
        worst["fp32_value_vs_oracle"] = _ratio(np.abs(value.cpu().double().numpy() - v_ref), vb)
        assert worst["fp32_value_vs_oracle"] <= 1.0
    assert worst["forward_vs_oracle"] <= 1.0, f"policy_forward vs oracle: {worst['forward_vs_oracle']:.3g}"
    # action and log-prob
    act = act_d.cpu().numpy()
    logp = g(rec["logp"]).cpu().numpy()
    ls32 = theta[-4:]
    ls_sum = np.float32(0)
    for o in range(4):
        ls_sum = np.float32(ls_sum + ls32[o])
    if det:
        assert (logp == np.float32(-ls_sum - np.float32(4 * HALF_LOG_2PI))).all(), "deterministic log-prob"
    else:
        ids = batch.env_offset + idx.cpu().numpy().astype(np.uint64)
        std = np.exp(ls32.astype(np.float64))
        mean_k = pm_h.reshape(K, m, 4)
        slack = 1e-5 if kernel == "warp" else 0.0
        wa, wl = 0.0, 0.0
        for k in range(K):
            z = philox.noise_normals(SEED, ids, t0 + k)
            ref_a = mean_k[k] + std * z
            ba = 2.0 ** -20 * std * np.abs(z) + 2.0 ** -24 * np.abs(act[k]) + slack + 1e-30
            wa = max(wa, _ratio(np.abs(act[k] - ref_a), ba))
            ref_lp = -0.5 * (z * z).sum(1) - ls32.astype(np.float64).sum() - 2 * np.log(2 * np.pi)
            bl = 2.0 ** -19 * (0.5 * (z * z).sum(1) + np.abs(ls32).sum() + 4)
            wl = max(wl, _ratio(np.abs(logp[k] - ref_lp), bl))
        worst["action"], worst["logp"] = wa, wl
        assert wa <= 1.0 and wl <= 1.0, f"action {wa:.3g} logp {wl:.3g}"
    # env transitions under the clipped actions
    o = obs_d.cpu().numpy()
    nxt = np.concatenate([o[1:], rec["last_obs"][idx].cpu().numpy()[None]], 0)
    reward, done = g(rec["reward"]).cpu().numpy(), g(rec["done"]).cpu().numpy().astype(bool)
    sub = {k: v[idx.cpu().numpy()] for k, v in st0.items()}
    rep = verify.check_rollout(o[0], np.clip(act, 0, MOTOR_MAX), nxt, reward, done, spec=do.SINGLE, seed=SEED,
                               env_ids=batch.env_offset + idx.cpu().numpy().astype(np.uint64),
                               ep_num0=sub["ep_num"], step0=sub["step"])
    worst["env"] = rep["worst_err_over_bound"]
    # state after the launch
    st1 = {k: v[idx.cpu().numpy()] for k, v in batch.get_state("step", "ep_num", "ep_len", "ep_ret").items()}
    step, ep_num, ep_len, ep_ret, rets, length_sum = _expected_after(sub, done, reward)
    assert np.array_equal(st1["step"], step) and np.array_equal(st1["ep_num"], ep_num) and np.array_equal(st1["ep_len"], ep_len)
    assert np.array_equal(st1["ep_ret"].view(np.uint32), ep_ret.view(np.uint32)), "ep_ret is not the float32 replay"
    return worst, rep, done, rets, length_sum


def _affine_ref(x, nz):
    from tests.test_gpu_normalize import _affine_ref as f
    return f(x, nz)


def _check_stats(stats, done, rets, length_sum, rep):
    assert stats["episodes"] == int(done.sum())
    assert stats["length_sum"] == length_sum
    assert rep["terminated"] <= stats["terminated"] <= rep["terminated"] + rep["terminated_slack"]
    assert stats["truncated"] == stats["episodes"] - stats["terminated"]
    flat = [r for env in rets for r in env]
    ref = float(np.sum(np.asarray(flat, np.float64)))
    tol = sum(max(len(env) - 1, 0) * 2.0 ** -24 * 1.01 * float(np.abs(np.asarray(env, np.float64)).sum()) for env in rets)
    tol += 1e-12 * (float(np.abs(np.asarray(flat, np.float64)).sum()) + 1.0)
    assert abs(stats["return_sum"] - ref) <= tol, f"return_sum {stats['return_sum']!r} vs {ref!r} (tol {tol:.3g})"


def _design():
    """10 cases per kernel, one per n; the other factors cycle with periods <= 4 from a per-kernel offset, so each
    kernel meets every level of every factor."""
    cases = []
    for ki, kernel in enumerate(KERNELS):
        for j, n in enumerate(NS):
            r = j + ki
            K = (1, 40, 230)[r % 3]
            if n * K > 1_100_000:
                K = 40
            cases.append(pytest.param(kernel, n, K, ("fresh", "mid")[r % 2], (0, 12345)[(r // 2) % 2],
                                      (0, 7 << 23)[((r + 1) // 2) % 2], (r % 4) in (1, 2), (r % 4) >= 2,
                                      16 if r % 3 == 1 else 15, "wide" if r % 4 == 3 else "hover",
                                      id=f"{kernel}-n{n}-K{K}-{('fresh', 'mid')[r % 2]}-gs{(0, 12345)[(r // 2) % 2]}"
                                         f"-off{(0, 7 << 23)[((r + 1) // 2) % 2]}-{'det' if (r % 4) in (1, 2) else 'stoch'}"
                                         f"-{'norm' if (r % 4) >= 2 else 'raw'}-s{16 if r % 3 == 1 else 15}"
                                         f"-{'wide' if r % 4 == 3 else 'hover'}"))
    return cases


def _setup(drl, n, start, gs, off, rng):
    b = drl.DroneBatch(n, drl.EnvConfig.single(), seed=SEED, env_offset=off)
    b.reset()
    if start == "mid":
        _mid_episode(b, rng)
    b.global_step = gs
    b.episode_stats(reset=True)
    return b


@pytest.mark.parametrize("kernel,n,K,start,gs,off,det,norm,stride,policy", _design())
def test_rollout_parity(drl, rollout_kernel_mode, kernel, n, K, start, gs, off, det, norm, stride, policy):
    rng = np.random.default_rng(n * 7 + K)
    theta = _policy(policy)
    theta_dev = torch.from_numpy(theta).cuda()
    nz = _norm_affine(n) if norm else None
    b = _setup(drl, n, start, gs, off, rng)
    st0 = b.get_state()
    rec = _launch(b, kernel, K, theta_dev, det, stride, None if nz is None else nz.affine, rollout_kernel_mode)
    stats = b.episode_stats(reset=True)
    assert b.global_step == gs + K
    worst, rep, done, rets, length_sum = _check_record(b, rec, theta, theta_dev, kernel, det, nz, st0, gs)
    _check_stats(stats, done, rets, length_sum, rep)
    if policy == "wide" and not det and n * K >= 1000:
        a = rec["actions"]
        assert bool((a < 0).any()) and bool((a > float(MOTOR_MAX)).any()), "the wide policy must cross both clip limits"
    if start == "mid" and K >= 15:
        assert rep["dones"] >= n, "every env reaches its time limit"
    if K == 230:
        assert (done.any(0)).all(), "every env ends an episode in 230 steps"
    if stride == 16:
        assert bool((rec["obs_store"][..., 15] == 1.0).all())
        # the packed run from the same state and clock: identical record
        b.set_state(**st0)
        b.global_step = gs
        packed = _launch(b, kernel, K, theta_dev, det, 15, None if nz is None else nz.affine, rollout_kernel_mode)
        for key in ("obs", "actions", "logp", "value", "reward", "done", "last_value", "last_obs"):
            assert torch.equal(rec[key], packed[key]), key
    print(f"{kernel} n={n} K={K}: worst err/bound " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items())
          + f"; dones {rep['dones']}, terminated {stats['terminated']}, borderline {rep['borderline_done']}")
    b.close()


@pytest.mark.parametrize("kernel,stride", [("tc", 15), ("tc", 16), ("thread", 15)])
def test_rollout_parity_at_production_size(drl, rollout_kernel_mode, kernel, stride):
    """1,048,576 envs x 32 steps (the c3 / c5 shapes): every check on a strided sample of envs and the last env of the
    last tile; the episode statistics over all envs (terminated: at least the dones before the time limit)."""
    n, K = 1 << 20, 32
    theta = _policy("hover")
    theta_dev = torch.from_numpy(theta).cuda()
    b = _setup(drl, n, "mid", 0, 0, np.random.default_rng(3))
    st0 = b.get_state()
    rec = _launch(b, kernel, K, theta_dev, False, stride, None, rollout_kernel_mode)
    stats = b.episode_stats(reset=True)
    cols = torch.cat([torch.arange(0, n, 997, device="cuda"), torch.tensor([n - 1], device="cuda")])
    worst, rep, _, _, _ = _check_record(b, rec, theta, theta_dev, kernel, False, None, st0, 0, cols=cols)
    # statistics over every env, on the device
    done = rec["done"].bool()
    assert stats["episodes"] == int(done.sum())
    any_done = done.any(0)
    last = K - 1 - torch.flip(done, [0]).int().argmax(0)
    ep_len0 = torch.from_numpy(st0["ep_len"]).cuda().long()
    assert stats["length_sum"] == int(torch.where(any_done, ep_len0 + last + 1, torch.zeros_like(ep_len0)).sum())
    # dones before the time limit are crashes; the return sum within each env's float32 sum over its episodes
    cnt = torch.from_numpy(st0["step"]).cuda().long()
    ret = torch.from_numpy(st0["ep_ret"]).cuda()
    early = 0
    rsum = torch.zeros(n, dtype=torch.float64, device="cuda")
    rabs = torch.zeros(n, dtype=torch.float64, device="cuda")
    for k in range(K):
        cnt += 1
        ret = ret + rec["reward"][k]
        early += int((done[k] & (cnt < 200)).sum())
        rsum += torch.where(done[k], ret, torch.zeros_like(ret)).double()
        rabs += torch.where(done[k], ret.abs(), torch.zeros_like(ret)).double()
        cnt = torch.where(done[k], torch.zeros_like(cnt), cnt)
        ret = torch.where(done[k], torch.zeros_like(ret), ret)
    assert early <= stats["terminated"] <= stats["episodes"]
    assert stats["truncated"] == stats["episodes"] - stats["terminated"]
    m_env = done.sum(0).double()
    tol = float(((m_env - 1).clamp(min=0) * 2.0 ** -24 * 1.01 * rabs).sum()) + 1e-12 * (1 + float(rabs.sum()))
    assert abs(stats["return_sum"] - float(rsum.sum())) <= tol
    assert torch.equal(ret[cols].cpu(), torch.from_numpy(b.get_state("ep_ret")["ep_ret"])[cols.cpu()])
    print(f"{kernel} stride {stride} n={n} K={K}: worst err/bound " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items())
          + f"; episodes {stats['episodes']}, terminated {stats['terminated']}")
    b.close()


@pytest.mark.parametrize("B", [1, 127, 128, 129, 38405, 1 << 20])
def test_tc_forward_within_bound(drl, B):
    """policy_forward on the tensor cores against the oracle/tc_bound.py bound, per element; the largest B on a
    strided sample of rows and the last tile."""
    theta = _policy("hover")
    theta_dev = torch.from_numpy(theta).cuda()
    g = torch.Generator(device="cuda").manual_seed(B)
    scales = torch.tensor([3.0] * 3 + [4.0] * 3 + [2.0] * 3 + [10.0] * 3 + [1.0] * 3, device="cuda")
    rows = torch.randn(B, 15, generator=g, device="cuda") * scales
    m, v = _forward(theta_dev, rows, True)
    sel = torch.arange(B, device="cuda") if B < 65536 else torch.cat([torch.arange(0, B, 31, device="cuda"),
                                                                      torch.arange(B - 128, B, device="cuda")])
    m_ref, v_ref, mb, vb = tc_forward_bound(theta, rows[sel].cpu().numpy())
    r = max(_ratio(np.abs(m[sel].cpu().double().numpy() - m_ref), mb), _ratio(np.abs(v[sel].cpu().double().numpy() - v_ref), vb))
    print(f"B={B}: worst err/bound {r:.3g}, median bound / max(1, |ref|) "
          f"{np.median(np.concatenate([(mb / np.maximum(1, np.abs(m_ref))).ravel(), vb / np.maximum(1, np.abs(v_ref))])):.2e}")
    assert r <= 1.0


def test_env_emits_non_finite_rows(drl, rollout_kernel_mode):
    """A finite state the policy can be handed through set_state -- body rates of 3e19 rad/s, inside the arena -- makes
    the env emit rows with inf and then NaN in them without ending the episode (the crash test looks at the position
    only, and NaN compares false), so the policy towers do see non-finite rows."""
    n = 32
    b = drl.DroneBatch(n, drl.EnvConfig.single(), seed=SEED)
    b.reset()
    b.set_state(omega=np.tile(np.array([3e19, 3e19, 3e19], np.float32), (n, 1)))
    rec = _launch(b, "thread", 4, torch.from_numpy(_policy("hover")).cuda(), True, 15, None, rollout_kernel_mode)
    obs, done = rec["obs"].cpu().numpy(), rec["done"].cpu().numpy()
    assert not done[:3].any()
    assert np.isinf(obs[1]).any() and np.isnan(obs[2:]).any()
    b.close()


def test_forward_on_non_finite_and_huge_rows(drl):
    """policy_forward (fp32 and tf32) on rows holding 1e30, +-inf, FLT_MAX and NaN, against torch float32 po.forward.
    fp32: the same NaN pattern and the same values within 2e-5.  tf32: the rows without NaN match within 2e-2 (1e30 and
    inf saturate the first tanh); a row holding NaN gives an unspecified output on the tensor cores (tc_mlp.cuh)."""
    theta = _policy("hover")
    theta_dev = torch.from_numpy(theta).cuda()
    g = torch.Generator().manual_seed(0)
    rows = torch.randn(12, 15, generator=g)
    rows[0, 3] = 1e30; rows[1, 9] = -1e30; rows[2, 0] = float("inf"); rows[3, 11] = float("-inf")
    rows[4, :] = 1e30; rows[5, 14] = float("inf"); rows[5, 2] = 1e30
    rows[6, 5] = float("nan"); rows[7, :] = float("nan")
    rows[8, 0] = torch.finfo(torch.float32).max; rows[9, 1] = -torch.finfo(torch.float32).max   # round to inf in tf32
    ref_m, ref_v, _ = po.forward(torch.from_numpy(theta), rows)
    nan_row = torch.isnan(rows).any(1)
    report = {}
    for tc in (False, True):
        m, v = (t.cpu() for t in _forward(theta_dev, rows.cuda(), tc))
        keep = ~nan_row if tc else torch.ones_like(nan_row)
        for got, ref in ((m, ref_m), (v, ref_v)):
            got, ref = got[keep], ref[keep]
            assert torch.equal(torch.isnan(got), torch.isnan(ref)), f"{'tf32' if tc else 'fp32'}: NaN pattern"
            fin = ~torch.isnan(ref)
            err = float(((got - ref).abs() / ref.abs().clamp(min=1))[fin].max())
            report[tc] = max(report.get(tc, 0.0), err)
        if tc:
            print(f"tf32 outputs of the NaN rows (unspecified): mean {m[nan_row].tolist()}, value {v[nan_row].tolist()}")
    print(f"worst scaled err: fp32 {report[False]:.3g}, tf32 {report[True]:.3g}")
    assert bool(torch.isnan(ref_m[nan_row]).all())
    assert report[False] <= 2e-5 and report[True] <= 2e-2
