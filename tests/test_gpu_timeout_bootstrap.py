"""The time-limit bootstrap (PPO(handle_timeout_termination=True), csrc/ppo_timeout.cuh, DESIGN.md section 11) on the GPU.

From the same state, seed and clock, a rollout with the flag on equals the rollout with the flag off in everything but the
rewards of truncated steps: observations, actions, log-probabilities, values, dones, last values, the env state afterwards,
the episode statistics, the normalisation statistics and per-env returns are bit-identical.  On a truncated step the reward
is f32(r + f32(f32(gamma) * V)) of the flag-off reward r and V = dronecu_policy_forward(norm(terminal row)), bit for bit
(tests/test_timeout_oracle.py pins that expression to SB3's).  The recorded terminal rows equal DroneBatch.step's
terminal_obs replaying the recorded actions, and the live slots equal its truncated mask.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ppo_oracle as po  # noqa: E402

pytestmark = pytest.mark.gpu
MAX_STEPS = 7


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


@pytest.fixture
def kernel_mode():
    from drone_rl_b200 import _lib
    lib = _lib.load()
    yield lambda kernel: _lib.check(lib.dronecu_set_rollout_kernel({"thread": 1, "warp": 2, "tc": 0}[kernel]))
    lib.dronecu_set_rollout_kernel(0)


def _theta():
    from tests.test_gpu_rollout_parity import _policy
    return torch.from_numpy(_policy("hover")).to(torch.float32).cuda()


def _bits(a):
    a = np.ascontiguousarray(a)
    b = a.view(np.uint32 if a.dtype == np.float32 else np.uint8).copy()
    if a.dtype == np.float32:
        b[np.isnan(a)] = 0x7FC00000
    return b


def _same(a, b):
    return np.array_equal(_bits(np.asarray(a)), _bits(np.asarray(b)))


def _expr(r, v, gamma):
    return (np.float32(r) + (np.float32(gamma) * np.asarray(v, np.float32)).astype(np.float32)).astype(np.float32)


def _forward_value(theta, rows):
    """dronecu_policy_forward's value of [B,15] float32 rows (host arrays)"""
    from drone_rl_b200 import _lib
    lib = _lib.load()
    x = torch.from_numpy(np.ascontiguousarray(rows, np.float32)).cuda()
    v = torch.empty(x.shape[0], device="cuda")
    _lib.check(lib.dronecu_policy_forward(0, x.shape[0], C.c_void_p(theta.data_ptr()), C.c_void_p(x.data_ptr()), None,
                                          C.c_void_p(v.data_ptr()), None))
    torch.cuda.synchronize()
    return v.cpu().numpy()


def _norm_rows(rows, aff):
    """norm_obs_row of the kernels: float32 subtract, multiply, np.clip"""
    y = ((np.asarray(rows, np.float32) - aff[:15]).astype(np.float32) * aff[15:30]).astype(np.float32)
    return np.clip(y, -aff[30], aff[30])


def _mid_episode(batch, seed, crash=()):
    """every env mid-episode, env 0 one step before the limit (a truncation at k = 0); `crash` envs below the floor"""
    rng = np.random.default_rng(seed)
    n = batch.n
    step = rng.integers(0, MAX_STEPS, n).astype(np.int32)
    step[0] = MAX_STEPS - 1
    if len(crash):
        step[list(crash)] = MAX_STEPS - 1      # crash and time limit on the same step
    batch.set_state(step=step, ep_len=step, ep_num=rng.integers(1, 50, n).astype(np.int32),
                    ep_ret=(-rng.uniform(0, 2, n)).astype(np.float32))
    if len(crash):
        pos = batch.get_state("pos")["pos"]
        pos[list(crash), 2] = -3.0
        batch.set_state(pos=pos)


# ---------------------------------------------------------------------------------------------------------------------
# the PPO rollout with the flag on against the flag off
# ---------------------------------------------------------------------------------------------------------------------
def _model(drl, n, K, kernel, norm, padded, flag, seed=3):
    from drone_rl_b200.ppo import PPO
    b = drl.DroneBatch(n, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=seed)
    m = PPO(b, n_steps=K, batch_size=n * K, n_epochs=1, gamma=0.93, seed=seed, padded_obs=bool(padded),
            rollout_precision="tf32" if kernel == "tc" else "fp32", norm_obs=norm >= 1, norm_reward=norm >= 2,
            clip_obs=4.0, handle_timeout_termination=flag)
    m.tc_min_envs = 0
    m.params.copy_(_theta())
    if m.normalizer is not None:           # statistics that are not the identity, the same in both models
        s = torch.zeros(34, dtype=torch.float64)
        s[:15] = torch.linspace(-1, 1, 15)
        s[15:30] = torch.linspace(0.5, 3, 15) ** 2
        s[30], s[31], s[32], s[33] = 100.0, -0.5, 4.0, 100.0
        m.normalizer.stats.copy_(s)
        m.normalizer._combine(None)
        m.normalizer.returns.copy_(torch.linspace(-1, 0, n, dtype=torch.float64))
    _mid_episode(b, seed, crash=(1,))
    return m


KERNELS = ("thread", "warp", "tc")
NORMS = (0, 1, 2)


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("norm", NORMS, ids=["raw", "obs", "obs+reward"])
@pytest.mark.parametrize("det", [1, 0], ids=["det", "stoch"])
@pytest.mark.parametrize("padded", [0, 1], ids=["rows15", "rows16"])
def test_flag_on_equals_flag_off_but_truncated_rewards(drl, kernel_mode, kernel, norm, det, padded):
    n = 1000 if kernel == "tc" else 257                 # not a multiple of 32 or 128
    K = 23
    theta = _theta()
    kernel_mode(kernel)
    off, on = (_model(drl, n, K, kernel, norm, padded, flag) for flag in (False, True))
    aff = None if on.normalizer is None or not on.normalizer.norm_obs else on.normalizer.affine.cpu().numpy()
    st0 = on.batch.get_state()
    l0 = (off.launches, on.launches)
    off.collect_rollouts(deterministic=bool(det))
    on.collect_rollouts(deterministic=bool(det))
    torch.cuda.synchronize()
    assert on.launches - l0[1] == off.launches - l0[0] + 1
    for name in ("obs_store", "actions", "logp", "value", "done", "last_value"):
        assert _same(getattr(on.buf, name).cpu().numpy(), getattr(off.buf, name).cpu().numpy()), name
    s_on, s_off = on.batch.get_state(), off.batch.get_state()
    for k in s_off:
        assert np.array_equal(s_on[k], s_off[k]), k
    e_on, e_off = on.batch.episode_stats(), off.batch.episode_stats()
    for key in ("episodes", "terminated", "truncated", "length_sum"):
        assert e_on[key] == e_off[key], key
    assert e_on["return_sum"] == pytest.approx(e_off["return_sum"], rel=1e-6)   # per-CTA double atomics: order not fixed
    if on.normalizer is not None:
        assert torch.equal(on.normalizer.stats, off.normalizer.stats)
        assert torch.equal(on.normalizer.returns, off.normalizer.returns)
    # the side buffer: live slots, in order, then -1
    T = -(-K // MAX_STEPS)
    rows = on.timeout_row.cpu().numpy()
    assert rows.shape == (T, n)
    live = rows >= 0
    assert (live[1:] <= live[:-1]).all(), "an env's slots fill from j = 0"
    assert (rows[live] % n == np.nonzero(live)[1]).all(), "slot j * n + i holds env i"
    trunc = np.zeros((K, n), bool)
    trunc[rows[live] // n, rows[live] % n] = True
    assert trunc[0, 0], "env 0 truncates at k = 0"
    assert not trunc[0, 1] and on.buf.done[0, 1].item() == 1, "env 1 crashes at the limit: no bootstrap"
    assert trunc.sum() > n // 2
    # rewards
    r_on, r_off = on.buf.reward.cpu().numpy(), off.buf.reward.cpu().numpy()
    assert _same(r_on[~trunc], r_off[~trunc])
    term = on.timeout_obs.cpu().numpy()[live][:, :15]
    assert (on.timeout_obs.cpu().numpy()[live][:, 15] == 1.0).all()
    v = _forward_value(theta, term if aff is None else _norm_rows(term, aff))
    ref = r_off.copy()
    ref[rows[live] // n, rows[live] % n] = _expr(r_off[rows[live] // n, rows[live] % n], v, on.gamma)
    assert _same(r_on, ref)
    # the terminal rows against the env's own step API, replaying the recorded clipped actions from the same state
    rep = drl.DroneBatch(n, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=3)
    rep.set_state(**st0)
    acts = torch.clamp(on.buf.actions, 0.0, rep.config.motor_max)
    tr_rep = np.zeros((K, n), bool)
    term_rep = np.zeros((K, n, 15), np.float32)
    for k in range(K):
        res = rep.step(acts[k].contiguous(), want_truncated=True, want_terminal_obs=True)
        tr_rep[k] = res["truncated"].cpu().numpy().astype(bool)
        term_rep[k] = res["terminal_obs"].cpu().numpy()
    assert np.array_equal(tr_rep, trunc)
    assert _same(term, term_rep[rows[live] // n, rows[live] % n])
    # values of the terminal rows within the float32 forward tolerance of the float64 tower
    x64 = torch.from_numpy((term if aff is None else _norm_rows(term, aff)).astype(np.float64))
    v64 = po.forward(theta.cpu().double(), x64)[1].numpy()
    assert np.abs(v - v64).max() <= 1e-4 * (1 + np.abs(v64).max())
    for m in (on, off):
        m.close()
        m.batch.close()
    rep.close()


# ---------------------------------------------------------------------------------------------------------------------
# the entry points directly: slot edge cases and argument checks
# ---------------------------------------------------------------------------------------------------------------------
def _raw_rollout(theta, batch, K, slots, kernel, det=1, aff=None, buf_obs=None):
    from drone_rl_b200 import _lib
    from drone_rl_b200._lib import PolicyOut, TimeoutBuf
    n = batch.n
    e = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device="cuda")  # noqa: E731
    r = {"obs": e(K, n, 15), "actions": e(K, n, 4), "logp": e(K, n), "value": e(K, n), "reward": e(K, n),
         "done": e(K, n, dt=torch.uint8), "last_value": e(n)}
    P = lambda t: t.data_ptr()  # noqa: E731
    out = PolicyOut(P(r["obs"]), P(r["actions"]), P(r["logp"]), P(r["value"]), P(r["reward"]), P(r["done"]),
                    P(r["last_value"]), None, 0, 0)
    r["tobs"] = torch.full((slots, n, 16), 7.0, device="cuda") if buf_obs is None else buf_obs
    r["trow"] = torch.full((slots, n), -5, dtype=torch.int32, device="cuda")
    tb = TimeoutBuf(P(r["tobs"]), P(r["trow"]), slots)
    rc = batch.lib.dronecu_rollout_policy_timeouts(batch._h, K, C.c_void_p(theta.data_ptr()), det, C.byref(out),
                                                   None if aff is None else C.c_void_p(aff.data_ptr()), int(kernel == "tc"),
                                                   C.byref(tb), None)
    torch.cuda.synchronize()
    r["rc"], r["tb"] = rc, tb
    if rc == 0:
        r["reward0"] = r["reward"].clone()
        _lib.check(batch.lib.dronecu_bootstrap_timeouts(0, C.c_void_p(theta.data_ptr()), C.byref(tb), n, None, C.c_float(0.99),
                                                        C.c_void_p(r["reward"].data_ptr()), None))
        torch.cuda.synchronize()
    return r


@pytest.mark.parametrize("kernel", KERNELS)
def test_every_slot_filled_and_spare_slots_read_minus_one(drl, kernel_mode, kernel):
    """K a multiple of max_steps and every env one step before the limit: truncations at k = 0, 7, ..., K - 7 fill all T
    slots; with two spare slots those read -1.  K = 22 adds a truncation at k = K - 1 = 21."""
    theta = _theta()
    kernel_mode(kernel)
    n = 300 if kernel != "tc" else 1000
    for K, extra in ((21, 0), (21, 2), (22, 0)):
        b = drl.DroneBatch(n, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=9)
        b.reset()
        b.set_state(step=np.full(n, MAX_STEPS - 1, np.int32), ep_len=np.full(n, MAX_STEPS - 1, np.int32))
        T = -(-K // MAX_STEPS)
        r = _raw_rollout(theta, b, K, T + extra, kernel)
        assert r["rc"] == 0
        rows = r["trow"].cpu().numpy()
        done = r["done"].cpu().numpy().astype(bool)
        full = np.all(rows[:T] >= 0, axis=0)
        assert full.mean() > 0.9                                      # hover: nearly every env reaches every limit
        want = np.arange(0, K, MAX_STEPS)[:, None] * n + np.arange(n)[None]
        assert np.array_equal(rows[:T][:, full], want[:, full])
        assert (rows[T:] == -1).all()
        if K == 22:
            assert done[K - 1][full].all()
        r0, r1 = r["reward0"].cpu().numpy(), r["reward"].cpu().numpy()
        live = rows >= 0
        k, i = rows[live] // n, rows[live] % n
        term = r["tobs"].cpu().numpy()[live][:, :15]
        assert _same(r1[k, i], _expr(r0[k, i], _forward_value(theta, term), 0.99))
        mask = np.ones_like(r0, bool)
        mask[k, i] = False
        assert _same(r1[mask], r0[mask])
        b.close()


def test_too_few_slots_and_bad_buffers_are_rejected(drl):
    from drone_rl_b200._lib import TimeoutBuf
    theta = _theta()
    n, K = 64, 15
    b = drl.DroneBatch(n, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=1)
    b.reset()
    st0 = b.get_state()
    r = _raw_rollout(theta, b, K, 2, "warp")                # ceil(15 / 7) = 3
    assert r["rc"] == -1
    assert np.array_equal(b.get_state()["pos"], st0["pos"]), "a rejected launch must not step the envs"
    base = torch.empty(3 * n * 16 + 1, device="cuda")
    r = _raw_rollout(theta, b, K, 3, "warp", buf_obs=base[1:].view(3, n, 16))    # 4-byte aligned only
    assert r["rc"] == -1
    lib = b.lib
    th = C.c_void_p(theta.data_ptr())
    rew = torch.zeros(K, n, device="cuda")
    tb = TimeoutBuf(None, None, 3)
    assert lib.dronecu_bootstrap_timeouts(0, th, C.byref(tb), n, None, C.c_float(0.99), C.c_void_p(rew.data_ptr()), None) == -1
    assert lib.dronecu_bootstrap_timeouts(0, th, None, n, None, C.c_float(0.99), C.c_void_p(rew.data_ptr()), None) == -1
    b.close()


@pytest.mark.parametrize("kernel", KERNELS)
def test_non_finite_terminal_row_gives_nan_reward(drl, kernel_mode, kernel):
    """body rates of 3e19 rad/s make the state inf, then NaN; NaN compares false, so those envs are never 'crashed' and
    truncate at the limit with a NaN terminal row: V is NaN and so is the reward, as SB3's expression gives"""
    theta = _theta()
    kernel_mode(kernel)
    n, K = (1000 if kernel == "tc" else 128), 9
    b = drl.DroneBatch(n, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=4)
    b.reset()
    om = np.zeros((n, 3), np.float32)
    om[::4] = 3e19
    b.set_state(omega=om, step=np.full(n, 2, np.int32), ep_len=np.full(n, 2, np.int32))
    r = _raw_rollout(theta, b, K, 2, kernel)
    assert r["rc"] == 0
    rows = r["trow"].cpu().numpy()
    live = rows >= 0
    k, i = rows[live] // n, rows[live] % n
    term = r["tobs"].cpu().numpy()[live][:, :15]
    bad = ~np.isfinite(term).all(1)
    assert bad.any() and (i[bad] % 4 == 0).all()
    r0, r1 = r["reward0"].cpu().numpy(), r["reward"].cpu().numpy()
    v = _forward_value(theta, term)
    assert _same(r1[k, i], _expr(r0[k, i], v, 0.99))
    assert np.isnan(r1[k[np.isnan(v)], i[np.isnan(v)]]).all() and np.isnan(v[np.isnan(term).any(1)]).all()
    b.close()


# ---------------------------------------------------------------------------------------------------------------------
# the training loop, teacher-forced per rollout, and the flag through checkpoints and train.py
# ---------------------------------------------------------------------------------------------------------------------
def _sync(dst, src):
    """give the flag-off model the flag-on model's parameters, env state, clock and normaliser before a rollout"""
    dst.params.copy_(src.params)
    dst.batch.set_state(**src.batch.get_state())
    dst.batch.global_step = src.batch.global_step
    if src.normalizer is not None:
        dst.normalizer.stats.copy_(src.normalizer.stats)
        dst.normalizer.affine.copy_(src.normalizer.affine)
        dst.normalizer.returns.copy_(src.normalizer.returns)
        dst.normalizer.training = src.normalizer.training


@pytest.mark.parametrize("shape", [(257, 32, "fp32"), (2048, 16, "tf32")], ids=["n257-K32-fp32", "n2048-K16-tf32"])
@pytest.mark.parametrize("mode", [(0, 0), (1, 0), (1, 1)], ids=["raw", "obs", "both"])
def test_ppo_loop_follows_the_oracle_with_bootstrap(drl, shape, mode):
    """Per rollout (train, train, evaluate, train): the flag-on buffer rewards equal the flag-off rewards of the same rollout
    plus the pinned bootstrap of dronecu_policy_forward's value, and that value is within the float32 forward tolerance of
    the float64 oracle tower on the same normalised row."""
    from drone_rl_b200.ppo import PPO
    n, K, prec = shape
    kw = dict(n_steps=K, batch_size=min(n * K, 4096), n_epochs=1, gamma=0.95, seed=6, rollout_precision=prec,
              norm_obs=bool(mode[0]), norm_reward=bool(mode[1]), clip_obs=5.0, clip_reward=3.0, norm_epsilon=1e-3)
    mk = lambda flag: PPO(drl.DroneBatch(n, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=6),  # noqa: E731
                          handle_timeout_termination=flag, **kw)
    on, off = mk(True), mk(False)
    _mid_episode(on.batch, 6)
    worst = 0.0
    for it, training in enumerate((True, True, False, True)):
        on.training = training
        _sync(off, on)
        aff = on.normalizer.affine.cpu().numpy() if mode[0] else None
        on.collect_rollouts()
        off.collect_rollouts()
        torch.cuda.synchronize()
        rows = on.timeout_row.cpu().numpy()
        live = rows >= 0
        assert live.sum() > 0, f"iteration {it}: the 7-step limit must be reached"
        k, i = rows[live] // n, rows[live] % n
        term = on.timeout_obs.cpu().numpy()[live][:, :15]
        x = term if aff is None else _norm_rows(term, aff)
        v = _forward_value(on.params, x)
        r_on, r_off = on.buf.reward.cpu().numpy(), off.buf.reward.cpu().numpy()
        ref = r_off.copy()
        ref[k, i] = _expr(r_off[k, i], v, on.gamma)
        assert _same(r_on, ref), f"rewards, iteration {it}"
        v64 = po.forward(on.params.cpu().double(), torch.from_numpy(x.astype(np.float64)))[1].numpy()
        err = np.abs(v - v64).max() / (1e-4 * (1 + np.abs(v64).max()))
        worst = max(worst, float(err))
        assert err <= 1.0
        on.train()
    print(f"n {n} K {K} {prec} mode {mode}: worst value err / tolerance {worst:.3g}")
    for m in (on, off):
        m.close()


def test_flag_round_trips_through_checkpoints_and_train_py(drl, tmp_path, monkeypatch):
    from drone_rl_b200.ppo import PPO
    from drone_rl_b200 import sb3_zip
    m = PPO(drl.DroneBatch(8, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=2), n_steps=16, batch_size=64, n_epochs=1,
            handle_timeout_termination=True)
    assert m.state_dict()["handle_timeout_termination"] is True
    for suffix in (".zip", ".pt"):
        path = str(tmp_path / f"m{suffix}")
        m.save(path)
        a = PPO.load(path, drl.DroneBatch(8, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=2))
        assert a.handle_timeout_termination and a.timeout_row is not None
        b = PPO.load(path, drl.DroneBatch(8, drl.EnvConfig.single(max_steps=MAX_STEPS), seed=2), handle_timeout_termination=False)
        assert not b.handle_timeout_termination and b.timeout_row is None
        a.close()
        b.close()
    assert sb3_zip.import_zip(str(tmp_path / "m.zip"))["hyper"]["handle_timeout_termination"] is True
    m.close()
    # train.py: the flag reaches the model and the archive
    from drone_rl_b200 import train
    monkeypatch.chdir(tmp_path)
    seen = {}
    orig = PPO.__init__

    def spy(self, *a, **k):
        seen.update(k)
        orig(self, *a, **k)
    monkeypatch.setattr(PPO, "__init__", spy)
    train.main(["--handle-timeout-termination", "--total-timesteps", "64", "--n-envs", "4", "--n-steps", "16", "--n-epochs",
                "1", "--save", str(tmp_path / "t"), "--resume", str(tmp_path / "none.zip"), "--quiet",
                "--tensorboard-root", str(tmp_path / "tb")])
    assert seen.get("handle_timeout_termination") is True
    assert sb3_zip.import_zip(str(tmp_path / "t.zip"))["hyper"]["handle_timeout_termination"] is True
