"""GPU parity tests: the CUDA env (through the C ABI / its Python mirror) against the oracle
and the golden vectors generated from the unmodified reference.

Tolerance (north-star: "<= 1e-5 relative per step" for state, obs, reward; bit-exact for
done / reset / indexing), teacher-forced -- both sides start every compared step from the
SAME float32-representable state and action, the oracle continues in float64:

    |gpu - ref| <= 1e-5 * max(|ref|, 1)                 (TOL_REL, unit floor)

with two documented carve-outs (SURVEY.md section 7 "hard parts"):
  * rows with |cos(pitch)| < 1e-3: tan/sec amplify a 1-ulp float32 difference in cos(pitch)
    by 1/cos^2; there roll/yaw are checked with the bound scaled by 1/cos(pitch)^2.
  * |angle| > 1e4 rad: sincosf of a float32 angle is exact to 2 ulp of the RESULT, the
    comparison is still against the float64 sin of the same float32 angle, so no carve-out
    is needed -- it is covered.
Done flags are compared wherever the float64 margin to a threshold exceeds the float32
rounding of the compared quantity; the remaining (borderline) rows are counted and must be rare.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import drone_oracle as do  # noqa: E402
from oracle import philox  # noqa: E402

TOL_REL = 1e-5
np.seterr(all="ignore")


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    return drone_rl_b200


def _cfg(drl, spec):
    return drl.EnvConfig.single() if spec is do.SINGLE else drl.EnvConfig.vector()


def _tf_step(drl, spec, pos, vel, euler, omega, target, action, step_count, auto_reset=None, seed=0, ep_num=None):
    """Teacher-forced single step on GPU and oracle from the same f32 state."""
    n = pos.shape[0]
    cfg = _cfg(drl, spec)
    if auto_reset is not None:
        cfg.auto_reset = auto_reset
    b = drl.DroneBatch(n, cfg, seed=seed)
    kw = dict(pos=pos, vel=vel, euler=euler, omega=omega, step=step_count, ep_len=step_count,
              ep_ret=np.zeros(n, np.float32))
    if spec is do.SINGLE:
        kw["target"] = target
    if ep_num is not None:
        kw["ep_num"] = ep_num
    b.set_state(**kw)
    act = torch.from_numpy(np.ascontiguousarray(action)).to(b.device)
    out = b.step(act, want_truncated=True, want_terminal_obs=True, want_episode=True)
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["state"] = b.get_state()

    spec_o = spec if auto_reset is None else do.Spec(spec.name, spec.obs_dim, spec.max_steps, spec.bonus_radius,
                                                     spec.curriculum, spec.random_start, spec.shared_step, auto_reset)
    o = do.BatchedDroneOracle(n, spec_o, seed=seed)
    o.set_state(pos, vel, euler, omega, target if spec is do.SINGLE else None, step_count=step_count, ep_num=ep_num)
    o.ep_length[:] = step_count
    o.ep_return[:] = 0
    obs, rew, done, info = o.step(action)
    b.close()
    return res, dict(obs=obs, reward=rew, done=done, info=info, env=o)


def _assert_close(got, ref, scale=1.0, what=""):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), f"{what}: NaN pattern differs"
    inf = np.isinf(ref)
    assert np.array_equal(got[inf], ref[inf]), f"{what}: inf pattern differs"
    ok = np.isfinite(ref)
    err = np.abs(got[ok] - ref[ok])
    bound = TOL_REL * np.maximum(np.abs(ref[ok]), 1.0) * (scale[ok] if isinstance(scale, np.ndarray) else scale)
    bad = err > bound
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} outside tolerance, worst ratio {np.max(err / bound):.3g}"
    return float(np.max(err / bound)) if err.size else 0.0


def _done_margin_ok(o_env, spec):
    """rows whose done decision is not within float32 rounding of a threshold."""
    z = o_env.pos[:, 2]
    rad = np.linalg.norm(o_env.pos, axis=1)
    return (np.abs(z) > 1e-5 * np.maximum(1.0, np.abs(z))) & (np.abs(rad - 50.0) > 1e-4) | ~np.isfinite(rad)


@pytest.mark.parametrize("spec", [do.SINGLE, do.VECTOR], ids=["single", "vector"])
def test_teacher_forced_golden(drl, golden, spec):
    """2048 one-step cases incl. crash / out-of-range / bonus / near-singular pitch / NaN / inf /
    huge angles / unclipped actions / time limit -- against the unmodified reference's outputs."""
    g = golden("teacher_forced")
    n = g["pos"].shape[0]
    res, orc = _tf_step(drl, spec, g["pos"], g["vel"], g["euler"], g["omega"], g["target"], g["action"],
                        g["step_count"], auto_reset=False)
    if spec is do.VECTOR:
        ref_state = np.concatenate([g["vec_pos"], g["vec_vel"], g["vec_euler"], g["vec_omega"]], 1)
        ref_rew, ref_done = g["vec_reward"], g["vec_done"]
        # shared counter: the golden ran at current_step 0 -> 1; ours ran at step_count+1 < 1000
    else:
        ref_state = g["single_state"]
        ref_rew, ref_done = g["single_reward"], g["single_done"]
    st = res["state"]
    got_state = np.concatenate([st["pos"], st["vel"], st["euler"], st["omega"]], 1)

    cosp = np.cos(g["euler"][:, 1].astype(np.float64))
    amp = np.ones((n, 12))
    sing = np.abs(cosp) < 1e-3
    amp[sing, 6] = amp[sing, 8] = 1.0 / cosp[sing] ** 2          # roll, yaw rates carry tan / sec
    worst = _assert_close(got_state, ref_state, amp, "state")
    # reward: |d reward| = 0.01 |d dist|
    _assert_close(res["reward"], ref_rew, 1.0, "reward")
    # observation == float32(state) (+ target - pos)
    margin = _done_margin_ok(orc["env"], spec)
    both = ref_done & res["done"].astype(bool)
    _assert_close(res["terminal_obs"][both][:, :12], ref_state[both], amp[both], "terminal_obs")
    assert margin.mean() > 0.995
    assert np.array_equal(res["done"].astype(bool)[margin], ref_done[margin])
    if spec is do.SINGLE:
        assert res["done"].astype(bool)[g["step_count"] == 199].all()
        trunc = res["truncated"].astype(bool)
        assert np.array_equal(trunc[margin], orc["info"]["truncated"][margin])
    print(f"[{spec.name}] worst err/bound = {worst:.3f}")


def test_nan_inf_semantics(drl, golden):
    """NaN position never 'crashes' (drone.py:154), 0*inf -> NaN in the Euler-rate / body-rate
    terms (drone.py:138,181-186): identical non-finite pattern and done bits."""
    g = golden("teacher_forced")
    rows = np.flatnonzero(~np.isfinite(g["single_state"]).all(1) | ~np.isfinite(g["pos"]).all(1)
                          | ~np.isfinite(g["euler"]).all(1) | ~np.isfinite(g["omega"]).all(1))
    assert rows.size >= 3
    sel = lambda a: np.ascontiguousarray(a[rows])
    res, _ = _tf_step(drl, do.SINGLE, sel(g["pos"]), sel(g["vel"]), sel(g["euler"]), sel(g["omega"]), sel(g["target"]),
                      sel(g["action"]), sel(g["step_count"]), auto_reset=False)
    st = res["state"]
    got = np.concatenate([st["pos"], st["vel"], st["euler"], st["omega"]], 1)
    assert np.array_equal(np.isnan(got), np.isnan(g["single_state"][rows]))
    assert np.array_equal(res["done"].astype(bool), g["single_done"][rows])
    assert np.array_equal(np.isnan(res["reward"]), np.isnan(g["single_reward"][rows]))


def _teacher_forced_trajectory(drl, spec, actions, seed, env_offset, n):
    """Walk the oracle's float64 trajectory; at every step restart the GPU (and a float64 shadow
    oracle) from the float32 rounding of the trajectory state and compare one step."""
    cfg = _cfg(drl, spec)
    gpu = drl.DroneBatch(n, cfg, seed=seed, env_offset=env_offset)
    traj = do.BatchedDroneOracle(n, spec, seed=seed, env_offset=env_offset)
    shadow = do.BatchedDroneOracle(n, spec, seed=seed, env_offset=env_offset)
    obs_g = gpu.reset().cpu().numpy()
    obs_o = traj.reset()
    assert np.array_equal(obs_g, obs_o), "reset observation must be bit-identical"
    worst, n_border, n_done = 0.0, 0, 0
    f32 = lambda a: a.astype(np.float32)
    for t in range(actions.shape[0]):
        st = dict(pos=f32(traj.pos), vel=f32(traj.vel), euler=f32(traj.euler), omega=f32(traj.omega),
                  target=f32(traj.target))
        gpu.set_state(step=traj.step_count.astype(np.int32), ep_num=traj.ep_num.astype(np.int32),
                      ep_len=traj.ep_length.astype(np.int32), ep_ret=traj.ep_return.copy(), **st)
        shadow.set_state(st["pos"], st["vel"], st["euler"], st["omega"], st["target"],
                         step_count=traj.step_count, ep_num=traj.ep_num)
        shadow.ep_length[:] = traj.ep_length
        shadow.ep_return[:] = traj.ep_return
        a = actions[t]
        out = gpu.step(torch.from_numpy(a).to(gpu.device), want_truncated=True, want_terminal_obs=True, want_episode=True)
        res = {k: v.cpu().numpy() for k, v in out.items()}
        obs, rew, done, info = shadow.step(a)
        margin = _done_margin_ok_from(info["terminal_obs"])
        n_border += int((~margin).sum())
        d_g = res["done"].astype(bool)
        assert np.array_equal(d_g[margin], done[margin]), f"step {t}"
        same = d_g == done
        worst = max(worst, _assert_close(res["reward"][same], rew[same], 1.0, f"reward t={t}"))
        # post-reset observation of done rows is bit-exact (start position / target from Philox);
        # other rows follow the tolerance
        both_done = same & done
        live = same & ~done
        worst = max(worst, _assert_close(res["obs"][live], obs[live], 1.0, f"obs t={t}"))
        if both_done.any():
            n_done += int(both_done.sum())
            if spec.auto_reset:
                assert np.array_equal(res["obs"][both_done], obs[both_done]), f"reset obs t={t}"
            _assert_close(res["terminal_obs"][both_done], info["terminal_obs"][both_done], 1.0, f"terminal t={t}")
            assert np.array_equal(res["episode_l"][both_done], info["episode_l"][both_done])
            _assert_close(res["episode_r"][both_done], info["episode_r"][both_done], 1.0, f"episode_r t={t}")
            assert np.array_equal(res["truncated"].astype(bool)[both_done], info["truncated"][both_done])
        traj.step(a)
    gpu.close()
    return worst, n_border, n_done


def _done_margin_ok_from(term_obs):
    z = term_obs[:, 2].astype(np.float64)
    rad = np.linalg.norm(term_obs[:, :3].astype(np.float64), axis=1)
    return ((np.abs(z) > 1e-5) & (np.abs(rad - 50.0) > 1e-4)) | ~np.isfinite(rad)


def test_golden_single_rollout_teacher_forced(drl, golden):
    """The 8-env / 400-step DummyVecEnv+VecMonitor rollout generated from the real reference."""
    g = golden("single_rollout")
    T, n = g["actions"].shape[:2]
    worst, n_border, n_done = _teacher_forced_trajectory(drl, do.SINGLE, g["actions"], int(g["seed"]),
                                                         int(g["env_offset"]), n)
    assert n_done >= 50 and n_border <= 2
    print(f"single rollout: worst err/bound {worst:.3f}, dones {n_done}, borderline {n_border}")


def test_golden_vector_rollout_teacher_forced(drl, golden):
    g = golden("vector_rollout")
    T, n = g["actions"].shape[:2]
    worst, n_border, n_done = _teacher_forced_trajectory(drl, do.VECTOR, g["actions"], 0, 0, n)
    assert n_border <= 4
    print(f"vector rollout: worst err/bound {worst:.3f}, borderline {n_border}")


def test_const_action_demo_open_loop(drl, golden):
    """drone.py:288-294 demo, open loop on the GPU: vertical climb is not chaotic, so the whole
    158-step float32 trajectory stays within 1e-5 relative and terminates at the same step."""
    g = golden("single_const_action")
    env = drl.DroneGymEnv(seed=int(g["seed"]), env_id=int(g["env_id"]))
    obs0 = env.reset()
    assert np.array_equal(obs0, g["obs0"])
    for t in range(g["obs"].shape[0]):
        obs, rew, done, info = env.step(g["action"])
        np.testing.assert_allclose(obs, g["obs"][t], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(rew, g["reward"][t], rtol=1e-5, atol=1e-6)
        assert done == bool(g["done"][t]), t
        assert obs.dtype == np.float32 and isinstance(rew, float) and isinstance(done, bool) and info == {}
    assert done and t == 157
    env.close()


def test_rollout_equals_repeated_step(drl):
    """K fused steps in one launch == K single-step launches, bit for bit (state stays in registers)."""
    n, K = 5000, 37        # ragged: not a multiple of 256 / 32 / 4
    rng = np.random.default_rng(0)
    acts = rng.uniform(0, 7.3575, (K, n, 4)).astype(np.float32)
    a_dev = torch.from_numpy(acts).cuda()
    b1 = drl.DroneBatch(n, drl.EnvConfig.single(), seed=3)
    b2 = drl.DroneBatch(n, drl.EnvConfig.single(), seed=3)
    obs0 = b1.empty(n, 15); nxt = b1.empty(K, n, 15); rew = b1.empty(K, n)
    done = b1.empty(K, n, dtype=torch.uint8); trunc = b1.empty(K, n, dtype=torch.uint8)
    b1.rollout(K, a_dev, obs0=obs0, next_obs=nxt, reward=rew, done=done, truncated=trunc)
    assert torch.equal(obs0, b2.reset(mask=torch.zeros(n, dtype=torch.uint8, device="cuda")))
    for k in range(K):
        out = b2.step(a_dev[k], want_truncated=True)
        assert torch.equal(out["obs"], nxt[k]), k
        assert torch.equal(out["reward"], rew[k]) and torch.equal(out["done"], done[k])
        assert torch.equal(out["truncated"], trunc[k])
    s1, s2 = b1.get_state(), b2.get_state()
    for k in s1:
        assert np.array_equal(s1[k], s2[k], equal_nan=True), k
    e1, e2 = b1.episode_stats(), b2.episode_stats()
    assert e1["episodes"] == e2["episodes"] == int(done.sum().item()) > 0
    assert e1["length_sum"] == e2["length_sum"] and e1["env_steps"] == n * K
    b1.close(); b2.close()


def test_shard_invariance(drl):
    """Results depend on the GLOBAL env id only: one handle over [0,n) == two handles over
    [0,n/2), [n/2,n) (what 2 GPUs would hold), incl. Philox actions and resets."""
    n, K = 3000, 64
    whole = drl.DroneBatch(n, drl.EnvConfig.single(), seed=11, env_offset=1 << 33)
    parts = [drl.DroneBatch(1000, drl.EnvConfig.single(), seed=11, env_offset=(1 << 33)),
             drl.DroneBatch(2000, drl.EnvConfig.single(), seed=11, env_offset=(1 << 33) + 1000)]
    outs = []
    for b in [whole] + parts:
        nxt = b.empty(K, b.n, 15); act = b.empty(K, b.n, 4); dn = b.empty(K, b.n, dtype=torch.uint8)
        b.rollout(K, None, next_obs=nxt, out_actions=act, done=dn)
        outs.append((nxt.cpu(), act.cpu(), dn.cpu()))
    for j in range(3):
        assert torch.equal(outs[0][j], torch.cat([outs[1][j], outs[2][j]], dim=1))
    assert outs[0][2].sum() > 0
    for b in [whole] + parts:
        b.close()


def test_philox_actions_and_resets_bit_exact(drl):
    """In-kernel Philox == oracle/philox.py: random-policy actions and reset draws are bit-identical."""
    n, K, seed, off = 777, 5, 2**40 + 17, 123456789012
    b = drl.DroneBatch(n, drl.EnvConfig.single(), seed=seed, env_offset=off)
    st = b.get_state()
    ids = np.arange(off, off + n, dtype=np.uint64)
    u = philox.reset_uniforms(seed, ids, np.ones(n, np.uint64))
    assert np.array_equal(st["pos"][:, 0], (u[0] - 0.5).astype(np.float32))
    assert np.array_equal(st["pos"][:, 1], (u[1] - 0.5).astype(np.float32))
    assert (st["pos"][:, 2] == 1).all() and (st["ep_num"] == 1).all()
    assert np.array_equal(st["target"], np.tile(np.float32([0, 0, 1]), (n, 1)))     # eps == 0
    act = b.empty(K, n, 4)
    b.rollout(K, None, out_actions=act)
    for k in range(K):
        ref = (philox.action_uniforms(seed, ids, k).astype(np.float32) * np.float32(7.3575))
        assert np.array_equal(act[k].cpu().numpy(), ref), k
    assert b.global_step == K
    b.close()


def test_curriculum_targets_bit_exact(drl, golden):
    """eps schedule (drone.py:68-73): after the reset that makes ep_num 2000 / 4000 / 6000 the
    target is float32(eps * u) with eps accumulated in float64 -- equal to the reference's values."""
    g = golden("curriculum")
    seed, env_id = int(g["seed"]), int(g["env_id"])
    b = drl.DroneBatch(1, drl.EnvConfig.single(auto_reset=False), seed=seed, env_offset=env_id)
    for k, ep in enumerate(g["ep_num"]):
        b.set_state(ep_num=np.int32([ep - 1]))
        b.reset()
        st = b.get_state("pos", "target", "ep_num")
        assert st["ep_num"][0] == ep
        assert np.array_equal(st["pos"][0], g["pos"][k].astype(np.float32))
        assert np.array_equal(st["target"][0], g["target"][k].astype(np.float32)), ep
    b.close()


def test_vecenv_surface(drl):
    """SB3 VecEnv duck-type: shapes, dtypes, infos with terminal_observation / episode, get_attr."""
    n = 16
    env = drl.DroneVecEnv(n, seed=5)
    assert env.num_envs == n and env.observation_space.shape == (15,) and env.action_space.shape == (4,)
    assert np.isclose(env.action_space.high[0], 7.3575)
    obs = env.reset()
    assert obs.shape == (n, 15) and obs.dtype == np.float32
    rng = np.random.default_rng(0)
    seen_done = 0
    for t in range(120):
        a = rng.uniform(0, 7.3575, (n, 4)).astype(np.float32)
        env.step_async(a)
        obs, rew, done, infos = env.step_wait()
        assert rew.dtype == np.float32 and done.dtype == np.bool_ and len(infos) == n
        for i in np.flatnonzero(done):
            seen_done += 1
            assert infos[i]["terminal_observation"].shape == (15,)
            assert infos[i]["episode"]["l"] >= 1 and "r" in infos[i]["episode"]
            assert "TimeLimit.truncated" not in infos[i]
            # fresh episode: zero velocity, z = 1
            assert obs[i, 2] == 1.0 and (obs[i, 3:12] == 0).all()
    assert seen_done > 10
    pos = env.get_attr("pos")
    assert len(pos) == n and pos[0].shape == (3,)
    assert env.get_attr("mass") == [1.0] * n and env.env_is_wrapped(object) == [False] * n
    st = env.episode_stats()
    assert st["episodes"] == seen_done
    env.close()


def test_vectorized_gym_env_surface(drl, golden):
    """VectorizedDroneGymEnv: numpy in/out with the reference's dtypes; hover env stays put and
    the shared 1000-step limit flips every done flag (vectorized_drone.py:212-213)."""
    B = 8
    env = drl.VectorizedDroneGymEnv(batch_size=B)
    obs = env.reset()
    assert obs.shape == (B, 12) and obs.dtype == np.float32
    assert np.allclose(obs[:, :3], 0.1) and (obs[:, 3:] == 0).all()
    hover = np.full((B, 4), 9.81 / 4, np.float32)
    for t in range(1000):
        obs, rew, done, info = env.step(hover)
        if t < 999:
            assert not done.any()
    assert done.all() and rew.dtype == np.float64 and done.dtype == np.bool_ and info == {}
    assert env.current_step == 1000
    env.close()


def test_gymnasium_surface(drl):
    env = drl.DroneGymnasiumEnv()
    obs, info = env.reset(seed=3)
    assert obs.shape == (15,) and info == {}
    term = trunc = False
    steps = 0
    while not (term or trunc):
        obs, r, term, trunc, info = env.step(np.full(4, 9.81 / 4 * 1.0005, np.float32))
        steps += 1
    assert steps == 200 and trunc and not term        # gentle climb: only the time limit ends it
    env.close()


def test_errors_are_loud(drl):
    b = drl.DroneBatch(8)
    with pytest.raises(ValueError):
        b.step(torch.zeros(8, 4))                       # CPU tensor
    with pytest.raises(ValueError):
        b.step(torch.zeros(7, 4, device="cuda"))
    with pytest.raises(drl.DronecuError):
        drl.DroneBatch(0)
    with pytest.raises(drl.DronecuError):
        drl.DroneBatch(4, drl.EnvConfig.single(obs_dim=13))
    b.close()


def test_full_size_rollout_properties(drl):
    """BASELINE size (1M envs, the C3 batch): K-fusion invariance, shard invariance and episode
    bookkeeping at full size, plus every transition of a strided 4k-env sample checked against the
    float64 oracle teacher-forced from the record (oracle/verify.py)."""
    from oracle import verify
    n, K, seed = 1 << 20, 40, 5          # episodes last ~32 steps under random actions (SURVEY section 6)
    b = drl.DroneBatch(n, drl.EnvConfig.single(), seed=seed)
    obs0 = b.reset()
    nxt = b.empty(K, n, 15); act = b.empty(K, n, 4); rew = b.empty(K, n); done = b.empty(K, n, dtype=torch.uint8)
    b.rollout(K, None, next_obs=nxt, out_actions=act, reward=rew, done=done)
    st = b.episode_stats()
    assert st["episodes"] == int(done.sum().item()) and st["env_steps"] == n * K
    sel = torch.arange(0, n, 257, device="cuda")
    rep = verify.check_rollout(obs0[sel].cpu().numpy(), act[:, sel].cpu().numpy(), nxt[:, sel].cpu().numpy(),
                               rew[:, sel].cpu().numpy(), done[:, sel].cpu().numpy().astype(bool),
                               spec=do.SINGLE, seed=seed, env_ids=sel.cpu().numpy())
    assert rep["dones"] > 100 and rep["borderline_done"] <= 3
    # same global ids from a second handle covering only the tail quarter, in two launches
    q = n // 4
    b2 = drl.DroneBatch(q, drl.EnvConfig.single(), seed=seed, env_offset=3 * q)
    b2.reset()
    nxt2 = b2.empty(K, q, 15)
    b2.rollout(K // 2, None, next_obs=nxt2[: K // 2])
    b2.rollout(K - K // 2, None, next_obs=nxt2[K // 2:])
    assert torch.equal(nxt2, nxt[:, 3 * q:])
    print("full-size:", rep)
    b.close(); b2.close()


def test_chunked_host_step_equals_device_step(drl):
    """dronecu_step_host cuts large batches into 1M-env chunks on two streams (H2D / kernel / D2H
    overlap); the result must be bit-identical to the single device-pointer launch, ragged tail included.
    Both specs, the 15-dim auto-resetting one and the 12-dim fixed-start one, 2 steps short of their time
    limit, so the chunks carry timeouts with and without a reset."""
    n = (1 << 21) + 1000
    rng = np.random.default_rng(3)
    acts = rng.uniform(0, 7.3575, (n, 4)).astype(np.float32)
    a_dev = torch.from_numpy(acts).cuda()
    for cfg in (drl.EnvConfig.single(), drl.EnvConfig.vector()):
        venv = drl.DroneVecEnv(n, seed=9, info_mode="arrays", copy=False, config=cfg)
        ref = drl.DroneBatch(n, cfg, seed=9)
        o_h = venv.reset().copy()
        o_d = ref.reset()
        assert np.array_equal(o_h, o_d.cpu().numpy())
        for b in (venv.batch, ref):
            b.set_state(step=np.full(n, cfg.max_steps - 2, np.int32))
        n_done = 0
        for _ in range(3):
            obs, rew, done, info = venv.step(acts)
            out = ref.step(a_dev, want_truncated=True)
            assert np.array_equal(obs, out["obs"].cpu().numpy())
            assert np.array_equal(rew, out["reward"].cpu().numpy())
            assert np.array_equal(done, out["done"].cpu().numpy().astype(bool))
            assert np.array_equal(info["truncated"], out["truncated"].cpu().numpy().astype(bool))
            n_done += int(done.sum())
        assert n_done > 0
        assert venv.batch.global_step == ref.global_step == 3
        assert venv.episode_stats()["env_steps"] == 3 * n
        assert venv.episode_stats()["episodes"] == ref.episode_stats()["episodes"] == n_done
        venv.close(); ref.close()


@pytest.mark.parametrize("scale", [1.0, 50.0, 3e3, 1.0e5, 1.056e5, 1.0e7, 5.0e8, 1.05e9, 3.0e9, 1.0e15])
def test_euler_angle_range_of_sincos(drl, scale):
    """The kernel's own sin/cos of the three Euler angles (float Cody-Waite by pi/2 below 105615 rad, float64 Cody-Waite
    up to 2^30, libm above) against the float64 oracle, teacher-forced, for angles from +-1 rad up to +-1e7 rad -- the reference
    never wraps its angles (drone.py:131), so every magnitude a long episode can reach must stay within 1e-5
    relative.  Mixed rows (one angle above the fast-path limit, two below) exercise the shared range check."""
    rng = np.random.default_rng(int(scale) % 9973)
    n = 8192
    pos = rng.uniform(-5, 5, (n, 3)).astype(np.float32); pos[:, 2] = np.abs(pos[:, 2]) + 1
    vel = rng.uniform(-3, 3, (n, 3)).astype(np.float32)
    euler = (rng.uniform(-1, 1, (n, 3)) * scale).astype(np.float32)
    euler[::7, rng.integers(0, 3)] *= 0.01                    # mixed magnitudes within a row
    # keep pitch away from the tan / sec singularity: the amplification there is covered by the golden cases
    c = np.cos(euler[:, 1].astype(np.float64))
    euler[np.abs(c) < 0.05, 1] += np.float32(0.3)
    omega = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
    target = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    action = rng.uniform(0, 7.3575, (n, 4)).astype(np.float32)
    res, orc = _tf_step(drl, do.SINGLE, pos, vel, euler, omega, target, action, np.zeros(n, np.int32), auto_reset=False)
    st, o = res["state"], orc["env"]
    got = np.concatenate([st["pos"], st["vel"], st["euler"], st["omega"]], 1)
    ref = np.concatenate([o.pos, o.vel, o.euler, o.omega], 1)
    cosp = np.cos(euler[:, 1].astype(np.float64))
    amp = np.ones((n, 12))
    amp[:, 6] = amp[:, 8] = np.maximum(1.0, 1.0 / cosp ** 2)      # roll / yaw rates carry tan / sec of the pitch
    worst = _assert_close(got, ref, amp, f"state at |angle| <= {scale:g}")
    _assert_close(res["reward"], orc["reward"], 1.0, "reward")
    print(f"scale {scale:g}: worst err/bound = {worst:.3f}")


def test_sb3_vecenv_adapter_against_stub_interface(drl, monkeypatch):
    """make_sb3_vec_env builds a genuine subclass of SB3's abstract VecEnv.  stable-baselines3 / gymnasium are not in this
    image, so the abstract interface (SB3's published one) is stubbed: every abstract method must be implemented, the
    constructor arguments are (num_envs, observation_space, action_space), and the step protocol returns SB3's types."""
    import abc
    import sys
    import types
    from drone_rl_b200 import envs

    class VecEnv(abc.ABC):
        def __init__(self, num_envs, observation_space, action_space):
            self.num_envs, self.observation_space, self.action_space = num_envs, observation_space, action_space

        @abc.abstractmethod
        def reset(self): ...
        @abc.abstractmethod
        def step_async(self, actions): ...
        @abc.abstractmethod
        def step_wait(self): ...
        @abc.abstractmethod
        def close(self): ...
        @abc.abstractmethod
        def get_attr(self, attr_name, indices=None): ...
        @abc.abstractmethod
        def set_attr(self, attr_name, value, indices=None): ...
        @abc.abstractmethod
        def env_method(self, method_name, *method_args, indices=None, **method_kwargs): ...
        @abc.abstractmethod
        def env_is_wrapped(self, wrapper_class, indices=None): ...

        def step(self, actions):
            self.step_async(actions)
            return self.step_wait()

    class Box:
        def __init__(self, low, high, shape, dtype):
            self.low, self.high, self.shape, self.dtype = low, high, shape, dtype

    sb3, common, vec = types.ModuleType("stable_baselines3"), types.ModuleType("stable_baselines3.common"), types.ModuleType("stable_baselines3.common.vec_env")
    vec.VecEnv = VecEnv
    gymn, spaces = types.ModuleType("gymnasium"), types.ModuleType("gymnasium.spaces")
    spaces.Box = Box
    gymn.spaces = spaces
    for name, mod in (("stable_baselines3", sb3), ("stable_baselines3.common", common), ("stable_baselines3.common.vec_env", vec),
                      ("gymnasium", gymn), ("gymnasium.spaces", spaces)):
        monkeypatch.setitem(sys.modules, name, mod)
    env = envs.make_sb3_vec_env(64, seed=3)
    assert isinstance(env, VecEnv) and env.num_envs == 64
    assert env.observation_space.shape == (15,) and env.action_space.shape == (4,) and abs(env.action_space.high - 7.3575) < 1e-6
    obs = env.reset()
    assert obs.shape == (64, 15) and obs.dtype == np.float32
    seen = 0
    for _ in range(80):
        obs, rew, done, infos = env.step(np.random.default_rng(0).uniform(0, 7.3575, (64, 4)))   # float64 in, like SB3's clipped actions
        assert rew.dtype == np.float32 and done.dtype == np.bool_ and isinstance(infos, list) and len(infos) == 64
        for i in np.flatnonzero(done):
            assert infos[i]["terminal_observation"].shape == (15,) and {"r", "l", "t"} <= set(infos[i]["episode"])
            seen += 1
    assert seen > 0
    assert len(env.get_attr("pos")) == 64 and env.env_is_wrapped(object) == [False] * 64
    env.close()


def test_render_returns_the_reference_scenes(drl):
    """DroneGymEnv.render / VectorizedDroneGymEnv.render (drone.py:205-248, vectorized_drone.py:218-243): Pillow images of the
    reference's scenes; recording collects one frame per render call."""
    env = drl.DroneGymEnv(seed=1)
    env.reset()
    env.start_record("unused.gif", fps=10)
    for _ in range(3):
        env.step(np.full(4, 2.5, np.float32))
        img = env.render()
    assert img.size == (480, 480) and len(env._recorder.frames) == 3
    px = np.asarray(img).reshape(-1, 3)
    assert bool((px == np.array((220, 0, 0))).all(1).any())           # the drone centre
    env._recorder = None                                              # do not write a file from the test
    env.close()
    venv = drl.VectorizedDroneGymEnv(batch_size=7)
    venv.reset()
    imgb = np.asarray(venv.render()).reshape(-1, 3)
    assert bool((imgb == np.array((0, 160, 0))).all(1).any()) and bool((imgb == np.array((220, 0, 0))).all(1).any())
    venv.close()


def test_vecenv_with_observations_kept_on_the_device(drl):
    """DroneVecEnv(obs_device=True): observations stay on the GPU (a CUDA tensor), rewards / dones arrive as numpy -- the
    same numbers as the numpy protocol, with numpy or CUDA actions."""
    n = 3000
    rng = np.random.default_rng(5)
    host = drl.DroneVecEnv(n, seed=12, info_mode="arrays")
    dev = drl.DroneVecEnv(n, seed=12, info_mode="arrays", obs_device=True)
    dev2 = drl.DroneVecEnv(n, seed=12, info_mode="none", obs_device=True, copy=False)
    o_h, o_d, o_d2 = host.reset(), dev.reset(), dev2.reset()
    assert isinstance(o_d, torch.Tensor) and o_d.is_cuda and np.array_equal(o_h, o_d.cpu().numpy()) and torch.equal(o_d, o_d2)
    n_done = 0
    for _ in range(40):
        a = rng.uniform(0, 7.3575, (n, 4)).astype(np.float32)
        oh, rh, dh, ih = host.step(a)
        od, rd, dd, idv = dev.step(a)
        od2, rd2, dd2, i2 = dev2.step(torch.from_numpy(a).cuda())            # actions already on the device: no copy at all
        assert np.array_equal(oh, od.cpu().numpy()) and np.array_equal(rh, rd) and np.array_equal(dh, dd)
        assert np.array_equal(ih["truncated"], idv["truncated"]) and i2 == {}
        assert torch.equal(od, od2) and np.array_equal(rd, rd2) and np.array_equal(dd, dd2)
        assert rd.dtype == np.float32 and dd.dtype == np.bool_
        n_done += int(dh.sum())
    assert n_done > 100
    with pytest.raises(ValueError):
        drl.DroneVecEnv(4, obs_device=True)                                  # SB3 info dicts need host terminal observations
    for e in (host, dev, dev2):
        e.close()
