"""Every environment kernel -- the 32 instantiations of rollout_kernel<OBS_DIM, RANDOMIZED, AUTORESET, ACT_MODE, RECORD>
and the 4 of reset_kernel<OBS_DIM, RANDOMIZED> (csrc/env_kernels.cuh) -- teacher-forced against float64 over a covering
design of launch shapes, CTA sizes, start states, clocks, output sets, output placements and env constants.  Every level
of every factor appears, and every instantiation meets every level of every other factor (test_env_dispatch.py
restates the dispatch rule of capi_env.cu and asserts it).

Checked in every rollout case:
  transitions         every (step, env), or a strided sample of envs plus the first and last warps at large n, through
                      oracle/verify.check_rollout with the config's constants; reset rows bit-exact
  actions             Philox: bit-exact philox.action_uniforms * motor_max of the config; streamed: the input, bit-exact
  output-set twin     a second handle with the same seed, offset, state and clock runs the full generic output set;
                      every output the case asked for, the final state planes and the counters of the episode statistics
                      are bit-identical to the twin's (return_sum is a double atomicAdd in arrival order: within tolerance)
  state after         step, ep_num, ep_len as the record implies; ep_ret bit-exact by a float32 replay of the rewards
  episode statistics  episodes, length_sum exactly; terminated within the borderline slack of the oracle's crash decisions;
                      truncated = episodes - terminated; return_sum within the float32 rounding of the per-env sums
  stray writes        guard regions around every output keep their sentinel; terminal_obs / episode_r / episode_l are
                      written on done rows only
"""
import dataclasses

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import drone_oracle as do  # noqa: E402
from oracle import philox, verify  # noqa: E402

SEED = 29
NS = (1, 31, 32, 33, 257, 4097, 18943, 18944, 75775, 75776, 1 << 20)
KS = (1, 2, 37, 256)
STARTS = ("fresh", "late", "edge", "bump")
CONFIGS = ("single", "vector", "A", "B")
OFFSETS = (0, (1 << 32) + 7)
CLOCKS = (0, 12345)
INSTANCES = [(D, R, AR, mode, rec) for D in (15, 12) for R in (True, False) for AR in (True, False)
             for mode in (0, 1) for rec in (True, False)]
GEN_OUTS = ("full", "subset_a", "subset_b", "none")
CHECKED = 30_000          # transitions checked against float64 per case (a strided sample of envs above this)
GUARD = 64                # guard elements before and after every output buffer

# two non-default constant sets: asymmetric inertia (dI_yaw != 0, invI[0] != invI[1]), mass != 1 (inv_mass != mass),
# other dt / arm / k_yaw / gravity / r_max / z_floor / bonus, timeouts and curriculum bumps inside a launch
CONFIG_KW = {
    "single": {},
    "vector": dict(bonus_radius=1.0, max_steps=1000),
    "A": dict(inertia=(0.004, 0.006, 0.011), mass=1.3, gravity=9.7, dt=0.015, arm_length=0.4, k_yaw=0.013, r_max=30.0,
              z_floor=0.25, bonus=0.5, bonus_radius=0.3, reward_scale=0.02, max_steps=23, curriculum_period=3,
              curriculum_step=0.07, start_z=1.5, target_z=2.0, fixed_start=(0.25, -0.5, 1.0), fixed_target=(1.0, -2.0, 5.0)),
    "B": dict(inertia=(0.007, 0.0045, 0.009), mass=0.8, dt=0.025, arm_length=0.6, k_yaw=0.008, r_max=20.0, z_floor=-0.5,
              bonus=2.0, bonus_radius=0.5, max_steps=57, curriculum_period=5, curriculum_step=0.25, start_z=0.75,
              target_z=1.25, fixed_start=(-0.125, 0.375, 0.5), fixed_target=(0.5, 0.25, 3.0)),
}


def block_for(n):
    """capi_env.cu block_for: the CTA size of a launch over n envs"""
    return 256 if n >= 148 * 256 * 2 else (64 if n >= 148 * 64 * 2 else 32)


def record_rule(outs, mode):
    """capi_env.cu launch_rollout: the RECORD specialisation runs for exactly next_obs + reward + done, plus the applied
    action iff it is generated in-kernel (dronecu_step always streams and always passes no out_actions)"""
    if "step" in outs:
        return False
    return ({"next_obs", "reward", "done"} <= outs and not ({"truncated", "terminal_obs", "episode_r", "episode_l"} & outs)
            and (mode == 1) == ("out_actions" in outs))


def output_set(level, mode):
    return {"record": {"next_obs", "reward", "done"} | ({"out_actions"} if mode == 1 else set()),
            "full": {"obs0", "next_obs", "out_actions", "reward", "done", "truncated"},
            "subset_a": {"obs0", "next_obs", "truncated"},
            "subset_b": {"reward", "done", "out_actions"},
            "none": set(),
            "step": {"step", "next_obs", "reward", "done", "truncated", "terminal_obs", "episode_r", "episode_l"}}[level]


def design():
    """One case per (instantiation, n); the other factors cycle over the case index with periods <= 4 from a
    per-instantiation offset, so every instantiation meets every level.  Plus, per non-auto-reset instantiation, one
    K = 1100 case at n = 33 that crosses max_steps = 1000 (done on every later step)."""
    cases = []
    for ii, (D, R, AR, mode, rec) in enumerate(INSTANCES):
        for j, n in enumerate(NS):
            K = KS[(j + ii) % 4]
            if n * K > 1 << 23:
                K = 2
            if rec:
                out = "record"
            elif K == 1 and mode == 0 and (j // 4 + ii) % 2 == 0:
                out = "step"
            else:
                out = GEN_OUTS[(j + ii // 2) % 4]
            cases.append(dict(inst=(D, R, AR, mode, rec), n=n, K=K, out=out, cfg=CONFIGS[(3 * j + ii + 1) % 4],
                              start=STARTS[(j // 2 + ii) % 4], t0=CLOCKS[(j // 4 + ii) % 2],
                              off=OFFSETS[((j + 1) // 3 + ii) % 2], misalign=(j + ii // 3) % 2 == 1))
        if not AR:
            cases.append(dict(inst=(D, R, AR, mode, rec), n=33, K=1100, out="record" if rec else "full", cfg="vector",
                              start="fresh", t0=CLOCKS[ii % 2], off=OFFSETS[ii % 2], misalign=ii % 3 == 0))
    return cases


def _case_id(c):
    D, R, AR, mode, rec = c["inst"]
    return (f"D{D}-{'rand' if R else 'fixed'}-{'ar' if AR else 'noar'}-{'philox' if mode else 'stream'}-"
            f"{'rec' if rec else 'gen'}-n{c['n']}-K{c['K']}-{c['out']}-{c['cfg']}-{c['start']}-t{c['t0']}-off{c['off']}"
            f"-{'mis' if c['misalign'] else 'al'}")


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    return drone_rl_b200


def make_config(drl, name, D, R, AR):
    return drl.EnvConfig.single(**CONFIG_KW[name], obs_dim=D, randomized=R, auto_reset=AR)


# ---------------------------------------------------------------------------------------------------------------------
# guarded output buffers
# ---------------------------------------------------------------------------------------------------------------------
_SENT = {torch.float32: 0x7FA5A5A5, torch.int32: 0x7FA5A5A5, torch.uint8: 0xA5}


class Guarded:
    """A [GUARD | shift | view | GUARD] buffer filled with a sentinel; ``shift`` = 1 element puts a float view at a
    4-byte offset from the 16-byte alignment of the allocation."""

    def __init__(self, shape, dtype=torch.float32, shift=0):
        count = int(np.prod(shape))
        self.raw = torch.empty(2 * GUARD + shift + count, dtype=dtype, device="cuda")
        self._bits().fill_(_SENT[dtype])
        self.lo, self.hi = GUARD + shift, GUARD + shift + count
        self.view = self.raw[self.lo:self.hi].view(*shape)

    def _bits(self):
        return self.raw.view(torch.int32) if self.raw.dtype == torch.float32 else self.raw

    def guards_intact(self):
        b, s = self._bits(), _SENT[self.raw.dtype]
        return bool((b[:self.lo] == s).all()) and bool((b[self.hi:] == s).all())

    def untouched(self):
        """[...] bool: which elements of the view still hold the sentinel"""
        b = self._bits()[self.lo:self.hi].view(*self.view.shape)
        return b == _SENT[self.raw.dtype]


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# start states
# ---------------------------------------------------------------------------------------------------------------------
def _start(b, cfg, start, rng):
    n = b.n
    b.reset()
    if start == "fresh":
        return
    if start == "late":      # time limits within 3 steps
        step = np.full(n, cfg.max_steps - 3, np.int32)
        b.set_state(step=step, ep_len=step, ep_ret=(-rng.uniform(0, 3, n)).astype(np.float32))
    elif start == "bump":    # the next reset makes ep_num a multiple of the curriculum period
        b.set_state(ep_num=np.full(n, cfg.curriculum_period - 1, np.int32), ep_len=np.full(n, 7, np.int32),
                    step=np.full(n, 7, np.int32), ep_ret=np.full(n, -0.25, np.float32))
    else:                    # edge: half the envs just above the floor falling, half just inside r_max flying outwards
        st = b.get_state("pos", "vel")
        pos, vel = st["pos"].astype(np.float64), st["vel"].astype(np.float64)
        low = rng.random(n) < 0.5
        pos[low, 2] = cfg.z_floor + rng.uniform(0.005, 0.05, int(low.sum()))
        vel[low, 2] = -rng.uniform(0.5, 2.0, int(low.sum()))
        m = int((~low).sum())
        u = rng.normal(size=(m, 3))
        u[:, 2] = np.abs(u[:, 2]) + 0.5
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        r = cfg.r_max - rng.uniform(0.01, 0.3, m)
        pos[~low] = u * r[:, None]
        vel[~low] = u * rng.uniform(1.0, 5.0, m)[:, None]
        b.set_state(pos=pos.astype(np.float32), vel=vel.astype(np.float32),
                    ep_len=np.full(n, 3, np.int32), step=np.full(n, 3, np.int32))


# ---------------------------------------------------------------------------------------------------------------------
# one launch
# ---------------------------------------------------------------------------------------------------------------------
def _launch(b, K, mode, actions, outs, shift):
    """Run the launch with the outputs ``outs`` in guarded buffers (obs0 / next_obs / terminal_obs at ``shift``)."""
    n, D = b.n, b.obs_dim
    bufs = {}
    if "obs0" in outs:
        bufs["obs0"] = Guarded((n, D), shift=shift)
    if "next_obs" in outs:
        bufs["next_obs"] = Guarded((K, n, D), shift=shift)
    if "out_actions" in outs:
        bufs["out_actions"] = Guarded((K, n, 4))
    if "reward" in outs:
        bufs["reward"] = Guarded((K, n))
    for key in ("done", "truncated"):
        if key in outs:
            bufs[key] = Guarded((K, n), torch.uint8)
    if "step" in outs:
        assert K == 1 and mode == 0
        bufs["terminal_obs"] = Guarded((n, D), shift=shift)
        bufs["episode_r"] = Guarded((n,))
        bufs["episode_l"] = Guarded((n,), torch.int32)
        flat = {"obs": bufs["next_obs"].view[0], "reward": bufs["reward"].view[0], "done": bufs["done"].view[0],
                "truncated": bufs["truncated"].view[0], "terminal_obs": bufs["terminal_obs"].view,
                "episode_r": bufs["episode_r"].view, "episode_l": bufs["episode_l"].view}
        b.step(actions[0], out=flat)
    else:
        b.rollout(K, actions if mode == 0 else None, **{k: bufs[k].view for k in bufs})
    torch.cuda.synchronize()
    return bufs


def _expected_state(st0, done, reward, auto_reset):
    from tests.test_gpu_rollout_parity import _expected_after
    step, ep_num, ep_len, ep_ret, rets, length_sum = _expected_after(st0, done, reward)
    if not auto_reset:        # no reset: the step counter runs on and ep_num stays; VecMonitor still zeroes on done
        K = done.shape[0]
        step, ep_num = st0["step"] + K, st0["ep_num"].copy()
    return step, ep_num, ep_len, ep_ret, rets, length_sum


def _columns(n, K):
    if n * K <= CHECKED:
        return np.arange(n)
    stride = max(1, (n * K) // CHECKED)
    return np.unique(np.concatenate([np.arange(0, n, stride), np.arange(min(n, 33)), np.arange(max(0, n - 33), n)]))


def run_case(drl, c):
    D, R, AR, mode, rec = c["inst"]
    n, K = c["n"], c["K"]
    cfg = make_config(drl, c["cfg"], D, R, AR)
    p = do.Params.from_config(cfg)
    outs = output_set(c["out"], mode)
    assert record_rule(outs, mode) == rec
    shift = 1 if c["misalign"] else 0
    rng = np.random.default_rng(n * 131 + K)
    b = drl.DroneBatch(n, cfg, seed=SEED, env_offset=c["off"])
    twin = drl.DroneBatch(n, cfg, seed=SEED, env_offset=c["off"])
    _start(b, cfg, c["start"], rng)
    st0 = b.get_state()
    twin.set_state(**st0)
    for h in (b, twin):
        h.global_step = c["t0"]
        h.episode_stats(reset=True)
    mm = np.float32(cfg.motor_max)
    actions = None
    if mode == 0:
        actions = torch.from_numpy(rng.uniform(0, float(mm), (K, n, 4)).astype(np.float32)).cuda()
    bufs = _launch(b, K, mode, actions, outs, shift)
    ref = _launch(twin, K, mode, actions, output_set("full", mode), shift)
    assert b.global_step == twin.global_step == c["t0"] + (1 if "step" in outs else K)

    # stray writes, output-set invariance
    for key, g in list(bufs.items()) + list(ref.items()):
        assert g.guards_intact(), f"guard region of {key} overwritten"
    for key, g in bufs.items():
        if key in ref:
            assert _bits_equal(g.view, ref[key].view), f"{key} differs from the full-output twin"
    st1, st_twin = b.get_state(), twin.get_state()
    for key in st1:
        assert np.array_equal(st1[key].view(np.uint32), st_twin[key].view(np.uint32)), f"final {key} differs from the twin"
    stats, stats_twin = b.episode_stats(reset=True), twin.episode_stats(reset=True)
    for key in ("episodes", "terminated", "truncated", "length_sum"):
        assert stats[key] == stats_twin[key], key

    # actions
    act = ref["out_actions"].view
    if mode == 0:
        assert torch.equal(act, actions)
    cols = _columns(n, K)
    ids = np.uint64(c["off"]) + cols.astype(np.uint64)
    act_h = act[:, torch.from_numpy(cols).cuda()].cpu().numpy()
    if mode == 1:
        for k in range(K):
            want = philox.action_uniforms(SEED, ids, c["t0"] + k).astype(np.float32) * mm
            assert np.array_equal(act_h[k], want), f"Philox action at step {k}"

    # transitions of the twin's record
    sel = torch.from_numpy(cols).cuda()
    obs0 = ref["obs0"].view[sel].cpu().numpy()
    nxt = ref["next_obs"].view[:, sel].cpu().numpy()
    done_full = ref["done"].view.cpu().numpy().astype(bool)
    reward_full = ref["reward"].view.cpu().numpy()
    trunc_full = ref["truncated"].view.cpu().numpy().astype(bool)
    sub = {k: v[cols] for k, v in st0.items()}
    rep = verify.check_rollout(obs0, act_h, nxt, reward_full[:, cols], done_full[:, cols], spec=p, seed=SEED, env_ids=ids,
                               ep_num0=sub["ep_num"], step0=sub["step"], target0=sub["target"])
    if c["start"] == "fresh":       # the constructor's reset and reset(): ep_num 2
        rp, rt = verify.reset_rows(p, SEED, ids, np.full(len(cols), 2))
        want = np.concatenate([rp, np.zeros((len(cols), 9), np.float32), rt - rp], 1)[:, :D]
        assert np.array_equal(obs0.view(np.uint32), want.view(np.uint32)), "reset observation"

    # state after the launch and the statistics, over every env
    step, ep_num, ep_len, ep_ret, rets, length_sum = _expected_state(st0, done_full, reward_full, AR)
    assert np.array_equal(st1["step"], step) and np.array_equal(st1["ep_num"], ep_num) and np.array_equal(st1["ep_len"], ep_len)
    assert _same_f32(st1["ep_ret"], ep_ret), "ep_ret is not the float32 replay"
    assert not (trunc_full & ~done_full).any(), "truncated without done"
    for st in (stats, stats_twin):
        if len(cols) == n:
            assert rep["terminated"] <= st["terminated"] <= rep["terminated"] + rep["terminated_slack"]
        _check_stats_sampled(st, done_full, rets, length_sum, st0, p.max_steps, AR)
    if AR is False and K == 1100:
        assert done_full[p.max_steps - 1 - int(st0["step"].max()):].all(), "done on every step past max_steps"

    # dronecu_step's info outputs: written on done rows only, equal to the oracle there
    if "step" in outs:
        d = done_full[0]
        for key in ("terminal_obs", "episode_r", "episode_l"):
            u = bufs[key].untouched().cpu().numpy()
            u = u.all(1) if u.ndim == 2 else u
            assert np.array_equal(u, ~d), f"{key} written off the done rows"
        rows = np.flatnonzero(d)
        if rows.size:
            assert np.array_equal(bufs["episode_l"].view.cpu().numpy()[rows], st0["ep_len"][rows] + 1)
            want_r = (st0["ep_ret"] + reward_full[0]).astype(np.float32)[rows]
            assert _same_f32(bufs["episode_r"].view.cpu().numpy()[rows], want_r)
            term = bufs["terminal_obs"].view.cpu().numpy()[rows]
            full_obs0 = ref["obs0"].view.cpu().numpy()[rows]
            verify.check_rollout(full_obs0, act[:, torch.from_numpy(rows).cuda()].cpu().numpy(), term[None],
                                 reward_full[:, rows], done_full[:, rows], spec=dataclasses.replace(p, auto_reset=False),
                                 seed=SEED, env_ids=np.uint64(c["off"]) + rows.astype(np.uint64),
                                 ep_num0=st0["ep_num"][rows], step0=st0["step"][rows], target0=st0["target"][rows])
    b.close()
    twin.close()
    return rep, stats


def _same_f32(a, b):
    """bit-identical float32, except that any NaN matches any NaN (the device's and numpy's NaN payloads differ)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def _check_stats_sampled(stats, done, rets, length_sum, st0, max_steps, auto_reset):
    """The statistics over every env: episodes, length_sum exact; terminated at least the dones before the time limit;
    return_sum within the float32 rounding of each env's sum (a non-finite sum: the same inf, or NaN, in any order)."""
    assert stats["episodes"] == int(done.sum())
    assert stats["length_sum"] == length_sum
    cnt = st0["step"].astype(np.int64).copy()
    early = 0
    for k in range(done.shape[0]):
        cnt += 1
        early += int((done[k] & (cnt < max_steps)).sum())
        if auto_reset:
            cnt[done[k]] = 0
    assert early <= stats["terminated"] <= stats["episodes"]
    assert stats["truncated"] == stats["episodes"] - stats["terminated"]
    flat = np.asarray([r for env in rets for r in env], np.float64)
    if not np.isfinite(flat).all():
        ref = float(flat.sum())
        assert stats["return_sum"] == ref or (np.isnan(ref) and np.isnan(stats["return_sum"])), (stats["return_sum"], ref)
        return
    tol = sum(max(len(env) - 1, 0) * 2.0 ** -24 * 1.01 * float(np.abs(np.asarray(env, np.float64)).sum()) for env in rets)
    tol += 1e-12 * (float(np.abs(flat).sum()) + 1.0)
    assert abs(stats["return_sum"] - float(flat.sum())) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("case", design(), ids=_case_id)
def test_env_rollout_parity(drl, case):
    rep, stats = run_case(drl, case)
    print(f"{_case_id(case)}: worst err/bound {rep['worst_err_over_bound']:.3g}, checked {rep['transitions']}, "
          f"dones {stats['episodes']}, terminated {stats['terminated']}, borderline {rep['borderline_done']}, "
          f"out of float32 range {rep['out_of_f32_range']}")


# ---------------------------------------------------------------------------------------------------------------------
# reset kernel
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [4097, 18944, 75776], ids=lambda n: f"n{n}-cta{block_for(n)}")
@pytest.mark.parametrize("D,R", [(15, True), (15, False), (12, True), (12, False)])
def test_reset_kernel_parity(drl, D, R, n):
    """reset_kernel<D, R> under no mask, a random mask and an all-zero mask, into aligned and misaligned observation
    rows, at each CTA size: observations bit-exact, rows outside the mask keep their state bit for bit, ep_num advances
    on masked rows only."""
    cfg = make_config(drl, "A", D, R, False)
    p = do.Params.from_config(cfg)
    off = (1 << 32) + 3
    rng = np.random.default_rng(D * 7 + n)
    b = drl.DroneBatch(n, cfg, seed=SEED, env_offset=off)
    f = lambda *s, lo=-2.0, hi=2.0: rng.uniform(lo, hi, s).astype(np.float32)
    b.set_state(pos=f(n, 3, lo=0.5, hi=5.0), vel=f(n, 3), euler=f(n, 3), omega=f(n, 3), target=f(n, 3),
                step=rng.integers(0, 20, n).astype(np.int32), ep_num=rng.integers(0, 40, n).astype(np.int32),
                ep_len=rng.integers(0, 20, n).astype(np.int32), ep_ret=f(n))
    st0 = b.get_state()
    ids = np.uint64(off) + np.arange(n, dtype=np.uint64)
    for kind in ("none", "random", "zero"):
        for shift in (0, 1):
            b.set_state(**st0)
            m = np.ones(n, bool) if kind == "none" else (rng.random(n) < 0.4 if kind == "random" else np.zeros(n, bool))
            mask = None if kind == "none" else torch.from_numpy(m.astype(np.uint8)).cuda()
            g = Guarded((n, D), shift=shift)
            b.reset(mask=mask, out=g.view)
            torch.cuda.synchronize()
            assert g.guards_intact()
            st1 = b.get_state()
            obs = g.view.cpu().numpy()
            rows, keep = np.flatnonzero(m), np.flatnonzero(~m)
            for key in st0:
                assert np.array_equal(st1[key][keep].view(np.uint32), st0[key][keep].view(np.uint32)), f"{kind}: {key} off the mask"
            assert np.array_equal(st1["ep_num"][rows], st0["ep_num"][rows] + 1)
            for key in ("vel", "euler", "omega"):
                assert (st1[key][rows] == 0).all()
            for key in ("step", "ep_len", "ep_ret"):
                assert (st1[key][rows] == 0).all()
            rp, rt = verify.reset_rows(p, SEED, ids[rows], st0["ep_num"][rows] + 1)
            assert np.array_equal(st1["pos"][rows], rp) and np.array_equal(st1["target"][rows], rt), kind
            want = np.concatenate([st1["pos"], st1["vel"], st1["euler"], st1["omega"], st1["target"] - st1["pos"]], 1)[:, :D]
            assert np.array_equal(obs.view(np.uint32), want.view(np.uint32)), f"{kind} shift {shift}: observation rows"
    b.close()


# ---------------------------------------------------------------------------------------------------------------------
# curriculum bump count at large ep_num
# ---------------------------------------------------------------------------------------------------------------------
EP_NUMS = (33_554_434, 58_720_262, 1_677_722_689, (1 << 24) - 1, 1 << 24, (1 << 24) + 1, (1 << 31) - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("period", [1, 7, 100, 2000])
def test_curriculum_bump_count_at_large_ep_num(drl, period):
    """The reset that makes ep_num E replays floor(E / period) curriculum steps for every 31-bit E: the values where a
    float32 estimate of E / period is off by 2 or more (33,554,434 and on at period 1, 58,720,262 at 7, 1,677,722,689 at
    100), 2^24 +- 1 and 2^31 - 1.  Start and target bit-exact against the oracle's float64 accumulation."""
    cfg = drl.EnvConfig.single(curriculum_period=period, curriculum_step=0.1, auto_reset=False)
    p = do.Params.from_config(cfg)
    n = len(EP_NUMS)
    b = drl.DroneBatch(n, cfg, seed=SEED, env_offset=77)
    e = np.asarray(EP_NUMS, np.int64)
    b.set_state(ep_num=(e - 1).astype(np.int32))
    b.reset()
    st = b.get_state("pos", "target", "ep_num")
    assert np.array_equal(st["ep_num"], e.astype(np.int32))
    rp, rt = verify.reset_rows(p, SEED, np.uint64(77) + np.arange(n, dtype=np.uint64), e)
    assert np.array_equal(st["pos"], rp)
    bad = np.flatnonzero((st["target"] != rt).any(1))
    assert bad.size == 0, f"period {period}: wrong curriculum target at ep_num {e[bad].tolist()}"
    b.close()
