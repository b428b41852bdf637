"""Observation and reward normalisation (csrc/obs_norm.cuh, drone_rl_b200/normalize.py) pinned against SB3 VecNormalize
restated in float64 (oracle/normalize_oracle.py) over a covering design of the pass's launch shapes, modes, settings,
statistics, data and done patterns: every level of every factor appears, and every mode (outputs x update) meets every
env count, step count and row stride.

Stated bounds (u = 2^-53, gamma_k = k u / (1 - k u)):
  normalised rows      bit-identical to normalize_obs_f32 with the kernel's own affine record (float32 subtract and
                       multiply, np.clip: NaN stays NaN, +-inf goes to +-clip_obs)
  rewards              bit-identical to normalize_reward_f32 = float32(clip(float64(r) / sqrt(ret_var + eps))) with the
                       kernel's ret_var (double / and sqrt are correctly rounded on both sides)
  per-env returns      bit-identical to the numpy recurrence ret * gamma + r (the kernel's __dmul_rn / __dadd_rn), zeroed
                       at dones; in evaluation not advanced, still zeroed at dones (SB3 step_wait)
  side rows, pad       exact
  CTA partials         counts exact; sum(x - c) and sum((x - c)^2) within gamma_{K + 14 + ref} of the magnitudes summed
                       (x - c is one rounding on both sides; K sequential adds, 5 shuffle levels, the 8-warp fold, the
                       fma; ref = the reference's long double pairwise sum and its rounding to float64, ~1)
  reduce               bit-identical to reduce_partials, the kernel's fixed order restated on the same partials
  combine              within combine_bound of SB3 update_from_moments given the kernel's moments (twice the forward error
                       of either evaluation: nvcc may contract the kernel's products and sums into FMAs)
  against the data     within one_pass_bound of SB3 update_from_moments on two-pass moments of the data (np.mean /
                       np.var summed pairwise in long double: numpy's float64 np.mean(axis=0) adds the rows one after
                       another, N roundings that would swamp the kernel's error): the shifted one-pass formula
                       errs relative to the spread about the shift, |e_var_b| <= gamma (2 s2 / cb + delta^2), which the
                       initial statistics (shift 0, position features far from it) exercise
  affine record        bit-identical to float32(mean), float32(1 / sqrt(var + eps)) and clip_obs
Each case prints its worst error as a fraction of its bound.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import normalize_oracle as no  # noqa: E402

FLT_MAX = float(np.finfo(np.float32).max)
NS = (1, 255, 256, 257, 7424, 7680, 7681, 15361, 1 << 20, (1 << 20) + 3)
MODES = tuple((o, r, u) for (o, r) in ((1, 1), (1, 0), (0, 1)) for u in (1, 0))      # (obs, rewards, update)
SIDES = ("off", "first", "last")
GAMMAS, CLIP_OBS, CLIP_REW, EPSILONS = (0.99, 0.95, 0.0), (10.0, 0.5, 1e30), (10.0, 0.1), (1e-8, 0.0, 1e-2)
STATS = ("initial", "near", "zero_var", "late")
DATA = ("recorded", "synthetic")
DONES = ("none", "all", "random", "every_step")
OFFSETS = np.array([1e3, -50, 20, 3, -2, 1, 0.5, 0, -0.3, 40, -40, 5, 0, 0, 7e3])
SCALES = np.array([5, 10, 2, 1, 4, 0.1, 0.5, 0.2, 0.3, 1, 1, 3, 8, 0.01, 1])
ZERO_VAR = [12, 13, 14]          # the columns held constant for the zero-variance statistics


def _design():
    """mode x env count in full; the step count and stride rotate with (env count + mode) so that every mode meets each;
    K = 2048 runs with n = 1 (the c1 shape) once per mode; every other factor is a balanced permutation of its levels."""
    cases = []
    for a, n in enumerate(NS):
        for b, mode in enumerate(MODES):
            Ks = (1, 2) if n >= 1 << 20 else (1, 2, 40)
            cases.append(dict(n=n, K=Ks[(a + b) % len(Ks)], mode=mode, stride=(15, 16)[(a + b) % 2]))
    for b, mode in enumerate(MODES):
        cases.append(dict(n=1, K=2048, mode=mode, stride=(15, 16)[b % 2]))
    levels = dict(side=SIDES, gamma=GAMMAS, clip_obs=CLIP_OBS, clip_reward=CLIP_REW, epsilon=EPSILONS, stats=STATS,
                  data=DATA, dones=DONES)
    for s, (name, lv) in enumerate(levels.items()):
        perm = np.random.default_rng(100 + s).permutation(len(cases))
        for i, c in enumerate(cases):
            c[name] = lv[perm[i] % len(lv)]
    return cases


CASES = _design()


def _case_id(c):
    o, r, u = c["mode"]
    return (f"n{c['n']}-K{c['K']}-{'obs' if o else ''}{'rew' if r else ''}-{'upd' if u else 'eval'}-s{c['stride']}-"
            f"{c['stats']}-{c['data']}-{c['dones']}")


def test_design_covers_every_level_and_pair():
    seen = {k: {c[k] for c in CASES} for k in ("n", "K", "mode", "stride", "side", "gamma", "clip_obs", "clip_reward",
                                                "epsilon", "stats", "data", "dones")}
    want = dict(n=set(NS), K={1, 2, 40, 2048}, mode=set(MODES), stride={15, 16}, side=set(SIDES), gamma=set(GAMMAS),
                clip_obs=set(CLIP_OBS), clip_reward=set(CLIP_REW), epsilon=set(EPSILONS), stats=set(STATS), data=set(DATA),
                dones=set(DONES))
    assert seen == want
    for shape in ("n", "K", "stride"):
        pairs = {(c["mode"], c[shape]) for c in CASES}
        assert pairs == {(m, s) for m in MODES for s in want[shape]}, shape


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


@pytest.fixture(scope="module")
def recorded(drl):
    """4096 envs x 64 steps of a real DroneBatch rollout under uniform random motor commands: rows, rewards, dones."""
    n, K = 4096, 64
    b = drl.DroneBatch(n, drl.EnvConfig.single(), seed=31)
    b.reset()
    g = torch.Generator(device="cuda").manual_seed(31)
    acts = torch.rand(K, n, 4, generator=g, device="cuda") * 7.3575
    nxt, rew, done = b.empty(K, n, 15), b.empty(K, n), b.empty(K, n, dtype=torch.uint8)
    b.rollout(K, acts, next_obs=nxt, reward=rew, done=done)
    torch.cuda.synchronize()
    b.close()
    obs = nxt.reshape(-1, 15).cpu().numpy()
    assert np.isfinite(obs).all() and done.any()
    return obs, rew.reshape(-1).cpu().numpy(), done.reshape(-1).cpu().numpy().astype(bool)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _bits(a):
    """the bit pattern of a float array, every NaN mapped to one pattern (payloads are not specified)"""
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        b = a.view(np.uint32).copy()
        b[np.isnan(a)] = 0x7FC00000
    else:
        b = a.astype(np.float64).view(np.uint64).copy()
        b[np.isnan(a)] = 0x7FF8000000000000
    return b


def _same(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    return got.shape == ref.shape and got.dtype == ref.dtype and np.array_equal(_bits(got), _bits(ref))


def _ratio(err, bound):
    err, bound = np.broadcast_arrays(np.abs(np.asarray(err, np.float64)), np.asarray(bound, np.float64))
    if not err.size:
        return 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / np.where(bound > 0, bound, 0.0))
    return float(np.max(np.nan_to_num(r, nan=np.inf)))


def _rms(s):
    """(obs RunningMeanStd, ret RunningMeanStd) holding the [34] statistics record s"""
    s = np.asarray(s, np.float64)
    o, r = no.RunningMeanStd((15,)), no.RunningMeanStd(())
    o.mean, o.var, o.count = s[:15].copy(), s[15:30].copy(), float(s[30])
    r.mean, r.var, r.count = np.float64(s[31]), np.float64(s[32]), float(s[33])
    return o, r


def _set_stats(nz, s):
    nz.stats.copy_(torch.as_tensor(np.asarray(s, np.float64)))
    nz._combine(None)


def _check_affine(aff, stats, eps, clip_obs):
    aff, stats = np.asarray(aff), np.asarray(stats, np.float64)
    assert _same(aff[:15], stats[:15].astype(np.float32)), "affine mean"
    assert _same(aff[15:30], (1.0 / np.sqrt(stats[15:30] + eps)).astype(np.float32)), "affine rstd"
    assert _same(aff[30:], np.array([clip_obs], np.float32)), "affine clip"


def _returns_ref(ret0, rew, done, gamma, update):
    """(returns after the rollout, the [K, n] returns fed to ret_rms): ret = ret * gamma + r (training), 0 at done"""
    ret, rets = ret0.copy(), np.empty(rew.shape, np.float64)
    for k in range(rew.shape[0]):
        if update:
            ret = ret * gamma + rew[k].astype(np.float64)
        rets[k] = ret
        ret[done[k]] = 0.0
    return ret, rets


def _cta_sums(d, K, n):
    """per-CTA sum(d), sum|d|, sum(d^2) of d [K, n, F], the reference side of the partial check: each CTA's K x 256
    values laid out contiguously and summed pairwise in long double (PARTIAL_REF_DEPTH float64 roundings at most)"""
    P = -(-n // 256)
    pad = np.zeros((K, P * 256) + d.shape[2:])
    pad[:, :n] = d
    pad = np.moveaxis(pad.reshape((K, P, 256, -1)), (0, 2), (2, 3)).reshape(P, -1, K * 256)
    out = []
    for f in (lambda a: a, np.abs, np.square):
        v = np.ascontiguousarray(f(pad)).astype(np.longdouble).sum(axis=-1).astype(np.float64)
        out.append(v.reshape((P,) + d.shape[2:]))
    return out


def _partial_depth(K):
    """float64 roundings behind one partial, kernel and reference: K steps, 5 shuffle levels, the 8-warp fold, the fma,
    and the reference's long double pairwise sum of K x 256 values and its final rounding"""
    return K + 14 + no.ref_depth(256 * K)


def _check_stats_update(worst, tag, s0, s1, m, raw_or_rets, K, n):
    """s1 against SB3 update_from_moments on the kernel's moments m = (s1, s2, cb) (combine bound) and against SB3
    update_from_moments on two_pass_moments of the data (one-pass bound)."""
    mean0, var0, c0, (ms1, ms2, cb) = s0[0], s0[1], s0[2], m
    ref = no.RunningMeanStd(np.shape(mean0))
    ref.mean, ref.var, ref.count = np.array(mean0, np.float64), np.array(var0, np.float64), c0
    no.combine_sb3(ref, ms1, ms2, cb)
    bm, bv = no.combine_bound(mean0, var0, c0, ms1, ms2, cb)
    worst[f"{tag}_combine"] = max(_ratio(s1[0] - ref.mean, bm), _ratio(s1[1] - ref.var, bv))
    ref = no.RunningMeanStd(np.shape(mean0))
    ref.mean, ref.var, ref.count = np.array(mean0, np.float64), np.array(var0, np.float64), c0
    ref.update_from_moments(*no.two_pass_moments(raw_or_rets), cb)
    bm, bv = no.one_pass_bound(mean0, var0, c0, ms2, cb, no.pass_depth(K, n))
    worst[f"{tag}_vs_data"] = max(_ratio(s1[0] - ref.mean, bm), _ratio(s1[1] - ref.var, bv))
    assert s1[2] == c0 + cb, f"{tag} count"
    assert worst[f"{tag}_combine"] <= 1.0 and worst[f"{tag}_vs_data"] <= 1.0, f"{tag}: {worst}"


# ---------------------------------------------------------------------------------------------------------------------
# the pass, reduce and combine over the covering design
# ---------------------------------------------------------------------------------------------------------------------
def _case_inputs(c, recorded, rng):
    n, K = c["n"], c["K"]
    if c["data"] == "recorded":
        obs, rew, done = recorded
        idx = rng.integers(0, obs.shape[0], K * n)
        raw, r, d_rec = obs[idx].reshape(K, n, 15), rew[idx].reshape(K, n), done[idx].reshape(K, n)
        mu, sd = obs.mean(0), np.maximum(obs.std(0), 1e-3)
    else:
        raw = (OFFSETS + SCALES * rng.standard_normal((K, n, 15))).astype(np.float32)
        r = (0.05 * rng.standard_normal((K, n)) * np.where(rng.random((K, n)) < 0.01, 100.0, 1.0)).astype(np.float32)
        d_rec = rng.random((K, n)) < 0.05
        mu, sd = OFFSETS, SCALES
    done = {"none": np.zeros((K, n), bool), "all": np.arange(K)[:, None] == np.full((1, n), K // 2),
            "random": d_rec, "every_step": np.ones((K, n), bool)}[c["dones"]]
    s = np.zeros(34)
    if c["stats"] == "initial":
        s[15:30], s[30], s[32], s[33] = 1.0, 1e-4, 1.0, 1e-4
    else:
        s[:15], s[15:30], s[30] = mu + 0.3 * sd, (1.7 * sd) ** 2, 50.0
        s[31:34] = 0.02, 0.0025, 50.0
        if c["stats"] == "late":
            s[30] = s[33] = 1e12
        if c["stats"] == "zero_var":             # constant columns, as the fixed target gives
            raw = raw.copy()
            raw[..., ZERO_VAR] = raw[0, 0, ZERO_VAR]
            s[ZERO_VAR], s[[15 + f for f in ZERO_VAR]] = raw[0, 0, ZERO_VAR].astype(np.float64), 0.0
    return np.ascontiguousarray(raw, np.float32), np.ascontiguousarray(r, np.float32), done, s


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[_case_id(c) for c in CASES])
def test_pass_reduce_combine(drl, recorded, c):
    from drone_rl_b200.normalize import ObsNormalizer
    dev = torch.device("cuda", 0)
    n, K, stride = c["n"], c["K"], c["stride"]
    do_obs, do_rew, upd = c["mode"]
    eps, gamma, clip_obs, clip_rew = c["epsilon"], c["gamma"], c["clip_obs"], c["clip_reward"]
    rng = np.random.default_rng(n * 7 + K)
    raw, rew, done, s0 = _case_inputs(c, recorded, rng)
    nz = ObsNormalizer(n, dev, norm_obs=bool(do_obs), norm_reward=bool(do_rew), clip_obs=clip_obs, clip_reward=clip_rew,
                       epsilon=eps, gamma=gamma)
    nz.training = bool(upd)
    _set_stats(nz, s0)
    aff0 = nz.affine.cpu().numpy()
    _check_affine(aff0, s0, eps, clip_obs)
    ret0 = 0.05 * rng.standard_normal(n)
    nz.returns.copy_(torch.from_numpy(ret0))
    nz.partials.fill_(float("nan"))
    store = torch.ones(K, n, stride, device=dev)
    store[..., :15] = torch.from_numpy(raw).to(dev)
    rew_d, done_d = torch.from_numpy(rew).to(dev), torch.from_numpy(done.astype(np.uint8)).to(dev)
    side_env = {"off": -1, "first": 0, "last": n - 1}[c["side"]]
    side = torch.full((K, 15), float("nan"), device=dev)
    launches = nz.process_rollout(store, rew_d, done_d, K, side_env=side_env,
                                  side_obs=None if side_env < 0 else side)
    assert launches == (3 if upd else 1)
    torch.cuda.synchronize()
    worst = {}
    # rows, pad column, side rows
    st = store.cpu().numpy()
    o_rms, r_rms = _rms(s0)
    if do_obs:
        assert _same(st[..., :15], no.normalize_obs_f32(raw, o_rms, clip_obs, eps)), "normalised rows"
    else:
        assert _same(st[..., :15], raw), "rows must stay raw"
    if stride == 16:
        assert (st[..., 15] == 1.0).all(), "pad column"
    sd = side.cpu().numpy()
    assert _same(sd, raw[:, side_env]) if side_env >= 0 else np.isnan(sd).all(), "side rows"
    del st, store
    # rewards and per-env returns
    ret_ref, rets = _returns_ref(ret0, rew, done, gamma, upd)
    got_rew = rew_d.cpu().numpy()
    if do_rew:
        assert _same(got_rew, no.normalize_reward_f32(rew, s0[32], clip_rew, eps)), "normalised rewards"
        assert _same(nz.returns.cpu().numpy(), ret_ref), "per-env returns"
    else:
        assert _same(got_rew, rew) and _same(nz.returns.cpu().numpy(), ret0), "rewards / returns must be untouched"
    s1, a1 = nz.stats.cpu().numpy(), nz.affine.cpu().numpy()
    if not upd:           # evaluation: statistics and record untouched
        assert _same(s1, s0) and _same(a1, aff0)
        print(f"{_case_id(c)}: evaluation, every check exact")
        return
    # CTA partials
    P = nz.n_partials
    part = nz.partials.cpu().numpy()
    envs = np.minimum(256, n - 256 * np.arange(P)).astype(np.float64)
    assert _same(part[:, 30], envs * K if do_obs else np.zeros(P)), "obs counts"
    assert _same(part[:, 33], envs * K if do_rew else np.zeros(P)), "return counts"
    g = no.gamma_n(_partial_depth(K))
    if do_obs:
        s_1, s_a, s_2 = _cta_sums(raw.astype(np.float64) - s0[:15], K, n)
        worst["partial_obs"] = max(_ratio(part[:, :15] - s_1, g * s_a), _ratio(part[:, 15:30] - s_2, g * s_2))
    else:
        assert (part[:, :30] == 0).all()
    if do_rew:
        s_1, s_a, s_2 = _cta_sums(rets - s0[31], K, n)
        worst["partial_ret"] = max(_ratio(part[:, 31] - s_1, g * s_a), _ratio(part[:, 32] - s_2, g * s_2))
    else:
        assert (part[:, 31:33] == 0).all()
    assert max(worst.values(), default=0.0) <= 1.0, worst
    # reduce: the fixed order restated
    m = nz.moments.cpu().numpy()
    assert _same(m, no.reduce_partials(part)), "reduce order"
    # combine: against SB3 given these moments and against the data; a part with zero count leaves its statistics as
    # they were
    if do_obs:
        _check_stats_update(worst, "obs", (s0[:15], s0[15:30], s0[30]), (s1[:15], s1[15:30], s1[30]),
                            (m[:15], m[15:30], m[30]), raw.reshape(-1, 15), K, n)
    else:
        assert _same(s1[:31], s0[:31])
    if do_rew:
        _check_stats_update(worst, "ret", (s0[31], s0[32], s0[33]), (s1[31], s1[32], s1[33]), (m[31], m[32], m[33]),
                            rets.reshape(-1), K, n)
    else:
        assert _same(s1[31:], s0[31:])
    _check_affine(a1, s1, eps, clip_obs)
    print(f"{_case_id(c)}: worst err / bound " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


@pytest.mark.gpu
def test_zero_count_moments_leave_the_statistics(drl):
    from drone_rl_b200.normalize import ObsNormalizer
    nz = ObsNormalizer(4, torch.device("cuda", 0), epsilon=1e-2, clip_obs=3.0)
    s0 = np.concatenate([np.linspace(-3, 4, 15), np.linspace(0.1, 9, 15), [77.0, 0.3, 0.5, 12.0]])
    _set_stats(nz, s0)
    m = torch.full((34,), 5.0, dtype=torch.float64, device="cuda")
    m[30] = m[33] = 0.0
    nz._combine(m)
    torch.cuda.synchronize()
    assert _same(nz.stats.cpu().numpy(), s0)
    _check_affine(nz.affine.cpu().numpy(), s0, 1e-2, 3.0)


# ---------------------------------------------------------------------------------------------------------------------
# non-finite inputs: np.clip semantics, and statistics that become NaN as SB3's do
# ---------------------------------------------------------------------------------------------------------------------
SPECIALS = np.array([np.nan, np.inf, -np.inf, FLT_MAX, -FLT_MAX], np.float32)


@pytest.mark.gpu
def test_pass_on_non_finite_rows_and_rewards(drl):
    from drone_rl_b200.normalize import ObsNormalizer
    dev = torch.device("cuda", 0)
    n, K, eps, clip_obs, clip_rew = 300, 3, 1e-8, 5.0, 2.0
    rng = np.random.default_rng(8)
    raw = (OFFSETS + SCALES * rng.standard_normal((K, n, 15))).astype(np.float32)
    rew = (0.1 * rng.standard_normal((K, n))).astype(np.float32)
    # feature f of env f holds special value f % 5 at step 1; rewards likewise; columns 10..14 stay finite
    for f in range(10):
        raw[1, f, f] = SPECIALS[f % 5]
        rew[1, 20 + f] = SPECIALS[f % 5]
    done = np.zeros((K, n), bool)
    done[2, 20:25] = True                      # NaN / inf returns end with their episode
    nz = ObsNormalizer(n, dev, clip_obs=clip_obs, clip_reward=clip_rew, epsilon=eps, gamma=0.9)
    _set_stats(nz, np.concatenate([OFFSETS, SCALES ** 2, [50.0, 0.0, 0.01, 50.0]]))
    s0, aff0 = nz.stats.cpu().numpy(), nz.affine.cpu().numpy()
    store = torch.from_numpy(raw).to(dev).contiguous()
    rew_d, done_d = torch.from_numpy(rew).to(dev), torch.from_numpy(done.astype(np.uint8)).to(dev)
    nz.process_rollout(store, rew_d, done_d, K)
    torch.cuda.synchronize()
    o_rms, _ = _rms(s0)
    got = store.cpu().numpy()
    ref = no.normalize_obs_f32(raw, o_rms, clip_obs, eps)
    assert np.isnan(ref[1, 0, 0]) and ref[1, 1, 1] == clip_obs and ref[1, 2, 2] == -clip_obs
    assert _same(got, ref), "rows: NaN stays NaN, +-inf and +-FLT_MAX go to +-clip"
    got_r, ref_r = rew_d.cpu().numpy(), no.normalize_reward_f32(rew, s0[32], clip_rew, eps)
    assert np.isnan(ref_r[1, 20]) and ref_r[1, 21] == clip_rew and ref_r[1, 22] == -clip_rew
    assert _same(got_r, ref_r), "rewards: NaN stays NaN"
    ret_ref, rets = _returns_ref(np.zeros(n), rew, done, 0.9, True)
    assert _same(nz.returns.cpu().numpy(), ret_ref)
    assert np.isnan(ret_ref[25]) and np.isinf(ret_ref[26]) and (ret_ref[20:25] == 0).all()
    # statistics as SB3 update() leaves them: NaN where a column held NaN, inf or both infinities; finite with FLT_MAX
    s1 = nz.stats.cpu().numpy()
    ref_o, ref_r = _rms(s0)
    with np.errstate(invalid="ignore", over="ignore"):
        ref_o.update_from_moments(*no.two_pass_moments(raw.reshape(-1, 15)), K * n)
        ref_r.update_from_moments(*no.two_pass_moments(rets.reshape(-1)), K * n)
    for got_v, ref_v in ((s1[:15], ref_o.mean), (s1[15:30], ref_o.var), (s1[31], ref_r.mean), (s1[32], ref_r.var)):
        got_v, ref_v = np.atleast_1d(got_v), np.atleast_1d(ref_v)
        assert np.array_equal(np.isnan(got_v), np.isnan(ref_v)), (got_v, ref_v)
        assert np.array_equal(np.isposinf(got_v), np.isposinf(ref_v)) and np.array_equal(np.isneginf(got_v), np.isneginf(ref_v))
    assert np.isnan(s1[15:15 + 3]).all() and np.isnan(s1[32])
    assert np.isfinite(s1[[3, 4, 10, 11, 12, 13, 14]]).all()
    fin = np.isfinite(ref_o.var)
    with np.errstate(invalid="ignore", over="ignore"):
        s2 = np.square(raw.astype(np.float64) - s0[:15]).reshape(-1, 15).sum(0)
        bm, bv = no.one_pass_bound(s0[:15], s0[15:30], s0[30], s2, K * n, no.pass_depth(K, n))
    assert _ratio((s1[15:30] - ref_o.var)[fin], bv[fin]) <= 1.0 and _ratio((s1[:15] - ref_o.mean)[fin], bm[fin]) <= 1.0
    _check_affine(nz.affine.cpu().numpy(), s1, eps, clip_obs)


@pytest.mark.gpu
def test_predict_normaliser_on_non_finite_rows(drl):
    from drone_rl_b200.normalize import ObsNormalizer
    nz = ObsNormalizer(1, torch.device("cuda", 0), clip_obs=4.0)
    s = np.concatenate([np.linspace(-3, 12, 15), np.linspace(0.5, 30, 15) ** 2, [50.0, 0.0, 1.0, 50.0]])
    _set_stats(nz, s)
    rows = np.random.default_rng(2).normal(0, 5, (40, 15)).astype(np.float32)
    for i in range(40):
        rows[i, i % 15] = SPECIALS[i % 5]
    got = nz.normalize_obs(torch.from_numpy(rows)).cpu().numpy()
    ref = no.normalize_obs_f32(rows, _rms(s)[0], 4.0, 1e-8)
    assert np.isnan(ref).sum() == 8 and _same(got, ref)


@pytest.fixture
def rollout_kernel_mode():
    from drone_rl_b200 import _lib
    lib = _lib.load()
    yield lambda mode: _lib.check(lib.dronecu_set_rollout_kernel(mode))
    lib.dronecu_set_rollout_kernel(0)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["thread", "warp", "tc"])
def test_rollout_towers_see_np_clip_of_non_finite_rows(drl, rollout_kernel_mode, kernel):
    """Body rates of 3e19 rad/s on every fourth env make it emit inf and then NaN rows (tests/test_gpu_rollout_parity.py);
    a record with rstd_f = FLT_MAX on feature 5 overflows every row there to +-inf.  The towers must see np.clip of them:
    the deterministic action and the value equal policy_forward on normalize_obs_f32 of the recorded raw rows (bit for
    bit on the thread-per-env and tensor-core kernels, within 1e-5 and with the same NaN pattern on the warp-per-env
    kernel).  Before, a NaN feature reached the towers as -clip_obs and gave a finite action."""
    from tests.test_gpu_rollout_parity import _forward, _launch, _policy
    from drone_rl_b200.normalize import ObsNormalizer
    n, K = (2048 if kernel == "tc" else 256), 4
    b = drl.DroneBatch(n, drl.EnvConfig.single(), seed=5)
    b.reset()
    om = np.zeros((n, 3), np.float32)
    om[::4] = 3e19
    b.set_state(omega=om)
    nz = ObsNormalizer(n, torch.device("cuda", 0), clip_obs=10.0)
    s = np.concatenate([np.linspace(-3, 12, 15), np.linspace(0.5, 30, 15) ** 2, [50.0, 0.0, 1.0, 50.0]])
    _set_stats(nz, s)
    nz.affine[15 + 5] = FLT_MAX
    aff = nz.affine.cpu().numpy()
    theta = torch.from_numpy(_policy("hover")).cuda()
    rec = _launch(b, kernel, K, theta, True, 16, nz.affine, rollout_kernel_mode)
    raw = rec["obs"].cpu().numpy().reshape(-1, 15)
    assert np.isnan(raw).any() and np.isinf(raw).any()
    x = ((raw - aff[:15]).astype(np.float32) * aff[15:30]).astype(np.float32)
    xn = np.clip(x, -aff[30], aff[30])
    assert np.isnan(xn).any() and (np.abs(xn[:, 5]) == 10.0).sum() > 0
    pm, pv = (t.cpu().numpy() for t in _forward(theta, torch.from_numpy(xn).cuda(), kernel == "tc"))
    act, val = rec["actions"].cpu().numpy().reshape(-1, 4), rec["value"].cpu().numpy().reshape(-1)
    nan_rows = np.isnan(xn).any(1)
    assert np.isnan(pv[nan_rows]).all() or kernel == "tc"
    if kernel == "warp":
        for got, ref in ((act, pm), (val, pv)):
            assert np.array_equal(np.isnan(got), np.isnan(ref))
            fin = ~np.isnan(ref)
            assert np.abs(got[fin] - ref[fin]).max() <= 1e-5
    else:
        assert _same(act, pm) and _same(val, pv)
    b.close()


# ---------------------------------------------------------------------------------------------------------------------
# the PPO loop against FrozenVecNormalize: train, train, evaluate, train
# ---------------------------------------------------------------------------------------------------------------------
def _spy(model):
    """capture (raw rows, raw rewards, dones, statistics and record before) at every normalisation pass"""
    nz, raw = model.normalizer, []
    orig = nz.process_rollout

    def spy(obs_store, reward, done, K, *a, **k):
        raw.append((obs_store[..., :15].cpu().numpy(), reward.cpu().numpy(), done.bool().cpu().numpy(),
                    nz.stats.cpu().numpy(), nz.affine.cpu().numpy()))
        return orig(obs_store, reward, done, K, *a, **k)
    nz.process_rollout = spy
    return raw


PPO_SHAPES = ((1, 2048, "fp32"), (257, 32, "fp32"), (2048, 16, "tf32"))
PPO_MODES = ((1, 0), (0, 1), (1, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PPO_SHAPES, ids=[f"n{s[0]}-K{s[1]}-{s[2]}" for s in PPO_SHAPES])
@pytest.mark.parametrize("mode", PPO_MODES, ids=["obs", "reward", "both"])
def test_ppo_loop_follows_the_oracle(drl, shape, mode):
    from drone_rl_b200.ppo import PPO
    n, K, prec = shape
    norm_obs, norm_rew = mode
    gamma, clip_obs, clip_rew, eps = 0.95, 5.0, 3.0, 1e-3
    model = PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=6), n_steps=K, batch_size=min(n * K, 4096), n_epochs=1,
                gamma=gamma, seed=6, rollout_precision=prec, norm_obs=bool(norm_obs), norm_reward=bool(norm_rew),
                clip_obs=clip_obs, clip_reward=clip_rew, norm_epsilon=eps)
    raw = _spy(model)
    ora = no.FrozenVecNormalize(n, gamma=gamma, norm_obs=bool(norm_obs), norm_reward=bool(norm_rew), clip_obs=clip_obs,
                                clip_reward=clip_rew, epsilon=eps)
    worst = {}
    for it, training in enumerate((True, True, False, True)):
        model.training = ora.training = training
        model.collect_rollouts()
        obs, rew, done, s0, aff0 = raw[-1]
        if not training:
            assert done.any(), "the evaluation rollout must end episodes"
        # teacher-forced: the oracle holds the statistics the kernel held before this rollout
        ora.obs_rms, ora.ret_rms = _rms(s0)
        _, rets = _returns_ref(ora.returns, rew, done, gamma, training)
        ora.apply(obs.astype(np.float64), rew.astype(np.float64), done)
        buf_obs, buf_rew = model.buf.obs.cpu().numpy(), model.buf.reward.cpu().numpy()
        s1 = model.normalizer.stats.cpu().numpy()
        if norm_obs:
            assert _same(buf_obs, no.normalize_obs_f32(obs, _rms(s0)[0], clip_obs, eps)), f"rows, iteration {it}"
        if norm_rew:
            assert _same(buf_rew, no.normalize_reward_f32(rew, s0[32], clip_rew, eps)), f"rewards, iteration {it}"
            assert _same(model.normalizer.returns.cpu().numpy(), ora.returns), f"returns, iteration {it}"
        if not training:
            assert _same(s1, s0)
        else:
            depth = no.pass_depth(K, n)
            if norm_obs:
                s2 = np.square(obs.astype(np.float64) - s0[:15]).reshape(-1, 15).sum(0)
                bm, bv = no.one_pass_bound(s0[:15], s0[15:30], s0[30], s2, K * n, depth)
                ref = _rms(s0)[0]
                ref.update_from_moments(*no.two_pass_moments(obs.reshape(-1, 15)), K * n)
                worst["obs"] = max(worst.get("obs", 0.0), _ratio(s1[:15] - ref.mean, bm), _ratio(s1[15:30] - ref.var, bv))
                assert s1[30] == ora.obs_rms.count
            if norm_rew:
                s2 = np.square(rets - s0[31]).sum()
                bm, bv = no.one_pass_bound(s0[31], s0[32], s0[33], s2, K * n, depth)
                ref = _rms(s0)[1]
                ref.update_from_moments(*no.two_pass_moments(rets.reshape(-1)), K * n)
                worst["ret"] = max(worst.get("ret", 0.0), _ratio(s1[31] - ref.mean, bm), _ratio(s1[32] - ref.var, bv))
                assert s1[33] == ora.ret_rms.count
            assert max(worst.values(), default=0.0) <= 1.0, worst
        model.train()
    print(f"n {n} K {K} {prec} obs {norm_obs} reward {norm_rew}: worst err / bound {worst}")
    model.close()


# ---------------------------------------------------------------------------------------------------------------------
# data parallel on one GPU: two normalisers play two ranks over the two halves of one buffer
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_ranks_on_one_gpu_equal_one_normaliser_over_the_union(drl, recorded):
    from drone_rl_b200 import _lib
    from drone_rl_b200.core import _ptr
    from drone_rl_b200.normalize import ObsNormalizer
    from tests.test_gpu_dp import _handles
    dev, lib = torch.device("cuda", 0), _lib.load()
    h, K, eps = 3000, 8, 1e-8
    n = 2 * h
    hs = _handles(lib, 2)
    streams = [torch.cuda.Stream() for _ in range(2)]
    ranks = [ObsNormalizer(h, dev, gamma=0.97) for _ in range(2)]
    one = ObsNormalizer(n, dev, gamma=0.97)
    rng = np.random.default_rng(4)
    obs_rec, rew_rec, done_rec = recorded
    for it in range(2):
        idx = rng.integers(0, obs_rec.shape[0], K * n)
        raw, rew = obs_rec[idx].reshape(K, n, 15), rew_rec[idx].reshape(K, n)
        done = torch.from_numpy(done_rec[idx].reshape(K, n).astype(np.uint8)).to(dev)
        s_one = one.stats.cpu().numpy()
        bufs = [(torch.from_numpy(raw[:, r * h:(r + 1) * h].copy()).to(dev), torch.from_numpy(rew[:, r * h:(r + 1) * h].copy()).to(dev),
                 done[:, r * h:(r + 1) * h].contiguous()) for r in range(2)]
        whole = (torch.from_numpy(raw).to(dev), torch.from_numpy(rew).to(dev), done)
        torch.cuda.synchronize()
        for r in range(2):
            with torch.cuda.stream(streams[r]):
                st = C.c_void_p(streams[r].cuda_stream)
                ar = (lambda t, r=r, st=st: _lib.check(lib.dronecu_ppo_dp_allreduce_f64(hs[r], _ptr(t), t.numel(), st)))
                ranks[r].process_rollout(*bufs[r], K, allreduce=ar)
        one.process_rollout(*whole, K)
        torch.cuda.synchronize()
        for r in range(2):
            assert torch.equal(ranks[r].returns, one.returns[r * h:(r + 1) * h])
            if it == 0:          # the same initial record; later ones differ from the union's by its reduce order
                assert torch.equal(bufs[r][0], whole[0][:, r * h:(r + 1) * h])
                assert torch.equal(bufs[r][1], whole[1][:, r * h:(r + 1) * h])
        s0, s1 = ranks[0].stats.cpu().numpy(), ranks[1].stats.cpu().numpy()
        assert _same(s0, s1) and torch.equal(ranks[0].affine, ranks[1].affine), "ranks must hold identical statistics"
        if it > 0:
            continue
        ref = one.stats.cpu().numpy()
        depth = no.pass_depth(K, n)
        m = one.moments.cpu().numpy()
        bm, bv = no.one_pass_bound(s_one[:15], s_one[15:30], s_one[30], m[15:30], K * n, depth)
        rm, rv = no.one_pass_bound(s_one[31], s_one[32], s_one[33], m[32], K * n, depth)
        worst = max(_ratio(s0[:15] - ref[:15], 2 * bm), _ratio(s0[15:30] - ref[15:30], 2 * bv),
                    _ratio(s0[31] - ref[31], 2 * rm), _ratio(s0[32] - ref[32], 2 * rv))
        assert s0[30] == ref[30] and s0[33] == ref[33]
        print(f"iteration {it}: two ranks vs one over the union, worst err / bound {worst:.3g}")
        assert worst <= 1.0
    for hh in hs:
        lib.dronecu_ppo_destroy(hh)


# ---------------------------------------------------------------------------------------------------------------------
# predict-time normaliser
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B", [0, 1, 127, 128, 129, (1 << 20) + 1])
def test_predict_normaliser(drl, B):
    from drone_rl_b200.normalize import ObsNormalizer
    dev = torch.device("cuda", 0)
    rows = (OFFSETS + SCALES * np.random.default_rng(B).standard_normal((B, 15))).astype(np.float32)
    s = np.concatenate([OFFSETS + 0.3 * SCALES, (1.7 * SCALES) ** 2, [50.0, 0.0, 1.0, 50.0]])
    on, off = ObsNormalizer(1, dev, clip_obs=2.0, epsilon=1e-2), ObsNormalizer(1, dev, norm_obs=False)
    _set_stats(on, s)
    _set_stats(off, s)
    got = on.normalize_obs(torch.from_numpy(rows)).cpu().numpy()
    assert _same(got, no.normalize_obs_f32(rows, _rms(s)[0], 2.0, 1e-2))
    x = torch.from_numpy(rows).to(dev)
    y = off.normalize_obs(x)
    assert _same(y.cpu().numpy(), rows) and (B == 0 or y.data_ptr() != x.data_ptr())
