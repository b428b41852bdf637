"""Every policy evaluation kernel -- thread per env, warp per env, tensor cores (csrc/ppo_eval.cuh), each instantiated for
RANDOMIZED x NORM -- against its rollout twin, and the twin against float64, over a covering design of launch shapes,
env constants, episode splits, probe chunkings, slot row strides (max_eps), start states, clocks, env offsets, modes and policies.
One case per (kernel, instantiation, n); the other factors cycle from a per-instantiation offset with periods <= 6, so
every instantiation meets every level (tests/test_policy_dispatch.py asserts it).

Per case, ``dronecu_evaluate_policy`` runs the case's launch sequence on one handle (outputs in guarded buffers), and a
twin handle with the same config, seed, offset, state and clock runs the same-flavour rollout kernel for the
evaluation's T steps with the full record.  Then:
  twin vs float64     every check of tests/test_gpu_rollout_parity.py (_check_record, _check_stats) on every env, or on a
                      strided sample of about CHECKED transitions that keeps the first and last warp / tile and every env
                      with a non-zero target of a sparse split
  launch contract     after every launch, steps and count exactly as oracle/eval_oracle.launch_sequence replays them over
                      the twin's record; after a probe, pending = the envs below target; a catch-up leaves pending alone
                      and brings every env to T
  episodes            ep_return bit-equal to the float32 replay of the rewards from the state's ep_ret, ep_length exact;
                      slots past count, rows of envs past their target and every guard region keep the sentinel
  state and clock     final state planes bit-identical to the twin's; the handle's clock and episode statistics untouched
  end to end          fresh single-shard cases: evaluation.evaluate_policy gives the lists and T of
                      eval_oracle.episodes_from_transitions on the twin's record
"""
import ctypes as C
import threading
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import eval_oracle as eo  # noqa: E402
from tests import test_gpu_rollout_parity as rp  # noqa: E402
from tests.test_gpu_env_parity import Guarded  # noqa: E402

SEED = rp.SEED
KERNELS = ("thread", "warp", "tc")
INSTANCES = [(k, R, norm) for k in KERNELS for R in (True, False) for norm in (False, True)]
NS = (1, 33, 129, 1025, 4097, 8193)
CONFIGS = ("single", "A", "B")
SPLITS = ("last", "half", "one", "many", "middle", "end")
CHUNKS = ("one", "plus1", "plus7")
STARTS = ("fresh", "mid")
CLOCKS = (0, 12345, (1 << 32) - 3)
OFFSETS = (0, (1 << 32) + 7)
POLICIES = ("hover", "wide")
CHECKED = 30_000          # twin transitions checked against float64 per case (a strided sample of envs above this)
FIRST_PROBE = 1 << 20     # the "one" chunking: a single probe past any T of the design


def split(name, n):
    """(n_eval_episodes, env_index0, n_global) of an episode split over a shard of n envs"""
    return {"last": (1, 0, n),                    # only the last env records
            "half": (-(-n // 2), 0, n),           # the first floor(n / 2) envs have target 0
            "one": (n, 0, n),
            "many": (3 * n + 5, 0, n),
            "middle": (2 * n + 3, n, 3 * n),      # the middle shard of three
            "end": (2 * n + 3, 2 * n, 3 * n)}[name]


def design():
    cases = []
    for ii, (kernel, R, norm) in enumerate(INSTANCES):
        for j, n in enumerate(NS):
            cases.append(dict(kernel=kernel, randomized=R, norm=norm, n=n, cfg=CONFIGS[(j + ii) % 3],
                              split=SPLITS[(j + ii) % 6], chunks=CHUNKS[(j // 2 + ii) % 3],
                              extra_eps=2 * ((j + ii // 3) % 2), start=STARTS[(j // 3 + ii) % 2],
                              t0=CLOCKS[(2 * j + ii) % 3], off=OFFSETS[((j + 1) // 3 + ii) % 2],
                              det=(j + ii // 2) % 2 == 1, policy=POLICIES[(j // 2 + ii) % 2]))
    return cases


def case_id(c):
    return (f"{c['kernel']}-{'rand' if c['randomized'] else 'fixed'}-{'norm' if c['norm'] else 'raw'}-n{c['n']}-{c['cfg']}"
            f"-{c['split']}-{c['chunks']}-eps+{c['extra_eps']}-{c['start']}-t{c['t0']}-off{c['off']}"
            f"-{'det' if c['det'] else 'stoch'}-{c['policy']}")


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


# ---------------------------------------------------------------------------------------------------------------------
# one evaluation through the C entry point
# ---------------------------------------------------------------------------------------------------------------------
def _start(b, cfg, start, rng):
    """fresh: after reset(); mid: steps within 3 of the time limit, ep_num just below curriculum bumps, ep_ret != 0"""
    b.reset()
    if start == "mid":
        n, ms, per = b.n, cfg.max_steps, cfg.curriculum_period
        step = rng.integers(ms - 3, ms, n).astype(np.int32)
        ep_num = rng.choice([per - 1, 2 * per - 1, 5 * per - 1], n).astype(np.int32)
        b.set_state(step=step, ep_len=step, ep_num=ep_num, ep_ret=(-rng.uniform(0.1, 3, n)).astype(np.float32))


class Evaluation:
    """The arguments and guarded outputs of one evaluation on handle ``b``; ``launch`` runs one probe or catch-up."""

    def __init__(self, b, theta_dev, affine, tc, n_eval, index0, n_global, max_eps, t0, det):
        n = b.n
        self.b, self.theta, self.affine, self.tc = b, theta_dev, affine, int(tc)
        self.steps, self.count = Guarded((n,), torch.int32), Guarded((n,), torch.int32)
        self.steps.view.zero_()
        self.count.view.zero_()
        self.ret, self.len = Guarded((n, max_eps)), Guarded((n, max_eps), torch.int32)
        self.pending = Guarded((1,), torch.int32)
        from drone_rl_b200 import _lib
        a = _lib.EvalArgs()
        a.t0, a.deterministic, a.max_eps = t0, int(det), max_eps
        a.env_index0, a.n_global, a.n_eval_episodes = index0, n_global, n_eval
        a.d_steps, a.d_count, a.d_ep_return, a.d_ep_length, a.d_pending = (
            g.view.data_ptr() for g in (self.steps, self.count, self.ret, self.len, self.pending))
        self.args = a

    def launch(self, limit, catch_up):
        from drone_rl_b200 import _lib
        self.args.limit, self.args.catch_up = int(limit), int(catch_up)
        self.pending.view.fill_(0 if not catch_up else -12345)
        aff = None if self.affine is None else C.c_void_p(self.affine.data_ptr())
        _lib.check(self.b.lib.dronecu_evaluate_policy(self.b._h, C.c_void_p(self.theta.data_ptr()), aff, self.tc,
                                                      C.byref(self.args), None), "dronecu_evaluate_policy")
        torch.cuda.synchronize()
        return {"steps": self.steps.view.cpu().numpy(), "count": self.count.view.cpu().numpy(),
                "pending": int(self.pending.view.item())}

    def guards_intact(self):
        return all(g.guards_intact() for g in (self.steps, self.count, self.ret, self.len, self.pending))


def run_probes(ev, chunks):
    """the case's probe limits, then the catch-up to T; returns [(limit, catch_up)] and what each launch left"""
    launches, got = [], []
    limit, k = 0, 0
    while True:
        if chunks == "one":
            limit = FIRST_PROBE
        else:
            limit += 1 if chunks == "plus1" else (7 if k != 1 else 0)     # plus7: the second probe repeats the first
        launches.append((limit, False))
        got.append(ev.launch(limit, False))
        k += 1
        if got[-1]["pending"] == 0:
            break
        assert k < 10_000, "the evaluation does not end"
    T = int(got[-1]["steps"].max())
    launches.append((T, True))
    got.append(ev.launch(T, True))
    return launches, got, T


# ---------------------------------------------------------------------------------------------------------------------
# the twin: the same-flavour rollout over the evaluation's T steps, checked against float64
# ---------------------------------------------------------------------------------------------------------------------
def sample_columns(n, T, kernel, always=()):
    """every env, or a strided sample of about CHECKED transitions with the first and last warp (tensor cores: tile)"""
    if n * T <= CHECKED:
        return np.arange(n)
    w = 128 if kernel == "tc" else 32
    stride = max(1, (n * T) // CHECKED)
    return np.unique(np.concatenate([np.arange(0, n, stride), np.arange(min(n, w)), np.arange(max(0, n - w), n),
                                     np.asarray(always, np.int64)]))


def run_twin(twin, kernel, T, theta, theta_dev, det, nz, t0, set_mode, cols, max_transitions=8_000_000):
    """T steps of the twin in launches of at most ``max_transitions``; every launch checked on ``cols`` (the episode
    statistics over every env).  Returns reward [T, n], done [T, n], the worst err/bound per check and whether the
    recorded actions crossed 0 and motor_max."""
    n = twin.n
    Kc = max(1, min(T, max_transitions // n))
    rewards, dones, worst = [], [], {}
    mm = float(np.float32(twin.config.motor_max))
    below = above = False
    sel = None if len(cols) == n else torch.from_numpy(cols).cuda()
    k0 = 0
    while k0 < T:
        K = min(Kc, T - k0)
        st0 = twin.get_state()
        rec = rp._launch(twin, kernel, K, theta_dev, det, 15, None if nz is None else nz.affine, set_mode)
        stats = twin.episode_stats(reset=True)
        w, rep, done_s, rets, length_sum = rp._check_record(twin, rec, theta, theta_dev, kernel, det, nz, st0, t0 + k0,
                                                            cols=sel)
        reward, done = rec["reward"].cpu().numpy(), rec["done"].cpu().numpy().astype(bool)
        if sel is None:
            rp._check_stats(stats, done, rets, length_sum, rep)
        else:
            from tests.test_gpu_env_parity import _check_stats_sampled
            _, _, _, _, rets_all, ls_all = rp._expected_after(st0, done, reward)
            _check_stats_sampled(stats, done, rets_all, ls_all, st0, twin.config.max_steps, True)
        for key, v in w.items():
            worst[key] = max(worst.get(key, 0.0), v)
        a = rec["actions"]
        below, above = below or bool((a < 0).any()), above or bool((a > mm).any())
        rewards.append(reward)
        dones.append(done)
        del rec
        k0 += K
    return np.concatenate(rewards), np.concatenate(dones), worst, (below, above)


def same_lists(a, b):
    """two (returns, lengths) list pairs: the returns bit-identical as float32 (a NaN matching a NaN), the lengths equal"""
    return len(a[0]) == len(b[0]) and rp._same_f32(a[0], b[0]) and list(a[1]) == list(b[1])


def _theta_and_norm(case, cfg, n):
    theta = rp._policy(case["policy"], cfg.motor_max)
    nz = rp._norm_affine(n) if case["norm"] else None
    return theta, torch.from_numpy(theta).cuda(), nz


def _stand_in_model(theta_dev, nz, kernel):
    """what evaluation.evaluate_policy reads of a model"""
    return types.SimpleNamespace(params=theta_dev, normalizer=nz, rollout_precision="tf32" if kernel == "tc" else "fp32",
                                 tc_min_envs=0 if kernel == "tc" else 1 << 62)


def run_case(drl, c, set_mode):
    kernel, n = c["kernel"], c["n"]
    cfg = rp.make_config(drl, c["cfg"], c["randomized"])
    n_eval, index0, n_global = split(c["split"], n)
    targets = eo.shard_targets(n_eval, index0, n_global, n)
    max_eps = -(-n_eval // n_global) + c["extra_eps"]
    rng = np.random.default_rng(n * 17 + len(case_id(c)))
    theta, theta_dev, nz = _theta_and_norm(c, cfg, n)
    if kernel != "tc":
        set_mode({"thread": 1, "warp": 2}[kernel])

    b = drl.DroneBatch(n, cfg, seed=SEED, env_offset=c["off"])
    twin = drl.DroneBatch(n, cfg, seed=SEED, env_offset=c["off"])
    _start(b, cfg, c["start"], rng)
    st0 = b.get_state()
    twin.set_state(**st0)
    for h in (b, twin):
        h.global_step = c["t0"]
        h.episode_stats(reset=True)

    ev = Evaluation(b, theta_dev, None if nz is None else nz.affine, kernel == "tc", n_eval, index0, n_global, max_eps,
                    c["t0"], c["det"])
    launches, got, T = run_probes(ev, c["chunks"])
    assert T >= 1
    assert b.global_step == c["t0"], "the evaluation kernels keep no clock"
    stats = b.episode_stats()
    assert stats["episodes"] == 0 and stats["env_steps"] == 0, "the evaluation kernels keep no episode statistics"
    assert ev.guards_intact(), "a guard region was overwritten"

    # the twin, pinned against float64
    cols = sample_columns(n, T, kernel, np.flatnonzero(targets) if c["split"] in ("last", "half") else ())
    reward, done, worst, (below, above) = run_twin(twin, kernel, T, theta, theta_dev, c["det"], nz, c["t0"], set_mode, cols)
    if c["policy"] == "wide" and not c["det"] and n * T >= 1000:
        assert below and above, "the wide policy must cross both clip limits"

    # every launch against the bookkeeping over the twin's record
    after, want_r, want_l, written = eo.launch_sequence(reward, done, targets, launches, max_eps,
                                                        st0["ep_ret"], st0["ep_len"])
    for k, ((limit, catch_up), g, w) in enumerate(zip(launches, got, after)):
        what = f"launch {k} ({'catch-up' if catch_up else 'probe'} to {limit})"
        assert np.array_equal(g["steps"], w["steps"]), f"{what}: steps"
        assert np.array_equal(g["count"], w["count"]), f"{what}: count"
        if catch_up:
            assert g["pending"] == -12345, f"{what}: a catch-up wrote pending"
            assert (g["steps"] == T).all()
        else:
            assert g["pending"] == w["pending"], f"{what}: pending {g['pending']}, envs below target {w['pending']}"
    assert np.array_equal(got[-1]["count"], targets)
    untouched_r = ev.ret.untouched().cpu().numpy()
    untouched_l = ev.len.untouched().cpu().numpy()
    assert np.array_equal(~untouched_r, written) and np.array_equal(~untouched_l, written), "slots written off the record"
    got_r, got_l = ev.ret.view.cpu().numpy(), ev.len.view.cpu().numpy()
    assert rp._same_f32(got_r[written], want_r[written]), "episode returns"
    assert np.array_equal(got_l[written], want_l[written]), "episode lengths"
    st_b, st_t = b.get_state(), twin.get_state()
    for key in st_b:
        assert np.array_equal(st_b[key].view(np.uint32), st_t[key].view(np.uint32)), f"final {key} differs from the twin"
    assert twin.global_step == c["t0"] + T

    # fresh, one shard: the SB3 bookkeeping and evaluation.evaluate_policy end to end
    if c["start"] == "fresh" and n_global == n:
        ref_r, ref_l, ref_T = eo.episodes_from_transitions(reward, done, n_eval)
        assert ref_T == T
        lists = eo.sb3_order(eo.episode_lists(got[-1]["count"], got_r, got_l))
        assert same_lists(lists, (ref_r, ref_l))
        from drone_rl_b200 import evaluation
        e2e = drl.DroneBatch(n, cfg, seed=SEED, env_offset=c["off"])
        e2e.global_step = c["t0"]
        chunk = evaluation.PROBE_CHUNK
        evaluation.PROBE_CHUNK = {"one": chunk, "plus1": 1, "plus7": 7}[c["chunks"]]     # several probes per evaluation
        try:
            r, l = evaluation.evaluate_policy(_stand_in_model(theta_dev, nz, kernel), e2e, n_eval, deterministic=c["det"],
                                              return_episode_rewards=True)
        finally:
            evaluation.PROBE_CHUNK = chunk
        assert same_lists((r, l), (ref_r, ref_l)) and e2e.global_step == c["t0"] + T
        st_e = e2e.get_state()
        for key in st_e:
            assert np.array_equal(st_e[key].view(np.uint32), st_t[key].view(np.uint32)), f"end to end: final {key}"
        e2e.close()
    b.close()
    twin.close()
    return T, len(launches), len(cols), worst


@pytest.mark.gpu
@pytest.mark.parametrize("case", design(), ids=case_id)
def test_eval_parity(drl, rollout_kernel_mode, case):
    T, nl, m, worst = run_case(drl, case, rollout_kernel_mode)
    print(f"{case_id(case)}: T {T}, launches {nl}, envs checked {m}; worst err/bound "
          + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# automatic kernel choice, production size
# ---------------------------------------------------------------------------------------------------------------------
def _rollout_lists(drl, cfg, n, st0, t0, T, theta_dev, mode, set_mode, n_eval):
    twin = drl.DroneBatch(n, cfg, seed=SEED, env_offset=0)
    twin.set_state(**st0)
    twin.global_step = t0
    rec = rp._launch(twin, "thread" if mode == 1 else "warp", T, theta_dev, True, 15, None, set_mode)
    reward, done = rec["reward"].cpu().numpy(), rec["done"].cpu().numpy().astype(bool)
    del rec
    try:
        lists = eo.episodes_from_transitions(reward, done, n_eval)
    except ValueError:               # this flavour's envs had not all reached their targets after the evaluation's T
        lists = None
    out = lists, twin.get_state()
    twin.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n,expect", [(8192, "warp"), (8193, "thread")])
def test_auto_dispatch(drl, rollout_kernel_mode, n, expect):
    """dronecu_set_rollout_kernel(0): one warp per env up to kWarpRolloutMaxEnvs = 8192 envs, one thread per env above.
    The kernel that ran is the flavour whose rollout twin it matches bit for bit (the warp kernel's head sums are warp
    reductions, so the two flavours part in the last bits and then in the trajectories)."""
    cfg = rp.make_config(drl, "single")
    theta_dev = torch.from_numpy(rp._policy("hover")).cuda()
    b = drl.DroneBatch(n, cfg, seed=SEED)
    b.reset()
    st0 = b.get_state()
    rollout_kernel_mode(0)
    ev = Evaluation(b, theta_dev, None, False, 2 * n, 0, n, 2, 0, True)
    _, got, T = run_probes(ev, "one")
    lists = eo.sb3_order(eo.episode_lists(got[-1]["count"], ev.ret.view.cpu().numpy(), ev.len.view.cpu().numpy()))
    st_b = b.get_state()
    match = {}
    for mode, name in ((1, "thread"), (2, "warp")):
        ref, st_t = _rollout_lists(drl, cfg, n, st0, 0, T, theta_dev, mode, rollout_kernel_mode, 2 * n)
        rollout_kernel_mode(0)
        match[name] = (ref is not None and same_lists(lists, ref[:2]) and ref[2] == T
                       and all(np.array_equal(st_b[k].view(np.uint32), st_t[k].view(np.uint32)) for k in st_b))
    assert match == {"thread": expect == "thread", "warp": expect == "warp"}, match
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["thread", "tc"])
def test_eval_parity_at_production_size(drl, rollout_kernel_mode, kernel):
    """2^20 + 1 envs under config A (23-step episodes keep T short), one episode each, stochastic: every check of
    test_eval_parity, the twin on a strided sample of envs plus the first and last warp / tile."""
    c = dict(kernel=kernel, randomized=True, norm=False, n=(1 << 20) + 1, cfg="A", split="one", chunks="plus7",
             extra_eps=0, start="fresh", t0=(1 << 32) - 3, off=OFFSETS[1], det=False, policy="wide")
    T, nl, m, worst = run_case(drl, c, rollout_kernel_mode)
    print(f"{case_id(c)}: T {T}, launches {nl}, envs checked {m}; worst err/bound "
          + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# three shards on one GPU through evaluation.py's distributed branch
# ---------------------------------------------------------------------------------------------------------------------
class ThreadGroup:
    """The collectives evaluation.py calls, for ``world`` threads of one process: all_gather, all_reduce (SUM, MAX),
    all_gather_object, each synchronised by a barrier.  ``_dist()`` gives every thread its own rank."""

    class ReduceOp:
        SUM, MAX = "sum", "max"

    def __init__(self, world):
        self.world, self.barrier, self.local = world, threading.Barrier(world, timeout=600), threading.local()
        self.slots = [None] * world

    def _exchange(self, value):
        self.slots[self.local.rank] = value
        self.barrier.wait()
        every = list(self.slots)
        self.barrier.wait()
        return every

    def all_gather(self, out, t):
        for o, v in zip(out, self._exchange(t.clone())):
            o.copy_(v)

    def all_reduce(self, t, op="sum"):
        every = self._exchange(t.clone())
        acc = every[0].clone()
        for v in every[1:]:
            acc = acc + v if op == "sum" else torch.maximum(acc, v)
        t.copy_(acc)

    def all_gather_object(self, out, obj):
        out[:] = self._exchange(obj)

    def dist(self):
        return self, self.local.rank, self.world


@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 1025])
@pytest.mark.parametrize("kernel", ["thread", "tc"])
def test_three_shards_equal_one_batch(drl, rollout_kernel_mode, monkeypatch, kernel, n):
    """Three DroneBatch shards of n envs (env_offset r n), one thread each through evaluation.evaluate_policy with the
    collectives of ThreadGroup, equal one batch of 3n envs: the lists, T, the clock and every shard's final state
    against its slice."""
    from drone_rl_b200 import evaluation
    world, n_eval = 3, 2 * 3 * n + 5
    cfg = rp.make_config(drl, "B")
    theta_dev = torch.from_numpy(rp._policy("hover", cfg.motor_max)).cuda()
    model = _stand_in_model(theta_dev, None, kernel)
    if kernel != "tc":
        rollout_kernel_mode(1)
    t0 = 12345
    one = drl.DroneBatch(world * n, cfg, seed=SEED)
    one.global_step = t0
    r1, l1 = evaluation.evaluate_policy(model, one, n_eval, deterministic=False, return_episode_rewards=True)
    group = ThreadGroup(world)
    monkeypatch.setattr(evaluation, "_dist", group.dist)
    shards = [drl.DroneBatch(n, cfg, seed=SEED, env_offset=r * n) for r in range(world)]
    results, errors = [None] * world, []

    def worker(r):
        group.local.rank = r
        try:
            shards[r].global_step = t0
            results[r] = evaluation.evaluate_policy(model, shards[r], n_eval, deterministic=False, return_episode_rewards=True)
        except BaseException as e:          # noqa: BLE001  (reported below, after every thread has ended)
            errors.append(e)
            group.barrier.abort()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    assert len(r1) == n_eval
    for r in range(world):
        assert same_lists(results[r], (r1, l1)), f"rank {r}: lists differ from one batch"
        assert shards[r].global_step == one.global_step > t0
    st1, T = one.get_state(), one.global_step - t0
    for r in range(world):
        st = shards[r].get_state()
        for key in st:
            assert np.array_equal(st[key].view(np.uint32), st1[key][r * n:(r + 1) * n].view(np.uint32)), (r, key)
        shards[r].close()
    one.close()
    print(f"{kernel} 3 x {n} envs, {n_eval} episodes: T {T}")
