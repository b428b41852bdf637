"""The covering designs of tests/test_gpu_eval_parity.py and tests/test_gpu_rollout_parity.py against the kernel
dispatch of csrc/capi_ppo.cu: each of the 12 policy evaluation and 12 policy rollout kernels (thread per env, warp per
env, tensor cores, each for RANDOMIZED x NORM) runs, and meets every level of every other factor of its design."""
import pytest

pytest.importorskip("torch")

from oracle import eval_oracle as eo  # noqa: E402
from tests import test_gpu_eval_parity as evp  # noqa: E402
from tests import test_gpu_rollout_parity as rp  # noqa: E402

K_WARP_ROLLOUT_MAX_ENVS = 8192     # capi_ppo.cu kWarpRolloutMaxEnvs
TILE = 128                         # kPolBlock = tc::kTile: envs per CTA of the thread-per-env and tensor-core kernels
SMALL_WARPS = 4                    # kSmallWarps: envs per CTA of the warp-per-env kernels


def test_eval_design_reaches_every_instantiation():
    cases = evp.design()
    got = {(c["kernel"], c["randomized"], c["norm"]) for c in cases}
    assert got == set(evp.INSTANCES) and len(got) == 12
    ns = {c["n"] for c in cases}
    # both sides of one CTA / tile, a partial warp-kernel CTA, and both sides of the automatic warp / thread switch
    assert {1, TILE + 1} <= ns and any(n % SMALL_WARPS for n in ns) and K_WARP_ROLLOUT_MAX_ENVS + 1 in ns
    assert all(c["n"] <= K_WARP_ROLLOUT_MAX_ENVS + 1 for c in cases)


def test_eval_design_meets_every_level_with_every_instantiation():
    cases = evp.design()
    levels = {"n": set(evp.NS), "cfg": set(evp.CONFIGS), "split": set(evp.SPLITS), "chunks": set(evp.CHUNKS),
              "extra_eps": {0, 2}, "start": set(evp.STARTS), "t0": set(evp.CLOCKS), "off": set(evp.OFFSETS),
              "det": {False, True}, "policy": set(evp.POLICIES)}
    for inst in evp.INSTANCES:
        mine = [c for c in cases if (c["kernel"], c["randomized"], c["norm"]) == inst]
        assert len(mine) == len(evp.NS)
        for factor, want in levels.items():
            assert {c[factor] for c in mine} == want, (inst, factor)
    # the clock that crosses 32 bits meets the stochastic mode, under which the noise index matters
    assert any(c["t0"] == (1 << 32) - 3 and not c["det"] for c in cases)
    # every kernel meets the non-default constants under the wide policy
    for k in evp.KERNELS:
        assert {c["cfg"] for c in cases if c["kernel"] == k and c["policy"] == "wide"} >= {"A", "B"}, k


@pytest.mark.parametrize("n", evp.NS)
def test_splits(n):
    """the splits are what their names say"""
    t = {name: eo.shard_targets(*evp.split(name, n), n) for name in evp.SPLITS}
    assert t["last"].tolist() == [0] * (n - 1) + [1]
    assert (t["half"] == 0).sum() == n // 2 and set(t["half"].tolist()) <= {0, 1}
    assert (t["one"] == 1).all() and (t["many"] >= 3).all() and (t["many"] > 3).any()
    for name in ("middle", "end"):
        n_eval, index0, n_global = evp.split(name, n)
        union = eo.shard_targets(n_eval, 0, n_global, n_global)
        assert index0 in (n, 2 * n) and t[name].tolist() == union[index0:index0 + n].tolist()


def test_rollout_design_reaches_every_instantiation_and_level():
    cases = rp.design()
    got = {(c["kernel"], c["randomized"], c["norm"]) for c in cases}
    assert len(got) == 12
    levels = {"n": set(rp.NS), "K": {1, 40, 230}, "start": {"fresh", "mid"}, "gs": {0, 12345}, "off": {0, 7 << 23},
              "det": {False, True}, "norm": {False, True}, "stride": {15, 16}, "policy": {"hover", "wide"},
              "cfg": set(rp.CONFIGS), "randomized": {False, True}}
    for k in rp.KERNELS:
        mine = [c for c in cases if c["kernel"] == k]
        assert len(mine) == len(rp.NS)
        for factor, want in levels.items():
            assert {c[factor] for c in mine} == want, (k, factor)
