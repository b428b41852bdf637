"""The covering design of tests/test_gpu_env_parity.py against the kernel dispatch of csrc/capi_env.cu: every one of the
32 rollout_kernel instantiations and every CTA size is reached, and every instantiation meets every level of every
other factor of the design."""
import itertools

import pytest

pytest.importorskip("torch")

from tests import test_gpu_env_parity as ep  # noqa: E402


def _instantiation(case):
    """capi_env.cu launch_rollout restated: (D, RANDOMIZED, AUTORESET) from the config flags, ACT_MODE from the entry point
    (dronecu_step always streams), RECORD from the output pointers"""
    D, R, AR, mode, _ = case["inst"]
    outs = ep.output_set(case["out"], mode)
    if "step" in outs:
        mode = 0
    return D, R, AR, mode, ep.record_rule(outs, mode)


def test_design_reaches_every_instantiation_and_cta_size():
    cases = ep.design()
    got = {_instantiation(c) for c in cases}
    want = set(itertools.product((15, 12), (True, False), (True, False), (0, 1), (True, False)))
    assert got == want and len(want) == 32
    for c in cases:
        assert _instantiation(c) == c["inst"], ep._case_id(c)
    assert {ep.block_for(c["n"]) for c in cases} == {32, 64, 256}
    # both sides of both CTA-size switches
    assert ep.block_for(18943) == 32 and ep.block_for(18944) == 64
    assert ep.block_for(75775) == 64 and ep.block_for(75776) == 256


def test_design_meets_every_level_with_every_instantiation():
    cases = ep.design()
    levels = {"n": set(ep.NS), "K": set(ep.KS), "cfg": set(ep.CONFIGS), "start": set(ep.STARTS), "t0": set(ep.CLOCKS),
              "off": set(ep.OFFSETS), "misalign": {False, True}}
    for inst in ep.INSTANCES:
        mine = [c for c in cases if c["inst"] == inst]
        for factor, want in levels.items():
            assert {c[factor] for c in mine} >= want, (inst, factor)
        _, _, AR, mode, rec = inst
        outs = {c["out"] for c in mine}
        if rec:
            assert outs == {"record"}
        else:
            assert outs >= set(ep.GEN_OUTS) | ({"step"} if mode == 0 else set()), (inst, outs)
        if not AR:
            assert any(c["K"] >= 1000 for c in mine)
    assert any(c["n"] > 148 * 256 for c in cases)        # more than 128 CTAs: statistics slots are shared
