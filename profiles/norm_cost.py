#!/usr/bin/env python
"""Cost of observation / reward normalisation (PPO(norm_obs=True, norm_reward=True)) on one GPU, off and on alternated in
the same process, CUDA events around whole calls after a warm-up:
    c3  1,048,576 envs x 32 steps, tensor-core rollout: collect_rollouts (rollout + GAE) vs (rollout + pass + reduce +
        combine + GAE), plus the pass + reduce + combine alone
    c5  the same size, full iteration: collect + 10 epochs x 4 minibatches, bf16 update
    c1  1 env x 2048 steps (fp32, warp-per-env rollout): the pass is one thread walking 2048 steps
    python profiles/norm_cost.py OUT.json"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / reps


def pair(make, step, rounds, reps, extra=None):
    """ms per call of `step` for the plain and the normalising model, alternated `rounds` times; median per model."""
    models = {"off": make(False), "on": make(True)}
    for m in models.values():
        step(m)
        step(m)
    torch.cuda.synchronize()
    t = {k: [] for k in models}
    t_extra = []
    for _ in range(rounds):
        for k, m in models.items():
            t[k].append(timed(lambda: step(m), reps))
        if extra is not None:
            t_extra.append(timed(lambda: extra(models["on"]), reps))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
    out = {"ms_off": med["off"], "ms_on": med["on"], "overhead_ms": med["on"] - med["off"],
           "overhead_pct": 100.0 * (med["on"] - med["off"]) / med["off"], "ms_off_all": t["off"], "ms_on_all": t["on"]}
    if extra is not None:
        out["norm_pass_reduce_combine_ms"] = sorted(t_extra)[len(t_extra) // 2]
    for m in models.values():
        m.close()
    torch.cuda.empty_cache()
    return out


def main(path):
    import drone_rl_b200 as drl
    from drone_rl_b200.ppo import PPO
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    res = {"card": card, "torch": torch.__version__}
    n, K = 1 << 20, 32

    def c3(norm):
        return PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=0), n_steps=K, batch_size=n * K // 4, n_epochs=10, seed=0,
                   rollout_precision="tf32", update_precision="bf16", padded_obs=False, norm_obs=norm, norm_reward=norm)
    b = lambda m: m.normalizer.process_rollout(m.buf.obs_store, m.buf.reward, m.buf.done, K)
    res["c3"] = pair(c3, lambda m: m.collect_rollouts(), rounds=5, reps=10, extra=b)
    print("c3", {k: v for k, v in res["c3"].items() if not k.endswith("_all")}, flush=True)

    def c5(norm):
        return PPO(drl.DroneBatch(n, drl.EnvConfig.single(), seed=0), n_steps=K, batch_size=n * K // 4, n_epochs=10, seed=0,
                   rollout_precision="tf32", update_precision="bf16", norm_obs=norm, norm_reward=norm)

    def it(m):
        m.collect_rollouts()
        m.train()
    res["c5"] = pair(c5, it, rounds=5, reps=3)
    print("c5", {k: v for k, v in res["c5"].items() if not k.endswith("_all")}, flush=True)

    def c1(norm):
        return PPO(drl.DroneBatch(1, drl.EnvConfig.single(), seed=0), n_steps=2048, batch_size=64, n_epochs=10, seed=0,
                   norm_obs=norm, norm_reward=norm)
    b1 = lambda m: m.normalizer.process_rollout(m.buf.obs_store, m.buf.reward, m.buf.done, 2048)
    res["c1_rollout"] = pair(c1, lambda m: m.collect_rollouts(), rounds=5, reps=5, extra=b1)
    print("c1_rollout", {k: v for k, v in res["c1_rollout"].items() if not k.endswith("_all")}, flush=True)
    res["_doc"] = __doc__
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    json.dump(res, open(path, "w"), indent=1)
    print(card)


if __name__ == "__main__":
    main(sys.argv[1])
