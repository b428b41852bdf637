#!/usr/bin/env python
"""Cost of the time-limit bootstrap (PPO(handle_timeout_termination=True)) on one GPU, flag off and on alternated in the
same process, CUDA events around whole calls after a warm-up:
    c5      1,048,576 envs x 32 steps, full iteration (collect + 10 epochs x 4 minibatches), tf32 rollout, bf16 update, from
            the initial policy (episodes mostly crash before the 200-step limit)
    stress  the c3 shape with max_steps = 8: T = 4 slots per env and every env truncates whenever it survives 8 steps
    c3      1,048,576 envs x 32 steps, tensor-core rollout alone (collect_rollouts: rollout [+ bootstrap] + GAE)
Each also times the bootstrap launch alone, and counts the truncated rows of the last rollout.
    python profiles/timeout_cost.py OUT.json"""
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


def pair(make, step, rounds, reps):
    """ms per call of `step` for the plain and the bootstrapping model, alternated `rounds` times; median per model."""
    models = {"off": make(False), "on": make(True)}
    for m in models.values():
        step(m)
        step(m)
    torch.cuda.synchronize()
    t = {k: [] for k in models}
    t_boot = []
    for _ in range(rounds):
        for k, m in models.items():
            t[k].append(timed(lambda: step(m), reps))
        t_boot.append(timed(models["on"]._bootstrap_timeouts, reps))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
    on = models["on"]
    out = {"ms_off": med["off"], "ms_on": med["on"], "overhead_ms": med["on"] - med["off"],
           "overhead_pct": 100.0 * (med["on"] - med["off"]) / med["off"], "bootstrap_ms": sorted(t_boot)[len(t_boot) // 2],
           "slots": int(on.timeout_row.numel()), "truncated_rows_last_rollout": int((on.timeout_row >= 0).sum()),
           "env_steps_per_rollout": on.n_envs * on.n_steps, "ms_off_all": t["off"], "ms_on_all": t["on"]}
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

    def model(flag, max_steps=200):
        return PPO(drl.DroneBatch(n, drl.EnvConfig.single(max_steps=max_steps), seed=0), n_steps=K, batch_size=n * K // 4,
                   n_epochs=10, seed=0, rollout_precision="tf32", update_precision="bf16", handle_timeout_termination=flag)

    def it(m):
        m.collect_rollouts()
        m.train()
    res["c5"] = pair(model, it, rounds=5, reps=3)
    print("c5", {k: v for k, v in res["c5"].items() if not k.endswith("_all")}, flush=True)
    res["stress_max_steps_8"] = pair(lambda f: model(f, 8), lambda m: m.collect_rollouts(), rounds=5, reps=10)
    print("stress", {k: v for k, v in res["stress_max_steps_8"].items() if not k.endswith("_all")}, flush=True)
    res["c3"] = pair(model, lambda m: m.collect_rollouts(), rounds=5, reps=10)
    print("c3", {k: v for k, v in res["c3"].items() if not k.endswith("_all")}, flush=True)
    res["_doc"] = __doc__
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    json.dump(res, open(path, "w"), indent=1)
    print(card)


if __name__ == "__main__":
    main(sys.argv[1])
