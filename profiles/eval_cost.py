#!/usr/bin/env python
"""Cost of policy evaluation (drone_rl_b200.evaluation.evaluate_policy, csrc/ppo_eval.cuh) on one GPU, same process, after
a warm-up, evaluation and rollout alternated:
    big    1,048,576 eval envs, one deterministic episode each (fp32 thread-per-env kernel, and tf32 tensor-core kernel):
           the evaluation kernels (probe and catch-up launches, CUDA events around each, summed) against a deterministic
           dronecu_rollout_policy[_tc] of the same T steps with no buffer outputs on an identical env (CUDA events);
           env-steps/s = n * T / time.  Also the whole evaluate_policy call (reset, launches, readbacks, the episode
           lists built on the host) with a host clock; it ends in a device synchronise
    small  EvalCallback's default shape: 1 env x 5 episodes (fp32 warp-per-env kernel), wall time per evaluation
The policy is the initial one with the action-head bias at the hover thrust per motor (m g / 4), so that episodes last long.
    python profiles/eval_cost.py OUT.json"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def hover_model(drl, precision):
    from drone_rl_b200.ppo import PPO
    from oracle import ppo_oracle as po
    model = PPO(drl.DroneBatch(16, drl.EnvConfig.single(), seed=1), n_steps=8, seed=1, rollout_precision=precision)
    flat = po.init_params(5, torch.float64)
    off = po.offsets()["pi.b3"][0]
    flat[off:off + 4] = 9.81 / 4
    model.params.copy_(flat.float())
    return model


def med(v):
    return sorted(v)[len(v) // 2]


def main(path):
    import drone_rl_b200 as drl
    from drone_rl_b200 import _lib
    from drone_rl_b200.evaluation import evaluate_policy
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    res = {"card": card, "torch": torch.__version__}
    n = 1 << 20
    for precision in ("fp32", "tf32"):
        model = hover_model(drl, precision)
        ev = drl.DroneBatch(n, drl.EnvConfig.single(), seed=0)
        ro = drl.DroneBatch(n, drl.EnvConfig.single(), seed=0)
        fn = model.lib.dronecu_rollout_policy_tc if precision == "tf32" else model.lib.dronecu_rollout_policy

        real, events = ev.lib, []

        class Timed:                            # CUDA events around every evaluation launch
            def __getattr__(self, name):
                return getattr(real, name)

            def dronecu_evaluate_policy(self, *a):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                rc = real.dronecu_evaluate_policy(*a)
                e.record()
                events.append((s, e))
                return rc
        ev.lib = Timed()

        def evaluate():
            t0 = ev.global_step
            events.clear()
            torch.cuda.synchronize()
            w = time.perf_counter()
            evaluate_policy(model, ev, n, deterministic=True)
            torch.cuda.synchronize()
            wall = time.perf_counter() - w
            return sum(s.elapsed_time(e) for s, e in events) / 1e3, wall, len(events), ev.global_step - t0

        def rollout(T):
            ro.reset()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            _lib.check(fn(ro._h, T, C.c_void_p(model.params.data_ptr()), 1, None, None), "dronecu_rollout_policy")
            e.record()
            e.synchronize()
            return s.elapsed_time(e) / 1e3

        T = evaluate()[-1]                      # warm-up of both, and T
        rollout(T)
        t_ev, t_wall, t_ro, Ts, launches = [], [], [], [], []
        for _ in range(5):
            dt, wall, nl, T_i = evaluate()
            t_ev.append(dt)
            t_wall.append(wall)
            launches.append(nl)
            Ts.append(T_i)
            t_ro.append(rollout(T_i))
        r = {"n_envs": n, "T": Ts, "eval_launches": launches, "eval_kernels_s": t_ev, "eval_call_wall_s": t_wall,
             "rollout_s": t_ro, "eval_env_steps_per_s": n * Ts[0] / med(t_ev),
             "eval_call_env_steps_per_s": n * Ts[0] / med(t_wall), "rollout_env_steps_per_s": n * Ts[0] / med(t_ro)}
        r["ratio_eval_over_rollout"] = r["eval_env_steps_per_s"] / r["rollout_env_steps_per_s"]
        res[precision] = r
        print(precision, {k: v for k, v in r.items() if not isinstance(v, list)}, "T", Ts, flush=True)
        model.close(); ev.close(); ro.close()
        torch.cuda.empty_cache()

    model = hover_model(drl, "fp32")
    small = drl.DroneBatch(1, drl.EnvConfig.single(), seed=0)
    evaluate_policy(model, small, 5)
    walls = []
    for _ in range(20):
        torch.cuda.synchronize()
        w = time.perf_counter()
        evaluate_policy(model, small, 5)
        walls.append(time.perf_counter() - w)
    res["eval_callback_default"] = {"n_envs": 1, "n_eval_episodes": 5, "wall_s_median": med(walls), "wall_s_all": walls}
    print("eval_callback_default", med(walls), flush=True)
    model.close(); small.close()
    res["_doc"] = __doc__
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    json.dump(res, open(path, "w"), indent=1)
    print(card)


if __name__ == "__main__":
    main(sys.argv[1])
