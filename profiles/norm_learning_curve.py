#!/usr/bin/env python
"""The round-2 learning-curve command (4096 envs x 64 steps, batch 65,536, 1e8 env-steps; fp32 and tf32 rollout precision;
seeds 0-3) with and without --norm-obs --norm-reward; final ep_rew_mean / ep_len_mean / explained_variance per run:
    python profiles/norm_learning_curve.py OUT.json [total_timesteps]"""
import json
import os
import subprocess
import sys
import tempfile

out = sys.argv[1]
total = sys.argv[2] if len(sys.argv) > 2 else "1e8"
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
runs = {}
keep = ("step", "rollout/ep_rew_mean", "rollout/ep_len_mean", "train/explained_variance", "train/value_loss", "train/std", "time/fps")
for norm in (False, True):
    for prec in ("fp32", "tf32"):
        for seed in range(4):
            d = tempfile.mkdtemp()
            cmd = [sys.executable, "-m", "drone_rl_b200.train", "--n-envs", "4096", "--n-steps", "64", "--batch-size", "65536",
                   "--total-timesteps", total, "--precision", prec, "--seed", str(seed), "--quiet", "--tensorboard-root", d,
                   "--save", os.path.join(d, "m"), "--resume", os.path.join(d, "none.zip")] + (["--norm-obs", "--norm-reward"] if norm else [])
            subprocess.check_call(cmd, cwd=root, stdout=subprocess.DEVNULL)
            rows = [json.loads(l) for l in open(os.path.join(d, "drone_runs_1", "progress.jsonl"))]
            key = f"{'norm' if norm else 'raw'}/{prec}/seed{seed}"
            runs[key] = {"first": {k: rows[0].get(k) for k in keep}, "final": {k: rows[-1].get(k) for k in keep}}
            print(key, runs[key]["final"], flush=True)
os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
json.dump({"_doc": __doc__, "card": card, "total_timesteps": total, "runs": runs}, open(out, "w"), indent=1)
