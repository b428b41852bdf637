"""``python -m drone_rl_b200.train`` -- the reference's training driver (train.py:10-70) on the GPU path.

Same flow as the reference script:
  * resume from ``./dd.zip`` when it exists (``PPO.load(path, env, n_steps=2048 // n_envs, batch_size=64,
    learning_rate=3e-4)``, train.py:11-31), else a fresh ``PPO("MlpPolicy")`` with SB3's defaults (train.py:33-43);
  * a numbered run directory ``./tensorboard/drone_runs_<n>`` (helper.py:6-21 ``make_run_dir``);
  * scalars under SB3's key names (``rollout/ep_rew_mean``, ``train/value_loss`` ...) to stdout and to
    ``progress.csv`` / ``progress.jsonl`` and a TensorBoard event file (``events.out.tfevents.*``, written by
    ``tb_events.py`` -- the ``tensorboard`` package itself is not needed) in the run dir;
  * the trajectory callback (traj_tb.py:31-73): every ``record_interval``-th finished episode of env 0 is
    buffered and every ``block_size`` episodes the overlays XY / XZ / YZ are written -- here from the rollout
    buffer itself (``obs[:, 0, 0:3]`` is the position before each step: ONE device->host copy per rollout instead
    of one ``get_attr('pos')`` per env step), as ``.npz`` + a Pillow-drawn ``.png`` (matplotlib is absent);
  * ``total_timesteps = 2e6`` and ``model.save("ppo_drone_rel_obs_pos_reward")`` (train.py:11, :63-70).

Differences, on purpose: ``--n-envs`` (default 1 = the reference) scales the rollout to many GPU envs with
``n_steps = 2048 // n_envs`` exactly as the reference's resume branch spells it; under ``torchrun`` every rank
trains its shard and the gradient is all-reduced (SURVEY.md section 8e).
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import re
import time

import numpy as np


def make_run_dir(root_dir: str, prefix: str = "drone_runs_") -> str:
    """helper.py:6-21: next free ``<root>/<prefix><n>`` (n = 1 + the largest existing index), created."""
    os.makedirs(root_dir, exist_ok=True)
    pat = re.compile(rf"^{re.escape(prefix)}(\d+)$")
    taken = [int(m.group(1)) for m in (pat.match(name) for name in os.listdir(root_dir)) if m]
    run_dir = os.path.join(root_dir, f"{prefix}{max(taken, default=0) + 1}")
    os.makedirs(run_dir, exist_ok=True)
    return run_dir


class RunLogger:
    """stdout table + progress.csv + progress.jsonl + TensorBoard event file, SB3 key names."""

    def __init__(self, run_dir: str, stdout: bool = True):
        self.run_dir, self.stdout, self.rows, self.keys = run_dir, stdout, 0, None
        self.jsonl = open(os.path.join(run_dir, "progress.jsonl"), "w")
        self.csv_path = os.path.join(run_dir, "progress.csv")
        from .tb_events import EventFileWriter
        self.tb = EventFileWriter(run_dir)               # TensorBoard scalars (own writer: the package is not needed)

    def dump(self, values: dict, step: int):
        self.jsonl.write(json.dumps({"step": step, **values}) + "\n")
        self.jsonl.flush()
        if self.keys is None:
            self.keys = list(values)
            with open(self.csv_path, "w", newline="") as f:
                csv.writer(f).writerow(["step"] + self.keys)
        elif any(k not in self.keys for k in values):
            # keys that first appear now (eval/* after the first evaluation): rewrite the header with the extended key set
            # and pad the earlier rows, as SB3's CSV writer does
            self.keys += [k for k in values if k not in self.keys]
            with open(self.csv_path, newline="") as f:
                old = list(csv.reader(f))[1:]
            with open(self.csv_path, "w", newline="") as f:
                w = csv.writer(f)
                w.writerow(["step"] + self.keys)
                w.writerows(row + [""] * (len(self.keys) + 1 - len(row)) for row in old)
        with open(self.csv_path, "a", newline="") as f:
            csv.writer(f).writerow([step] + [values.get(k, "") for k in self.keys])
        self.tb.add_scalars(values, step)
        if self.stdout:
            groups: dict = {}
            for k, v in values.items():
                g, _, name = k.partition("/")
                groups.setdefault(g, []).append((name, v))
            width = 24
            print("-" * (2 * width + 7))
            for g in sorted(groups):
                print(f"| {g + '/':<{width}} | {'':<{width}} |")
                for name, v in sorted(groups[g]):
                    txt = f"{v:.3g}" if isinstance(v, float) else str(v)
                    print(f"|    {name:<{width - 3}} | {txt:<{width}} |")
            print("-" * (2 * width + 7), flush=True)
        self.rows += 1

    def close(self):
        self.jsonl.close()
        self.tb.close()


class TrajectoryCallback:
    """traj_tb.py:7-73 restated over the rollout buffer: positions of env 0, episode by episode."""

    def __init__(self, run_dir: str, record_interval: int = 25, block_size: int = 500, env_index: int = 0, tb=None):
        self.run_dir, self.record_interval, self.block_size, self.env_index = run_dir, record_interval, block_size, env_index
        self.tb = tb                           # EventFileWriter: the overlays also go to TensorBoard, as traj_tb.py:66 does
        self.positions: list = []
        self.episode_count = 0
        self.buffered: list = []
        self.blocks_written = 0

    def __call__(self, model) -> bool:
        # position BEFORE step t (drone.py:77-79); with norm_obs the buffer is normalised and the raw rows come from the tap
        tap = getattr(model, "side_obs", None)
        rows = tap if tap is not None and model.side_env == self.env_index else model.buf.obs[:, self.env_index]
        pos = rows[:, 0:3].cpu().numpy()
        done = model.buf.done[:, self.env_index].cpu().numpy().astype(bool)
        for t in range(pos.shape[0]):
            self.positions.append(pos[t])
            if done[t]:
                self.episode_count += 1
                traj = np.array(self.positions)
                if self.episode_count % self.record_interval == 0:
                    self.buffered.append(traj)
                if self.episode_count % self.block_size == 0 and self.buffered:
                    self._write_block(model.num_timesteps)
                self.positions = []
        return True

    def _write_block(self, step: int):
        block = self.episode_count // self.block_size
        base = os.path.join(self.run_dir, f"trajectory_block{block}")
        np.savez_compressed(base + ".npz", step=step, **{f"ep_{(i + 1) * self.record_interval}": t
                                                         for i, t in enumerate(self.buffered)})
        try:
            from PIL import Image, ImageDraw
            size, pad = 360, 24
            img = Image.new("RGB", (3 * size, size), "white")
            d = ImageDraw.Draw(img)
            allp = np.concatenate(self.buffered)
            lo, hi = allp.min(0), allp.max(0)
            span = np.maximum(hi - lo, 1e-6)
            for p, (i, j, tag) in enumerate([(0, 1, "XY"), (0, 2, "XZ"), (1, 2, "YZ")]):
                d.text((p * size + 6, 4), f"Overlay_{tag} block {block}", fill="black")
                for r, t in enumerate(self.buffered):
                    xs = p * size + pad + (t[:, i] - lo[i]) / span[i] * (size - 2 * pad)
                    ys = size - pad - (t[:, j] - lo[j]) / span[j] * (size - 2 * pad)
                    col = ((53 * r) % 200, (97 * r) % 200, (151 * r) % 200)
                    if len(xs) > 1:
                        d.line(list(zip(xs.tolist(), ys.tolist())), fill=col, width=1)
            img.save(base + ".png")
            if self.tb is not None:
                for p, tag in enumerate(("Overlay_XY", "Overlay_XZ", "Overlay_YZ")):
                    self.tb.add_image(f"Trajectory/{tag}_block{block}", img.crop((p * size, 0, (p + 1) * size, size)), step)
        except Exception:                                   # Pillow missing: the .npz is the record
            pass
        self.buffered = []
        self.blocks_written += 1


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--resume", default="./dd.zip", help="archive to resume from when it exists (train.py:10)")
    ap.add_argument("--total-timesteps", type=float, default=2e6)
    ap.add_argument("--n-envs", type=int, default=1, help="envs per GPU (reference: 1)")
    ap.add_argument("--n-steps", type=int, default=None, help="default 2048 // n_envs (train.py:14)")
    ap.add_argument("--batch-size", type=int, default=64)
    ap.add_argument("--n-epochs", type=int, default=10)
    ap.add_argument("--learning-rate", type=float, default=3e-4)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32"], help="policy MLP in the rollout: CUDA cores (parity path) or tcgen05")
    ap.add_argument("--update-precision", default=None, choices=["fp32", "tf32", "bf16"],
                    help="minibatch gradient: fp32 CUDA cores, tcgen05 all-tf32, or tcgen05 with bf16 weight-gradient operands "
                         "(default: fp32 with --precision fp32, bf16 with --precision tf32)")
    ap.add_argument("--norm-obs", action="store_true", help="normalise observations (SB3 VecNormalize norm_obs) in the rollout")
    ap.add_argument("--norm-reward", action="store_true", help="normalise rewards by the running std of the discounted return")
    ap.add_argument("--clip-obs", type=float, default=10.0, help="clip of the normalised observations")
    ap.add_argument("--handle-timeout-termination", action="store_true",
                    help="bootstrap time-limit ends with gamma * V(terminal observation), as SB3 does for Gymnasium time limits")
    ap.add_argument("--eval-freq", type=int, default=0,
                    help="evaluate the policy every this many vec-env steps (SB3 EvalCallback; 0 = no evaluation)")
    ap.add_argument("--n-eval-episodes", type=int, default=5)
    ap.add_argument("--n-eval-envs", type=int, default=1, help="evaluation envs per GPU")
    ap.add_argument("--eval-stochastic", action="store_true", help="evaluate with sampled actions instead of the mean")
    ap.add_argument("--tensorboard-root", default="./tensorboard")
    ap.add_argument("--save", default="ppo_drone_rel_obs_pos_reward")
    ap.add_argument("--quiet", action="store_true")
    args = ap.parse_args(argv)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from . import DroneBatch, EnvConfig
    from .ppo import PPO

    n_steps = args.n_steps or max(1, 2048 // args.n_envs)
    env = DroneBatch(args.n_envs, EnvConfig.single(), device=local, seed=args.seed, env_offset=rank * args.n_envs)
    kw = dict(n_steps=n_steps, batch_size=args.batch_size, learning_rate=args.learning_rate, n_epochs=args.n_epochs,
              seed=args.seed, rollout_precision=args.precision,
              update_precision=args.update_precision or ("bf16" if args.precision == "tf32" else "fp32"))
    if args.norm_obs or args.norm_reward:       # else: PPO.load takes the archive's own settings
        kw.update(norm_obs=args.norm_obs, norm_reward=args.norm_reward, clip_obs=args.clip_obs)
    if args.handle_timeout_termination:        # else: PPO.load takes the archive's own setting
        kw.update(handle_timeout_termination=True)
    if os.path.exists(args.resume):
        model = PPO.load(args.resume, env, **kw)
        if rank == 0:
            print(f"resumed from {args.resume} at {model.num_timesteps} timesteps")
    else:
        model = PPO(env, **kw)

    t0 = time.time()
    model.collect_rollouts()
    torch.cuda.synchronize()
    if rank == 0:
        print("Wall-clock per iter:", time.time() - t0)        # train.py:46-53 prints the same probe
    # the probe is not counted (learn() restarts the counter); it does advance the envs by one rollout, as the reference's
    # probe advances its env by one step (train.py:46-50)

    logger = cb = None
    if rank == 0:
        run_dir = make_run_dir(args.tensorboard_root, prefix="drone_runs_")
        logger = RunLogger(run_dir, stdout=not args.quiet)
        cb = TrajectoryCallback(run_dir, tb=logger.tb)
        if model.normalizer is not None and model.normalizer.norm_obs:
            model.set_raw_obs_tap(cb.env_index)

    eval_cb = None
    if args.eval_freq > 0:
        from .evaluation import EvalCallback
        run_dirs = [logger.run_dir if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(run_dirs, src=0)
        eval_env = DroneBatch(args.n_eval_envs, EnvConfig.single(), device=local, seed=args.seed + 1,
                              env_offset=rank * args.n_eval_envs)
        eval_cb = EvalCallback(eval_env, n_eval_episodes=args.n_eval_episodes, eval_freq=args.eval_freq,
                               deterministic=not args.eval_stochastic, log_path=run_dirs[0], best_model_save_path=run_dirs[0],
                               verbose=int(rank == 0 and not args.quiet))

    def on_iteration(m):
        if eval_cb is not None:
            eval_cb(m)
        if rank == 0:
            cb(m)
            logger.dump(dict(m.logger_values), m.num_timesteps)
        for k in [k for k in m.logger_values if k.startswith("eval/")]:      # SB3 records them for the evaluation's row only
            del m.logger_values[k]
        return True

    # SB3 semantics (reset_num_timesteps=True): total_timesteps MORE steps, also after a resume (train.py:22-30, :63-68)
    model.learn(total_timesteps=int(args.total_timesteps), callback=on_iteration)
    model.save(args.save)            # rank 0: the archive; other ranks: their env / curriculum shard next to it
    if rank == 0:
        logger.close()
        print(f"saved {args.save}.zip; run dir {logger.run_dir}")
    model.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
