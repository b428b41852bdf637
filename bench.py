#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused quadcopter env step and of the PPO rollout + update on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--workload c4|c2|k1|c3|c5|c1] [--only] [--impl reference] [--dump-outputs DIR]

ONE JSON line on stdout.  Its top level is the step-only workload `c4` (configs[3]'s per-GPU shard: the configuration the
metric's "at 1/2/4/8 B200" is quoted on); `"workloads"` carries the other halves of the metric measured in the same run:

  c4 (top level) configs[3] per-GPU shard: 8,388,608 envs per GPU (= 64M over 8 GPUs, weak scaling), DroneGymEnv spec
                 (15-dim obs, curriculum target, auto-reset), in-kernel Philox random actions, 32 env steps fused per launch.
  c2             configs[1]: VectorizedDroneEnv spec, 4096 envs x 1000 steps, random actions streamed from HBM, one launch
                 (N = 1 only: the config is "1 x B200").
  c3             configs[2]: 1,048,576 envs per GPU, fused K-step rollout with the PPO MLP policy / value forward in-kernel:
                 tcgen05 path (tf32) and the fp32 parity path, both reported.
  c5             configs[4]: full PPO iteration (rollout + GAE + 10 epochs x 4 minibatches; for N > 1 the gradient exchange
                 + clip + Adam over NVLink peer memory): tensor-core paths and the fp32 parity path, both reported.
  k1 / c1        on request (--workload): the K = 1 SB3 boundary; configs[0], the reference's own shape (1 env).

One bench "step" = ONE pass of the workload's hot path over its batch (c4 / c2 / k1: one launch of the fused kernel; c3: one
rollout launch + GAE; c5 / c1: one PPO iteration).  `value` = env-steps/s over all ranks with inputs resident in HBM, timed
with CUDA events on the launching stream, max over ranks; `roofline` = the dominant kernel against the measured peak, from
CUDA events inside the run; `e2e` = the same metric through the reference-facing API with host buffers / host results
(wall clock, copies inside); `cpu_baseline` = the reference's CPU path for that workload on this box's host cores.

--steps K times K steps of every workload's value (the e2e, sustained and fp32 parity-path figures keep their own counts).
A full run therefore times K PPO iterations of c3 and of c5 at 1M envs, and the reference arm runs K iterations of its CPU
PPO loop for each: at large K that, not the step-only workloads, sets the wall time of a run.
--only runs just the workload named by --workload (A/B timing, ncu captures).
--dump-outputs DIR writes, for every workload timed in the run, what its timed path returned in its last step as
DIR/<workload>_<name>.npy (float32; float64 for the env index): all envs, or a fixed sample of env columns where the full
arrays exceed 12 MB (<workload>_env_index.npy says which; a --fuse at which one env alone exceeds it is refused), so a run
writes at most 64 MB.  Inputs are seeded (--seed), so two builds run with the same arguments can be compared output for
output.
--impl reference times the reference's CPU implementation: the UNMODIFIED reference env staged by oracle/make_ref.py
(oracle/_ref/reference_py.zip; kind "reference") where the reference has the path, the oracle port otherwise (the PPO loop
lives in stable-baselines3, which is not installable here: kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STATE_BYTES = 80                              # 5 quads per env, read once + written once per launch
MLP_FLOP = 20864.0                            # policy + value forward per env-step (2 x (15*64 + 64*64) + 64*4 + 64) x 2
MOTOR_MAX = 7.3575
DUMP_BYTES = 12 << 20                         # --dump-outputs, per workload: the four workloads of one run stay under 64 MB


def json_safe(o):
    """Strict JSON has no NaN / Infinity: non-finite floats (an undefined explained variance, an empty episode mean) become null."""
    if isinstance(o, float):
        return o if np.isfinite(o) else None
    if isinstance(o, (np.floating,)):
        return float(o) if np.isfinite(o) else None
    if isinstance(o, (np.integer,)):
        return int(o)
    if isinstance(o, dict):
        return {k: json_safe(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [json_safe(v) for v in o]
    return o


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return json.load(open(p)) if os.path.isfile(p) else {}


def hbm_peak():
    d = measured_peaks()
    if "hbm_gbs" in d:
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def tensor_peak():
    d = measured_peaks()
    if "bf16_tflops_sustained" in d:
        return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md)"


def static_traffic(key):
    """ncu dram__bytes of the dominant kernel per launch: a STATIC number from a committed capture (profiles/), not measured in
    this run -- the source is named next to it."""
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(prof))
        return d.get(key), d.get(f"_{key}_source")
    except Exception:
        return None, None


# ------------------------------------------------------------------------------------------------
# plumbing: stdout hygiene, clocks sampler
# ------------------------------------------------------------------------------------------------
class stdout_to_stderr:
    """NCCL (and torch's process group) print a version banner on STDOUT when the communicator is created; the contract is ONE
    JSON line on stdout, so file descriptor 1 points at stderr while the process group initialises and runs its first collective."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)


class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.ok = [], set(), False
        self._stop = threading.Event()
        if os.environ.get("DRONECU_NO_CLOCKS") == "1":          # debugging aid: no sampler thread
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.ok:
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.ok:
            self.t.join()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": float(self.max),
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU legs: the reference's own env (staged archive) or the numpy port, on the host cores
# ------------------------------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(kind, spec_name, n_envs, seed):
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    np.seterr(all="ignore")
    rng = np.random.default_rng(seed)
    # a small pool of pre-drawn action batches: drawing random numbers is not part of the env step being timed
    _W["acts"] = [rng.uniform(0, MOTOR_MAX, (n_envs, 4)).astype(np.float32).astype(np.float64) for _ in range(4)]
    _W["n"] = n_envs
    if kind == "reference":
        from oracle import ref_import
        _, vd = ref_import.load()
        _W["env"] = vd.VectorizedDroneEnv(n_envs)          # vectorized_drone.py:12-216, unmodified
    else:
        from oracle import drone_oracle as do
        spec = do.SINGLE if spec_name == "single" else do.VECTOR
        _W["env"] = do.BatchedDroneOracle(n_envs, spec, seed=seed, env_offset=seed * n_envs)
    _W["env"].reset()


def _cpu_worker_steps(k_inner):
    env, acts = _W["env"], _W["acts"]
    for i in range(k_inner):
        env.step(acts[i & 3])
    return _W["n"] * k_inner


class CpuEnvPool:
    """`cores` worker processes, each stepping its own batch of the reference env (or of its numpy port)."""

    def __init__(self, cores, envs_per_core, kind, spec_name):
        import multiprocessing as mp
        self.cores, self.envs_per_core, self.kind, self.spec_name = cores, envs_per_core, kind, spec_name
        ctx = mp.get_context("spawn")
        self.pools = [ctx.Pool(1, initializer=_cpu_worker_init, initargs=(kind, spec_name, envs_per_core, i)) for i in range(cores)]

    def step(self, k_inner):
        res = [p.apply_async(_cpu_worker_steps, (k_inner,)) for p in self.pools]
        return sum(r.get() for r in res)

    def time(self, budget_s, k_inner=8):
        self.step(2)                                  # warm-up (imports, first touch)
        t0, units = time.perf_counter(), 0
        while True:
            units += self.step(k_inner)
            dt = time.perf_counter() - t0
            if dt > budget_s:
                return units / dt, units, dt

    def close(self):
        for p in self.pools:
            p.terminate()


def reference_available():
    try:
        from oracle import ref_import
        return ref_import.available()
    except Exception:
        return False


def time_reference_gym_env(budget_s=2.0):
    """The reference's DroneGymEnv (drone.py:254-274), ONE env on one core, manual reset on done -- how train.py steps it."""
    from oracle import ref_import
    drone, _ = ref_import.load()
    env = drone.DroneGymEnv()
    env.reset()
    a = np.full(4, 2.0, dtype=np.float32)
    t0, n = time.perf_counter(), 0
    while time.perf_counter() - t0 < budget_s:
        for _ in range(200):
            _, _, done, _ = env.step(a)
            if done:
                env.reset()
        n += 200
    return n / (time.perf_counter() - t0)


def cpu_baseline_env(wl, cores, budget_s=8.0):
    """cpu_baseline of a step-only workload.  c4 / k1: the reference's fastest batched path (VectorizedDroneEnv.step, no
    auto-reset: a conservative denominator) on all cores, the numpy port of the DroneGymEnv spec (with auto-reset: the spec
    the GPU runs) beside it.  c2: VectorizedDroneEnv(4096) in ONE process, as the reference runs it, and on all cores."""
    have_ref = reference_available()
    kind = "reference" if have_ref else "port"
    out = {"unit": "env-steps/s", "cores": cores, "kind": kind}
    if wl == "c2":
        one = CpuEnvPool(1, 4096, kind, "vector")
        v1, u1, d1 = one.time(budget_s / 2)
        one.close()
        many = CpuEnvPool(cores, 4096, kind, "vector")
        vN, uN, dN = many.time(budget_s / 2)
        many.close()
        out.update(value=vN, value_1_process=v1,
                   sample=f"VectorizedDroneEnv(4096).step ({kind}), float64 numpy: {cores} processes x 4096 envs, {uN} env-steps in "
                          f"{dN:.1f}s; 1 process (how the reference runs configs[1]): {u1} env-steps in {d1:.1f}s")
        return out
    pool = CpuEnvPool(cores, 16384, kind, "vector")
    v, u, d = pool.time(budget_s * 0.6)
    pool.close()
    port = CpuEnvPool(cores, 16384, "port", "single")
    vp, up, dp = port.time(budget_s * 0.4)
    port.close()
    out.update(value=v, port_value_gym_spec=vp,
               sample=f"VectorizedDroneEnv.step ({kind}; the reference's batched path, no auto-reset): {cores} processes x 16384 envs, "
                      f"{u} env-steps in {d:.1f}s | numpy port of the DroneGymEnv spec + DummyVecEnv auto-reset (what the GPU "
                      f"workload computes): {up} env-steps in {dp:.1f}s")
    if have_ref:
        out["reference_gym_env_1_core"] = time_reference_gym_env()
        out["sample"] += " | reference DroneGymEnv, one env on one core (train.py's shape)"
    return out


PPO_CPU_SAMPLE = dict(n_envs=4096, n_steps=32, n_epochs=10, minibatches=4)


def cpu_baseline_ppo(wl, cores, budget_s=8.0):
    """The restated SB3 loop (oracle/ppo_loop.py: torch CPU on all host threads + the numpy env port): SB3 is not installable,
    so this leg is the port.  Batched like the GPU workload, and (c5 / c1) in the reference's own shape (train.py:33-43)."""
    import torch
    from oracle import ppo_loop
    out = {"unit": "env-steps/s", "cores": cores, "kind": "port"}
    if wl == "c1":
        v1, its1, dt1 = ppo_loop.time_loop(1, 2048, 64, 10, budget_s=2 * budget_s, update=True)
        out.update(value=v1, sample=f"restated SB3 loop on CPU (torch {torch.get_num_threads()} threads + numpy env port), the "
                                    f"reference's own config: 1 env, n_steps 2048, batch 64, 10 epochs; {its1} iterations in {dt1:.1f}s")
        return out
    c, update = PPO_CPU_SAMPLE, wl == "c5"
    v, its, dt = ppo_loop.time_loop(c["n_envs"], c["n_steps"], c["n_envs"] * c["n_steps"] // c["minibatches"], c["n_epochs"],
                                    budget_s=budget_s, update=update)
    sample = (f"restated SB3 loop on CPU (torch {torch.get_num_threads()} threads + numpy env port): {c['n_envs']} envs x {c['n_steps']} steps" +
              (f", {c['n_epochs']} epochs x {c['minibatches']} minibatches" if update else ", rollout only") + f"; {its} iterations in {dt:.1f}s")
    out.update(value=v, sample=sample)
    if update:
        v1, its1, dt1 = ppo_loop.time_loop(1, 2048, 64, 10, budget_s=budget_s, update=True)
        out["value_reference_shape"] = v1
        out["sample"] += f" | the reference's own config (1 env, n_steps 2048, batch 64, 10 epochs): {its1} iterations in {dt1:.1f}s"
    return out


WORKLOAD_NAMES = {
    "c4": "configs[3] shard: step-only fused rollout, 8388608 envs/GPU (64M over 8), DroneGymEnv spec, Philox actions",
    "c2": "configs[1]: vectorized step-only, 4096 envs x 1000 steps, random actions streamed from HBM",
    "k1": "SB3 boundary: one env step per launch (dronecu_step), 8388608 envs/GPU, streamed actions",
    "c3": "configs[2]: 1048576 envs fused K-step rollout with the PPO MLP policy/value forward in-kernel",
    "c5": "configs[4]: full PPO loop (in-kernel-policy rollout + GAE + 10-epoch minibatch update, gradient exchange over NVLink for N > 1)",
    "c1": "configs[0]: the reference's own shape -- ONE env, n_steps 2048, batch 64, 10 epochs (train.py defaults), full PPO loop",
}


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------
def reference_env_line(args, wl, cores):
    have_ref = reference_available()
    kind = "reference" if have_ref else "port"
    k_inner = 8
    per = 4096 if wl == "c2" else 16384
    pool = CpuEnvPool(cores, per, kind, "vector")
    for _ in range(max(1, args.warmup)):
        pool.step(k_inner)
    t0, units = time.perf_counter(), 0
    for _ in range(args.steps):
        units += pool.step(k_inner)
    dt = time.perf_counter() - t0
    pool.close()
    v = units / dt
    sample = (f"VectorizedDroneEnv.step ({'unmodified reference, oracle/_ref' if have_ref else 'numpy port'}), float64: {cores} processes x {per} "
              f"envs x {k_inner} env steps per bench step")
    return {"impl": "reference", "metric": "env_steps_per_sec", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD_NAMES[wl], "sample": sample},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def reference_ppo_line(args, wl, cores):
    from oracle import ppo_loop
    c = PPO_CPU_SAMPLE if wl != "c1" else dict(n_envs=1, n_steps=2048, n_epochs=10, minibatches=32)
    update = wl != "c3"
    loop = ppo_loop.PPOLoopOracle(c["n_envs"], c["n_steps"], c["n_envs"] * c["n_steps"] // c["minibatches"], c["n_epochs"])

    def one():
        loop.collect_rollouts()
        if update:
            loop.train()
    for _ in range(max(1, min(args.warmup, 2))):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    dt = time.perf_counter() - t0
    v = args.steps * c["n_envs"] * c["n_steps"] / dt
    sample = (f"restated SB3 loop on CPU (torch, all host threads + numpy env port; SB3 itself is not installable): {c['n_envs']} envs x "
              f"{c['n_steps']} steps per bench step" + (f", {c['n_epochs']} epochs x {c['minibatches']} minibatches" if update else ", rollout only"))
    return {"impl": "reference", "metric": "env_steps_per_sec", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_NAMES[wl], "sample": sample},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def run_reference(args):
    """Reference arm: the reference's CPU path on all host cores, same metric; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = os.cpu_count() or 1
    wl = args.workload
    line = reference_ppo_line(args, wl, cores) if wl in ("c3", "c5", "c1") else reference_env_line(args, wl, cores)
    if wl == "c4" and not args.only:
        extra = {}
        for w in (["c2"] if args.gpus == 1 else []) + ["c3", "c5"]:
            sub = reference_ppo_line(args, w, cores) if w in ("c3", "c5") else reference_env_line(args, w, cores)
            extra[w] = {k: sub[k] for k in ("value", "unit", "ms_per_step", "steps", "dtype", "config", "cpu_baseline")}
        line["workloads"] = extra
    print(json.dumps(json_safe(line), allow_nan=False), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, dump=False):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.dump = {} if dump else None          # name -> array, filled by capture()
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device and no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            with stdout_to_stderr():
                dist.init_process_group("nccl", device_id=self.dev)
                dist.barrier()                           # creates the communicator (and prints NCCL's banner) now
                torch.cuda.synchronize()
        import drone_rl_b200 as drl
        self.drl = drl

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()

    def capture(self, wl, arrays):
        """--dump-outputs: host float32 copies of `arrays` ({name: device tensor [steps, n, ...]}, what a caller of the timed path
        receives) -- every env, or a fixed, seeded sample of env columns where the arrays exceed DUMP_BYTES."""
        if self.dump is None:
            return
        torch = self.torch
        n = next(iter(arrays.values())).shape[1]
        per_env = 4 * sum(t[:, 0].numel() for t in arrays.values())
        if per_env > DUMP_BYTES:
            raise SystemExit(f"bench.py --dump-outputs: one env of {wl} returns {per_env} bytes per step, more than the "
                             f"{DUMP_BYTES}-byte sample; use a smaller --fuse")
        m = min(n, DUMP_BYTES // per_env)
        idx = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
        sel = torch.from_numpy(idx).to(self.dev)
        self.dump[f"{wl}_env_index"] = idx.astype(np.float64)
        for name, t in arrays.items():
            self.dump[f"{wl}_{name}"] = t.index_select(1, sel).float().cpu().numpy()


def bench_env(ctx, args, wl, steps, warmup, want_cpu):
    """c4 / c2 / k1: one launch of the fused kernel per bench step."""
    torch, drl, dev, world, rank = ctx.torch, ctx.drl, ctx.dev, ctx.world, ctx.rank
    if wl == "c2":
        n, fuse, cfg = 4096, 1000, drl.EnvConfig.vector()
    else:
        n, fuse, cfg = args.envs_per_gpu, (1 if wl == "k1" else args.fuse), drl.EnvConfig.single()
    D = cfg.obs_dim
    batch = drl.DroneBatch(n, cfg, device=ctx.local, seed=args.seed, env_offset=rank * n)
    nxt = torch.empty(fuse, n, D, device=dev)
    rew = torch.empty(fuse, n, device=dev)
    done = torch.empty(fuse, n, dtype=torch.uint8, device=dev)
    if wl == "c4":
        acts_in, acts_out = None, torch.empty(fuse, n, 4, device=dev)
    else:
        gen = torch.Generator(device=dev).manual_seed(args.seed + rank)
        acts_in, acts_out = torch.rand(fuse, n, 4, device=dev, generator=gen) * MOTOR_MAX, None

    def one_step():
        if wl == "k1":
            batch.step(acts_in[0], out={"obs": nxt[0], "reward": rew[0], "done": done[0]})
        else:
            batch.rollout(fuse, acts_in, next_obs=nxt, out_actions=acts_out, reward=rew, done=done)
        if wl == "c2":
            batch.reset()                  # configs[1] is ONE 1000-step episode of the shared counter: start the next pass fresh

    for _ in range(warmup):
        one_step()
    ctx.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps)]
    l0 = batch.launch_count
    with ClockSampler(ctx.local) as clocks:
        for i in range(steps):
            ev[2 * i].record()
            if wl == "k1":
                batch.step(acts_in[0], out={"obs": nxt[0], "reward": rew[0], "done": done[0]})
            else:
                batch.rollout(fuse, acts_in, next_obs=nxt, out_actions=acts_out, reward=rew, done=done)
            ev[2 * i + 1].record()
            if wl == "c2":
                batch.reset()
        ctx.barrier()
    launches = batch.launch_count - l0
    last = slice(0, 1 if wl == "k1" else fuse)
    ctx.capture(wl, dict(next_obs=nxt[last], reward=rew[last], done=done[last],
                         **({"actions": acts_out} if acts_out is not None else {})))
    per = [ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(steps)]      # ms per launch of the dominant kernel
    sustained = None
    if wl == "c4" and args.sustain_s > 0:
        # the timed region is short (steps x ~4 ms): also show the behaviour over seconds -- same launches back to back,
        # clocks sampled every 20 ms (a separate figure: it is not the headline value)
        reps = max(steps, int(args.sustain_s / max(np.mean(per) * 1e-3, 1e-6)))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(ctx.local) as sclk:
            s0.record()
            for _ in range(reps):
                batch.rollout(fuse, acts_in, next_obs=nxt, out_actions=acts_out, reward=rew, done=done)
            s1.record()
            ctx.barrier()
        s_ms = ctx.max_over_ranks(s0.elapsed_time(s1))
        sustained = {"launches": reps, "seconds": s_ms * 1e-3, "value": n * fuse * reps * world / (s_ms * 1e-3), "unit": "env-steps/s",
                     "clocks": sclk.summary()}
    total_ms = ctx.max_over_ranks(ev[0].elapsed_time(ev[-1]))
    units = n * fuse * steps * world
    value = units / (total_ms * 1e-3)

    in_bytes = 16 if acts_in is not None else 0
    out_bytes = D * 4 + 4 + 1 + (16 if acts_out is not None else 0)
    alg_bytes_per_launch = n * (fuse * (in_bytes + out_bytes) + 2 * STATE_BYTES)
    avg_ms = float(np.mean(per))
    peak, peak_src = hbm_peak()
    achieved = alg_bytes_per_launch / (avg_ms * 1e-3) / 1e9
    traffic, traffic_src = static_traffic(wl)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": (traffic_src + " (ncu, static: not measured in this run)") if traffic else None,
                "peak_source": peak_src, "kernel": "rollout_kernel" if wl != "k1" else "step_kernel",
                "algorithmic_bytes_per_env_step": in_bytes + out_bytes + 2 * STATE_BYTES / fuse,
                "avg_launch_ms": avg_ms, "min_launch_ms": float(np.min(per))}
    if wl == "c2":
        # 4096 envs = 128 warps on 148 SMs: one warp per SM, every env a chain of 1000 DEPENDENT steps -- the bound is the
        # latency of one step's dependent instruction chain, not HBM (DESIGN.md section 4.1, profiles/r02_c2_chain_model.md)
        sm_hz = 1.965e9
        roofline["latency_model"] = {"bound": "dependent chain (one warp per SM)", "cycles_per_env_step_per_warp": avg_ms * 1e-3 * sm_hz / fuse,
                                     "note": "hbm frac is reported for the contract; the kernel cannot be HBM-bound at 128 warps"}

    del nxt, rew, done, acts_in, acts_out
    torch.cuda.empty_cache()
    e2e = None if args.no_e2e else e2e_env(ctx, args, wl, n, cfg, steps)
    batch.close()
    res = {"value": value, "unit": "env-steps/s", "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps, "dtype": "f32",
           "config": {"workload": WORKLOAD_NAMES[wl], "envs_per_gpu": n, "env_steps_per_launch": fuse, "obs_dim": D,
                      "outputs": "next_obs+action+reward+done" if wl == "c4" else "next_obs+reward+done",
                      "l2": "inputs larger than L2 (state %.0f MB, outputs %.1f GB per launch)" % (n * STATE_BYTES / 1e6, n * fuse * out_bytes / 1e9)
                      if wl != "c2" else "every launch streams 65.5 MB of actions in and 213 MB of records out (L2 126 MB): nothing is reused"},
           "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks.summary()}
    if sustained:
        res["sustained"] = sustained
    if want_cpu:
        res["cpu_baseline"] = cpu_baseline_env(wl, os.cpu_count() or 1)
    return res


def e2e_env(ctx, args, wl, n, cfg, steps):
    """The reference-facing call with HOST buffers, wall clock, every call copies its inputs H2D and its results D2H.
    c4 / k1: DroneVecEnv.step (SB3 VecEnv surface; arrays instead of 8M dicts) with pinned numpy buffers.
    c2: VectorizedDroneGymEnv(4096).step -- the reference's own API for configs[1] (vectorized_drone.py:251-269): one env
    step per call, fresh numpy arrays returned."""
    torch, drl = ctx.torch, ctx.drl
    D = cfg.obs_dim
    if wl == "c2":
        env = drl.VectorizedDroneGymEnv(n, device=ctx.local)
        acts = np.random.default_rng(0).uniform(0, MOTOR_MAX, (n, 4)).astype(np.float32)
        calls, api = 1000, "VectorizedDroneGymEnv(4096).step (numpy in, fresh numpy out; 1000 calls = one episode of the shared counter)"
    else:
        env = drl.DroneVecEnv(n, seed=args.seed, device=ctx.local, env_offset=ctx.rank * n, info_mode="arrays", copy=False, config=cfg)
        acts = torch.empty(n, 4, pin_memory=True).uniform_(0, MOTOR_MAX).numpy()
        calls, api = max(3, min(steps, 10)), "DroneVecEnv.step (numpy, pinned; info as arrays)"
    env.reset()
    for _ in range(3):
        env.step(acts)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(calls):
        obs, rew, done, _ = env.step(acts)
    ctx.barrier()
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    checksum = float(np.asarray(rew[: min(n, 1024)], dtype=np.float64).sum())
    env.close()
    h2d, d2h = n * 16, n * (D * 4 + 4 + 1 + (1 if wl != "c2" else 0))
    res = {"value": n * calls * ctx.world / dt, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "api": api, "calls": calls, "ms_per_call": 1e3 * dt / calls, "reward_checksum": checksum}
    if wl != "c2":
        # the ceiling of this call on this box: the SAME bytes as plain pinned cudaMemcpyAsync copies (H2D on one stream, D2H
        # on another: PCIe is full duplex), no kernel, all ranks at once -- what the host / PCIe side allows at this N
        dev = ctx.dev
        hb_in = torch.empty(h2d, dtype=torch.uint8, pin_memory=True)
        hb_out = torch.empty(d2h, dtype=torch.uint8, pin_memory=True)
        db_in, db_out = torch.empty(h2d, dtype=torch.uint8, device=dev), torch.empty(d2h, dtype=torch.uint8, device=dev)
        s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

        def copies():
            with torch.cuda.stream(s_in):
                db_in.copy_(hb_in, non_blocking=True)
            with torch.cuda.stream(s_out):
                hb_out.copy_(db_out, non_blocking=True)
        copies()
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(calls):
            copies()
        ctx.barrier()
        dtc = ctx.max_over_ranks(time.perf_counter() - t0)
        res["copy_ceiling"] = {"value": n * calls * ctx.world / dtc, "unit": "env-steps/s", "d2h_gbs_per_gpu": d2h * calls / dtc / 1e9,
                               "h2d_gbs_per_gpu": h2d * calls / dtc / 1e9,
                               "what": "the same H2D + D2H bytes as bare pinned cudaMemcpyAsync on two streams, all ranks concurrently"}
        res["frac_of_copy_ceiling"] = res["value"] / res["copy_ceiling"]["value"]
        del hb_in, hb_out, db_in, db_out
        # callers whose policy lives on the GPU keep the observations there: actions H2D, reward + done D2H only
        env = drl.DroneVecEnv(n, seed=args.seed, device=ctx.local, env_offset=ctx.rank * n, info_mode="none", copy=False, config=cfg,
                              obs_device=True)
        env.reset()
        for _ in range(3):
            env.step(acts)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(calls):
            obs_d, rew, done, _ = env.step(acts)
        ctx.barrier()
        dto = ctx.max_over_ranks(time.perf_counter() - t0)
        env.close()
        res["obs_on_device"] = {"value": n * calls * ctx.world / dto, "unit": "env-steps/s", "h2d_bytes_per_step": n * 16,
                                "d2h_bytes_per_step": n * 5, "api": "DroneVecEnv(obs_device=True).step: numpy actions in, CUDA obs + numpy reward / done out",
                                "ms_per_call": 1e3 * dto / calls}
        torch.cuda.empty_cache()
    return res


def ppo_variant(ctx, args, wl, n, K, minibatches, epochs, rollout_precision, update_precision, steps, warmup, want_e2e,
                dump=False):
    """One precision variant of c3 / c5 / c1: timed region + the dominant kernel's CUDA-event time."""
    torch, drl, dev, world = ctx.torch, ctx.drl, ctx.dev, ctx.world
    from drone_rl_b200.ppo import PPO
    env = drl.DroneBatch(n, drl.EnvConfig.single(), device=ctx.local, seed=args.seed, env_offset=ctx.rank * n)
    full = wl in ("c5", "c1")
    # c3 collects rollouts only: no update kernel follows, so the buffer keeps SB3's packed 60-byte observation rows (the 64-byte
    # rows are the bf16 update kernel's input format: c5 / c1 take the model's default)
    model = PPO(env, n_steps=K, batch_size=n * K // minibatches, n_epochs=epochs, seed=args.seed,
                rollout_precision=rollout_precision, update_precision=update_precision, dp_backend=args.dp_backend,
                padded_obs=None if full else False)

    debug = os.environ.get("DRONECU_BENCH_DEBUG") == "1"

    def one_step():
        model.collect_rollouts()
        if full:
            model.train()
            if debug:
                print("[debug]", rollout_precision, update_precision, "param checksum %.15g" % float(model.params.double().sum()),
                      {k.split("/")[1]: v for k, v in model.logger_values.items() if k.split("/")[1] in ("policy_gradient_loss", "value_loss", "std")},
                      file=sys.stderr, flush=True)

    for _ in range(warmup):
        one_step()
    ctx.barrier()
    l0 = env.launch_count + model.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    graphs = model._graph is not None                       # the epoch replays a CUDA graph: no per-launch events inside
    in_region = wl == "c5" and not graphs
    model.grad_events = [] if in_region else None
    roll_events = []
    with ClockSampler(ctx.local) as clocks:
        ev0.record()
        for _ in range(steps):
            if wl == "c3":
                e = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                e[0].record()
            one_step()
            if wl == "c3":
                e[1].record()
                roll_events.append(e)
        ev1.record()
        ctx.barrier()
    launches = env.launch_count + model.launches - l0
    if dump and ctx.dump is not None:
        b = model.buf
        ctx.capture(wl, dict(obs=b.obs, actions=b.actions, logp=b.logp, value=b.value, reward=b.reward, done=b.done, adv=b.adv,
                             ret=b.ret, last_value=b.last_value[None]))
        if full:
            ctx.dump[f"{wl}_params"] = model.params.cpu().numpy()
    total_ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    value = n * K * steps * world / (total_ms * 1e-3)
    up = update_precision
    how = "CUDA events around every launch inside the timed region"
    if wl == "c5" and not in_region:
        # the timed region replayed CUDA graphs; time the gradient launches of ONE extra (eager) epoch right after it
        model.grad_events = []
        saved, model.n_epochs = model.n_epochs, 1
        model.train()
        model.n_epochs = saved
        torch.cuda.synchronize()
        how = "CUDA events around the gradient launches of one eager epoch right after the timed region (the region itself replays CUDA graphs)"
    if wl == "c1":
        ms, units, kflop = [total_ms / steps], float(n * K), MLP_FLOP * (1 + 3 * epochs)
        kname = "whole iteration (latency-bound: 2048 sequential env steps + one CUDA graph per epoch)"
    elif wl == "c5":
        ms = [a.elapsed_time(b) for a, b, _ in model.grad_events]
        units = float(np.mean([m for _, _, m in model.grad_events]))
        kflop = 3 * MLP_FLOP
        kname = {"tf32": "ppo_grad_tc_kernel", "bf16": "ppo_grad_bf16_kernel", "fp32": "ppo_grad_kernel"}[up] + " (+ its fixed-order reduce)"
    else:
        ms = [a.elapsed_time(b) for a, b in roll_events]
        units, kflop = float(n * K), MLP_FLOP
        kname = ("policy_rollout_tc_kernel" if rollout_precision == "tf32" else "policy_rollout_kernel") + " (+ gae_kernel)"
    model.grad_events = None
    k_ms = float(np.mean(ms))
    k_tflops = units * kflop / (k_ms * 1e-3) / 1e12
    tensor = (wl == "c3" and rollout_precision == "tf32") or (wl != "c3" and up in ("tf32", "bf16"))
    peak, peak_src = tensor_peak()
    traffic, traffic_src = static_traffic(f"{wl}_{up if wl != 'c3' else rollout_precision}")
    roofline = {"bound": "tensor", "achieved": k_tflops, "peak": peak, "unit": "TFLOP/s", "frac": k_tflops / peak,
                "traffic": traffic, "traffic_source": (traffic_src + " (ncu, static: not measured in this run)") if traffic else None,
                "peak_source": peak_src, "kernel": kname, "avg_launch_ms": k_ms, "units_per_launch": units,
                "algorithmic_flop_per_unit": kflop, "timed_by": how,
                "note": ("tcgen05 MMAs; the denominator is the measured dense bf16 peak (tf32 dense peak is half of it)" if tensor else
                         "fp32 CUDA-core parity path (nominal 74.4 TFLOP/s FMA peak: frac_of_fp32 = %.3f); the denominator is the "
                         "measured bf16 tensor peak" % (k_tflops / 74.4))}
    e2e = None
    if want_e2e:
        # the public API (PPO.learn / PPO.collect_rollouts), wall clock, every iteration reads its result (episode statistics +
        # train/* scalars) back to the host.  The simulator lives on the GPU, so an iteration has no host input: h2d is 0.
        its = max(1, min(steps, 5))
        ctx.barrier()
        t0 = time.perf_counter()
        if full:
            model.learn(total_timesteps=its * n * K * world)
            d2h = 19 * 4 + 128 * 64 + 5 * 8
        else:
            for _ in range(its):
                model.collect_rollouts()
                env.episode_stats(reset=True)
            d2h = 128 * 64
        ctx.barrier()
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": its * n * K * world / dt, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h,
               "api": "PPO.learn" if full else "PPO.collect_rollouts + episode_stats", "iterations": its,
               "note": "GPU-resident simulator: no host inputs per iteration; the result read back is the episode statistics "
                       "(128 slots x 64 B)" + (" and the train/* scalars" if full else "")}
    res = {"value": value, "ms_per_step": total_ms / steps, "steps": steps, "warmup": warmup,
           "rollout_precision": rollout_precision, "update_precision": up if full else None,
           "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks.summary(), "cuda_graph_epochs": graphs,
           "train": {k: v for k, v in model.logger_values.items() if k.startswith("train/")}}
    if world > 1 and full:
        res["dp_backend"] = model.dp_backend
    model.close()
    env.close()
    torch.cuda.empty_cache()
    return res


def bench_ppo(ctx, args, wl, steps, warmup, want_cpu, both=True):
    """c3 / c5 / c1: the tensor-core variant is the workload's value; the fp32 parity-path variant sits beside it."""
    if wl == "c1":
        n, K, mb, ep = 1, 2048, 32, 10
    else:
        n, K, mb, ep = args.ppo_envs, args.fuse, args.ppo_minibatches, args.ppo_epochs
    rp, up = args.precision, (args.update_precision or args.precision)
    main = ppo_variant(ctx, args, wl, n, K, mb, ep, rp, up, steps, warmup, not args.no_e2e, dump=True)
    res = {"value": main["value"], "unit": "env-steps/s", "steps": main["steps"], "warmup": warmup, "ms_per_step": main["ms_per_step"],
           "dtype": ("f32" if rp == "fp32" else "tf32 (fp32 accumulate)") if wl == "c3" else
                    "rollout MLP %s, update %s (fp32 accumulate; env step, loss, Adam in f32)" % (rp, up),
           "config": {"workload": WORKLOAD_NAMES[wl], "envs_per_gpu": n, "n_steps": K, "n_epochs": ep, "minibatches_per_epoch": mb,
                      "policy": "MlpPolicy 15-64-64-{4,1} tanh, random init",
                      "l2": ("rollout buffers %.1f GB per iteration, larger than L2" % (n * K * 93 / 1e9)) if wl != "c1" else
                            "latency-bound workload (190 KB of buffers): no L2 effect to flush"},
           "tensor_core_path": {k: main[k] for k in ("value", "ms_per_step", "rollout_precision", "update_precision", "cuda_graph_epochs")},
           "roofline": main["roofline"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "clocks": main["clocks"],
           "train": main["train"]}
    if "dp_backend" in main:
        res["config"]["dp_backend"] = main["dp_backend"]
    if both and (rp != "fp32" or (wl != "c3" and up != "fp32")):
        # the parity path (what tests/test_gpu_ppo.py pins at 2e-5 .. 2e-4): fewer steps, it is 10-15x slower
        s32 = max(2, min(steps, 3)) if wl != "c1" else steps
        p32 = ppo_variant(ctx, args, wl, n, K, mb, ep, "fp32", "fp32", s32, 3 if wl == "c1" else 1, False)
        res["fp32_parity_path"] = {k: p32[k] for k in ("value", "ms_per_step", "steps", "warmup", "roofline", "clocks", "gpu_launches")}
    if want_cpu:
        res["cpu_baseline"] = cpu_baseline_ppo(wl, os.cpu_count() or 1)
    return res


def main():
    # NCCL prints its version banner on STDOUT when NCCL_DEBUG=VERSION (some images export it): keep stdout = the JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=list(WORKLOAD_NAMES))
    ap.add_argument("--only", action="store_true", help="run only --workload (no 'workloads' object)")
    ap.add_argument("--envs-per-gpu", type=int, default=8_388_608)
    ap.add_argument("--fuse", type=int, default=32)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e legs (A/B kernel timing only)")
    ap.add_argument("--sustain-s", type=float, default=2.0, help="c4: seconds of back-to-back launches for the 'sustained' figure (0 = skip)")
    ap.add_argument("--ppo-envs", type=int, default=1_048_576)
    ap.add_argument("--ppo-epochs", type=int, default=10)
    ap.add_argument("--ppo-minibatches", type=int, default=4)
    ap.add_argument("--precision", default="tf32", choices=["fp32", "tf32"], help="policy MLP in the rollout: CUDA cores or tcgen05")
    ap.add_argument("--update-precision", default="bf16", choices=["fp32", "tf32", "bf16"], help="PPO minibatch gradient: fp32 = CUDA cores (parity path), tf32 = tcgen05 all-tf32, bf16 = tcgen05 with bf16 weight-gradient operands, three tiles per SM (default)")
    ap.add_argument("--dp-backend", default="peer", choices=["peer", "nccl"], help="N > 1: gradient exchange + clip + Adam as one kernel over NVLink peer memory (default), or NCCL all-reduce between the kernels")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what each timed path returned in its last step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs: not with --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    ctx = Ctx(dump=bool(args.dump_outputs))
    wl = args.workload
    want_cpu = ctx.world == 1 and not args.no_cpu and ctx.rank == 0
    if wl in ("c3", "c5", "c1"):
        top = bench_ppo(ctx, args, wl, args.steps, args.warmup, want_cpu)
    else:
        top = bench_env(ctx, args, wl, args.steps, args.warmup, want_cpu)
    extra = {}
    if wl == "c4" and not args.only:
        # the rest of the metric in the same run
        if ctx.world == 1:
            extra["c2"] = bench_env(ctx, args, "c2", args.steps, args.warmup, want_cpu)
        extra["c3"] = bench_ppo(ctx, args, "c3", args.steps, args.warmup, want_cpu)
        extra["c5"] = bench_ppo(ctx, args, "c5", args.steps, args.warmup, want_cpu)
    if ctx.rank == 0 and ctx.dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in ctx.dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if ctx.rank == 0:
        line = {"metric": "env_steps_per_sec", "value": top["value"], "unit": "env-steps/s", "n_gpus": ctx.world,
                "steps": top["steps"], "warmup": top["warmup"], "ms_per_step": top["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": top["dtype"], "data": "synthetic"}
        line.update({k: v for k, v in top.items() if k not in line})
        if extra:
            line["workloads"] = extra
        print(json.dumps(json_safe(line), allow_nan=False), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
