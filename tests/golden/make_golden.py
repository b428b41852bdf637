"""Generate the golden vectors in this directory FROM THE UNMODIFIED REFERENCE.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference ships no fixtures or tests (SURVEY.md section 4), so the pins are its own
outputs: every array written here comes out of ``drone.DroneGymEnv`` /
``vectorized_drone.VectorizedDroneEnv`` imported unmodified (oracle/ref_import.py).  The
only things injected are (a) the actions and (b) the uniforms ``np.random.rand()`` returns
inside ``DroneEnv.reset`` (our Philox stream, oracle/philox.py), and (c) for the
teacher-forced set, the state attributes before a step.  float32 actions are upcast to
float64 before they are handed to the reference (dtype convention, oracle/drone_oracle.py).
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import philox, ref_import  # noqa: E402
from oracle.vecenv_oracle import DummyVecEnvOracle, VecMonitorOracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
MOTOR_MAX = 3 * 1.0 * 9.81 / 4.0


class PhiloxFedEnv:
    """A real reference ``DroneGymEnv`` whose reset draws come from our Philox stream."""

    def __init__(self, drone_mod, stream, seed, env_id):
        self.stream, self.seed, self.env_id = stream, seed, env_id
        self._feed(1)
        self.env = drone_mod.DroneGymEnv()      # constructor resets once (drone.py:46)

    def _feed(self, ep_num):
        u = philox.reset_uniforms(self.seed, np.array([self.env_id], dtype=np.uint64),
                                  np.array([ep_num], dtype=np.uint64))[:, 0]
        self.stream.feed(u)

    def reset(self):
        self._feed(self.env.ep_num + 1)
        return self.env.reset()

    def step(self, action):
        return self.env.step(action)


def gen_single_rollout(drone_mod, n_envs=8, n_steps=400, seed=1234, env_offset=100):
    stream = ref_import.UniformStream()
    with ref_import.patched_rand(stream):
        envs = [PhiloxFedEnv(drone_mod, stream, seed, env_offset + i) for i in range(n_envs)]
        venv = VecMonitorOracle(DummyVecEnvOracle(envs))
        obs0 = venv.reset()
        rng = np.random.default_rng(7)
        actions = rng.uniform(0, MOTOR_MAX, (n_steps, n_envs, 4)).astype(np.float32)
        # mix in gentler actions so some episodes live long and hit the 200-step limit
        hover = np.float32(9.81 / 4.0)
        actions[:, n_envs // 2:, :] = hover + 0.02 * (actions[:, n_envs // 2:, :] - hover)
        actions[:, -1, :] = hover * np.float32(1.001)
        obs = np.zeros((n_steps, n_envs, 15), np.float32)
        rew = np.zeros((n_steps, n_envs), np.float32)
        rew64 = np.zeros((n_steps, n_envs), np.float64)
        done = np.zeros((n_steps, n_envs), bool)
        term_obs = np.zeros((n_steps, n_envs, 15), np.float32)
        ep_r = np.zeros((n_steps, n_envs), np.float32)
        ep_l = np.zeros((n_steps, n_envs), np.int32)
        for t in range(n_steps):
            # capture the float64 reward the env itself returned
            a64 = actions[t].astype(np.float64)
            o, r, d, infos = venv.step(a64)
            obs[t], rew[t], done[t] = o, r, d
            for i, info in enumerate(infos):
                if d[i]:
                    term_obs[t, i] = info["terminal_observation"]
                    ep_r[t, i] = info["episode"]["r"]
                    ep_l[t, i] = info["episode"]["l"]
        ep_num = np.array([e.env.ep_num for e in envs])
        assert stream.queue == [], "every injected uniform must have been consumed"
    np.savez_compressed(os.path.join(HERE, "single_rollout.npz"), seed=seed, env_offset=env_offset,
                        obs0=obs0, actions=actions, obs=obs, reward=rew, done=done,
                        terminal_obs=term_obs, episode_r=ep_r, episode_l=ep_l, final_ep_num=ep_num)
    print("single_rollout: dones", int(done.sum()), "timeouts", int((ep_l == 200).sum()))


def gen_const_action(drone_mod, seed=5, env_id=0):
    """The reference's own demo (drone.py:288-294): 2x hover thrust until done."""
    stream = ref_import.UniformStream()
    with ref_import.patched_rand(stream):
        env = PhiloxFedEnv(drone_mod, stream, seed, env_id)
        obs0 = env.reset()
        act = np.full(4, np.float32((env.env.mass * env.env.g) / 4.0 * 2)).astype(np.float64)  # f32-representable
        obs, rew, done = [], [], []
        for _ in range(300):
            o, r, d, _ = env.step(act)
            obs.append(o), rew.append(r), done.append(d)
            if d:
                break
    np.savez_compressed(os.path.join(HERE, "single_const_action.npz"), seed=seed, env_id=env_id,
                        obs0=obs0, action=act.astype(np.float32), obs=np.array(obs),
                        reward=np.array(rew), done=np.array(done))
    print("const_action: done at step", len(done))


def gen_vector_rollout(vd_mod, batch=16, n_steps=1003):
    env = vd_mod.VectorizedDroneEnv(batch)
    obs0 = env.reset()
    rng = np.random.default_rng(11)
    actions = rng.uniform(0, MOTOR_MAX, (n_steps, batch, 4)).astype(np.float32)
    hover = np.float32(9.81 / 4.0)
    actions[:, batch // 2:, :] = hover + 0.01 * (actions[:, batch // 2:, :] - hover)
    actions[:, -2:, :] = hover * np.float32(1.5)     # climbs to the target at z = 10 (bonus zone)
    actions[:, -3, :] = hover                        # hovers: still alive when the time limit hits
    obs = np.zeros((n_steps, batch, 12), np.float32)
    rew = np.zeros((n_steps, batch), np.float64)
    done = np.zeros((n_steps, batch), bool)
    with np.errstate(all="ignore"):
        for t in range(n_steps):
            obs[t], rew[t], done[t], _ = env.step(actions[t].astype(np.float64))
    np.savez_compressed(os.path.join(HERE, "vector_rollout.npz"), obs0=obs0, actions=actions,
                        obs=obs, reward=rew, done=done)
    print("vector_rollout: bonus steps", int((rew > 0).sum()), "done frac", float(done.mean()))


def teacher_forced_rows(n_drawn=4096, n_corner=16, n_keep=2048):
    """The rows of the teacher-forced draw that are stored (the file stays under 1 MB): the hand-made corner cases at the
    front, then a fixed, seeded sample of the random rows.  Every row is an independent one-step case."""
    rest = np.random.default_rng(4).choice(np.arange(n_corner, n_drawn), n_keep - n_corner, replace=False)
    return np.concatenate([np.arange(n_corner), np.sort(rest)])


def gen_teacher_forced(drone_mod, vd_mod, n=4096):
    """One step from injected float32-representable states, through BOTH reference envs (the rows teacher_forced_rows keeps)."""
    rng = np.random.default_rng(3)
    f32 = np.float32
    pos = (rng.normal(0, 3, (n, 3))).astype(f32)
    pos[:, 2] = np.abs(pos[:, 2]) + f32(0.05)
    vel = rng.normal(0, 4, (n, 3)).astype(f32)
    scale = 10.0 ** rng.uniform(-2, 3.2, (n, 1))           # |angles| from 1e-2 to ~1.5e3 rad
    euler = (rng.normal(0, 1, (n, 3)) * scale).astype(f32)
    omega = (rng.normal(0, 1, (n, 3)) * 10.0 ** rng.uniform(-1, 2, (n, 1))).astype(f32)
    target = np.concatenate([rng.uniform(0, 0.5, (n, 2)), 1 + rng.uniform(0, 0.5, (n, 1))], 1).astype(f32)
    action = rng.uniform(0, MOTOR_MAX, (n, 4)).astype(f32)
    # hand-made corner cases ---------------------------------------------------------------
    k = 0
    pos[k] = [0, 0, 0.001]; vel[k] = [0, 0, -1]; k += 1                 # crosses z < 0
    pos[k] = [30, 40, 0.5]; vel[k] = [5, 5, 0]; k += 1                  # |pos| crosses 50
    pos[k] = target[k] + f32(0.01); vel[k] = 0; action[k] = f32(9.81 / 4); euler[k] = 0; omega[k] = 0; k += 1  # bonus zone
    euler[k, 1] = f32(np.pi / 2); k += 1                                # cos(pitch) ~ -4.4e-8
    euler[k, 1] = f32(np.pi / 2 + 1e-3); k += 1
    euler[k, 1] = f32(-np.pi / 2 + 1e-4); k += 1
    pos[k] = [np.nan, 0, 1]; k += 1                                     # NaN -> never "crashed"
    omega[k] = [np.inf, 0, 0]; k += 1                                   # 0*inf -> NaN (drone.py:138)
    euler[k] = [np.inf, 0, 0]; k += 1
    euler[k] = [1e6, -2e6, 3e6]; k += 1                                  # unwrapped huge angles
    euler[k] = [3e4, 1e5, -7e4]; k += 1
    action[k] = 0; k += 1
    action[k] = f32(MOTOR_MAX); k += 1
    action[k] = [20, -5, 100, 0]; k += 1                                 # env never clips (SURVEY 8b)
    step_count = rng.integers(0, 198, n)
    step_count[k] = 199; k += 1                                          # time limit this step
    step_count[k] = 198; k += 1

    keep = teacher_forced_rows(n, k)
    pos, vel, euler, omega, target, action, step_count = (a[keep] for a in (pos, vel, euler, omega, target, action, step_count))
    n = keep.size
    out = {"pos": pos, "vel": vel, "euler": euler, "omega": omega, "target": target,
           "action": action, "step_count": step_count.astype(np.int32)}
    with np.errstate(all="ignore"):
        # (a) VectorizedDroneEnv: inject state, one step
        env = vd_mod.VectorizedDroneEnv(n)
        env.pos, env.vel = pos.astype(np.float64), vel.astype(np.float64)
        env.euler, env.omega = euler.astype(np.float64), omega.astype(np.float64)
        o, r, d, _ = env.step(action.astype(np.float64))
        out.update(vec_pos=env.pos, vec_vel=env.vel, vec_euler=env.euler, vec_omega=env.omega,
                   vec_obs=o, vec_reward=r, vec_done=d)
        # (b) DroneGymEnv: inject state, one step each
        env1 = drone_mod.DroneGymEnv()
        s_state = np.zeros((n, 12)); s_obs = np.zeros((n, 15), f32)
        s_rew = np.zeros(n); s_done = np.zeros(n, bool)
        for i in range(n):
            env1.pos, env1.vel = pos[i].astype(np.float64), vel[i].astype(np.float64)
            env1.euler, env1.omega = euler[i].astype(np.float64), omega[i].astype(np.float64)
            env1.target = target[i].astype(np.float64)
            env1.current_step = int(step_count[i])
            o1, r1, d1, _ = env1.step(action[i].astype(np.float64))
            s_state[i] = np.concatenate([env1.pos, env1.vel, env1.euler, env1.omega])
            s_obs[i], s_rew[i], s_done[i] = o1, r1, d1
        out.update(single_state=s_state, single_obs=s_obs, single_reward=s_rew, single_done=s_done)
    np.savez_compressed(os.path.join(HERE, "teacher_forced.npz"), **out)
    print("teacher_forced: n", n, "single done", int(s_done.sum()), "nan rows",
          int(np.isnan(s_state).any(1).sum()))


def gen_curriculum(drone_mod, seed=99, env_id=7):
    """eps / target schedule across 6001 resets of ONE reference env (drone.py:61-73)."""
    stream = ref_import.UniformStream()
    probe = [1, 2, 1999, 2000, 2001, 3999, 4000, 4001, 5999, 6000, 6001]
    with ref_import.patched_rand(stream):
        env = PhiloxFedEnv(drone_mod, stream, seed, env_id)
        rows = []
        if env.env.ep_num in probe:
            rows.append((env.env.ep_num, env.env.eps, *env.env.pos, *env.env.target))
        while env.env.ep_num < 6001:
            env.reset()
            if env.env.ep_num in probe:
                rows.append((env.env.ep_num, env.env.eps, *env.env.pos, *env.env.target))
    arr = np.array(rows)
    np.savez_compressed(os.path.join(HERE, "curriculum.npz"), seed=seed, env_id=env_id,
                        ep_num=arr[:, 0].astype(np.int64), eps=arr[:, 1], pos=arr[:, 2:5],
                        target=arr[:, 5:8])
    print("curriculum eps:", dict(zip(arr[:, 0].astype(int).tolist(), arr[:, 1].tolist())))


def main():
    np.seterr(all="ignore")
    drone_mod, vd_mod = ref_import.load()
    gen_const_action(drone_mod)
    gen_single_rollout(drone_mod)
    gen_vector_rollout(vd_mod)
    gen_teacher_forced(drone_mod, vd_mod)
    gen_curriculum(drone_mod)


if __name__ == "__main__":
    main()
