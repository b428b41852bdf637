"""TEST INFRASTRUCTURE: float64 numpy restatement of the reference quadcopter env.

This is the CPU oracle the CUDA path is checked against.  It restates, in one batched
function set, the arithmetic of BOTH reference environments (SURVEY.md section 2.2 shows
the physics is the same function; only the obs/reward/reset/termination epilogue differs):

  * ``DroneEnv``            /root/reference/drone.py:13-186           -> ``SINGLE`` spec
  * ``VectorizedDroneEnv``  /root/reference/vectorized_drone.py:12-216 -> ``VECTOR`` spec

Every function cites the reference lines it follows.  The temporaries the reference
builds (full (B,3,3) rotation and Euler-rate matrices, the einsum contractions with the
zero thrust components) are kept on purpose: they decide inf/NaN propagation
(``0 * inf``) and make this restatement bit-identical to ``VectorizedDroneEnv.step`` --
tests/test_oracle_vs_reference.py asserts exactly that, and tests/golden/*.npz hold
vectors generated from the unmodified reference (tests/golden/make_golden.py).

dtype convention: the reference never casts its inputs; with float32 actions the result
depends on the numpy version's promotion rules (SURVEY.md section 7).  The oracle -- and the
golden vectors -- fix one convention: the float32 action is upcast to float64 first, all
arithmetic is float64, only the observation is cast to float32 (drone.py:79).
"""
from __future__ import annotations

from dataclasses import dataclass, replace

import numpy as np

from . import philox

# ----------------------------------------------------------------------------------------
# constants: drone.py:21-43 == vectorized_drone.py:18-33
# ----------------------------------------------------------------------------------------
MASS = 1.0
GRAVITY = 9.81
INERTIA = np.array([0.005, 0.005, 0.01])
ARM_LENGTH = 0.5
K_YAW = 0.01
DT = 0.02
MOTOR_MAX = 3 * MASS * GRAVITY / 4.0  # drone.py:263, vectorized_drone.py:259


@dataclass(frozen=True)
class Spec:
    name: str
    obs_dim: int          # 15: drone.py:79,259   12: vectorized_drone.py:61,256
    max_steps: int        # 200: drone.py:43      1000: vectorized_drone.py:33
    bonus_radius: float   # 0.05: drone.py:147    1.0: vectorized_drone.py:207
    curriculum: bool      # per-episode random target (drone.py:68-73) vs fixed [0,0,10] (vec :30)
    random_start: bool    # drone.py:57 vs vectorized_drone.py:50
    shared_step: bool     # vectorized_drone.py:56,200: ONE counter for the whole batch
    auto_reset: bool      # SB3 DummyVecEnv semantics around DroneGymEnv (train.py:18-20)


SINGLE = Spec("single", 15, 200, 0.05, True, True, False, True)
VECTOR = Spec("vector", 12, 1000, 1.0, False, False, True, False)


@dataclass(frozen=True)
class Params:
    """Every constant of the env, field for field as ``EnvConfig`` (drone_rl_b200/core.py) holds them; the defaults are
    the reference's literals (drone.py:21-43, :57-73, :147-156) and ``SINGLE``'s epilogue.  ``randomized`` selects the
    Philox start with the curriculum target (drone.py:57-73) over ``fixed_start`` / ``fixed_target``
    (vectorized_drone.py:30,50); ``auto_reset`` the DummyVecEnv reset on done."""
    dt: float = DT
    mass: float = MASS
    gravity: float = GRAVITY
    inertia: tuple = tuple(INERTIA.tolist())
    arm_length: float = ARM_LENGTH
    k_yaw: float = K_YAW
    reward_scale: float = 0.01
    bonus_radius: float = 0.05
    bonus: float = 1.0
    z_floor: float = 0.0
    r_max: float = 50.0
    fixed_target: tuple = (0.0, 0.0, 10.0)
    fixed_start: tuple = (0.1, 0.1, 0.1)
    start_z: float = 1.0
    target_z: float = 1.0
    curriculum_step: float = 0.1
    curriculum_period: int = 2000
    max_steps: int = 200
    obs_dim: int = 15
    randomized: bool = True
    auto_reset: bool = True

    @property
    def motor_max(self):
        return 3 * self.mass * self.gravity / 4.0      # drone.py:263

    @classmethod
    def of(cls, spec=None, **kw):
        """A ``Params`` as it is, or the one of a ``Spec`` (default constants), with ``kw`` replaced."""
        if spec is None:
            spec = SINGLE
        if isinstance(spec, Params):
            return replace(spec, **kw) if kw else spec
        base = dict(obs_dim=spec.obs_dim, max_steps=spec.max_steps, bonus_radius=spec.bonus_radius,
                    randomized=spec.random_start, auto_reset=spec.auto_reset)
        base.update(kw)
        return cls(**base)

    @classmethod
    def from_config(cls, cfg):
        """The record of an ``EnvConfig`` (any object with its attribute names)."""
        return cls(**{f: (tuple(getattr(cfg, f)) if isinstance(getattr(cfg, f), (tuple, list)) else getattr(cfg, f))
                      for f in cls.__dataclass_fields__})


DEFAULT = Params()


# ----------------------------------------------------------------------------------------
# physics: one batched Euler step
# ----------------------------------------------------------------------------------------
def rotor_mix(action, p=DEFAULT):
    """Thrust and body torques from the four motor forces.

    drone.py:106-117 / vectorized_drone.py:154-166.  ``action`` float64 [B,4].
    """
    f1, f2, f3, f4 = action[:, 0], action[:, 1], action[:, 2], action[:, 3]
    thrust = np.sum(action, axis=1)
    lever = p.arm_length / np.sqrt(2)
    tau_roll = lever * (f1 + f2 - f3 - f4)
    tau_pitch = lever * (-f1 + f2 + f3 - f4)
    tau_yaw = p.k_yaw * (f1 - f2 + f3 - f4)
    return thrust, tau_roll, tau_pitch, tau_yaw


def body_to_inertial(euler):
    """ZYX rotation matrices [B,3,3] (drone.py:161-174 / vectorized_drone.py:63-98)."""
    roll, pitch, yaw = euler[:, 0], euler[:, 1], euler[:, 2]
    cr, sr = np.cos(roll), np.sin(roll)
    cp, sp = np.cos(pitch), np.sin(pitch)
    cy, sy = np.cos(yaw), np.sin(yaw)
    rot = np.empty((euler.shape[0], 3, 3))
    rot[:, 0, 0] = cy * cp
    rot[:, 0, 1] = cy * sp * sr - sy * cr
    rot[:, 0, 2] = cy * sp * cr + sy * sr
    rot[:, 1, 0] = sy * cp
    rot[:, 1, 1] = sy * sp * sr + cy * cr
    rot[:, 1, 2] = sy * sp * cr - cy * sr
    rot[:, 2, 0] = -sp
    rot[:, 2, 1] = cp * sr
    rot[:, 2, 2] = cp * cr
    return rot


def euler_rates(euler, omega):
    """d(euler)/dt = T(roll,pitch) @ omega (drone.py:176-186 / vectorized_drone.py:100-133).

    No guard at cos(pitch) -> 0: tan and 1/cos overflow exactly as the reference's do.
    """
    roll, pitch = euler[:, 0], euler[:, 1]
    tan_p = np.tan(pitch)
    sec_p = 1 / np.cos(pitch)
    tm = np.empty((euler.shape[0], 3, 3))
    tm[:, 0, 0] = 1.0
    tm[:, 0, 1] = np.sin(roll) * tan_p
    tm[:, 0, 2] = np.cos(roll) * tan_p
    tm[:, 1, 0] = 0.0
    tm[:, 1, 1] = np.cos(roll)
    tm[:, 1, 2] = -np.sin(roll)
    tm[:, 2, 0] = 0.0
    tm[:, 2, 1] = np.sin(roll) * sec_p
    tm[:, 2, 2] = np.cos(roll) * sec_p
    return np.einsum("bij,bj->bi", tm, omega)


def dynamics_step(pos, vel, euler, omega, action, dt=None, p=DEFAULT):
    """One step of the reference integrator; returns NEW arrays (inputs untouched).

    Order (drone.py:119-139 / vectorized_drone.py:168-197): acceleration from the OLD
    attitude; v += a dt; p += v_new dt (semi-implicit); euler += T(old euler) old_omega dt;
    omega += omega_dot(old omega) dt.  ``dt`` (default ``p.dt``) overrides the record's step.
    """
    dt = p.dt if dt is None else dt
    inertia = np.asarray(p.inertia, dtype=np.float64)
    action = np.asarray(action, dtype=np.float64)
    thrust, tau_roll, tau_pitch, tau_yaw = rotor_mix(action, p)
    n = action.shape[0]

    rot = body_to_inertial(euler)
    thrust_body = np.zeros((n, 3))
    thrust_body[:, 2] = thrust
    thrust_world = np.einsum("bij,bj->bi", rot, thrust_body)
    accel = np.tile(np.array([0, 0, -p.gravity]), (n, 1)) + (thrust_world / p.mass)

    vel = vel + accel * dt
    pos = pos + vel * dt

    new_euler = euler + euler_rates(euler, omega) * dt

    wdot = np.empty_like(omega)
    wdot[:, 0] = (tau_roll - (inertia[1] - inertia[2]) * omega[:, 1] * omega[:, 2]) / inertia[0]
    wdot[:, 1] = (tau_pitch - (inertia[2] - inertia[0]) * omega[:, 0] * omega[:, 2]) / inertia[1]
    wdot[:, 2] = (tau_yaw - (inertia[0] - inertia[1]) * omega[:, 0] * omega[:, 1]) / inertia[2]
    new_omega = omega + wdot * dt
    return pos, vel, new_euler, new_omega


def reward_and_crash(pos, target, bonus_radius, p=DEFAULT):
    """reward (float64 [B]) and the crash/out-of-range flag (bool [B]).

    drone.py:142-148,154 / vectorized_drone.py:204-207,211.  NaN position -> both
    comparisons False -> not crashed.  ``bonus_radius`` overrides ``p.bonus_radius`` (None: the record's).
    """
    bonus_radius = p.bonus_radius if bonus_radius is None else bonus_radius
    dist = np.linalg.norm(pos - target, axis=1)
    reward = -p.reward_scale * dist
    reward[dist < bonus_radius] += p.bonus
    crashed = (pos[:, 2] < p.z_floor) | (np.linalg.norm(pos, axis=1) > p.r_max)
    return reward, crashed


def build_obs(pos, vel, euler, omega, target, obs_dim):
    """float32 observation (drone.py:77-79: 15 with target-pos; vectorized_drone.py:59-61: 12)."""
    parts = [pos, vel, euler, omega]
    if obs_dim == 15:
        parts.append(target - pos)
    return np.concatenate(parts, axis=1).astype(np.float32)


def curriculum_eps(ep_num, period=2000, step=0.1):
    """eps after the reset that made the episode counter ``ep_num`` (drone.py:61,68-70).

    The reference accumulates ``eps += 0.1`` each time ep_num hits a multiple of 2000, in
    float64 (0.1, 0.2, 0.30000000000000004, ...): reproduce the accumulation, not 0.1*n.
    One sequential float64 sum up to the largest bump count, read off at every distinct count
    (an ep_num of 2^31 - 1 at period 1 takes 2^31 additions).
    """
    ep_num = np.asarray(ep_num)
    bumps = ep_num // period
    out = np.zeros(ep_num.shape, dtype=np.float64)
    eps, done = 0.0, 0
    for b in np.unique(bumps):
        eps, done = _accumulate(eps, step, int(b) - done), int(b)
        out[bumps == b] = eps
    return out


def _accumulate(eps, step, count, chunk=1 << 22):
    """((eps + step) + step) + ... with ``count`` float64 additions in order (ufunc.accumulate is sequential)."""
    while count > 0:
        m = min(count, chunk)
        a = np.full(m + 1, step, dtype=np.float64)
        a[0] = eps
        eps = float(np.add.accumulate(a)[-1])
        count -= m
    return eps


# ----------------------------------------------------------------------------------------
# batched env with the semantics the CUDA env implements
# ----------------------------------------------------------------------------------------
class BatchedDroneOracle:
    """n independent reference envs (SINGLE spec, each wrapped the way SB3's DummyVecEnv
    wraps ``DroneGymEnv``: train.py:18-20) or one ``VectorizedDroneEnv`` (VECTOR spec).

    Randomness: env ``i`` (global id ``env_offset + i``) draws its five reset uniforms from
    the Philox stream keyed by (seed, global id, ep_num) -- see oracle/philox.py.
    """

    def __init__(self, n_envs, spec=SINGLE, seed=0, env_offset=0, dt=None):
        """``spec``: a ``Spec`` (the reference's constants) or a ``Params`` record; ``dt`` overrides its step."""
        self.p = Params.of(spec) if dt is None else Params.of(spec, dt=dt)
        self.n, self.spec, self.seed, self.dt = int(n_envs), spec, int(seed), self.p.dt
        self.env_ids = np.arange(env_offset, env_offset + self.n, dtype=np.uint64)
        self.pos = np.zeros((self.n, 3))
        self.vel = np.zeros((self.n, 3))
        self.euler = np.zeros((self.n, 3))
        self.omega = np.zeros((self.n, 3))
        self.target = np.tile(np.array(self.p.fixed_target, dtype=np.float64), (self.n, 1))  # vectorized_drone.py:30
        self.step_count = np.zeros(self.n, dtype=np.int64)
        self.ep_num = np.zeros(self.n, dtype=np.int64)
        # VecMonitor accumulators (SURVEY.md appendix C)
        self.ep_return = np.zeros(self.n, dtype=np.float32)   # SB3 VecMonitor keeps float32
        self.ep_length = np.zeros(self.n, dtype=np.int64)
        self.reset()  # both constructors reset once: drone.py:46, vectorized_drone.py:36

    # -- reset ---------------------------------------------------------------------------
    def _reset_rows(self, rows):
        """drone.py:48-75 (SINGLE) / vectorized_drone.py:38-57 (VECTOR) for a row subset."""
        if rows.size == 0:
            return
        self.vel[rows] = 0.0
        self.euler[rows] = 0.0
        self.omega[rows] = 0.0
        self.ep_num[rows] += 1
        self.step_count[rows] = 0
        p = self.p
        if p.randomized:
            u = philox.reset_uniforms(self.seed, self.env_ids[rows], self.ep_num[rows])
            self.pos[rows, 0] = u[0] - 0.5
            self.pos[rows, 1] = u[1] - 0.5
            self.pos[rows, 2] = p.start_z
            eps = curriculum_eps(self.ep_num[rows], p.curriculum_period, p.curriculum_step)
            self.target[rows, 0] = eps * u[2]
            self.target[rows, 1] = eps * u[3]
            self.target[rows, 2] = eps * u[4] + p.target_z + 0
        else:
            self.pos[rows] = np.array(p.fixed_start, dtype=np.float64)
            self.target[rows] = np.array(p.fixed_target, dtype=np.float64)   # VECTOR: [0,0,10]

    def reset(self, mask=None):
        rows = np.arange(self.n) if mask is None else np.flatnonzero(np.asarray(mask))
        self._reset_rows(rows)
        self.ep_return[rows] = 0.0
        self.ep_length[rows] = 0
        return self.obs()

    def obs(self):
        return build_obs(self.pos, self.vel, self.euler, self.omega, self.target, self.p.obs_dim)

    # -- state injection for teacher-forced tests ---------------------------------------------
    def set_state(self, pos=None, vel=None, euler=None, omega=None, target=None,
                  step_count=None, ep_num=None):
        for name, val in (("pos", pos), ("vel", vel), ("euler", euler), ("omega", omega),
                          ("target", target)):
            if val is not None:
                getattr(self, name)[...] = np.asarray(val, dtype=np.float64)
        if step_count is not None:
            self.step_count[...] = step_count
        if ep_num is not None:
            self.ep_num[...] = ep_num

    # -- step ------------------------------------------------------------------------------
    def step(self, action):
        """Returns (obs f32[n,D], reward f64[n], done bool[n], info dict of arrays).

        info: ``terminated`` (crash / out of range), ``truncated`` (time limit only),
        ``terminal_obs`` f32[n,D] (the pre-reset observation, meaningful where done),
        ``episode_r`` / ``episode_l`` (VecMonitor totals, meaningful where done).
        """
        with np.errstate(all="ignore"):
            self.pos, self.vel, self.euler, self.omega = dynamics_step(
                self.pos, self.vel, self.euler, self.omega, action, self.dt, self.p)
            reward, crashed = reward_and_crash(self.pos, self.target, None, self.p)
            self.step_count += 1                                   # drone.py:155 / vec :200
            timeout = self.step_count >= self.p.max_steps           # drone.py:156 / vec :212
            done = crashed | timeout
            obs = self.obs()
        info = {"terminated": crashed.copy(), "truncated": timeout & ~crashed,
                "terminal_obs": obs.copy()}
        # VecMonitor: accumulate (in float32) the float32 reward DummyVecEnv stored
        self.ep_return += reward.astype(np.float32)
        self.ep_length += 1
        info["episode_r"] = self.ep_return.copy()
        info["episode_l"] = self.ep_length.copy()
        # VecMonitor zeroes its accumulators on every done, whether or not the env resets
        rows = np.flatnonzero(done)
        self.ep_return[rows] = 0.0
        self.ep_length[rows] = 0
        if self.p.auto_reset and rows.size:
            self._reset_rows(rows)
            obs = self.obs()
        return obs, reward, done, info
