"""TEST INFRASTRUCTURE: check a recorded rollout transition-by-transition against the oracle.

Open-loop float32 and float64 trajectories of this system separate exponentially under random
motor forces (SURVEY.md section 7: the reference against itself drifts 0.2 rad in 26 steps when only the
action dtype changes), so a K-step record is verified *teacher-forced from its own rows*: the
float64 oracle is restarted from the recorded float32 observation of step k-1 and must reproduce
the recorded observation / reward / done of step k within the per-step tolerance.  Rows that were
auto-reset are checked bit-exactly against the Philox-fed reset (drone.py:48-75).
"""
from __future__ import annotations

import numpy as np

from . import drone_oracle as do
from . import philox

TOL_REL = 1e-5
# float32 rows past this magnitude (or non-finite) leave the range in which float32 arithmetic can follow float64:
# products of two such values, (Iyy - Izz) q r or dx^2, overflow to inf where float64 stays finite, and inf - inf
# then gives NaN.  Such rows (a body spinning up without bound once nothing resets it) are counted, not compared.
F32_SAFE = 1e18


def check_rollout(obs0, actions, next_obs, reward, done, *, spec=do.SINGLE, seed=0, env_ids=None,
                  ep_num0=None, step0=None, tol=TOL_REL, sing_cos=1e-3, target0=None):
    """obs0 [n,D]; actions [K,n,4]; next_obs [K,n,D]; reward [K,n]; done [K,n] (bool).

    spec: a ``drone_oracle.Spec`` (the default constants) or a ``drone_oracle.Params`` record.
    ep_num0 / step0: episode number (default 2: constructor reset + reset()) and step counter
    (default 0) of every env before the first step.  target0 [n,3]: the float32 target of every env
    before the first step, needed for D = 12 (it is not in the observation; default: the fixed target);
    D = 15 reads it from each row.
    Returns a dict with the worst error/bound ratio and the counts of borderline decisions; "terminated" counts the
    recorded dones the oracle calls a crash (at the time limit too) away from the crash borderline, and
    "terminated_slack" the recorded dones on the borderline, whose crash flag is not decided here.
    Raises AssertionError on a violation.
    """
    K, n = actions.shape[:2]
    p = do.Params.of(spec)
    D = p.obs_dim
    inertia = np.asarray(p.inertia, dtype=np.float64)
    dI = np.abs(np.array([(inertia[1] - inertia[2]) / inertia[0], (inertia[2] - inertia[0]) / inertia[1],
                          (inertia[0] - inertia[1]) / inertia[2]]))
    tgt = np.tile(np.asarray(p.fixed_target, np.float32), (n, 1)) if target0 is None else np.asarray(target0, np.float32).copy()
    env_ids = np.arange(n, dtype=np.uint64) if env_ids is None else np.asarray(env_ids, dtype=np.uint64)
    ep_num = np.broadcast_to(np.asarray(2 if ep_num0 is None else ep_num0, dtype=np.int64), (n,)).copy()
    step = np.zeros(n, dtype=np.int64) if step0 is None else np.broadcast_to(np.asarray(step0, dtype=np.int64), (n,)).copy()
    prev = np.asarray(obs0, dtype=np.float32)
    worst, borderline, n_done, n_sing, n_term, term_slack, n_wild = 0.0, 0, 0, 0, 0, 0, 0
    # the tolerance has a unit floor (1e-5 * max(|ref|, 1)); to make the floor visible also track the worst PURE relative
    # error |got - ref| / |ref| -- over all finite non-zero reference entries outside the near-singular rows, and over those
    # with |ref| >= 1e-3 (below that the quantity is a difference of O(1) terms and its relative error is cancellation)
    pure = {"all": (0.0, 0.0), "ref_ge_1e-3": (0.0, 0.0), "ref_ge_1": (0.0, 0.0)}
    with np.errstate(all="ignore"):
        for k in range(K):
            p64 = prev.astype(np.float64)
            pos, vel, eul, om = p64[:, 0:3], p64[:, 3:6], p64[:, 6:9], p64[:, 9:12]
            target = (p64[:, 12:15] + pos) if D == 15 else tgt.astype(np.float64)
            npos, nvel, neul, nom = do.dynamics_step(pos, vel, eul, om, actions[k].astype(np.float64), p=p)
            rew, crashed = do.reward_and_crash(npos, target, None, p)
            step += 1
            timeout = step >= p.max_steps
            d_ref = crashed | timeout
            d_got = np.asarray(done[k]).astype(bool)
            rad = np.linalg.norm(npos, axis=1)
            wild = ~(np.abs(p64) <= F32_SAFE).all(1)
            n_wild += int(wild.sum())
            margin = (((np.abs(npos[:, 2] - p.z_floor) > 1e-5 * max(1.0, abs(p.z_floor)))
                       & (np.abs(rad - p.r_max) > 2e-6 * max(50.0, p.r_max))) | ~np.isfinite(rad)) & ~wild
            assert np.array_equal(d_got[margin], d_ref[margin]), f"done mismatch at step {k}"
            borderline += int((~margin & ~wild).sum())
            n_term += int((d_got & crashed & margin).sum())
            term_slack += int((d_got & ~margin).sum())
            live = ((~d_got & ~d_ref) if p.auto_reset else (d_got == d_ref)) & ~wild
            ref_obs = do.build_obs(npos, nvel, neul, nom, target, D).astype(np.float64)
            got_obs = np.asarray(next_obs[k], dtype=np.float64)
            # Tolerance: |gpu - ref| <= tol * max(|ref|, 1, T) where T = the sum of the MAGNITUDES of the terms that are added
            # to form that output (float32 addition errs relative to its operands, not to a cancelling result): for roll / yaw
            # T = dt (|p| + |tan(pitch)| (|q sin(roll)| + |r cos(roll)|)) resp. dt |sec(pitch)| (...), which is what blows up
            # next to the pitch singularity (drone.py:182-184 has no guard); for the body rates T = dt |dI w w / I|.
            # No separate carve-out for |cos(pitch)| < sing_cos any more: the rows are only counted.
            sphi, cphi, cosp = np.sin(eul[:, 0]), np.cos(eul[:, 0]), np.cos(eul[:, 1])
            tanp, secp = np.tan(eul[:, 1]), 1.0 / cosp
            mix = np.abs(om[:, 1] * sphi) + np.abs(om[:, 2] * cphi)
            scale = np.maximum(np.abs(ref_obs), 1.0)
            T = np.zeros((n, D))
            T[:, 6] = np.abs(eul[:, 0]) + p.dt * (np.abs(om[:, 0]) + np.abs(tanp) * mix)
            T[:, 7] = np.abs(eul[:, 1]) + p.dt * mix
            T[:, 8] = np.abs(eul[:, 2]) + p.dt * np.abs(secp) * mix
            T[:, 9] = np.abs(om[:, 0]) + p.dt * dI[0] * np.abs(om[:, 1] * om[:, 2])      # |dI / I| = 1 for roll, pitch
            T[:, 10] = np.abs(om[:, 1]) + p.dt * dI[1] * np.abs(om[:, 0] * om[:, 2])     # at the default inertia
            if dI[2] != 0:
                T[:, 11] = np.abs(om[:, 2]) + p.dt * dI[2] * np.abs(om[:, 0] * om[:, 1])
            scale = np.maximum(scale, np.where(np.isfinite(T), T, 0.0))
            sing = np.abs(cosp) < sing_cos
            n_sing += int(sing.sum())
            amp = np.ones((n, D))
            # the recorded target-pos is float32(t - p): reconstructing t adds one float32 rounding
            if D == 15:
                amp[:, 12:15] = 2.0
            fin = np.isfinite(ref_obs) & live[:, None]
            assert np.array_equal(np.isnan(got_obs[live]), np.isnan(ref_obs[live])), f"NaN pattern, step {k}"
            err = np.where(fin, np.abs(got_obs - ref_obs), 0.0)
            bound = tol * scale * amp
            if fin.any():
                ratio_all = err / bound
                ratio = float(ratio_all.max())
                worst = max(worst, ratio)
                if ratio > 1.0:
                    i, j = np.unravel_index(int(np.argmax(ratio_all)), ratio_all.shape)
                    raise AssertionError(f"obs outside tolerance at step {k}: err/bound {ratio:.3g} (env row {i}, column {j}: got "
                                         f"{got_obs[i, j]!r} ref {ref_obs[i, j]!r}, previous state {prev[i].tolist()}, action "
                                         f"{actions[k][i].tolist()}, cos(pitch) {cosp[i]:.3g})")
            reg = fin & ~sing[:, None] & (ref_obs != 0)
            if reg.any():
                e, r = np.abs(got_obs - ref_obs)[reg], np.abs(ref_obs)[reg]
                for name, lo in (("all", 0.0), ("ref_ge_1e-3", 1e-3), ("ref_ge_1", 1.0)):
                    m = r >= lo
                    if m.any():
                        j = int(np.argmax(e[m] / r[m]))
                        if e[m][j] / r[m][j] > pure[name][0]:
                            pure[name] = (float(e[m][j] / r[m][j]), float(r[m][j]))
            both = (d_got == d_ref) & ~wild
            rfin = np.isfinite(rew) & both
            rerr = np.abs(np.asarray(reward[k], dtype=np.float64) - rew)[rfin]
            rbound = 2 * tol * np.maximum(np.abs(rew[rfin]), 1.0)
            assert not (rerr > rbound).any(), f"reward outside tolerance at step {k}"
            # auto-reset rows: bit-exact Philox-fed (randomized) or fixed reset observation
            rows = np.flatnonzero(d_got)
            n_done += rows.size
            if p.auto_reset and rows.size:
                ep_num[rows] += 1
                step[rows] = 0
                rp32, rt32 = reset_rows(p, seed, env_ids[rows], ep_num[rows])
                tgt[rows] = rt32
                ref_reset = np.concatenate([rp32, np.zeros((rows.size, 9), np.float32), rt32 - rp32], 1)
                got_reset = np.asarray(next_obs[k])[rows]
                if not np.array_equal(got_reset, ref_reset[:, :D]):
                    bad = np.flatnonzero((got_reset != ref_reset[:, :D]).any(1))
                    i = rows[bad[0]]
                    raise AssertionError(f"reset obs at step {k}: {bad.size} of {rows.size} rows differ; env id {env_ids[i]}, "
                                         f"ep_num {ep_num[i]}: got {got_reset[bad[0]].tolist()} ref {ref_reset[bad[0], :D].tolist()}")
            prev = np.asarray(next_obs[k], dtype=np.float32)
    return {"worst_err_over_bound": worst, "borderline_done": borderline, "dones": n_done, "out_of_f32_range": n_wild,
            "terminated": n_term, "terminated_slack": term_slack,
            "near_singular_rows": n_sing, "transitions": K * n,
            "worst_pure_relative": {k: {"rel_err": v[0], "at_abs_ref": v[1]} for k, v in pure.items()}}


def reset_rows(p, seed, env_ids, ep_num):
    """float32 (start position, target) [m, 3] of the resets that make the episode counters ``ep_num``: the Philox start
    with the curriculum target (drone.py:57-73) when ``p.randomized``, else ``p.fixed_start`` / ``p.fixed_target``
    (vectorized_drone.py:30,50).  The CUDA env stores both in float32 and forms target - pos in float32."""
    m = np.asarray(ep_num).size
    if not p.randomized:
        return (np.tile(np.asarray(p.fixed_start, np.float32), (m, 1)), np.tile(np.asarray(p.fixed_target, np.float32), (m, 1)))
    u = philox.reset_uniforms(seed, env_ids, ep_num)
    eps = do.curriculum_eps(ep_num, p.curriculum_period, p.curriculum_step)
    rp = np.stack([u[0] - 0.5, u[1] - 0.5, np.full(m, float(np.float32(p.start_z)))], 1)
    rt = np.stack([eps * u[2], eps * u[3], eps * u[4] + float(np.float32(p.target_z))], 1)
    return rp.astype(np.float32), rt.astype(np.float32)
