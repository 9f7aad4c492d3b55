"""Helpers shared by the GPU parity tests: drive the CUDA path (through the C ABI) and the
CPU oracle with the same seeded inputs and compare.

Stated tolerances (FP32 CUDA path vs FP64 oracle; SURVEY.md section 8c):
over a 240-substep (1 s) open-loop horizon  |dpos| <= 1e-4 m, |dvel| <= 1e-3 m/s,
|dquat| <= 1e-4, |dobs| <= 1e-4, |dreward| <= 1e-3 (the shaped reward has a 3000x gain on
the distance difference); discrete outputs (done bits, found_targets) exact, except where
the oracle itself sits within MARGIN_TOL of a threshold (near-tie), which is counted,
reported and excluded.
"""
from __future__ import annotations

import numpy as np

POS_TOL, VEL_TOL, QUAT_TOL, OBS_TOL, REW_TOL = 1e-4, 1e-3, 1e-4, 1e-4, 1e-3
# obs[9:12] is ang_v / |ang_v| (PBDroneEnv.py:383-384): the direction of a nearly-zero vector is
# ill-conditioned (bang-bang torques cancel to ~1e-7 rad/s residues, in the reference too), so those
# three entries are compared as  |d| <= OBS_TOL + ANGV_ABS_TOL / |ang_v_oracle|, i.e. an absolute
# angular-velocity tolerance of 1e-4 rad/s over the horizon (rates reach ~50 rad/s: 6e-8 * 50 * sqrt(240))
ANGV_ABS_TOL = 1e-4
# Roll and yaw (obs[3], obs[5]) are ill-conditioned near gimbal lock: d(roll, yaw) ~ d(quat) / cos(pitch).  Among 65 536 tumbling
# environments some always sit within a degree of |pitch| = 90 deg (cos ~ 5e-3), so in the full-size tests those two entries
# are compared as  |d| <= OBS_TOL + EULER_COND_TOL / cos(pitch_oracle)  (in units of pi; the quaternion itself has its own bound)
EULER_COND_TOL = 5e-6
# FP32 orientation error grows with the rotation traversed (relative error ~2e-6 of the angle): an environment tumbling at
# 200 rad/s turns 30 revolutions within one horizon.  Beyond EULER_RATE_REF the Euler-angle tolerance scales with |omega|.
EULER_RATE_REF = 60.0
MARGIN_TOL = 2e-5          # oracle margin below which an FP32/FP64 discrete disagreement is a near-tie
HORIZON_SUBSTEPS = 240


def oracle_state_arrays(envs):
    """Stack oracle env states into the row-major arrays dn_set_state takes."""
    keys = ("pos", "quat", "vel", "rpy_rates", "ang_v", "prev_vel", "prev_ang_v")
    st = [e.get_state() for e in envs]
    out = {k: np.stack([s[k] for s in st]).astype(np.float32) for k in keys}
    out["dist"] = np.array([s["dist"] for s in st], np.float32)
    out["prev_dist"] = np.array([s["prev_dist"] for s in st], np.float32)
    out["target_idx"] = np.array([s["target_idx"] for s in st], np.int32)
    out["steps"] = np.array([s["steps"] for s in st], np.int32)
    out["just_found"] = np.array([s["just_found"] for s in st], np.uint8)
    return out


def upload_oracle_state(gpu_env, workers):
    st = oracle_state_arrays([w.env for w in workers])
    st["ep_return"] = np.array([w.ep_return for w in workers], np.float32)
    st["ep_length"] = np.array([w.ep_len for w in workers], np.int32)
    if getattr(gpu_env, "_optional", {}).get("pid"):   # DSLPIDControl state (PID action types)
        st["pid"] = np.stack([np.concatenate([w.env.ctrl.integral_pos_e, w.env.ctrl.integral_rpy_e, w.env.ctrl.last_rpy])
                              for w in workers]).astype(np.float32)
    if gpu_env.uses_drag:
        st["last_rpm_sum"] = np.array([float(np.sum(w.env.last_clipped_action)) for w in workers], np.float32)
    gpu_env.set_state(st)


def return_sum_bound(abs_sum, n_terms, max_per_lane):
    """|return_sum - FP64 sum| bound of the Monitor statistics (dn_episode_stats) over `n_terms` finished episodes whose
    returns have absolute sum `abs_sum`.  A lane adds its finished episodes (at most `max_per_lane` between two flushes) one
    after another in FP32, a warp adds its 32 lanes in a 5-level shuffle tree, and the warp sums are added as FP64:
    (k - 1 + 5) u sum|r| with u = 2^-24, plus 2^-53 sum|r| per FP64 addition.  dn_step has k = 1."""
    return (max_per_lane - 1 + 5) * 2.0 ** -24 * abs_sum + (n_terms + 1) * 2.0 ** -53 * abs_sum


def _np(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def obs_error(a, b, ang_v_norm=None, report=None, tol=OBS_TOL):
    """max |a - b| over an observation row; the three Euler-angle entries (3..5, in units of pi) are
    compared modulo 2 so that a +-pi wrap of atan2 on either side is not a discrepancy; the ang_v
    direction entries are de-weighted by their conditioning (see ANGV_ABS_TOL).  `report` counts the entries
    that passed only because of that de-weighting."""
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
    d[3:6] = np.minimum(d[3:6], np.abs(2.0 - d[3:6]))
    if ang_v_norm is not None:
        plain = d[9:12].copy()
        d[9:12] = np.maximum(d[9:12] - ANGV_ABS_TOL / max(ang_v_norm, 1e-30), 0.0)
        if report is not None:
            report.carved["ang_v_direction"] += int(((plain > tol) & (d[9:12] <= tol)).sum())
    if report is not None:
        report.obs_entries += d.size
    return float(d.max())


def min_margin(env):
    m = [abs(float(x)) for x in env.margins if np.isfinite(x)]
    return min(m) if m else np.inf


class ParityReport:
    def __init__(self):
        self.max_obs = self.max_rew = self.max_pos = self.max_vel = self.max_quat = 0.0
        self.near_ties = 0
        self.env_steps = 0
        self.dones = 0
        self.captures = 0
        # coverage lost to the carve-outs above: entry comparisons whose PLAIN error exceeded the stated tolerance and that
        # passed only because of the named rule (obs entries compared = `obs_entries`)
        self.obs_entries = 0
        self.carved = {"ang_v_direction": 0, "euler_gimbal_conditioning": 0, "euler_gimbal_branch": 0, "euler_tumbling_rate": 0}

    def __str__(self):
        carved = " ".join(f"{k}={v}" for k, v in self.carved.items())
        return (f"env_steps={self.env_steps} dones={self.dones} captures={self.captures} near_ties={self.near_ties} "
                f"max|dobs|={self.max_obs:.2e} max|drew|={self.max_rew:.2e} max|dpos|={self.max_pos:.2e} "
                f"max|dvel|={self.max_vel:.2e} max|dquat|={self.max_quat:.2e} | obs entries compared={self.obs_entries}, "
                f"passed only by a carve-out: {carved}")


def run_lockstep(gpu_env, workers, actions, resync_every, report=None, check_state=True,
                 obs_tol=OBS_TOL, rew_tol=REW_TOL):
    """Steps the CUDA env and the oracle workers in lock-step on `actions` [T, N, 4].

    Every `resync_every` control steps (= HORIZON_SUBSTEPS / S) the continuous state is
    compared against the horizon tolerances and the oracle state is uploaded again, so
    each comparison window is one stated horizon.  A discrete disagreement is accepted only
    if the oracle's own threshold margin at that step is < MARGIN_TOL; the env is then
    re-synchronised from the oracle.
    """
    rep = report or ParityReport()
    T, N = actions.shape[0], actions.shape[1]
    on_gpu = hasattr(gpu_env, "device")
    if on_gpu:
        import torch
        a_dev = torch.from_numpy(actions).to(gpu_env.device)
    for t in range(T):
        o, r, d, f = [_np(x).copy() for x in gpu_env.step(a_dev[t] if on_gpu else actions[t])]
        term_obs = _np(gpu_env.terminal_obs)
        has_ep = hasattr(gpu_env, "episode_return")
        ep_r = _np(gpu_env.episode_return) if has_ep else None
        ep_l = _np(gpu_env.episode_length) if has_ep else None
        need_resync = False
        for i, w in enumerate(workers):
            prev_idx = w.env._current_target_index
            oo, rr, dd, info = w.step(actions[t, i])
            rep.env_steps += 1
            angn = w.last_step_ang_v_norm
            want_bits = (1 if w.last_terminated else 0) | (2 if w.last_truncated else 0)
            assert bool(want_bits) == bool(dd)
            tie = min_margin(w.env) < MARGIN_TOL
            discrete_ok = (int(d[i]) == want_bits) and (int(f[i]) == info["found_targets"])
            if not discrete_ok:
                assert tie, (f"discrete mismatch at t={t} env={i}: gpu done={d[i]} found={f[i]} vs oracle "
                             f"{want_bits}/{info['found_targets']}, oracle margin={min_margin(w.env):.3e}")
                rep.near_ties += 1
                need_resync = True
                continue
            rew_err = abs(float(r[i]) - float(np.float32(rr)))
            if rew_err > rew_tol:
                # orientation / smoothness thresholds only change the reward, not the state
                assert tie, f"reward mismatch at t={t} env={i}: {r[i]} vs {rr} (margin {min_margin(w.env):.3e})"
                rep.near_ties += 1
            else:
                rep.max_rew = max(rep.max_rew, rew_err)
            rep.max_obs = max(rep.max_obs, obs_error(o[i], oo, angn, rep, obs_tol))
            assert rep.max_obs <= obs_tol, f"obs drift {rep.max_obs:.3e} at t={t} env={i}\n gpu {o[i]}\n ref {oo}"
            if dd:
                rep.dones += 1
                e = obs_error(term_obs[i], info["terminal_observation"], angn, rep, obs_tol)
                assert e <= obs_tol, f"terminal obs mismatch {e:.3e} at t={t} env={i}"
                if has_ep:
                    assert int(ep_l[i]) == info["episode"]["l"]
                    assert abs(float(ep_r[i]) - info["episode"]["r"]) <= max(5e-3, 1e-5 * abs(info["episode"]["r"]))
            if info["found_targets"] > prev_idx:
                rep.captures += 1
        if check_state and ((t + 1) % resync_every == 0 or need_resync or t == T - 1):
            st = {k: _np(v) for k, v in gpu_env.get_state().items()}
            ref = oracle_state_arrays([w.env for w in workers])
            if not need_resync:
                rep.max_pos = max(rep.max_pos, float(np.max(np.abs(st["pos"] - ref["pos"]))))
                rep.max_vel = max(rep.max_vel, float(np.max(np.abs(st["vel"] - ref["vel"]))))
                qd = np.minimum(np.abs(st["quat"] - ref["quat"]).max(axis=1), np.abs(st["quat"] + ref["quat"]).max(axis=1))
                rep.max_quat = max(rep.max_quat, float(qd.max()))
                assert rep.max_pos <= POS_TOL and rep.max_vel <= VEL_TOL and rep.max_quat <= QUAT_TOL, str(rep)
                np.testing.assert_array_equal(st["target_idx"], ref["target_idx"])
                np.testing.assert_array_equal(st["steps"], ref["steps"])
                np.testing.assert_array_equal(st["just_found"], ref["just_found"])
            upload_oracle_state(gpu_env, workers)
    return rep


# (model, action type, track, S, control steps, re-synchronisation period)
CONTROLLER_CASES = [
    ("cf2p", "rpm", "circle", 8, 90, 30), ("racer", "rpm", "reaching", 8, 90, 30), ("racer", "one_d_rpm", "circle", 1, 240, 240),
    ("cf2x", "one_d_pid", "circle", 8, 120, 30), ("cf2x", "vel", "circle", 8, 90, 1), ("cf2p", "pid", "reaching", 1, 240, 1),
]


def controller_lockstep_case(make_env, N, model, act, track, S, T, resync, get_pid):
    """Airframes other than CF2X and BaseSingleAgentAviary's action types, FP32 implementation against the oracle in
    lock-step.  PID and VEL close a loop whose roll axis is a POSITIVE feedback under the reference's DYN torque signs
    (BaseAviary.py:931 vs the DSLPIDControl mixer, DSLPIDControl.py:47-53; see DESIGN.md), so those two are
    re-synchronised every step -- one-step errors are what is compared; the vertical ONE_D_PID loop is stable and runs
    whole horizons.  The oracle's RPM map runs with the float32 semantics of the reference's pinned numpy 1.26."""
    from oracle.dyn_oracle import OracleWorker, circle_track, make_reference_env, reaching_track
    targets, init, dim = circle_track() if track == "circle" else reaching_track()
    env = make_env(N, targets, init, dim)
    workers = [OracleWorker(make_reference_env(track, pyb_freq=240, ctrl_freq=240 // S, act=act, drone_model=model,
                                               normalize_actions=False), normalize_obs=False) for _ in range(N)]
    obs = _np(env.reset())
    for i, w in enumerate(workers):
        o, _ = w.reset()
        if obs.any():      # (the host emulator has no reset kernel and returns zeros)
            np.testing.assert_allclose(obs[i], o, atol=1e-6)
    rng = np.random.default_rng(1234 + S + len(act))
    if act in ("rpm", "one_d_rpm"):
        a = rng.uniform(-1, 1, size=(T, N, 4))
    else:
        a = np.repeat(rng.uniform(-1, 1, size=((T + 9) // 10, N, 4)), 10, axis=0)[:T]
        if act == "pid":
            a = np.concatenate([init[0] + 0.5 * a[..., :3], a[..., 3:]], axis=-1)
    rep = run_lockstep(env, workers, a.astype(np.float32), resync_every=resync)
    print(f"\n[{model} {act} {track} S={S}] {rep}")
    assert rep.near_ties <= 2 and rep.env_steps == T * N
    if act in ("pid", "vel", "one_d_pid"):
        want = np.stack([np.concatenate([w.env.ctrl.integral_pos_e, w.env.ctrl.integral_rpy_e, w.env.ctrl.last_rpy]) for w in workers])
        np.testing.assert_allclose(get_pid(env), want, atol=1e-5)
    return env, workers


def run_lockstep_batched(env, B, actions, resync_every, obs_tol=OBS_TOL, rew_tol=REW_TOL):
    """FULL-SIZE lock-step: the FP32 implementation `env` (CUDA BatchedDroneEnv, or the host emulator) against the batched
    FP64 oracle `B` (oracle/batched_oracle.py) on `actions` [T, N, 4], every environment compared at every step.  Same
    rules as run_lockstep: continuous quantities within the stated horizon tolerances, the oracle state uploaded again every
    `resync_every` control steps (one stated horizon), discrete outputs exact unless the oracle's own margin to the
    threshold involved is below MARGIN_TOL (near-tie: counted, environment re-synchronised)."""
    rep = ParityReport()
    T, N = actions.shape[:2]
    on_gpu = hasattr(env, "device")
    if on_gpu:
        import torch
        a_dev = torch.from_numpy(actions).to(env.device)
    for t in range(T):
        o, r, d, f = [_np(x).copy() for x in env.step(a_dev[t] if on_gpu else actions[t])]
        term = _np(env.terminal_obs).copy()
        prev_idx = B.idx.copy()
        oo, rr, bits, found, tt, ep_r, ep_l = B.step(actions[t])
        rep.captures += int((found > prev_idx).sum())
        rep.env_steps += N
        tie = B.margin < MARGIN_TOL
        bad = (d != bits) | (f != found)
        assert not (bad & ~tie).any(), (f"discrete mismatch at t={t}, envs {np.nonzero(bad & ~tie)[0][:8]}: "
                                        f"done {d[bad & ~tie][:8]} vs {bits[bad & ~tie][:8]}, margins {B.margin[bad & ~tie][:8]}")
        rep.near_ties += int(bad.sum())
        ok = ~bad
        rew_err = np.abs(r.astype(np.float64) - np.float32(rr).astype(np.float64))
        gimbal = B.gimbal_margin < MARGIN_TOL               # Bullet's |sarg| >= 0.99999 Euler branch near its tie: obs[3:6] and the
        rep.near_ties += int(gimbal.sum())                  # forward vector of the orientation reward jump, the state does not
        soft = tie | gimbal | (B.rew_margin < MARGIN_TOL)   # a reward-only threshold (orientation, smoothness) near its tie
        assert (rew_err[ok & ~soft] <= rew_tol).all(), f"reward mismatch at t={t}: {rew_err[ok & ~soft].max():.3e}"
        rep.near_ties += int((ok & soft & (rew_err > rew_tol)).sum())
        rep.max_rew = max(rep.max_rew, float(rew_err[ok & ~soft].max(initial=0.0)))
        done = bits != 0
        for got, want, sel in ((np.where(done[:, None], term, o), tt, ok), (o, oo, ok & done)):     # step obs; reset obs where done
            e = np.abs(got.astype(np.float64) - want.astype(np.float64))
            e[:, 3:6] = np.minimum(e[:, 3:6], np.abs(2.0 - e[:, 3:6]))

            def over():                                      # entries of the selected rows still above the plain tolerance
                return int((e[sel] > obs_tol).sum())
            n0 = over()
            e[:, 9:12] = np.maximum(e[:, 9:12] - ANGV_ABS_TOL / np.maximum(B.last_ang_v_norm, 1e-30)[:, None], 0.0)
            n1 = over()
            cond = EULER_COND_TOL / np.maximum(np.cos(np.pi * want[:, 4].astype(np.float64)), 1e-5)
            e[:, 3], e[:, 5] = np.maximum(e[:, 3] - cond, 0.0), np.maximum(e[:, 5] - cond, 0.0)
            n2 = over()
            e[gimbal, 3:6] = 0.0
            n3 = over()
            e[:, 3:6] /= np.maximum(1.0, B.last_ang_v_norm / EULER_RATE_REF)[:, None]
            n4 = over()
            rep.obs_entries += int(sel.sum()) * e.shape[1]
            for key, n in (("ang_v_direction", n0 - n1), ("euler_gimbal_conditioning", n1 - n2), ("euler_gimbal_branch", n2 - n3),
                           ("euler_tumbling_rate", n3 - n4)):
                rep.carved[key] += n
            if sel.any():
                m = float(e[sel].max())
                rep.max_obs = max(rep.max_obs, m)
                assert m <= obs_tol, f"obs drift {m:.3e} at t={t} env {int(np.argmax(e.max(axis=1) * sel))}"
        rep.dones += int(done.sum())
        if (t + 1) % resync_every == 0 or bad.any() or t == T - 1:
            st = {k: _np(v) for k, v in env.get_state().items()}
            ref = B.state()
            sel = ok
            rep.max_pos = max(rep.max_pos, float(np.abs(st["pos"] - ref["pos"])[sel].max()))
            rep.max_vel = max(rep.max_vel, float(np.abs(st["vel"] - ref["vel"])[sel].max()))
            qd = np.minimum(np.abs(st["quat"] - ref["quat"]).max(axis=1), np.abs(st["quat"] + ref["quat"]).max(axis=1))
            rep.max_quat = max(rep.max_quat, float(qd[sel].max()))
            assert rep.max_pos <= POS_TOL and rep.max_vel <= VEL_TOL and rep.max_quat <= QUAT_TOL, str(rep)
            for k in ("target_idx", "steps", "just_found"):
                np.testing.assert_array_equal(np.asarray(st[k])[sel], np.asarray(ref[k])[sel])
            env.set_state({k: v for k, v in ref.items() if k not in ("ep_return", "ep_length") or on_gpu})
    return rep
