"""Fixtures minted from the REFERENCE'S OWN CODE (tests/golden/ref_*.npz; generator tests/golden/make_ref_golden.py
imports the original project unmodified behind import shims for the absent third-party packages).

 - not gpu: (1) if a checkout of the original project is present (make_ref_golden.REF), the generator still reproduces the committed
            fixtures bit for bit; (2) the oracle restatement matches them to FP64 round-off
            (obs: identical float32 values; reward 1e-12; done bits / found_targets / Monitor lengths exact);
            (3) the host build of the device step logic matches them within the stated FP32 tolerances.
 - gpu:     the CUDA path, through the C ABI, matches them within the stated FP32 tolerances.
"""
import glob
import os

import numpy as np
import pytest

from tests.golden.make_ref_golden import CASES, HAVE_REF

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ref_*.npz")))
IDS = [os.path.basename(p)[:-4] for p in GOLD]


REWARD_IDS = {"default": 0, "dummy": 1, "thrustenv": 2, "her": 3, "reaching": 4, "progress": 5, "hover": 6, "flythrugate": 7,
              "bootstrapped": 8, "champ": 9}


def _meta(g):
    m = [str(x) for x in g["meta"]]
    m = m + ["default", "0", "0", "1", "1", "thrust", "cf2x"][len(m) - 5:]
    track, S, mode, max_steps, norm, reward, norm_rew, clip_rew, dist, nact, act, model = m[:12]
    return dict(track=track, S=int(S), mode=mode, max_steps=int(max_steps), norm=(norm == "1"), reward=reward,
                norm_rew=(norm_rew == "1"), clip_rew=(clip_rew == "1"), include_distance=(dist == "1"), normalize_actions=(nact == "1"),
                act=act, model=model)


ACT_IDS = {"thrust": 0, "rpm": 1, "one_d_rpm": 2, "pid": 3, "vel": 4, "one_d_pid": 5}
MODEL_IDS = {"cf2x": 0, "cf2p": 1, "racer": 2}


def test_fixtures_exist():
    assert sorted(IDS) == sorted(CASES)


@pytest.mark.skipif(not HAVE_REF, reason="needs a checkout of the original project (DN_REFERENCE_ROOT)")
def test_reference_reproduces_fixtures():
    """Re-runs the reference for a few of the cases (each one exercises every function on the path)."""
    import subprocess
    import sys
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import tests.golden.make_ref_golden as M; "
            "ref = M._import_reference(); "
            "[np.savez(sys.argv[1] + '/' + n + '.npz', **M.run(ref, *M.CASES[n])) for n in sys.argv[2:]]"
            % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import tempfile
    names = ["ref_circle_s8_saturating", "ref_reaching_s8_saturating", "ref_circle_s1_truncate", "ref_circle_s8_normobs",
             "ref_circle_s8_cf2p_pid", "ref_reaching_s8_race_rpm"]
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([sys.executable, "-W", "ignore", "-c", code, tmp] + names, check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        for n in names:
            new, old = np.load(os.path.join(tmp, n + ".npz")), np.load(os.path.join(os.path.dirname(__file__), "golden", n + ".npz"))
            for k in old.files:
                np.testing.assert_array_equal(new[k], old[k], err_msg=f"{n}:{k}")


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_oracle_matches_reference(path):
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    g = np.load(path)
    m = _meta(g)
    norm = m["norm"]
    T, N = g["reward"].shape
    ws = [OracleWorker(make_reference_env(m["track"], pyb_freq=240, ctrl_freq=240 // m["S"], max_steps=m["max_steps"],
                                          reward_id=m["reward"], include_distance=m["include_distance"],
                                          normalize_actions=m["normalize_actions"], act=m["act"], drone_model=m["model"]),
                       normalize_obs=norm, normalize_reward=m["norm_rew"], clip_reward=10.0 if m["clip_rew"] else 0.0)
          for _ in range(N)]
    for w in ws:
        w.env.numpy_legacy_cast = False          # the fixtures were minted under numpy 2.x (float64 RPM map)
    # the PID family feeds the state back through gains of up to 7e4: the scipy Euler round trip restated in numpy and
    # the 1e-16 differences in summation order are amplified, the loop being unstable in roll (see DESIGN.md)
    pid = m["act"] in ("pid", "vel", "one_d_pid")
    tol = 1e4 if pid else 1.0
    obs0 = np.stack([w.reset()[0] for w in ws])
    np.testing.assert_allclose(obs0, g["obs0"], rtol=0, atol=1e-12)
    ep_checked = 0
    for t in range(T):
        for i, w in enumerate(ws):
            o, r, d, info = w.step(g["actions"][t, i])
            bits = (1 if w.last_terminated else 0) | (2 if w.last_truncated else 0)
            assert bits == g["done"][t, i], (t, i)
            assert info["found_targets"] == g["found_targets"][t, i], (t, i)
            np.testing.assert_allclose(o, g["obs"][t, i], rtol=0, atol=1e-9 if norm else (1e-7 if pid else 0))
            assert abs(float(r) - g["reward"][t, i]) <= 1e-12 * tol * max(1.0, abs(g["reward"][t, i]))
            if d:
                np.testing.assert_allclose(info["terminal_observation"], g["terminal_obs"][t, i], rtol=0, atol=1e-9 if norm else (1e-7 if pid else 0))
                assert info["episode"]["l"] == g["ep_length"][t, i]
                assert abs(info["episode"]["r"] - g["ep_return"][t, i]) <= 1e-5 + 1e-9 * abs(g["ep_return"][t, i])   # Monitor rounds to 6 decimals
                ep_checked += 1
            else:
                # physical state right after a non-terminal step (after a done the oracle worker has already reset)
                if pid:
                    np.testing.assert_allclose(np.float64(w.env.last_clipped_action), g["rpm"][t, i], rtol=0, atol=1e-5)
                    c = w.env.ctrl
                    np.testing.assert_allclose(np.concatenate([c.integral_pos_e, c.integral_rpy_e, c.last_rpy]), g["pid"][t, i], rtol=0, atol=1e-9)
                else:
                    np.testing.assert_array_equal(np.float64(w.env.last_clipped_action), g["rpm"][t, i])   # action map: exact
                np.testing.assert_allclose(w.env.pos, g["pos"][t, i], rtol=0, atol=1e-13 * tol)
                np.testing.assert_allclose(w.env.vel, g["vel"][t, i], rtol=0, atol=1e-12 * tol)
                np.testing.assert_allclose(w.env.rpy_rates, g["rpy_rates"][t, i], rtol=0, atol=1e-10 * tol)
                np.testing.assert_allclose(w.env.ang_v, g["ang_v"][t, i], rtol=0, atol=1e-10 * tol)
                q, qr = w.env.quat, g["quat"][t, i]
                assert min(np.abs(q - qr).max(), np.abs(q + qr).max()) <= 1e-13 * tol
                assert abs(w.env._distance_to_target - g["dist"][t, i]) <= 1e-13 * tol
    assert ep_checked == int((g["done"] != 0).sum())


# ---- FP32 implementations against the reference fixtures ---------------------------------------------------------
# Open loop over the whole fixture without re-synchronisation (up to 480 substeps = 2x the stated 1 s horizon;
# the saturating-action cases reach |rates| ~ 60 rad/s): |dobs| <= 1e-3, |dreward| <= 1e-2, discrete outputs exact.
OBS_TOL, REW_TOL = 1e-3, 1e-2
# The STATED tolerance (north_star / SURVEY 8c / parity_utils.py): |dobs| <= 1e-4, |dreward| <= 1e-3 over a 240-substep (1 s)
# open-loop horizon.  Asserted directly against the reference fixtures on the first 240 substeps of every one of them.
STATED_OBS_TOL, STATED_REW_TOL, STATED_SUBSTEPS = 1e-4, 1e-3, 240
NORM_OBS_TOL = 2e-4          # normalised observations (abs + rel), FP64 running statistics on both sides


def _resync(g, t, get_state, set_state):
    """PID-family fixtures: the reference's DYN x-torque has the opposite sign of what the DSLPIDControl mixer assumes
    (BaseAviary.py:931 vs DSLPIDControl.py:47-53), so the roll loop is a POSITIVE feedback with gains of 7e4 -- rounding
    differences grow by orders of magnitude within an episode and, the controller state surviving resets, across
    episodes.  These fixtures are therefore compared step by step: after step t the physical and controller state is
    re-seeded from the fixture (running envs only; an env that just finished keeps its own reset state)."""
    cur = get_state()
    run = (g["done"][t] == 0)
    st = {}
    for k in ("pos", "quat", "vel", "rpy_rates", "ang_v", "dist"):
        v = np.array(cur[k], dtype=np.float32, copy=True)
        v[run] = g[k][t][run]
        st[k] = v
    # the stored quaternion is the unit read-back; the fixture's may be its negative (same rotation): keep the sign
    flip = (np.sum(st["quat"] * np.asarray(cur["quat"]), axis=1) < 0)
    st["quat"][flip] *= -1
    st["pid"] = g["pid"][t].astype(np.float32)
    set_state(st)


def _compare_fp32(g, step_fn, obs0, norm, rel_reward=False, resync=None):
    np.testing.assert_allclose(obs0, g["obs0"], atol=2e-4 if norm else 1e-6)
    T, N = g["reward"].shape
    worst_obs = worst_rew = 0.0
    stated_steps = STATED_SUBSTEPS // _meta(g)["S"]           # control steps inside the stated horizon
    stated = {"obs": 0.0, "rew": 0.0, "steps": 0}
    for t in range(T):
        o, r, d, f, term = step_fn(g["actions"][t])
        if resync is not None:
            _resync(g, t, *resync)
        np.testing.assert_array_equal(d, g["done"][t])
        np.testing.assert_array_equal(f, g["found_targets"][t])
        for i in range(N):
            rows = [(o[i], g["obs"][t, i])]
            if d[i] and term is not None:
                rows.append((term[i], g["terminal_obs"][t, i]))
            for a, b in rows:
                e = np.abs(a.astype(np.float64) - b)
                if norm:
                    # NormalizeObservation divides by sqrt(var + 1e-8) of a per-env running variance that is tiny for the
                    # first steps of an episode (gain up to 1e4 on the raw observation's FP32 error).  The statistics
                    # themselves are FP64 on the device, like the reference's.
                    keep = list(range(9)) + ([12] if a.size > 12 else [])
                    stated["norm"] = max(stated.get("norm", 0.0), float(np.max(e[keep] / (1.0 + np.abs(b[keep])))))
                    np.testing.assert_allclose(a[keep], b[keep], atol=NORM_OBS_TOL, rtol=NORM_OBS_TOL)
                    continue
                e[3:6] = np.minimum(e[3:6], np.abs(2 - e[3:6]))        # +-pi wrap of the Euler angles
                worst_obs = max(worst_obs, e[:9].max(), e[12] if e.size > 12 else 0.0)
                if t < stated_steps:
                    stated["obs"] = max(stated["obs"], e[:9].max(), e[12] if e.size > 12 else 0.0)
                # obs[9:12] = ang_v/|ang_v| is ill-conditioned near |ang_v| = 0; bounded by the absolute ang_v error
                angn = float(np.linalg.norm(g["ang_v"][t, i]))
                if not d[i]:
                    assert (e[9:12] <= 1e-3 + 1e-4 / max(angn, 1e-30)).all(), (t, i, e[9:12], angn)
        if rel_reward:
            # NormalizeReward divides by sqrt(var + 1e-8) of a running variance that starts near 0 (gain up to 1e4), and
            # the HER reward reaches 1e6: relative tolerance on top of the absolute one
            np.testing.assert_allclose(r, g["reward"][t], rtol=2e-3, atol=REW_TOL)
        else:
            worst_rew = max(worst_rew, float(np.abs(r - g["reward"][t]).max()))
            if t < stated_steps:
                stated["rew"] = max(stated["rew"], float(np.abs(r - g["reward"][t]).max()))
        if t < stated_steps:
            stated["steps"] = t + 1
    assert worst_obs < OBS_TOL and worst_rew < REW_TOL, (worst_obs, worst_rew)
    # the stated tolerance, CUDA / host build vs REFERENCE fixture directly (not via the oracle).  Skipped only where the
    # comparison above is relative by construction (normalised observations / normalised or 1e6-sized rewards) and for the
    # step-by-step re-synchronised PID fixtures (their horizon is one step).
    if not norm and resync is None:
        assert stated["steps"] == min(T, stated_steps)
        assert stated["obs"] <= STATED_OBS_TOL, ("stated obs tolerance", stated)
        if not rel_reward:
            assert stated["rew"] <= STATED_REW_TOL, ("stated reward tolerance", stated)
    return worst_obs, worst_rew, stated


def _env_args(g):
    from oracle.dyn_oracle import circle_track, reaching_track
    m = _meta(g)
    targets, init, dim = circle_track() if m["track"] == "circle" else reaching_track()
    kw = dict(target_points=targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=240 // m["S"],
              circle=(m["track"] == "circle"), include_distance=m["include_distance"], normalize_actions=m["normalize_actions"],
              max_steps=m["max_steps"],
              reward_id=REWARD_IDS[m["reward"]], normalize_reward=m["norm_rew"], clip_reward=10.0 if m["clip_rew"] else 0.0)
    kw["_act"], kw["_model"] = m["act"], m["model"]
    return kw, m["norm"], (m["norm_rew"] or m["reward"] == "her")


_NO_OBS_NORM = [p for p in GOLD if not _meta(np.load(p))["norm"]]        # the host emulator has no NormalizeObservation path


@pytest.mark.parametrize("path", _NO_OBS_NORM, ids=[os.path.basename(p)[:-4] for p in _NO_OBS_NORM])
def test_device_logic_matches_reference(path):
    """csrc/dn_device.cuh compiled for the host (tests/host_emu) against the reference fixtures."""
    from tests.host_emu import HostEmuEnv
    g = np.load(path)
    kw, norm, rel = _env_args(g)
    kw["act_type"], kw["drone_model"] = ACT_IDS[kw.pop("_act")], MODEL_IDS[kw.pop("_model")]
    env = HostEmuEnv(g["reward"].shape[1], kw.pop("target_points"), **kw)

    def step(a):
        o, r, d, f = env.step(a)
        return o, r, d, f, env.terminal_obs.copy()
    pid = "pid" in g.files
    print(_compare_fp32(g, step, g["obs0"], norm, rel, resync=(env.get_state, env.set_state) if pid else None))
    if pid:
        np.testing.assert_allclose(env.get_pid(), g["pid"][-1], atol=1e-6)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_cuda_matches_reference(path):
    import torch
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    g = np.load(path)
    from drl_dronenavigation_b200.enums import ActionType, DroneModel
    kw, norm, rel = _env_args(g)
    kw["act"], kw["drone_model"] = ActionType(kw.pop("_act")), DroneModel(kw.pop("_model"))
    env = BatchedDroneEnv(g["reward"].shape[1], kw.pop("target_points"), normalize_obs=norm, **kw)
    obs0 = env.reset().cpu().numpy()

    def step(a):
        o, r, d, f = env.step(torch.from_numpy(a).cuda())
        return o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy(), f.cpu().numpy(), env.terminal_obs.cpu().numpy()
    pid = "pid" in g.files
    get = lambda: {k: v.cpu().numpy() for k, v in env.get_state().items()}
    print(_compare_fp32(g, step, obs0, norm, rel, resync=(get, env.set_state) if pid else None))
    if pid:
        np.testing.assert_allclose(get()["pid"], g["pid"][-1], atol=1e-6)
    assert env.launch_count > g["reward"].shape[0]
    env.close()
