"""Pins of what used to be restated only (VERDICT r1, "next" item 3):

 * the drag / ground-effect force formulas against the reference's OWN ``BaseAviary._drag`` / ``_groundEffect``
   (tests/golden/forces_ref.npz: arguments they hand to ``p.applyExternalForce``, recorded by the pybullet shim);
 * the reward the ``hover`` fixture carries is the reference's own ``HoverAviary._computeReward`` function object;
 * the three Bullet quaternion helpers (restated from bullet3 in the shim AND in the oracle) against an independent
   implementation, ``scipy.spatial.transform.Rotation``;
 * the one genuine SB3-written PPO archive the reference ships loads through ``checkpoint.load_sb3_zip``.
"""
import json
import os

import numpy as np
import pytest

from tests.golden.make_ref_golden import HAVE_REF, REF

HERE = os.path.dirname(os.path.abspath(__file__))
ARCHIVE = os.path.join(REF, "Sol", "pyfly", "ppo_quadx_waypoints.zip")


# ---------------------------------------------------------------------------------------------------------------------
# drag / ground effect (SURVEY a7)
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_env_at(g, i):
    from oracle.dyn_oracle import make_reference_env
    env = make_reference_env("circle", pyb_freq=240, ctrl_freq=30)
    env.reset()
    env.pos, env.quat, env.vel = g["pos"][i].copy(), g["quat"][i].copy(), g["vel"][i].copy()
    # float32, as in the reference: BaseAviary.step stores the float32 output of the THRUST action map (BaseAviary.py:442),
    # so `2 * np.pi * rpm / 60` and its sum are float32 arithmetic in _drag
    env.last_clipped_action = g["last_rpm"][i].astype(np.float32)
    return env


def test_oracle_constants_are_the_references():
    from oracle.dyn_oracle import CF2X
    g = np.load(os.path.join(HERE, "golden", "forces_ref.npz"))
    kf, gnd_coeff, prop_r, h_clip, dxy, dxy2, dz = g["constants"]
    assert (CF2X.KF, CF2X.GND_EFF_COEFF, CF2X.PROP_RADIUS) == (kf, gnd_coeff, prop_r)
    assert abs(CF2X.GND_EFF_H_CLIP - h_clip) < 1e-15
    assert (CF2X.DRAG_COEFF_XY, CF2X.DRAG_COEFF_XY, CF2X.DRAG_COEFF_Z) == (dxy, dxy2, dz)
    np.testing.assert_array_equal(np.asarray(CF2X.PROP_XY), g["link_offsets"][:4, :2])


def test_oracle_drag_and_ground_effect_match_the_references_functions():
    """45 states (a DYN rollout that ends up tumbling + hand-placed edge states: height clip, |roll| / |pitch| beyond pi/2)."""
    from oracle.dyn_oracle import bullet_matrix_from_quaternion
    g = np.load(os.path.join(HERE, "golden", "forces_ref.npz"))
    n = g["pos"].shape[0]
    assert n >= 45 and 0 < int(g["gnd_applied"].sum()) < n          # both branches of the rpy test are present
    for i in range(n):
        env = _oracle_env_at(g, i)
        R = bullet_matrix_from_quaternion(env.quat)
        # forceObj of p.applyExternalForce(..., linkIndex=4, flags=LINK_FRAME), BaseAviary.py:855-865
        np.testing.assert_allclose(env._drag_link(R), g["drag_force_link"][i], rtol=1e-12, atol=1e-18)
        # LINK_FRAME: Bullet rotates the vector by the link (= base) orientation before applying it
        np.testing.assert_allclose(env._drag(R), R @ g["drag_force_link"][i], rtol=1e-12, atol=1e-18)
        # forceObj[2] of the four per-propeller calls (or no call at all), BaseAviary.py:820-834
        np.testing.assert_allclose(env._ground_effect(g["rpm"][i], R), g["gnd_force_z"][i], rtol=1e-12, atol=1e-18)


@pytest.mark.skipif(not HAVE_REF, reason="needs a checkout of the original project (DN_REFERENCE_ROOT)")
def test_force_fixture_is_reproduced_by_the_reference():
    import subprocess
    import sys
    import tempfile
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import tests.golden.make_ref_golden as M; "
            "ref = M._import_reference(); np.savez(sys.argv[1], **M.mint_forces(ref)); "
            "print('HOVER_FROM_REFERENCE', ref[-1])" % os.path.dirname(HERE))
    with tempfile.TemporaryDirectory() as tmp:
        out = subprocess.run([sys.executable, "-W", "ignore", "-c", code, os.path.join(tmp, "f.npz")], check=True, capture_output=True, text=True)
        # the hover fixture binds the reference's own HoverAviary._computeReward (not a hand-written copy)
        assert "HOVER_FROM_REFERENCE True" in out.stdout
        new, old = np.load(os.path.join(tmp, "f.npz")), np.load(os.path.join(HERE, "golden", "forces_ref.npz"))
        for k in old.files:
            np.testing.assert_array_equal(new[k], old[k], err_msg=k)


# ---------------------------------------------------------------------------------------------------------------------
# Bullet quaternion helpers against scipy (independent implementation)
# ---------------------------------------------------------------------------------------------------------------------
def _random_quats(n, seed):
    q = np.random.default_rng(seed).normal(size=(n, 4))
    return q / np.linalg.norm(q, axis=1, keepdims=True)


def test_bullet_quaternion_helpers_agree_with_scipy():
    from scipy.spatial.transform import Rotation
    from oracle.dyn_oracle import bullet_euler_from_quaternion, bullet_matrix_from_quaternion, bullet_quaternion_from_euler
    from tests.golden import ref_shims
    shim = ref_shims._PyBullet()
    q = _random_quats(100000, 0)
    rot = Rotation.from_quat(q)                      # scipy: scalar-last (x, y, z, w), like Bullet
    m_ref = rot.as_matrix()
    e_ref = rot.as_euler("xyz")                      # extrinsic x-y-z = Bullet's roll, pitch, yaw (R = Rz Ry Rx)
    away = np.abs(np.abs(e_ref[:, 1]) - np.pi / 2) > 1e-2        # away from the gimbal branch (|sarg| >= 0.99999)
    assert away.mean() > 0.98
    worst_m = worst_e = worst_q = 0.0
    for i in range(q.shape[0]):
        m = bullet_matrix_from_quaternion(q[i])
        worst_m = max(worst_m, float(np.abs(m - m_ref[i]).max()))
        if away[i]:
            e = bullet_euler_from_quaternion(q[i])
            worst_e = max(worst_e, float(np.abs(e - e_ref[i]).max()))
            back = bullet_quaternion_from_euler(e)
            worst_q = max(worst_q, float(min(np.abs(back - q[i]).max(), np.abs(back + q[i]).max())))
        if i < 2000:                                 # the shim's copies (plain-float code path) on a sample
            np.testing.assert_allclose(np.array(shim.getMatrixFromQuaternion(q[i])).reshape(3, 3), m_ref[i], atol=1e-14)
            if away[i]:
                np.testing.assert_allclose(shim.getEulerFromQuaternion(q[i]), e_ref[i], atol=1e-9)
                b = np.array(shim.getQuaternionFromEuler(e_ref[i]))
                assert min(np.abs(b - q[i]).max(), np.abs(b + q[i]).max()) < 1e-9
    assert worst_m < 1e-14 and worst_e < 1e-9 and worst_q < 1e-9, (worst_m, worst_e, worst_q)
    # un-normalised input: Bullet's setRotation divides by |q|^2 (BaseAviary.py:920 passes the integrator's quaternion as is)
    for scale in (0.5, 1.7):
        np.testing.assert_allclose(bullet_matrix_from_quaternion(scale * q[0]), m_ref[0], atol=1e-14)


# ---------------------------------------------------------------------------------------------------------------------
# the reference's genuine SB3 archive
# ---------------------------------------------------------------------------------------------------------------------
MANIFEST = os.path.join(HERE, "golden", "ppo_quadx_waypoints_manifest.json")


def test_sb3_archive_manifest_loads_into_a_learner():
    """Key / shape manifest of the original project's Sol/pyfly/ppo_quadx_waypoints.zip::policy.pth (committed: the archive
    itself is not part of this repository): a learner with that architecture accepts exactly those keys and shapes through the SB3 name map."""
    import torch
    from drl_dronenavigation_b200.checkpoint import policy_to_sb3_state_dict, sb3_state_dict_to_policy
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    man = json.load(open(MANIFEST))
    L = PPOLearner(man["obs_dim"], man["act_dim"], PPOConfig(pi_arch=tuple(man["pi_arch"]), vf_arch=tuple(man["vf_arch"]), update_impl="torch"))
    ours = policy_to_sb3_state_dict(L.policy)
    assert {k: list(v.shape) for k, v in ours.items()} == man["policy_pth"]
    fake = {k: torch.full(shape, 0.25) for k, shape in man["policy_pth"].items()}
    sb3_state_dict_to_policy(L.policy, fake, strict=True)
    assert all(float(p.detach().min()) == 0.25 for p in L.policy.parameters())


@pytest.mark.skipif(not os.path.exists(ARCHIVE), reason="needs the original project's SB3 archive (DN_REFERENCE_ROOT)")
def test_reference_sb3_archive_loads():
    """The archive SB3 itself wrote (members data, policy.pth, policy.optimizer.pth, pytorch_variables.pth, ...)."""
    import io
    import zipfile
    import torch
    from drl_dronenavigation_b200.checkpoint import load_sb3_zip, policy_to_sb3_state_dict
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    path = ARCHIVE
    man = json.load(open(MANIFEST))
    with zipfile.ZipFile(path) as zf:
        assert {"data", "policy.pth", "policy.optimizer.pth", "pytorch_variables.pth"} <= set(zf.namelist())
        sd = torch.load(io.BytesIO(zf.read("policy.pth")), map_location="cpu", weights_only=True)
    assert {k: list(v.shape) for k, v in sd.items()} == man["policy_pth"]
    L = PPOLearner(man["obs_dim"], man["act_dim"], PPOConfig(pi_arch=tuple(man["pi_arch"]), vf_arch=tuple(man["vf_arch"]), update_impl="torch"))
    data = load_sb3_zip(path, L, load_optimizer=True)
    back = policy_to_sb3_state_dict(L.policy)
    for k, v in sd.items():
        assert torch.equal(back[k], v), k
    # the loaded policy is a function: deterministic action of a fixed observation is finite and reproducible
    obs = torch.linspace(-1, 1, man["obs_dim"]).repeat(3, 1)
    a1, _, v1 = L.policy.act(obs, deterministic=True)
    assert torch.isfinite(a1).all() and torch.isfinite(v1).all() and a1.shape == (3, man["act_dim"])
    assert isinstance(data, dict)
    # SB3's optimiser state (positional, log_std first) is re-indexed into this repo's parameter order
    st = L.opt.state_dict()["state"]
    if st:
        for i, p in enumerate(L.policy.parameters()):
            assert tuple(st[i]["exp_avg"].shape) == tuple(p.shape)
