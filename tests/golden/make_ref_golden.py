"""Mints ``tests/golden/ref_*.npz`` by stepping the REFERENCE'S OWN code (imported unmodified from a checkout of
eRGiBi/DRL-DroneNavigation named by $DN_REFERENCE_ROOT), so that the oracle restatement and the CUDA path are pinned against what the
reference computes rather than against our reading of it.

Run (only the committed ``.npz`` fixtures are part of this repository, not that checkout):

    DN_REFERENCE_ROOT=<checkout> python tests/golden/make_ref_golden.py

What executes: ``Sol.Model.Environments.PBDroneEnv.PBDroneEnv`` (``step``, ``reset``, ``rescale_action``,
``_preprocessAction``, ``_computeObs``, ``_clipAndNormalizeState``, ``_computeReward``, ``orientation_reward``,
``smoothness_reward``, ``_computeTerminated``, ``is_out_of_cylinder_bounds``, ``_computeTruncated``,
``_update_state_post_step``), ``Sol.PyBullet.BaseAviary.BaseAviary`` (``step``, ``_dynamics``, ``_integrateQ``,
``_housekeeping``, ``_updateAndStoreKinematicInformation``, ``_parse_urdf_parameters`` on the reference's
own ``cf2x.urdf``), ``Sol.Model.env_utils`` (``cmd2pwm``, ``pwm2rpm``), ``Sol.Model.Environments.normalize``
(``NormalizeObservation``, ``RunningMeanStd``) and ``Sol.Utilities.Waypoints`` (``circle``, ``reaching``, ``Track``).

The three things that are NOT the reference (each unavoidable, each documented in DESIGN.md section 2):

1. third-party packages absent from this image are shimmed (``tests/golden/ref_shims.py``): pybullet becomes a
   state store with Bullet's quaternion maths restated; gymnasium/gym a minimal ``Env``/``Box``;
2. ``BaseAviary.py:418`` overwrites ``self.PHYSICS`` with ``Physics.PYB`` inside the substep loop, which makes
   the DYN branch unreachable.  ``_DynEnv`` below pins the attribute to ``Physics.DYN`` (a read-only property in
   a subclass; the assignment at :418 becomes a no-op), i.e. the loop runs as written minus that line;
3. ``BaseAviary.py:944`` reads the undefined ``self.TIMESTEP``; the subclass defines it as ``PYB_TIMESTEP``.

For the ``*_act_*`` / ``*_cf2p_*`` / ``*_race_*`` cases (action types and airframes PBDroneEnv itself never selects) three more,
all in ``make_env`` / ``_BsaAct`` below: the action type and its controller are attached after construction (PBDroneEnv drops
the ``act`` keyword), ``_saveLastAction`` stores 3- and 1-element actions as given (``BaseAviary.py:1013`` would raise), and
the CF2P / RACE constants are read from the reference's own URDFs and assigned to a CF2X-constructed env.

The SubprocVecEnv worker's auto-reset and the Monitor accumulators are SB3 code (absent); the loop in ``run``
restates that contract (reset on done, returned obs = reset obs, terminal obs kept aside).
"""
import contextlib
import copy
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("DN_REFERENCE_ROOT", "")          # a checkout of the original project; tests that re-run it skip without one
HAVE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "Sol"))
HOVER = 0.092227

CASES = {
    # name: (track, S, action mode, envs, steps, seed, max_steps, normalize_obs[, reward function, norm_rew, clip_rew])
    "ref_circle_s1_saturating": ("circle", 1, "saturating", 4, 160, 21, 4096, False),
    "ref_circle_s8_mixed": ("circle", 8, "mixed", 4, 60, 22, 4096, False),
    "ref_circle_s8_saturating": ("circle", 8, "saturating", 4, 40, 26, 4096, False),
    "ref_reaching_s8_saturating": ("reaching", 8, "saturating", 4, 50, 23, 4096, False),
    "ref_reaching_s1_hover": ("reaching", 1, "hover_band", 2, 200, 24, 4096, False),
    "ref_circle_s1_scripted": ("circle", 1, "scripted", 3, 120, 0, 4096, False),
    "ref_circle_s1_truncate": ("circle", 1, "hover", 2, 30, 0, 12, False),
    "ref_circle_s8_normobs": ("circle", 8, "mixed", 3, 60, 25, 4096, True),
    "ref_circle_s1_normobs_resets": ("circle", 1, "saturating", 3, 140, 27, 4096, True),
    # reward wrappers of make_env (PBDroneSimulator.py:190-195): clip to +-10, then the reference's NormalizeReward
    "ref_circle_s8_normrew": ("circle", 8, "mixed", 3, 60, 28, 4096, False, "default", True, False),
    "ref_reaching_s8_cliprew_normrew": ("reaching", 8, "saturating", 3, 50, 29, 4096, True, "default", True, True),
    # other reward functions of the reference, run inside the same PBDroneEnv step machine (SURVEY a19)
    "ref_reaching_s8_rw_dummy": ("reaching", 8, "mixed", 3, 50, 30, 4096, False, "dummy", False, False),
    "ref_circle_s8_rw_thrustenv": ("circle", 8, "mixed", 3, 50, 31, 4096, False, "thrustenv", False, False),
    "ref_reaching_s8_rw_thrustenv": ("reaching", 8, "hover_band", 2, 40, 32, 4096, False, "thrustenv", False, False),
    "ref_reaching_s8_rw_her": ("reaching", 8, "mixed", 3, 50, 33, 4096, False, "her", False, False),
    "ref_circle_s8_rw_her": ("circle", 8, "saturating", 3, 40, 34, 4096, False, "her", False, False),
    "ref_reaching_s8_rw_reaching": ("reaching", 8, "mixed", 3, 50, 35, 4096, False, "reaching", False, False),
    "ref_circle_s1_rw_reaching": ("circle", 1, "saturating", 3, 140, 36, 4096, False, "reaching", False, False),
    "ref_circle_s8_rw_hover": ("circle", 8, "mixed", 2, 40, 37, 4096, False, "hover", False, False),
    "ref_circle_s8_rw_flythrugate": ("circle", 8, "mixed", 2, 40, 38, 4096, False, "flythrugate", False, False),
    # the other constructor switches of PBDroneEnv: 12-dim observation (include_distance=False) and the physical action
    # space (normalize_actions=False: actions are per-motor thrusts in newtons, no rescale_action)
    "ref_circle_s8_obs12_physact": ("circle", 8, "physical", 3, 60, 39, 4096, False, "default", False, False, False, False),
    "ref_reaching_s1_obs12": ("reaching", 1, "hover_band", 2, 120, 40, 4096, False, "default", False, False, False, True),
    # the two literature reward calculators of Rewarder.py ("yet unused" in the reference): the reference's own calculator objects
    # fed from PBDroneEnv's waypoint machine (_Literature below)
    "ref_reaching_s8_rw_bootstrapped": ("reaching", 8, "mixed", 3, 50, 50, 4096, False, "bootstrapped", False, False),
    "ref_circle_s8_rw_champ": ("circle", 8, "mixed", 3, 50, 51, 4096, False, "champ", False, False),
    "ref_reaching_s1_rw_champ": ("reaching", 1, "hover_band", 2, 150, 52, 4096, False, "champ", False, False),
    # BaseSingleAgentAviary._preprocessAction (the branches PBDroneEnv overrides) bound onto the same step machine:
    # RPM / ONE_D_RPM maps, and the PID family through the reference's DSLPIDControl (with the real scipy Rotation)
    "ref_circle_s8_act_rpm": ("circle", 8, "rpm", 3, 60, 41, 4096, False, "default", False, False, True, False, "rpm", "cf2x"),
    "ref_reaching_s1_act_one_d_rpm": ("reaching", 1, "rpm", 2, 150, 42, 4096, False, "default", False, False, True, False, "one_d_rpm", "cf2x"),
    "ref_circle_s8_act_pid": ("circle", 8, "pid", 3, 80, 43, 4096, False, "default", False, False, True, False, "pid", "cf2x"),
    "ref_reaching_s1_act_pid": ("reaching", 1, "pid", 3, 200, 44, 4096, False, "default", False, False, True, False, "pid", "cf2x"),
    "ref_circle_s8_act_vel": ("circle", 8, "vel", 3, 80, 45, 4096, False, "default", False, False, True, False, "vel", "cf2x"),
    "ref_circle_s8_act_one_d_pid": ("circle", 8, "one_d", 3, 120, 46, 4096, False, "default", False, False, True, False, "one_d_pid", "cf2x"),
    # the other airframes of BaseAviary._dynamics (:927-935), constants parsed from the reference's own URDFs
    "ref_circle_s8_cf2p_rpm": ("circle", 8, "rpm", 3, 60, 47, 4096, False, "default", False, False, True, False, "rpm", "cf2p"),
    "ref_reaching_s8_race_rpm": ("reaching", 8, "rpm", 3, 60, 48, 4096, False, "default", False, False, True, False, "rpm", "racer"),
    "ref_circle_s8_cf2p_pid": ("circle", 8, "pid", 3, 80, 49, 4096, False, "default", False, False, True, False, "pid", "cf2p"),
}


def actions(mode, T, N, seed, track="circle"):
    u = np.random.default_rng(seed).uniform(-1, 1, size=(T, N, 4))
    if mode == "scripted":     # SURVEY 8c scenarios: hover band, max thrust, min thrust
        a = np.zeros((T, N, 4))
        a[:, 0], a[:, 1], a[:, 2] = 0.0922265, 1.0, -1.0
        return a.astype(np.float32)
    if mode == "hover":
        return np.full((T, N, 4), 0.0922265, np.float32)
    if mode == "rpm":          # BaseSingleAgentAviary RPM map: rpm = HOVER_RPM (1 + 0.05 a)
        return (0.6 * u).astype(np.float32)
    if mode in ("pid", "vel", "one_d"):   # piecewise-constant commands, held for 10 control steps
        h = np.repeat(np.random.default_rng(seed + 1000).uniform(-1, 1, size=((T + 9) // 10, N, 4)), 10, axis=0)[:T]
        if mode == "pid":      # destinations within ~0.5 m of the spawn point
            base = np.array([1.0, 0.0, 1.0, 0.0]) if track == "circle" else np.array([-0.5, 0.9, 1.2, 0.0])
            return (base + 0.5 * h).astype(np.float32)
        return h.astype(np.float32)
    if mode == "physical":     # per-motor thrust in newtons around the hover thrust 0.06615 N (physical bounds 0.0282 .. 0.1483 N)
        return (0.06615 + 0.02 * u).astype(np.float32)
    return {"saturating": u, "hover_band": HOVER + 0.002 * u, "mixed": HOVER + 0.006 * u}[mode].astype(np.float32)


def _import_reference():
    sys.path.insert(0, REPO)
    from tests.golden import ref_shims
    ref_shims.install(REF)
    os.chdir(REF)                      # BaseAviary.py:99 opens "Sol/resources/safegym/cf2x.urdf" relative to the cwd
    with contextlib.redirect_stdout(io.StringIO()):
        from Sol.Model.Environments.PBDroneEnv import PBDroneEnv
        from Sol.Model.Environments import normalize
        from Sol.PyBullet.enums import ActionType, Physics
        from Sol.Utilities import Waypoints

    class _DynEnv(PBDroneEnv):
        PHYSICS = property(lambda self: Physics.DYN, lambda self, value: None)        # see (2) above
        TIMESTEP = property(lambda self: self.PYB_TIMESTEP)                           # see (3) above

    # ---- the reference's OTHER reward functions, bound unmodified onto the same step machine ------------------
    with contextlib.redirect_stdout(io.StringIO()):
        from Sol.Model.Environments import dummy_env, ThrustEnv, HerPBDroneEnv
        from Sol.PyBullet.FlyThruGateAviary import FlyThruGateAviary
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "_ref_hover", os.path.join(REF, "Sol/PyBullet/GymPybulletDronesMain/gym_pybullet_drones/envs/single_agent_rl/HoverAviary.py"))
    try:
        # HoverAviary.py:3-4 imports `gym_pybullet_drones.utils.enums` (fine) and
        # `gym_pybullet_drones.envs.single_agent_rl.BaseSingleAgentAviary`, whose vendored copy cannot be imported by anyone:
        # its line 8 reads `sys.path.append(....gym_pybullet_drones)` (attribute access on Ellipsis -> AttributeError), and the
        # package __init__ files import it.  The base-class module (and the two package levels above it) are therefore stubbed
        # with the reference's OWN working copy of the same class, Sol/PyBullet/BaseSingleAgentAviary.py; HoverAviary.py itself
        # is then executed unmodified and its `_computeReward` function object is what the fixture binds.
        import types
        sys.path.insert(1, os.path.join(REF, "Sol/PyBullet/GymPybulletDronesMain"))   # the vendored upstream package tree
        with contextlib.redirect_stdout(io.StringIO()):
            import gym_pybullet_drones.utils.enums  # noqa: F401  (the real vendored module)
            from Sol.PyBullet import BaseSingleAgentAviary as sol_bsa
        for pkg in ("gym_pybullet_drones.envs", "gym_pybullet_drones.envs.single_agent_rl"):
            if pkg not in sys.modules:
                m = types.ModuleType(pkg)
                m.__path__ = []
                sys.modules[pkg] = m
        stub = types.ModuleType("gym_pybullet_drones.envs.single_agent_rl.BaseSingleAgentAviary")
        stub.ActionType, stub.ObservationType, stub.BaseSingleAgentAviary = sol_bsa.ActionType, sol_bsa.ObservationType, sol_bsa.BaseSingleAgentAviary
        sys.modules[stub.__name__] = stub
        hover_mod = importlib.util.module_from_spec(spec)
        with contextlib.redirect_stdout(io.StringIO()):
            spec.loader.exec_module(hover_mod)
        hover_reward = hover_mod.HoverAviary._computeReward
    except Exception as ex:    # noqa: BLE001
        print("HoverAviary import failed:", repr(ex), file=sys.stderr)
        hover_reward = None

    class _Dummy(_DynEnv):
        _computeReward = dummy_env.PBDroneEnv._computeReward
        smoothness_reward = dummy_env.PBDroneEnv.smoothness_reward

    class _Thrust(_DynEnv):
        _computeReward = ThrustEnv.ThrustEnv._computeReward

    class _Her(_DynEnv):
        def _computeReward(self):
            r = HerPBDroneEnv.PBDroneEnv._computeReward(self)        # (reward, reward + bonus) tuple, or -3000 on a crash
            return r[0] if isinstance(r, tuple) else r

    class _Reaching(_DynEnv):
        _computeReward = dummy_env.PBDroneEnv.progress_reward

        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self._last_position = self._current_position             # dummy_env.py __init__

        def _update_state_post_step(self, action):                   # dummy_env.update_state_post_step keeps _last_position
            self._last_position = copy.deepcopy(self._current_position)
            super()._update_state_post_step(action)

    class _Hover(_DynEnv):
        if hover_reward is not None:
            _computeReward = hover_reward
        else:
            def _computeReward(self):                                # HoverAviary.py:65-76 verbatim semantics
                state = self._getDroneStateVector(0)
                return -1 * np.linalg.norm(np.array([0, 0, 1]) - state[0:3]) ** 2

    class _FlyThru(_DynEnv):
        _computeReward = FlyThruGateAviary._computeReward

    with contextlib.redirect_stdout(io.StringIO()):
        from Sol.Model.Environments import Rewarder

    class _Literature(_DynEnv):
        """Rewarder.py's calculator classes, called with quantities of PBDroneEnv's waypoint machine (the wiring is ours: the
        reference never calls them; it is restated in oracle/dyn_oracle.py::_reward_literature and in the kernel)."""
        calculator = None

        def step(self, action):
            self._cur_action = np.array(action)
            return super().step(action)

        def _computeReward(self):
            crashed = bool(self._computeTerminated() and not self._is_done)
            passed = False
            if not crashed and self._distance_to_target <= self._threshold:
                self._current_target_index += 1
                passed = True
                if self._current_target_index == len(self._target_points):
                    self._is_done = True
            target = self._target_points[min(self._current_target_index, len(self._target_points) - 1)]
            v = np.array(target, dtype=np.float64) - np.array(self.pos[0])
            n = np.linalg.norm(v)
            delta_cam = float(np.arccos(np.clip(np.dot(self.get_forward_vector(), v / n), -1.0, 1.0))) if n > 0 else 0.0
            a_t, a_tm1 = np.asarray(self._cur_action, np.float64), np.asarray(self._last_action, np.float64)
            if isinstance(self.calculator, Rewarder.ChampRewardCalculator):
                r = self.calculator.calculate_reward(self._prev_distance_to_target, self._distance_to_target, delta_cam, a_t, a_tm1,
                                                     self.rpy_rates[0], self.pos[0][2], crashed)
            else:
                r = self.calculator.calculate_reward(self._prev_distance_to_target, self._distance_to_target, delta_cam, a_t, a_tm1,
                                                     self.rpy_rates[0], passed, crashed)
            if not crashed:
                self._prev_distance_to_target = self._distance_to_target
            return r

    class _Bootstrapped(_Literature):
        calculator = Rewarder.BootstrappedImiVisionRewardCalculator()

    class _Champ(_Literature):
        calculator = Rewarder.ChampRewardCalculator()

    with contextlib.redirect_stdout(io.StringIO()):
        from Sol.PyBullet.BaseSingleAgentAviary import BaseSingleAgentAviary
        from Sol.PyBullet.DSLPIDControl import DSLPIDControl
        from Sol.PyBullet.enums import DroneModel

    class _BsaAct(_DynEnv):
        """PBDroneEnv with BaseSingleAgentAviary's own action pre-processing (BaseSingleAgentAviary.py:153-225)."""
        _preprocessAction = BaseSingleAgentAviary._preprocessAction

        def _saveLastAction(self, action):
            # BaseAviary.py:1013 reshapes every action to (NUM_DRONES, 4) for the GUI's benefit, which raises for the
            # 3-element PID and 1-element ONE_D_* actions (upstream sizes it by the action space); stored as given
            self.last_action = np.array(action)

    _import_reference.extras = dict(BsaAct=_BsaAct, DSLPIDControl=DSLPIDControl, DroneModel=DroneModel)
    variants = {"default": _DynEnv, "dummy": _Dummy, "thrustenv": _Thrust, "her": _Her, "reaching": _Reaching,
                "hover": _Hover, "flythrugate": _FlyThru, "bootstrapped": _Bootstrapped, "champ": _Champ}
    return variants, normalize, ActionType, Physics, Waypoints, hover_reward is not None


def _urdf_constants(path):
    """The attributes BaseAviary._parse_urdf_parameters (BaseAviary.py:1123-1163) reads, minus the pwm ones that
    cf2p.urdf / racer.urdf do not have."""
    import xml.etree.ElementTree as etxml
    t = etxml.parse(path).getroot()
    a = t[0].attrib
    return dict(M=float(t[1][0][1].attrib["value"]), L=float(a["arm"]), T2W=float(a["thrust2weight"]),
                J=np.diag([float(t[1][0][2].attrib[k]) for k in ("ixx", "iyy", "izz")]), KF=float(a["kf"]), KM=float(a["km"]),
                MAX_SPEED_KMH=float(a["max_speed_kmh"]))


def make_env(ref, track, S, max_steps, normalize_obs, reward="default", norm_rew=False, clip_rew=False,
             include_distance=True, normalize_actions=True, act="thrust", model="cf2x"):
    variants, normalize, ActionType, Physics, Waypoints, _ = ref
    DynEnv = variants[reward] if act == "thrust" else _import_reference.extras["BsaAct"]
    if track == "circle":      # simulation_controller.py / PBDroneSimulator.py:111-130
        tr = Waypoints.Track(Waypoints.circle(radius=1, num_points=6, height=1), circle=True)
    else:
        tr = Waypoints.Track(Waypoints.reaching(), circle=False)
    targets = list(tr.waypoints)               # dilate_targets(.., 0) is the identity (PBDroneSimulator.py:89-105)
    if tr.is_circle:
        targets.pop(0)                         # PBDroneSimulator.py:129-130
    env = DynEnv(target_points=targets, threshold=0.3, discount=0.999, max_steps=max_steps, act=ActionType.THRUST,
                 gui=False, initial_xyzs=tr.initial_xyzs, save_folder=None, aviary_dim=tr.aviary_dim,
                 random_spawn=False, cylinder=True, circle=tr.is_circle, include_distance=include_distance,
                 normalize_actions=normalize_actions, collect_rollouts=False, physics=Physics.DYN,
                 pyb_freq=240, ctrl_freq=240 // S)       # PBDroneSimulator.py:154-172
    if model != "cf2x":
        # The reference cannot construct the other airframes itself (BaseAviary.py:99 looks for
        # Sol/resources/safegym/<model>.urdf, and cf2p.urdf / racer.urdf lack the pwm attributes its parser reads):
        # built as CF2X, then given the constants of ITS OWN URDF for that model, derived as BaseAviary.py:163-176 does
        k = _urdf_constants(os.path.join(REF, "Sol/resources", model + ".urdf"))
        env.DRONE_MODEL = _import_reference.extras["DroneModel"](model)
        env.M, env.L, env.THRUST2WEIGHT_RATIO, env.J, env.KF, env.KM = k["M"], k["L"], k["T2W"], k["J"], k["KF"], k["KM"]
        env.J_INV = np.linalg.inv(env.J)
        env.MAX_SPEED_KMH = k["MAX_SPEED_KMH"]
        env.GRAVITY = env.G * env.M
        env.HOVER_RPM = np.sqrt(env.GRAVITY / (4 * env.KF))
        env.MAX_RPM = np.sqrt((env.THRUST2WEIGHT_RATIO * env.GRAVITY) / (4 * env.KF))
        env.MAX_THRUST = (4 * env.KF * env.MAX_RPM ** 2)
    if act != "thrust":
        # PBDroneEnv.__init__ drops the `act` keyword on its way to BaseSingleAgentAviary.__init__ (PBDroneEnv.py:98-111),
        # so what BaseSingleAgentAviary.__init__ would have done for this action type (:67-75,:90-91) is done here
        env.ACT_TYPE = ActionType(act)
        if act in ("pid", "vel", "one_d_pid"):
            with contextlib.redirect_stdout(io.StringIO()):
                env.ctrl = _import_reference.extras["DSLPIDControl"](drone_model=_import_reference.extras["DroneModel"].CF2X)
            env.SPEED_LIMIT = 0.03 * env.MAX_SPEED_KMH * (1000 / 3600)
    env.reset(seed=0)                                    # :173
    raw = env
    if normalize_obs:
        env = normalize.NormalizeObservation(env)        # :181
    if clip_rew:                                         # :191-192 gym.wrappers.TransformReward (third party): restated
        env = _ClipReward(env)
    if norm_rew:                                         # :193-194 gym.wrappers.NormalizeReward (third party); the
        env = normalize.NormalizeReward(env)             # reference's own copy of the algorithm, normalize.py:100-147
    return env, raw


class _ClipReward:
    def __init__(self, env):
        self.env = env

    def step(self, action):
        o, r, te, tr, info = self.env.step(action)
        return o, np.clip(r, -10, 10), te, tr, info

    def reset(self, **kw):
        return self.env.reset(**kw)

    def __getattr__(self, name):
        return getattr(self.env, name)


def run(ref, track, S, mode, N, T, seed, max_steps, normalize_obs, reward="default", norm_rew=False, clip_rew=False,
        include_distance=True, normalize_actions=True, act="thrust", model="cf2x"):
    with contextlib.redirect_stdout(io.StringIO()):
        envs = [make_env(ref, track, S, max_steps, normalize_obs, reward, norm_rew, clip_rew, include_distance, normalize_actions,
                         act, model) for _ in range(N)]
        a = actions(mode, T, N, seed, track)
        obs0 = np.stack([np.asarray(e.reset()[0], np.float64) for e, _ in envs])   # VecEnv.reset()
        D = obs0.shape[1]
        out = dict(actions=a, obs0=obs0, obs=np.zeros((T, N, D)), terminal_obs=np.full((T, N, D), np.nan),
                   reward=np.zeros((T, N)), done=np.zeros((T, N), np.uint8), found_targets=np.zeros((T, N), np.int32),
                   ep_return=np.full((T, N), np.nan), ep_length=np.zeros((T, N), np.int32),
                   pos=np.zeros((T, N, 3)), quat=np.zeros((T, N, 4)), vel=np.zeros((T, N, 3)),
                   rpy_rates=np.zeros((T, N, 3)), ang_v=np.zeros((T, N, 3)), dist=np.zeros((T, N)),
                   rpm=np.zeros((T, N, 4)))
        if act in ("pid", "vel", "one_d_pid"):
            out["pid"] = np.zeros((T, N, 9))     # DSLPIDControl.integral_pos_e | integral_rpy_e | last_rpy after the step
        ep_ret, ep_len = np.zeros(N), np.zeros(N, np.int64)
        for t in range(T):
            for i, (e, raw) in enumerate(envs):
                o, r, term, trunc, info = e.step(a[t, i, :{"pid": 3, "one_d_rpm": 1, "one_d_pid": 1}.get(act, 4)])
                if "pid" in out:
                    out["pid"][t, i] = np.concatenate([raw.ctrl.integral_pos_e, raw.ctrl.integral_rpy_e, raw.ctrl.last_rpy])
                ep_ret[i] += float(r)
                ep_len[i] += 1
                out["reward"][t, i] = float(r)
                out["done"][t, i] = (1 if term else 0) | (2 if trunc else 0)
                out["found_targets"][t, i] = info["found_targets"]
                # physical state right after the step (before any reset)
                out["pos"][t, i], out["quat"][t, i], out["vel"][t, i] = raw.pos[0], raw.quat[0], raw.vel[0]
                out["rpy_rates"][t, i], out["ang_v"][t, i] = raw.rpy_rates[0], raw.ang_v[0]
                out["dist"][t, i] = raw._distance_to_target
                out["rpm"][t, i] = raw.last_clipped_action[0]
                if term or trunc:
                    out["terminal_obs"][t, i] = o
                    out["ep_return"][t, i], out["ep_length"][t, i] = ep_ret[i], ep_len[i]
                    ep_ret[i], ep_len[i] = 0.0, 0
                    o, _ = e.reset()
                out["obs"][t, i] = o
    out["meta"] = np.array([track, str(S), mode, str(max_steps), "1" if normalize_obs else "0", reward,
                            "1" if norm_rew else "0", "1" if clip_rew else "0", "1" if include_distance else "0",
                            "1" if normalize_actions else "0", act, model])
    return out


def _urdf_link_offsets(path):
    """xyz of the fixed joints' child links prop0..prop3 and center_of_mass, in link-index order (cf2x.urdf)."""
    import xml.etree.ElementTree as etxml
    root = etxml.parse(path).getroot()
    links = {l.attrib["name"]: l for l in root.findall("link")}
    out = []
    for name in ("prop0_link", "prop1_link", "prop2_link", "prop3_link", "center_of_mass_link"):
        origin = links[name].find("inertial").find("origin")
        out.append(tuple(float(v) for v in origin.attrib["xyz"].split()))
    return out


def mint_forces(ref, n_rollout=40, seed=77):
    """forces_ref.npz: the reference's OWN BaseAviary._drag (BaseAviary.py:838-865) and BaseAviary._groundEffect (:798-834)
    evaluated on states of a DYN rollout plus hand-placed edge states; what is stored is the argument each of them hands
    to p.applyExternalForce (recorded by the pybullet shim), next to the state it was computed from.  These two functions
    only run under Physics.PYB_* in the reference (which needs Bullet's integrator); the oracle / the kernel apply the same
    forces inside DYN as a documented extension, and this fixture pins the FORMULAS against the reference's code.
    Restated, not reference: the propeller link heights (Bullet forward kinematics over the fixed joints of the reference's
    cf2x.urdf, ref_shims.getLinkStates)."""
    import pybullet as p                                   # the shim
    p.link_offsets = _urdf_link_offsets(os.path.join(REF, "Sol/resources/safegym/cf2x.urdf"))
    with contextlib.redirect_stdout(io.StringIO()):
        env, raw = make_env(ref, "circle", 8, 4096, False)
    rng = np.random.default_rng(seed)
    acts = (HOVER + 0.006 * rng.uniform(-1, 1, size=(n_rollout, 4))).astype(np.float32)
    recs = []

    def record(rpm_now):
        st = dict(pos=np.array(raw.pos[0]), quat=np.array(raw.quat[0]), rpy=np.array(raw.rpy[0]), vel=np.array(raw.vel[0]),
                  last_rpm=np.array(raw.last_clipped_action[0], dtype=np.float64), rpm=np.array(rpm_now, dtype=np.float64))
        p.force_log = []
        raw._drag(raw.last_clipped_action[0, :], 0)        # BaseAviary.py:431,443: the PREVIOUS step's clipped action
        raw._groundEffect(np.array(rpm_now), 0)            # BaseAviary.py:425,437: this step's clipped action
        log, p.force_log = p.force_log, None
        drag = [e for e in log if e[2] == 4]
        gnd = sorted((e for e in log if e[2] < 4), key=lambda e: e[2])
        assert len(drag) == 1 and drag[0][5] == p.LINK_FRAME and len(gnd) in (0, 4)
        st["drag_force_link"] = np.array(drag[0][3])
        st["gnd_force_z"] = np.array([e[3][2] for e in gnd]) if gnd else np.zeros(4)
        st["gnd_applied"] = np.array(1 if gnd else 0)
        recs.append(st)

    with contextlib.redirect_stdout(io.StringIO()):
        for t in range(n_rollout):
            env.step(acts[t])
            record(raw.last_clipped_action[0] * rng.uniform(0.8, 1.1, size=4))
        # edge states: near the ground (height clip GND_EFF_H_CLIP), upside down (no ground effect), fast and tilted
        for pos, rpy, vel in (((0.3, -0.2, 0.012), (0.05, -0.1, 0.4), (0.4, 0.1, -0.3)),
                              ((0.0, 0.0, 0.05), (0.6, 0.4, -2.0), (1.5, -2.0, 0.5)),
                              ((0.1, 0.1, 0.2), (2.0, 0.1, 0.3), (0.2, 0.2, 0.2)),
                              ((0.1, 0.1, 0.2), (0.1, -1.7, 0.3), (-1.0, 0.7, 0.1)),
                              ((-0.5, 0.8, 1.6), (-0.9, 1.2, 3.0), (2.5, 2.5, -1.0))):
            quat = np.array(p.getQuaternionFromEuler(rpy))
            raw.pos[0], raw.quat[0], raw.rpy[0], raw.vel[0] = np.array(pos), quat, np.array(rpy), np.array(vel)
            p.resetBasePositionAndOrientation(raw.DRONE_IDS[0], pos, quat, physicsClientId=raw.CLIENT)
            raw.last_clipped_action[0] = rng.uniform(9000, 21000, size=4)
            record(rng.uniform(9000, 21000, size=4))
    out = {k: np.stack([r[k] for r in recs]) for k in recs[0]}
    out["constants"] = np.array([raw.KF, raw.GND_EFF_COEFF, raw.PROP_RADIUS, raw.GND_EFF_H_CLIP, *np.ravel(raw.DRAG_COEFF)], dtype=np.float64)
    out["link_offsets"] = np.array(p.link_offsets)
    return out


if __name__ == "__main__":
    if not HAVE_REF:
        sys.exit("DN_REFERENCE_ROOT must name a checkout of eRGiBi/DRL-DroneNavigation")
    ref = _import_reference()
    np.savez_compressed(os.path.join(HERE, "forces_ref.npz"), **mint_forces(ref))
    print("HoverAviary imported from the reference:", ref[-1], file=sys.stderr)
    for name, cfg in CASES.items():
        out = run(ref, *cfg)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(name, "dones", int((out["done"] != 0).sum()), "truncs", int((out["done"] & 2).astype(bool).sum()),
              "max found", int(out["found_targets"].max()), file=sys.stderr)
