"""The C-ABI library builds, loads and exports every symbol include/dronenav.h declares
(no compute calls: this file runs without a GPU)."""
import ctypes as C
import os
import re

from tests.conftest import ROOT


def _declared_functions():
    names = set()
    for header in ("dronenav.h", "dnppo.h"):
        text = open(os.path.join(ROOT, "include", header)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names |= set(re.findall(r"\b(dn_[a-z_]+)\s*\(", text))
    return sorted(names)


def test_header_declares_expected_entry_points():
    names = _declared_functions()
    for must in ("dn_create", "dn_destroy", "dn_reset", "dn_step", "dn_step_many", "dn_get_state",
                 "dn_set_state", "dn_episode_stats", "dn_last_error", "dn_abi_version"):
        assert must in names


def test_library_exports_every_declared_symbol(built_lib):
    from drl_dronenavigation_b200 import _lib
    names = _declared_functions()
    assert set(names) == set(_lib.SYMBOLS), "ctypes table and header disagree"
    for n in names:
        assert hasattr(built_lib, n), f"{n} not exported by libdronenav.so"
    assert built_lib.dn_abi_version() == _lib.DN_ABI_VERSION


def test_struct_layouts_match_header(built_lib):
    from drl_dronenavigation_b200 import _lib
    # sizes implied by include/dronenav.h on LP64
    assert C.sizeof(_lib.dn_step_io) == 8 * 8
    assert C.sizeof(_lib.dn_state_view) == 21 * 8
    assert C.sizeof(_lib.dn_stats) == 7 * 8
    assert C.sizeof(_lib.dn_config) == 4 + 4 + 8 + 8 + 12 * 4 + 2 * 8 + 12 * 8 + 4 + 4 + 2 * 8 + 8 + 4 + 4
    # include/dnppo.h
    assert C.sizeof(_lib.dn_ppo_config) == 6 * 4 + 8 * 4 + 4 * 4 + 10 * 4 + 20 * 8 + 2 * 8
    assert C.sizeof(_lib.dn_ppo_rollout) == 6 * 8
    assert C.sizeof(_lib.dn_ppo_stats) == 4 * 8 + 3 * 4 + 2 * 4 + 4      # + tail padding to 8


def test_ppo_update_rejects_bad_config_without_a_gpu(built_lib):
    from drl_dronenavigation_b200 import _lib
    h = C.c_void_p()
    cfg = _lib.dn_ppo_config()
    buf = (C.c_float * 8)()
    args = (C.byref(cfg), 0, buf, buf, buf, buf, buf, C.byref(h))
    cfg.abi_version = 999
    assert built_lib.dn_ppo_create(*args) == -1 and b"abi_version" in built_lib.dn_last_error()
    cfg.abi_version = _lib.DN_ABI_VERSION
    cfg.obs_dim, cfg.act_dim, cfg.max_rows, cfg.n_pi, cfg.n_vf = 13, 4, 100, 3, 3
    assert built_lib.dn_ppo_create(*args) == -1 and b"128" in built_lib.dn_last_error()
    cfg.max_rows = 256
    for i, w in enumerate((512, 500, 256)):
        cfg.pi_hidden[i] = cfg.vf_hidden[i] = w
    assert built_lib.dn_ppo_create(*args) == -1 and b"multiples of 128" in built_lib.dn_last_error()
    assert built_lib.dn_mlp_gemm(5, 3, 128, 64, 64, 1, buf, buf, buf, 1, None, buf, None, None) == -1


def test_comm_entry_points_reject_null_arguments_without_a_gpu(built_lib):
    """dn_ppo_comm_create / _connect / dn_ppo_allreduce check their pointers before they touch the handle or the device."""
    DN_EINVAL, DN_PPO_COMM_HANDLE_BYTES = -1, 64              # include/dronenav.h, include/dnppo.h
    buf = (C.c_ubyte * (DN_PPO_COMM_HANDLE_BYTES * 2))()
    not_null = C.cast(buf, C.c_void_p)        # stands in for a handle: a null buffer is refused before the handle is read
    for call in (lambda: built_lib.dn_ppo_comm_create(None, 0, 2, buf), lambda: built_lib.dn_ppo_comm_create(not_null, 0, 2, None),
                 lambda: built_lib.dn_ppo_comm_connect(None, buf), lambda: built_lib.dn_ppo_comm_connect(not_null, None),
                 lambda: built_lib.dn_ppo_allreduce(None, None)):
        assert call() == DN_EINVAL
        assert b"null" in built_lib.dn_last_error()


def test_fused_shape_rule_agrees_with_dn_ppo_create(built_lib):
    """FusedUpdate.shapes_ok accepts exactly the shapes dn_ppo_create validates, so PPOConfig(update_impl="auto") never picks a
    fused handle the library then refuses.  dn_ppo_create checks the whole configuration before it looks for a device: a shape it
    accepts gets DN_ECUDA without a device, and with device index -1 on a machine with one it gets "bad device index" -- either
    way it never allocates."""
    import itertools
    from drl_dronenavigation_b200 import _lib
    from drl_dronenavigation_b200.ppo import FusedUpdate
    archs = [(), (128,), (64,), (256, 128), (512, 512, 256), (512, 512, 256, 128), (128,) * 5, (1024, 512, 256), (512, 1024, 256),
             (512, 640), (640,), (384, 256), (192, 128), (500,), (0,)]
    buf = (C.c_float * 8)()
    h = C.c_void_p()
    accepted = 0
    for pi, vf, obs, act in itertools.product(archs, [(256, 128), (512, 512), (1024,), (128, 64)], (0, 1, 12, 64, 65), range(6)):
        cfg = _lib.dn_ppo_config()
        cfg.abi_version, cfg.max_rows, cfg.world_size = _lib.DN_ABI_VERSION, 256, 1
        cfg.obs_dim, cfg.act_dim, cfg.n_pi, cfg.n_vf = obs, act, len(pi), len(vf)
        for i, w in enumerate(pi[:_lib.DN_PPO_MAX_LAYERS]):
            cfg.pi_hidden[i] = w
        for i, w in enumerate(vf[:_lib.DN_PPO_MAX_LAYERS]):
            cfg.vf_hidden[i] = w
        rc = built_lib.dn_ppo_create(C.byref(cfg), -1, buf, buf, buf, buf, buf, C.byref(h))
        err = built_lib.dn_last_error()
        assert rc in (-1, -2) and not h.value, (pi, vf, obs, act, rc, err)
        lib_ok = rc == -2 or b"bad device index" in err
        assert FusedUpdate.shapes_ok(pi, vf, obs, act) == lib_ok, (pi, vf, obs, act, err)
        accepted += lib_ok
    assert accepted > 0


def test_bad_config_is_rejected_without_a_gpu(built_lib):
    from drl_dronenavigation_b200 import _lib
    h = C.c_void_p()
    cfg = _lib.dn_config()
    cfg.abi_version = 999
    assert built_lib.dn_create(C.byref(cfg), 0, C.byref(h)) == -1
    assert b"abi_version" in built_lib.dn_last_error()
    cfg.abi_version = _lib.DN_ABI_VERSION
    cfg.num_envs, cfg.pyb_freq, cfg.ctrl_freq = 4, 240, 7
    assert built_lib.dn_create(C.byref(cfg), 0, C.byref(h)) == -1
    assert b"divisible" in built_lib.dn_last_error()


def test_no_cpu_fallback_in_product_code():
    """The package never imports oracle/ (the oracle is test infrastructure only)."""
    pkg = os.path.join(ROOT, "drl-dronenavigation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_config_validation_messages(built_lib):
    """dn_create validates the whole configuration before it looks for a device, so these run without a GPU."""
    import numpy as np
    from drl_dronenavigation_b200 import _lib
    targets = np.ascontiguousarray([[0.0, 0.0, 1.0], [1.0, 0.0, 1.0]], dtype=np.float64)

    def cfg(**kw):
        c = _lib.dn_config()
        c.abi_version, c.num_envs, c.pyb_freq, c.ctrl_freq = _lib.DN_ABI_VERSION, 4, 240, 30
        c.num_targets, c.targets, c.max_steps = 2, targets.ctypes.data_as(C.POINTER(C.c_double)), 4096
        for k, v in kw.items():
            setattr(c, k, v)
        return c
    h = C.c_void_p()
    for kw, msg in ((dict(num_envs=0), b"num_envs"), (dict(num_targets=0), b"targets"), (dict(act_type=7), b"act_type"),
                    (dict(physics=64), b"physics"), (dict(spawn_mode=9), b"spawn_mode"), (dict(reward_id=99), b"reward_id"),
                    (dict(max_steps=1 << 21), b"max_steps"), (dict(spawn_mode=1, num_targets=1), b"random spawn"),
                    (dict(drone_model=3), b"drone_model"),
                    # only cf2x.urdf has the pwm attributes of the THRUST map; the reference builds a controller for CF2X / CF2P only
                    (dict(drone_model=_lib.DN_MODEL_CF2P, act_type=_lib.DN_ACT_THRUST), b"pwm2rpm"),
                    (dict(drone_model=_lib.DN_MODEL_RACE, act_type=_lib.DN_ACT_PID), b"no controller")):
        assert built_lib.dn_create(C.byref(cfg(**kw)), 0, C.byref(h)) == -1, kw
        assert msg in built_lib.dn_last_error(), (kw, built_lib.dn_last_error())
    # a valid configuration passes validation and then fails on the missing device (no CPU fallback) -- or succeeds on a GPU box
    for ok in (dict(), dict(drone_model=_lib.DN_MODEL_RACE, act_type=_lib.DN_ACT_RPM), dict(drone_model=_lib.DN_MODEL_CF2P, act_type=_lib.DN_ACT_VEL)):
        rc = built_lib.dn_create(C.byref(cfg(**ok)), 0, C.byref(h))
        assert rc in (0, -2), (ok, built_lib.dn_last_error())
        if rc == 0:
            built_lib.dn_destroy(h)
    rc = built_lib.dn_create(C.byref(cfg()), 0, C.byref(h))
    assert rc in (0, -2)
    if rc == 0:
        built_lib.dn_destroy(h)
    else:
        assert b"no CUDA device" in built_lib.dn_last_error() or b"CUDA" in built_lib.dn_last_error()
