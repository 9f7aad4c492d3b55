"""Device-resident batched environment: the thin Python layer over the C ABI.

``BatchedDroneEnv`` owns one ``dn_env`` handle (N environments on one GPU) plus the
caller-side I/O tensors, and exposes tensor-in / tensor-out ``reset`` / ``step`` /
``step_many``.  PyTorch is used for device memory and streams only; every number is
produced by libdronenav's kernels (csrc/dronenav.cu).  Constructor keywords are the
reference's ``PBDroneEnv.__init__`` ones (Sol/Model/Environments/PBDroneEnv.py:41-65).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib as L
from .enums import ActionType, DroneModel, ObservationType, Physics

_ACT = {ActionType.THRUST: L.DN_ACT_THRUST, ActionType.RPM: L.DN_ACT_RPM, ActionType.ONE_D_RPM: L.DN_ACT_ONE_D_RPM,
        ActionType.PID: L.DN_ACT_PID, ActionType.VEL: L.DN_ACT_VEL, ActionType.ONE_D_PID: L.DN_ACT_ONE_D_PID}
_MODEL = {DroneModel.CF2X: L.DN_MODEL_CF2X, DroneModel.CF2P: L.DN_MODEL_CF2P, DroneModel.RACE: L.DN_MODEL_RACE}
_PHYS = {
    Physics.DYN: L.DN_PHYS_DYN,
    Physics.PYB: L.DN_PHYS_DYN,          # the reference's default label; the maths integrated is DYN
    Physics.PYB_DRAG: L.DN_PHYS_DRAG,
    Physics.PYB_GND: L.DN_PHYS_GROUND_EFFECT,
    Physics.PYB_GND_DRAG_DW: L.DN_PHYS_DRAG | L.DN_PHYS_GROUND_EFFECT,
}

_STATE_DTYPES = {
    "pos": (torch.float32, 3), "quat": (torch.float32, 4), "vel": (torch.float32, 3),
    "rpy_rates": (torch.float32, 3), "ang_v": (torch.float32, 3), "prev_vel": (torch.float32, 3),
    "prev_ang_v": (torch.float32, 3), "dist": (torch.float32, 0), "prev_dist": (torch.float32, 0),
    "target_idx": (torch.int32, 0), "steps": (torch.int32, 0), "just_found": (torch.uint8, 0),
    "ep_return": (torch.float32, 0), "ep_length": (torch.int32, 0), "episode_count": (torch.int32, 0),
    "last_rpm_sum": (torch.float32, 0), "obs_rms": (torch.float64, -1),
    "aux": (torch.float32, 4), "rew_rms": (torch.float32, 4), "spawn": (torch.float32, 4), "pid": (torch.float32, 9),
}


class BatchedDroneEnv:
    """N waypoint-navigation environments (CF2X by default) stepped by one fused CUDA kernel."""

    def __init__(self, num_envs: int, target_points, threshold=0.3, discount=0.999, max_steps=4096,
                 aviary_dim=(-1, -1, 0, 1, 1, 1), initial_xyzs=None, initial_rpys=None,
                 drone_model: DroneModel = DroneModel.CF2X, physics: Physics = Physics.DYN,
                 pyb_freq: int = 240, ctrl_freq: int = 240,
                 obs: ObservationType = ObservationType.KIN, act: ActionType = ActionType.THRUST,
                 cylinder=True, circle=False, include_distance=False, normalize_actions=False,
                 normalize_obs=False, reward_id: int = L.DN_REWARD_DEFAULT, ground_contact=False,
                 normalize_reward=False, clip_reward: float = 0.0, reward_gamma: float = 0.99,
                 random_spawn=False, device=None, seed: int = 0, env_id_offset: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedDroneEnv needs a CUDA device: there is no CPU fallback")
        if drone_model not in _MODEL:
            raise ValueError(f"unknown drone model {drone_model}")
        if obs != ObservationType.KIN:
            raise NotImplementedError("only ObservationType.KIN is on the CUDA path")
        if act not in _ACT:
            raise ValueError(f"unknown action type {act}")
        if physics not in _PHYS:
            raise NotImplementedError(f"{physics}: multi-drone downwash is not on the CUDA path")
        lib = L.lib()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs = int(num_envs)
        self.env_id_offset = int(env_id_offset)     # global id of env 0 of this shard (Philox subsequences: spawn, dn_ppo_act)
        targets = np.ascontiguousarray(np.array(target_points, dtype=np.float64).reshape(-1, 3))
        self.target_points = targets
        c = L.dn_config()
        c.abi_version = L.DN_ABI_VERSION
        c.num_envs = self.num_envs
        c.env_id_offset = int(env_id_offset)
        c.seed = int(seed)
        c.pyb_freq, c.ctrl_freq = int(pyb_freq), int(ctrl_freq)
        c.act_type = _ACT[act]
        c.drone_model = _MODEL[drone_model]
        c.normalize_actions = int(bool(normalize_actions))
        c.physics = _PHYS[physics] | (L.DN_PHYS_GROUND_CONTACT if ground_contact else 0)
        c.reward_id = int(reward_id)
        c.include_distance = int(bool(include_distance))
        c.cylinder, c.circle = int(bool(cylinder)), int(bool(circle))
        c.max_steps = int(max_steps)
        # random_spawn=True: the reference's (commented-out) spawn around a random target-pair line (PBDroneEnv.py:622-629)
        # "midpoint": the other commented-out variant (PBDroneEnv.py:641-648)
        c.spawn_mode = {False: L.DN_SPAWN_FIXED, True: L.DN_SPAWN_LINE, "line": L.DN_SPAWN_LINE, "midpoint": L.DN_SPAWN_MIDPOINT}[random_spawn]
        c.normalize_obs = int(bool(normalize_obs))
        c.normalize_reward = int(bool(normalize_reward))       # args.norm_rew (PBDroneSimulator.py:193-194)
        c.clip_reward = float(clip_reward)                     # args.clip_rew -> 10 (PBDroneSimulator.py:191-192)
        c.reward_gamma = float(reward_gamma)
        c.threshold, c.discount = float(threshold), float(discount)
        c.aviary_dim = (C.c_double * 6)(*[float(v) for v in aviary_dim])
        if initial_xyzs is None:   # BaseAviary.py:248-253, single drone
            from .constants import CF2X
            initial_xyzs = [0.0, 0.0, CF2X.COLLISION_H / 2 - CF2X.COLLISION_Z_OFFSET + .1]
        init = np.array(initial_xyzs, dtype=np.float64).reshape(-1)[:3]
        rpy = np.zeros(3) if initial_rpys is None else np.array(initial_rpys, dtype=np.float64).reshape(-1)[:3]
        c.init_xyz = (C.c_double * 3)(*init)
        c.init_rpy = (C.c_double * 3)(*rpy)
        c.num_targets = targets.shape[0]
        c.targets = targets.ctypes.data_as(C.POINTER(C.c_double))
        self.INIT_XYZS = init.reshape(1, 3).copy()
        self.INIT_RPYS = rpy.reshape(1, 3).copy()
        self._cfg = c
        self._handle = C.c_void_p()
        L.check(lib.dn_create(C.byref(c), self.device.index, C.byref(self._handle)), "dn_create")
        self._lib = lib
        self.obs_dim = lib.dn_obs_dim(self._handle)
        self.substeps = int(pyb_freq) // int(ctrl_freq)
        self.normalize_obs = bool(normalize_obs)
        self.uses_drag = bool(c.physics & L.DN_PHYS_DRAG)
        self.normalize_reward = bool(normalize_reward)
        self.reward_id = int(reward_id)
        self._optional = {"last_rpm_sum": self.uses_drag, "obs_rms": self.normalize_obs,
                          "aux": self.reward_id in (L.DN_REWARD_REACHING, L.DN_REWARD_BOOTSTRAPPED, L.DN_REWARD_CHAMP), "rew_rms": self.normalize_reward,
                          "spawn": bool(random_spawn), "pid": c.act_type >= L.DN_ACT_PID}
        self.drone_model, self.act_type = drone_model, act
        N, D, dev = self.num_envs, self.obs_dim, self.device
        # the persistent output lines of dn_step, carved out of ONE zero-filled allocation (one fill kernel per handle)
        up = lambda b: (b + 255) & ~255
        sizes = [("obs", N * D * 4), ("terminal_obs", N * D * 4), ("reward", N * 4), ("found_targets", N * 4),
                 ("episode_return", N * 4), ("episode_length", N * 4), ("done", N)]
        self._out_mem = torch.zeros(sum(up(b) for _, b in sizes), dtype=torch.uint8, device=dev)
        views, off = {}, 0
        for name, b in sizes:
            views[name] = self._out_mem[off:off + b]
            off += up(b)
        self.obs = views["obs"].view(torch.float32).view(N, D)
        self.terminal_obs = views["terminal_obs"].view(torch.float32).view(N, D)
        self.reward = views["reward"].view(torch.float32)
        self.found_targets = views["found_targets"].view(torch.int32)
        self.episode_return = views["episode_return"].view(torch.float32)
        self.episode_length = views["episode_length"].view(torch.int32)
        self.done = views["done"]
        self._io = self._make_io(None, self.obs, self.reward, self.done, self.terminal_obs,
                                 self.found_targets, self.episode_return, self.episode_length)

    # ------------------------------------------------------------------ utils
    @staticmethod
    def _make_io(actions, obs, reward, done, terminal_obs=None, found=None, ep_ret=None, ep_len=None):
        io = L.dn_step_io()
        p = lambda t: None if t is None else t.data_ptr()
        io.actions, io.obs, io.reward, io.done = p(actions), p(obs), p(reward), p(done)
        io.terminal_obs, io.found_targets = p(terminal_obs), p(found)
        io.episode_return, io.episode_length = p(ep_ret), p(ep_len)
        return io

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_actions(self, actions: torch.Tensor, lead=()):
        want = tuple(lead) + (self.num_envs, 4)
        if not (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.float32
                and tuple(actions.shape) == want and actions.is_contiguous()):
            raise ValueError(f"actions must be a contiguous float32 CUDA tensor of shape {want}")
        if actions.device != self.device:
            raise ValueError("actions live on another device than the environment")

    @property
    def launch_count(self) -> int:
        return int(self._lib.dn_launch_count(self._handle))

    # -------------------------------------------------------------------- API
    def reset(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """PBDroneEnv.reset for all (or the masked) envs; returns the [N, obs_dim] obs tensor."""
        mptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mptr = mask.data_ptr()
        L.check(self._lib.dn_reset(self._handle, mptr, self.obs.data_ptr(), self._stream()), "dn_reset")
        return self.obs

    def step(self, actions: torch.Tensor):
        """One control step of every env (one kernel launch).  Returns views of the persistent
        output tensors: (obs, reward, done_bits, found_targets)."""
        self._check_actions(actions)
        self._io.actions = actions.data_ptr()
        L.check(self._lib.dn_step(self._handle, C.byref(self._io), self._stream()), "dn_step")
        return self.obs, self.reward, self.done, self.found_targets

    def step_host(self, host_io) -> None:
        """dn_step_host: one control step with HOST buffers (an ``_lib.dn_step_io`` of host pointers,
        see :meth:`_make_io`); returns when the results are in the host buffers."""
        L.check(self._lib.dn_step_host(self._handle, C.byref(host_io)), "dn_step_host")

    def host_buffers(self, with_episode_info: bool = False):
        """dn_host_buffers: the handle's pinned host slab as numpy views (``actions`` to write, the rest to read) plus the
        ``dn_step_io`` of their pointers.  ``step_host(io)`` / ``step_host_async(io)`` with that io replay one captured graph
        (one H2D DMA, the fused kernel, one D2H DMA) instead of a kernel that reads and writes host memory over PCIe."""
        io = L.dn_step_io()
        L.check(self._lib.dn_host_buffers(self._handle, int(bool(with_episode_info)), C.byref(io)), "dn_host_buffers")
        N, D = self.num_envs, self.obs_dim

        def view(ptr, ctype, shape, dtype):
            if not ptr:
                return None
            n = int(np.prod(shape))
            return np.frombuffer((ctype * n).from_address(ptr), dtype=dtype).reshape(shape)
        bufs = {"actions": view(io.actions, C.c_float, (N, 4), np.float32), "obs": view(io.obs, C.c_float, (N, D), np.float32),
                "reward": view(io.reward, C.c_float, (N,), np.float32), "done": view(io.done, C.c_uint8, (N,), np.uint8),
                "found_targets": view(io.found_targets, C.c_int32, (N,), np.int32),
                "terminal_obs": view(io.terminal_obs, C.c_float, (N, D), np.float32),
                "episode_return": view(io.episode_return, C.c_float, (N,), np.float32),
                "episode_length": view(io.episode_length, C.c_int32, (N,), np.int32)}
        return io, bufs

    def step_host_async(self, host_io) -> None:
        """dn_step_host_async (buffers of :meth:`host_buffers`, or pinned, device-mapped ones): returns once the step is launched.
        Until :meth:`step_host_wait`, every other call on the handle raises."""
        L.check(self._lib.dn_step_host_async(self._handle, C.byref(host_io)), "dn_step_host_async")

    def step_host_wait(self) -> None:
        L.check(self._lib.dn_step_host_wait(self._handle), "dn_step_host_wait")

    def host_server(self, idle_us: int) -> None:
        """dn_host_server: keep the step kernel resident between :meth:`step_host` calls on pinned, device-mapped buffers
        (no launch per step); it leaves after ``idle_us`` microseconds without a step.  0 switches it off."""
        L.check(self._lib.dn_host_server(self._handle, int(idle_us)), "dn_host_server")

    def host_server_stats(self):
        r, s = C.c_int64(0), C.c_int64(0)
        L.check(self._lib.dn_host_server_stats(self._handle, C.byref(r), C.byref(s)), "dn_host_server_stats")
        return {"residencies": int(r.value), "steps": int(s.value)}

    def step_many(self, actions: torch.Tensor, per_step_outputs: bool = True, out: Optional[Dict] = None):
        """T control steps in one launch (state stays in registers); actions [T, N, 4]."""
        T = int(actions.shape[0])
        self._check_actions(actions, lead=(T,))
        N, D, dev = self.num_envs, self.obs_dim, self.device
        lead = (T,) if per_step_outputs else ()
        if out is None:
            out = dict(obs=torch.empty(*lead, N, D, dtype=torch.float32, device=dev),
                       reward=torch.empty(*lead, N, dtype=torch.float32, device=dev),
                       done=torch.empty(*lead, N, dtype=torch.uint8, device=dev),
                       found_targets=torch.empty(*lead, N, dtype=torch.int32, device=dev))
        io = self._make_io(actions, out["obs"], out["reward"], out["done"], out.get("terminal_obs"),
                           out.get("found_targets"), out.get("episode_return"), out.get("episode_length"))
        L.check(self._lib.dn_step_many(self._handle, C.byref(io), T, int(per_step_outputs), self._stream()),
                "dn_step_many")
        return out

    def action_to_rpm(self, actions: torch.Tensor) -> torch.Tensor:
        """PBDroneEnv._preprocessAction(rescale_action(a)) elementwise (any shape, float32 CUDA)."""
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        out = torch.empty_like(a)
        L.check(self._lib.dn_action_to_rpm(self._handle, a.data_ptr(), out.data_ptr(), a.numel(), self._stream()),
                "dn_action_to_rpm")
        return out

    def _state_view(self, tensors: Dict[str, torch.Tensor]):
        v = L.dn_state_view()
        for name in L.STATE_FIELDS:
            t = tensors.get(name)
            setattr(v, name, None if t is None else t.data_ptr())
        return v

    def get_state(self) -> Dict[str, torch.Tensor]:
        N, dev = self.num_envs, self.device
        ts = {}
        for name, (dt, w) in _STATE_DTYPES.items():
            if not self._optional.get(name, True):
                continue
            if name == "obs_rms":
                ts[name] = torch.empty(N, 2 * self.obs_dim + 1, dtype=dt, device=dev)
            else:
                ts[name] = torch.empty((N, w) if w else (N,), dtype=dt, device=dev)
        v = self._state_view(ts)
        L.check(self._lib.dn_get_state(self._handle, C.byref(v), self._stream()), "dn_get_state")
        return ts

    def set_state(self, state: Dict) -> None:
        """Uploads any subset of the per-env state fields (numpy or torch, row-major)."""
        N, dev = self.num_envs, self.device
        ts = {}
        for name, val in state.items():
            if name not in _STATE_DTYPES:
                raise KeyError(name)
            dt, w = _STATE_DTYPES[name]
            t = torch.as_tensor(np.asarray(val) if not isinstance(val, torch.Tensor) else val)
            t = t.to(device=dev, dtype=dt).contiguous()
            shape = (N, 2 * self.obs_dim + 1) if name == "obs_rms" else ((N, w) if w else (N,))
            if tuple(t.shape) != shape:
                raise ValueError(f"{name}: expected shape {shape}, got {tuple(t.shape)}")
            ts[name] = t
        v = self._state_view(ts)
        L.check(self._lib.dn_set_state(self._handle, C.byref(v), self._stream()), "dn_set_state")
        torch.cuda.current_stream(self.device).synchronize()   # `ts` must outlive the kernel

    def episode_stats(self, clear: bool = False) -> Dict[str, float]:
        st = L.dn_stats()
        L.check(self._lib.dn_episode_stats(self._handle, C.byref(st), int(clear), self._stream()), "dn_episode_stats")
        return {k: getattr(st, k) for k, _ in L.dn_stats._fields_}

    def close(self) -> None:
        if getattr(self, "_handle", None) is not None and self._handle:
            torch.cuda.synchronize(self.device)
            self._lib.dn_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
