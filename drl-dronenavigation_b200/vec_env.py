"""SB3 ``VecEnv`` protocol over the fused CUDA step.

``GpuDroneVecEnv`` stands where the reference builds
``SubprocVecEnv([make_env(...) for i in range(num_envs)])``
(Sol/Model/PBDroneSimulator.py:653-681): same attributes (``num_envs``,
``observation_space``, ``action_space``), same numpy ``reset`` / ``step_async`` /
``step_wait`` contract with the worker's auto-reset semantics
(``terminal_observation``, ``TimeLimit.truncated``, Monitor's ``episode`` dict,
``found_targets``), but one kernel launch per vector step instead of N processes.
Host buffers are pinned.  By default (``host_path="zero_copy"``) every ``step`` is one
kernel launch that reads the actions from and writes the results to those buffers over
PCIe; ``host_path="slab"`` copies them with one H2D and one D2H DMA around the kernel, and
``host_path="server"`` keeps the kernel resident between steps.
"""
from __future__ import annotations

import pickle
import time
from typing import Any, List, Optional, Sequence

import numpy as np
import torch

from . import _lib as L
from .batched_env import BatchedDroneEnv
from .constants import CF2X
from .spaces import Box

try:  # pragma: no cover - SB3 is absent in the build image
    from stable_baselines3.common.vec_env import VecEnv as _SB3VecEnv  # type: ignore
    from stable_baselines3.common.monitor import Monitor as _SB3Monitor  # type: ignore
    _HAVE_SB3 = True
except Exception:  # noqa: BLE001
    _SB3VecEnv = object
    _SB3Monitor = None
    _HAVE_SB3 = False


def action_space(normalize_actions: bool) -> Box:
    """PBDroneEnv._actionSpace (PBDroneEnv.py:225-243)."""
    if normalize_actions:
        return Box(low=-1 * np.ones(4, dtype=np.float32), high=np.ones(4, dtype=np.float32), shape=(4,), dtype=np.float32)
    lo, hi = CF2X.physical_action_bounds()
    return Box(low=lo, high=hi, dtype=np.float32)


def observation_space(include_distance: bool) -> Box:
    """PBDroneEnv._observationSpace (PBDroneEnv.py:245-286)."""
    low = np.array([-1, -1, 0, -1, -1, -1, -1, -1, -1, -1, -1, -1], dtype=np.float32)
    high = np.ones(12, dtype=np.float32)
    if include_distance:
        low, high = np.append(low, 0).astype(np.float32), np.append(high, 1).astype(np.float32)
    return Box(low=low, high=high, dtype=np.float32)


class GpuDroneVecEnv(_SB3VecEnv):
    """Vectorised PBDroneEnv on one GPU.  Keyword arguments are PBDroneEnv's
    (PBDroneEnv.py:41-65); ``normalize_obs=True`` fuses the ``NormalizeObservation``
    wrapper that make_env always applies (PBDroneSimulator.py:181)."""

    def __init__(self, num_envs: int, target_points, threshold=0.3, discount=0.999, max_steps=4096,
                 aviary_dim=(-1, -1, 0, 1, 1, 1), include_distance=True, normalize_actions=True,
                 normalize_obs=True, device=None, collect_rollouts=False, rollout_dir="Sol/rollouts", **env_kwargs):
        # collect_rollouts (PBDroneEnv.py:152-157,811-821): every env appends "<13 obs floats>,<reward>" lines of the RAW
        # observation to its own Sol/rollouts/rollout_<n>.txt.  The raw rows are only on the host when the fused
        # NormalizeObservation is off, so in this (analysis) mode the wrapper runs on the host in numpy instead.
        self.collect_rollouts = bool(collect_rollouts)
        self._host_norm = bool(normalize_obs) and self.collect_rollouts
        self.host_path = env_kwargs.pop("host_path", "zero_copy")
        if self.host_path not in ("zero_copy", "slab", "server"):
            raise ValueError(f"host_path={self.host_path!r}")
        server_idle_us = int(env_kwargs.pop("server_idle_us", 2000))
        self.core = BatchedDroneEnv(num_envs, target_points, threshold=threshold, discount=discount,
                                    max_steps=max_steps, aviary_dim=aviary_dim,
                                    include_distance=include_distance, normalize_actions=normalize_actions,
                                    normalize_obs=bool(normalize_obs) and not self.collect_rollouts, device=device, **env_kwargs)
        obs_space, act_space = observation_space(include_distance), action_space(normalize_actions)
        if _HAVE_SB3:  # pragma: no cover
            super().__init__(num_envs, obs_space, act_space)
        else:
            self.num_envs, self.observation_space, self.action_space = num_envs, obs_space, act_space
        self.render_mode = None
        N, D = num_envs, self.core.obs_dim
        # one dn_step_host_async / dn_step_host_wait pair per vector step (include/dronenav.h).  Two forms of host buffers:
        #   "zero_copy" (default): pinned, device-mapped buffers of this object; the fused kernel reads the actions and writes the
        #                results over PCIe itself and its last CTA writes the completion word the host polls (measured faster
        #                at every batch size up to 4096 envs: 24 vs 35 us per step);
        #   "slab":      the handle's own pinned slab, one captured graph = H2D DMA, kernel, D2H DMA;
        #   "server":    the zero-copy buffers, stepped by the RESIDENT kernel (dn_host_server): no launch per step; the kernel
        #                leaves after `server_idle_us` without a step and comes back with the next one.  step_async only stores
        #                the actions; step_wait rings the doorbell and waits.
        if self.host_path == "slab":
            self._host_io, hb = self.core.host_buffers(with_episode_info=True)
        else:
            pin = lambda *shape, dtype: torch.empty(*shape, dtype=dtype).pin_memory().numpy()
            hb = {"actions": pin(N, 4, dtype=torch.float32), "obs": pin(N, D, dtype=torch.float32), "reward": pin(N, dtype=torch.float32),
                  "done": pin(N, dtype=torch.uint8), "terminal_obs": pin(N, D, dtype=torch.float32), "found_targets": pin(N, dtype=torch.int32),
                  "episode_return": pin(N, dtype=torch.float32), "episode_length": pin(N, dtype=torch.int32)}
            self._host_io = L.dn_step_io()
            for k, v in hb.items():
                setattr(self._host_io, k, v.ctypes.data)
            self._pinned = hb            # keeps the pinned storage alive (numpy views of pinned torch tensors hold their base)
        self._h_actions, self._h_obs, self._h_rew, self._h_done = hb["actions"], hb["obs"], hb["reward"], hb["done"]
        self._h_term, self._h_found, self._h_epr, self._h_epl = hb["terminal_obs"], hb["found_targets"], hb["episode_return"], hb["episode_length"]
        if self.collect_rollouts:
            import os
            os.makedirs(rollout_dir, exist_ok=True)
            base = sum(len(files) for _, _, files in os.walk(rollout_dir))          # PBDroneEnv.py:154-156
            self.rollout_paths = [os.path.join(rollout_dir, f"rollout_{base + 1 + i}.txt") for i in range(N)]
            self._rms_mean, self._rms_var = np.zeros((N, D)), np.ones((N, D))         # normalize.RunningMeanStd per env
            self._rms_count = np.full(N, 1e-4)
        if self.host_path == "server":
            self.core.host_server(server_idle_us)
        torch.cuda.synchronize(self.core.device)
        self._t_start = time.time()
        self._pending = False
        self.h2d_bytes_per_step = self._h_actions.size * 4
        self.d2h_bytes_per_step = 2 * self._h_obs.size * 4 + 4 * N * 4 + N          # obs, terminal obs, reward, found, episode r / l, done
        self._attrs = {"INIT_XYZS": self.core.INIT_XYZS, "INIT_RPYS": self.core.INIT_RPYS,
                       "CTRL_FREQ": env_kwargs.get("ctrl_freq", 240), "PYB_FREQ": env_kwargs.get("pyb_freq", 240),
                       "G": CF2X.G}

    # ------------------------------------------------------------- VecEnv API
    def _host_normalize(self, rows: np.ndarray, idx: np.ndarray) -> np.ndarray:
        """normalize.NormalizeObservation.normalize (normalize.py:94-97) for the envs `idx`: RunningMeanStd.update with
        a batch of one (:19-47), then (obs - mean) / sqrt(var + 1e-8); float64 statistics like the reference."""
        x = rows.astype(np.float64)
        mean, var, count = self._rms_mean[idx], self._rms_var[idx], self._rms_count[idx][:, None]
        delta, tot = x - mean, count + 1.0
        new_mean = mean + delta / tot
        new_var = (var * count + np.square(delta) * count / tot) / tot
        self._rms_mean[idx], self._rms_var[idx], self._rms_count[idx] = new_mean, new_var, tot[:, 0]
        return ((x - new_mean) / np.sqrt(new_var + 1e-8)).astype(np.float32)

    def _write_rollout_lines(self, raw: np.ndarray, rews: np.ndarray) -> None:
        for i, path in enumerate(self.rollout_paths):                # PBDroneEnv.collect_rollout, :811-821
            with open(path, mode="a+") as f:
                for x in raw[i].tolist():
                    f.write(str(np.format_float_positional(np.float32(x), unique=False, precision=32)) + ",")
                f.write(str(float(rews[i])))
                f.write("\n")

    def reset(self) -> np.ndarray:
        out = self.core.reset().cpu().numpy().copy()
        if self._host_norm:
            out = self._host_normalize(out, np.arange(self.num_envs))
        return out

    def step_async(self, actions: np.ndarray) -> None:
        a = np.asarray(actions, dtype=np.float32).reshape(self.num_envs, 4)
        self._h_actions[...] = a
        if self.host_path != "server":
            self.core.step_host_async(self._host_io)
        self._pending = True

    def step_wait(self):
        if not self._pending:
            raise RuntimeError("step_wait() called without step_async()")
        self._pending = False
        if self.host_path == "server":
            self.core.step_host(self._host_io)
        else:
            self.core.step_host_wait()
        obs = self._h_obs.copy()
        rews = self._h_rew.copy()
        bits = self._h_done
        dones = bits != 0
        found = self._h_found
        # one dict per env, as SB3 expects; built from Python ints (tolist) -- per-element numpy scalar conversion was
        # the most expensive line of the whole vector step at 4096 envs
        infos: List[dict] = [{"found_targets": f, "TimeLimit.truncated": False} for f in found.tolist()]
        term = self._h_term
        if self.collect_rollouts:
            raw = np.where(dones[:, None], term, obs)                # env.step's own observation (terminal one where done)
            self._write_rollout_lines(raw, rews)
            if self._host_norm:                                      # NormalizeObservation.step, then .reset where done
                all_idx = np.arange(self.num_envs)
                normed = self._host_normalize(raw, all_idx)
                d_idx = np.nonzero(dones)[0]
                if d_idx.size:
                    term = term.copy()
                    term[d_idx] = normed[d_idx]
                    normed[d_idx] = self._host_normalize(obs[d_idx], d_idx)
                obs = normed
        if dones.any():
            idx = np.nonzero(dones)[0]
            now = round(time.time() - self._t_start, 6)
            term_rows = term[idx]                                   # one gather (fancy indexing copies): rows are views of it
            trunc_only = (bits[idx] == L.DN_DONE_TRUNCATED).tolist()
            ep_r, ep_l = self._h_epr[idx].tolist(), self._h_epl[idx].tolist()
            for k, i in enumerate(idx.tolist()):
                info = infos[i]
                info["TimeLimit.truncated"] = trunc_only[k]
                info["terminal_observation"] = term_rows[k]
                info["episode"] = {"r": round(ep_r[k], 6), "l": ep_l[k], "t": now}
        return obs, rews, dones, infos

    def step(self, actions: np.ndarray):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        self.core.close()

    def seed(self, seed: Optional[int] = None) -> List[Optional[int]]:
        # the reference's env ignores seeds ("Seeding not implemented on pybullet side", PBDroneSimulator.py:690)
        return [None if seed is None else seed + i for i in range(self.num_envs)]

    def _indices(self, indices) -> Sequence[int]:
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return indices

    def get_attr(self, attr_name: str, indices=None) -> List[Any]:
        if attr_name == "render_mode":
            return [None for _ in self._indices(indices)]
        if attr_name in self._attrs:
            return [self._attrs[attr_name] for _ in self._indices(indices)]
        raise AttributeError(attr_name)

    def set_attr(self, attr_name: str, value: Any, indices=None) -> None:
        raise AttributeError(f"{attr_name}: per-env attributes of the GPU environment are read-only")

    def env_method(self, method_name: str, *args, indices=None, **kwargs) -> List[Any]:
        raise AttributeError(f"{method_name}: not available on the GPU environment")

    def env_is_wrapped(self, wrapper_class, indices=None) -> List[bool]:
        # Monitor's bookkeeping is fused into the kernel: info["episode"] is emitted on done
        is_monitor = _SB3Monitor is not None and wrapper_class is _SB3Monitor
        return [bool(is_monitor or getattr(wrapper_class, "__name__", "") == "Monitor") for _ in self._indices(indices)]

    def get_images(self):
        return [None] * self.num_envs

    def render(self, mode: Optional[str] = None):
        return None

    # the reference calls eval_env.save(path) (PBDroneSimulator.py:746): persist the running statistics of the wrappers
    def save(self, path: str) -> None:
        state = {k: v.cpu().numpy() for k, v in self.core.get_state().items()}
        with open(path, "wb") as f:
            pickle.dump({"obs_rms": state.get("obs_rms"), "rew_rms": state.get("rew_rms"), "obs_dim": self.core.obs_dim,
                         "num_envs": self.num_envs}, f)

    def load_running_stats(self, path: str) -> None:
        """Counterpart of save(): restores the per-env NormalizeObservation / NormalizeReward statistics (what
        VecNormalize.load(stats_path, env) does for the reference's evaluation runs, PBDroneSimulator.py:745-746)."""
        with open(path, "rb") as f:
            d = pickle.load(f)
        if d.get("num_envs") != self.num_envs or d.get("obs_dim") != self.core.obs_dim:
            raise ValueError("running statistics were saved for a different num_envs / observation size")
        st = {k: d[k] for k in ("obs_rms", "rew_rms") if d.get(k) is not None and self.core._optional.get(k)}
        if st:
            self.core.set_state(st)
