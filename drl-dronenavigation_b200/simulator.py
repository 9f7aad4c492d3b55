"""``PBDroneSimulator``: the reference's experiment manager (Sol/Model/PBDroneSimulator.py:108-995)
with its vectorised environments resolved to the GPU environment.

Kept: constructor signature, ``make_env`` keywords, ``setup_agent`` / ``run_full_training`` /
``run_test`` / ``test_saved`` method names, the hyper-parameters of the PPO branch (:251-286), the
evaluation protocol (stochastic actions, 10 episodes, :719-729).  The learner is the torch-native PPO
of ``ppo.py`` (SB3 is not installable here; when it is, ``make_env(multi=True)`` returns a VecEnv that
SB3's own PPO accepts unchanged).  Ray / CleanRL / TF-Agents launchers, wandb and plotting are out of
scope (SURVEY.md section 2).
"""
from __future__ import annotations

import os
import time
from datetime import datetime

import numpy as np
import torch

from .batched_env import BatchedDroneEnv
from .enums import ActionType
from .checkpoint import load_sb3_zip, save_sb3_zip
from .ppo import PPOConfig, PPOTrainer
from .vec_env import GpuDroneVecEnv
from .waypoints import Track, dilate_targets
from . import waypoints as Waypoints


class PBDroneSimulator:
    """Manage training and testing in the (GPU) PBDroneEnv environment."""

    def __init__(self, args, track: Track, target_factor: int = 0, plot: bool = True, discount: float = 0.999):
        self.args, self.plot, self.discount = args, plot, discount
        self.threshold = 0.3
        self.env_steps = args.max_env_steps
        self.num_envs = args.num_envs
        self.track = track
        self.initial_xyzs = track.initial_xyzs
        self.aviary_dim = track.aviary_dim
        self.targets = dilate_targets(track.waypoints, target_factor)
        if track.is_circle:
            self.targets.pop(0)
        self.pyb_freq = getattr(args, "pyb_freq", 240)
        self.ctrl_freq = getattr(args, "ctrl_freq", 240)
        # Example agent loaded from checkpoint by --run_type cont / saved (PBDroneSimulator.py:132-134)
        self.continued_agent = getattr(args, "model_path", None) or "Sol/model_chkpts/PPO_save_05.31.2024_03.06.57/best_model.zip"
        print(track)

    # ------------------------------------------------------------------ envs
    def _env_kwargs(self, initial_xyzs, aviary_dim, include_distance, normalize_actions):
        return dict(threshold=self.threshold, discount=self.discount, max_steps=self.env_steps,
                    aviary_dim=aviary_dim, initial_xyzs=self.initial_xyzs if initial_xyzs is None else initial_xyzs,
                    act=ActionType.THRUST, cylinder=True, circle=self.track.is_circle, include_distance=include_distance,
                    normalize_actions=normalize_actions, pyb_freq=self.pyb_freq, ctrl_freq=self.ctrl_freq,
                    # the reward wrappers make_env stacks between the env and Monitor (:190-195), fused into the kernel
                    clip_reward=10.0 if getattr(self.args, "clip_rew", False) else 0.0,
                    normalize_reward=bool(getattr(self.args, "norm_rew", False)),
                    reward_id=int(getattr(self.args, "reward_id", 0)))

    def make_env(self, multi=False, gui=False, initial_xyzs=None, aviary_dim=np.array([-1, -1, 0, 1, 1, 1]), rank: int = 0,
                 save_path: str = None, include_distance: bool = True, normalize_actions: bool = True,
                 collect_rollouts: bool = False, seed: int = 0, num_envs: int = 1):
        """make_env of the reference (:136-204).  ``multi=True`` returns a thunk, like the reference's
        SubprocVecEnv factories; calling it builds a ``GpuDroneVecEnv`` with the wrapper stack fused
        (NormalizeObservation always, Monitor always)."""
        if gui:
            raise NotImplementedError("the PyBullet GUI is outside the CUDA hot path")
        kw = self._env_kwargs(initial_xyzs, aviary_dim, include_distance, normalize_actions)

        def _init():
            return GpuDroneVecEnv(num_envs, self.targets, normalize_obs=True, collect_rollouts=collect_rollouts, **kw)
        return _init if multi else _init()

    def make_device_env(self, num_envs: int, normalize_obs: bool = None, device=None, env_id_offset: int = 0):
        """The device-resident shard the torch-native learner steps (no host hop).  Like every env ``make_env`` builds
        (PBDroneSimulator.py:181) it is wrapped in NormalizeObservation -- fused into the step kernel, per-env running
        statistics -- unless ``--no_norm_obs`` asks for raw observations (a labelled deviation)."""
        if normalize_obs is None:
            normalize_obs = not bool(getattr(self.args, "no_norm_obs", False))
        kw = self._env_kwargs(None, self.aviary_dim, True, True)
        return BatchedDroneEnv(num_envs, self.targets, normalize_obs=normalize_obs, device=device,
                               env_id_offset=env_id_offset, **kw)

    # ----------------------------------------------------------------- agent
    def setup_agent(self, tensorboard_path=None, train_env=None, chkpt_path=None):
        """PPO with the reference's hyper-parameters (:251-286).  The rollout length per env is n_steps=4096
        for the reference's 12 envs; with thousands of envs it is scaled so that one rollout holds about the
        same 12 x 4096 x (a few) samples per update unless --rollout_steps says otherwise."""
        if self.args.agent == "SAC":            # :290-331
            from .sac import SACConfig, SACTrainer
            impl = getattr(self.args, "rollout_impl", "torch")
            return SACTrainer(train_env, SACConfig(rollout_impl=impl) if impl != "torch" else SACConfig())
        if self.args.agent != "PPO":
            raise NotImplementedError(f"{self.args.agent}: the PPO and SAC branches are built on the device path")
        n = train_env.num_envs
        T = getattr(self.args, "rollout_steps", None) or max(16, min(4096, (12 * 4096 * 8) // max(n, 1)))
        cfg = PPOConfig(n_steps=T, batch_size=getattr(self.args, "minibatch", None) or max(512, (T * n) // 32),
                        n_epochs=getattr(self.args, "n_epochs", 10), rollout_impl=getattr(self.args, "rollout_impl", "torch"))
        return PPOTrainer(train_env, cfg, rollout_steps=T)

    # ------------------------------------------------------------------ runs
    def evaluate(self, trainer: PPOTrainer, n_eval_episodes: int = 10, n_envs: int = 64, max_steps: int = 20000):
        """EvalCallback's protocol (:719-729): stochastic actions, mean episode reward / length, plus the
        success rate defined in BASELINE.md (episodes ending with all targets found)."""
        env = self.make_device_env(n_envs, device=trainer.dev)
        # The reference's eval_env keeps ITS NormalizeObservation statistics across the periodic evaluations of a run, so they
        # converge; this eval env lives for one call, so it starts from the pooled statistics of the training shard instead of
        # (mean 0, var 1, count 1e-4) -- otherwise the first episodes of every evaluation would see badly scaled inputs
        src = getattr(trainer, "env", None)
        if getattr(env, "normalize_obs", False) and getattr(src, "normalize_obs", False) and src.obs_dim == env.obs_dim:
            env.set_state({"obs_rms": self._pool_obs_rms(src.get_state()["obs_rms"].double().cpu(), env.obs_dim, n_envs)})
        obs = env.reset()
        gen = torch.Generator(device=trainer.dev).manual_seed(123)
        sac = not hasattr(trainer.learner, "policy")
        with torch.no_grad():
            for k in range(max_steps):
                if sac:
                    a = trainer.learner.act(obs, generator=gen)
                else:
                    a, _, _ = trainer.learner.act(obs, generator=gen)
                obs, _, _, _ = env.step(a.clamp(-1, 1).contiguous())
                # statistics are read (one host sync) every 64 steps; run at least one full time-limit horizon so that
                # long (successful / truncated) episodes are not under-represented against quick crashes
                if k % 64 == 63 and k >= min(self.env_steps, max_steps - 1) and env.episode_stats()["episodes"] >= n_eval_episodes:
                    break
        st = env.episode_stats()
        env.close()
        e = max(st["episodes"], 1)
        return {"episodes": st["episodes"], "mean_reward": st["return_sum"] / e, "mean_ep_length": st["length_sum"] / e,
                "success_rate": st["successes"] / e, "mean_found_targets": st["found_targets"] / e}

    def run_full_training(self, max_seconds: float = None, log=print):
        args = self.args
        total = int(float(args.total_timesteps))
        # under torchrun every rank owns a contiguous shard of global env ids (SURVEY 8e); --num_envs is per GPU
        rank, world = getattr(args, "rank", 0), getattr(args, "world", 1)
        train_env = self.make_device_env(self.num_envs, env_id_offset=rank * self.num_envs)
        trainer = self.setup_agent(train_env=train_env)
        if args.run_type == "cont":              # continue from an SB3-format archive (:701-712)
            if not os.path.exists(self.continued_agent):
                raise FileNotFoundError(f"--run_type cont: {self.continued_agent} not found (pass --model_path)")
            load_sb3_zip(self.continued_agent, trainer.learner, load_optimizer=True)
            if self._load_obs_rms(train_env, self.continued_agent[:-4] + "_obs_rms.pt"):
                log("restored the NormalizeObservation statistics saved next to the archive")
            if args.agent == "SAC":              # model.load_replay_buffer(load_most_recent_replay_buffer(chkpt_path)), :357
                rb = load_most_recent_replay_buffer(os.path.dirname(self.continued_agent))
                if rb:
                    log(f"replay buffer {rb}: {trainer.buffer.load(rb)} transitions")
        chk = None
        if args.savemodel and rank == 0:           # one writer per job
            chk = os.path.join("Sol", "model_chkpts", f"{args.agent}_save_{datetime.now().strftime('%m.%d.%Y_%H.%M.%S')}")
            os.makedirs(chk, exist_ok=True)
        t0, it, best = time.time(), 0, -np.inf
        rb_saves = 0                               # SaveReplayBufferCallback(save_freq=100_000 env.step calls), :706-710
        max_seconds = max_seconds if max_seconds is not None else getattr(args, "max_seconds", None)
        # TensorBoard scalars under SB3's tag names (what Sol/Utilities/TensorboardManager.py reads back), SURVEY f.4
        tb = None
        if getattr(args, "tensorboard", None):
            from torch.utils.tensorboard import SummaryWriter
            tb = SummaryWriter(args.tensorboard)
        def keep_going():
            go = trainer.total_steps < total and (max_seconds is None or time.time() - t0 < max_seconds)
            if world > 1:                          # ranks must leave the loop together (the update all-reduces)
                import torch.distributed as dist
                flag = torch.tensor([1.0 if go else 0.0], device=trainer.dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                go = bool(flag.item() > 0)
            return go
        while keep_going():
            out = trainer.train_iteration()
            it += 1
            if it % 5 == 0 or trainer.total_steps >= total:
                st = train_env.episode_stats(clear=True)
                e = max(st["episodes"], 1)
                if tb is not None:
                    step = trainer.total_steps
                    tb.add_scalar("rollout/ep_rew_mean", st["return_sum"] / e, step)
                    tb.add_scalar("rollout/ep_len_mean", st["length_sum"] / e, step)
                    tb.add_scalar("rollout/success_rate", st["successes"] / e, step)
                    tb.add_scalar("time/fps", out.get("sps", 0.0), step)
                    for k_src, k_dst in (("approx_kl", "train/approx_kl"), ("clip_fraction", "train/clip_fraction"),
                                         ("entropy_loss", "train/entropy_loss"), ("policy_gradient_loss", "train/policy_gradient_loss"),
                                         ("value_loss", "train/value_loss"), ("std", "train/std")):
                        if k_src in out:
                            tb.add_scalar(k_dst, out[k_src], step)
                    for k_src, k_dst in (("critic_loss", "train/critic_loss"), ("actor_loss", "train/actor_loss"),
                                         ("ent_coef", "train/ent_coef"), ("ent_coef_loss", "train/ent_coef_loss")):      # SB3 SAC.train's tags
                        if k_src in out:
                            tb.add_scalar(k_dst, out[k_src], step)
                tail = (f"kl {out['approx_kl']:.4f}  std {out['std']:.3f}" if "approx_kl" in out else
                        f"critic_loss {out.get('critic_loss', float('nan')):.4g}  ent_coef {out.get('ent_coef', float('nan')):.4g}")
                log(f"[{time.time() - t0:7.1f}s] steps {trainer.total_steps:>12d}  sps {out['sps']:.3g}  ep_rew {st['return_sum'] / e:8.3f}  "
                    f"ep_len {st['length_sum'] / e:7.1f}  found {st['found_targets'] / e:5.2f}  success {st['successes'] / e:5.3f}  {tail}")
                # EvalCallback(best_model_save_path), :719-729.  The criterion here is the mean return of the training episodes that
                # finished since the last check (the reference runs a separate 10-episode evaluation); an interval without a single
                # finished episode says nothing and must not count as a return of 0
                if chk and st["episodes"] > 0 and st["return_sum"] / e > best:
                    best = st["return_sum"] / e
                    save_sb3_zip(os.path.join(chk, "best_model.zip"), trainer.learner)
                    self._save_obs_rms(train_env, os.path.join(chk, "best_model_obs_rms.pt"))
            if chk and args.agent == "SAC" and (trainer.total_steps // max(self.num_envs * world, 1)) // 100_000 > rb_saves:
                rb_saves = (trainer.total_steps // max(self.num_envs * world, 1)) // 100_000
                trainer.buffer.save(os.path.join(chk, "replay_buffer.pkl"))
        if chk:
            save_sb3_zip(os.path.join(chk, "success_model.zip"), trainer.learner)          # model.save(...), :741-746
            self._save_obs_rms(train_env, os.path.join(chk, "success_model_obs_rms.pt"))   # eval_env.save(...), :746
            if args.agent == "SAC":
                trainer.buffer.save(os.path.join(chk, "replay_buffer.pkl"))
        if tb is not None:
            tb.close()
        ev = self.evaluate(trainer, n_eval_episodes=1000, n_envs=256)
        log(f"final evaluation: {ev}")
        train_env.close()
        return trainer, ev

    @staticmethod
    def _save_obs_rms(env, path: str) -> None:
        """The running observation statistics belong to a policy trained on normalised observations (what ``VecNormalize.save``
        keeps in the reference, :746): per-env FP64 mean | var | count rows of the training shard."""
        if getattr(env, "normalize_obs", False):
            torch.save({"obs_rms": env.get_state()["obs_rms"].cpu(), "obs_dim": env.obs_dim}, path)

    @staticmethod
    def _load_obs_rms(env, path: str) -> bool:
        """Restores statistics saved by :meth:`_save_obs_rms` into an env of the same size (or broadcasts their mean over the
        envs otherwise: count-weighted pooled mean / variance of the saved rows)."""
        if not (getattr(env, "normalize_obs", False) and os.path.exists(path)):
            return False
        d = torch.load(path, map_location="cpu")
        rms = d["obs_rms"].double()
        if int(d.get("obs_dim", env.obs_dim)) != env.obs_dim:
            return False
        if rms.shape[0] != env.num_envs:
            rms = PBDroneSimulator._pool_obs_rms(rms, env.obs_dim, env.num_envs)
        env.set_state({"obs_rms": rms})
        return True

    @staticmethod
    def _pool_obs_rms(rms: torch.Tensor, D: int, n: int) -> torch.Tensor:
        """Count-weighted pooled mean / variance of per-env rows [*, 2 D + 1], replicated for `n` envs (count = the mean count)."""
        cnt = rms[:, 2 * D:]
        tot = cnt.sum()
        mean = (rms[:, :D] * cnt).sum(0) / tot
        var = ((rms[:, D:2 * D] + (rms[:, :D] - mean) ** 2) * cnt).sum(0) / tot
        return torch.cat([mean, var, (tot / rms.shape[0]).reshape(1)]).repeat(n, 1)

    def run_test(self, max_steps: int = 2000, log=print):
        """--run_type test (:390-436): constant action 0.1 on every motor on the `up` track until termination."""
        from .env import PBDroneEnv
        self.targets = Waypoints.up()[0]
        env = PBDroneEnv(target_points=self.targets, threshold=self.threshold, discount=self.discount, max_steps=self.env_steps,
                         aviary_dim=np.array([-2, -2, 0, 2, 2, 2]), initial_xyzs=np.array([[0, 0, 0.1]]), act=ActionType.THRUST,
                         cylinder=True, circle=self.track.is_circle, include_distance=True, normalize_actions=True,
                         pyb_freq=self.pyb_freq, ctrl_freq=self.ctrl_freq)
        log(env.G); log(env.INIT_XYZS)
        log(env.reset())
        action = np.array([0.1, 0.1, 0.1, 0.1], dtype=np.float32)
        rewards = []
        for i in range(1, max_steps + 1):
            ts = env.step(action)
            rewards.append(ts[1])
            log(f"step: {i} ------------------\n{ts}")
            if ts[2]:
                break
        env.close()
        return rewards

    def test_learning(self, total_timesteps: int = 500, log=print):
        """--run_type learning (:574-612): a 500-timestep PPO smoke run on ONE environment with the wider/deeper policy
        of that method (net_arch=[512, 512, dict(vf=[256, 128], pi=[256, 128])]; the shared trunk of old SB3 versions
        is unrolled into the two separate networks newer SB3 builds), n_steps = max_env_steps, batch_size = --batch_size."""
        env = self.make_device_env(1)
        T = min(int(self.args.max_env_steps), total_timesteps)
        cfg = PPOConfig(n_steps=T, batch_size=min(int(self.args.batch_size), T), pi_arch=(512, 512, 256, 128), vf_arch=(512, 512, 256, 128))
        trainer = PPOTrainer(env, cfg, rollout_steps=T)
        log(trainer.learner.policy)
        out = None
        while trainer.total_steps < total_timesteps:
            out = trainer.train_iteration()
        env.close()
        return trainer, out

    def test_saved(self, path: str = None, episodes: int = 50):
        """--run_type saved (:438-572): roll a saved policy and report episode statistics."""
        path = path or self.continued_agent
        env = self.make_device_env(64)
        trainer = self.setup_agent(train_env=env)
        if path.endswith(".zip"):            # an SB3 archive: the reference's best_model.zip / success_model.zip or one of ours
            load_sb3_zip(path, trainer.learner)
        else:
            trainer.learner.policy.load_state_dict(torch.load(path, map_location=trainer.dev))
        out = self.evaluate(trainer, n_eval_episodes=episodes)
        env.close()
        return out


def load_most_recent_replay_buffer(directory: str):
    """PBDroneSimulator.load_most_recent_replay_buffer (PBDroneSimulator.py:998-1017): the ``replay_buffer_<n>.pkl`` with the
    largest n in `directory`; the reference's own callback writes ``replay_buffer.pkl`` (Callbacks.py:30), which its loader's
    pattern does not match -- accepted here as the fallback.  Returns None when there is none."""
    import re
    if not directory or not os.path.isdir(directory):
        return None
    best, best_n = None, -1
    for f in os.listdir(directory):
        m = re.match(r"replay_buffer_(\d+)\.pkl$", f)
        if m and int(m.group(1)) > best_n:
            best, best_n = f, int(m.group(1))
    if best is None and os.path.exists(os.path.join(directory, "replay_buffer.pkl")):
        best = "replay_buffer.pkl"
    return os.path.join(directory, best) if best else None
