"""Torch-native SAC on the device-resident environment (SURVEY.md section 8 a20 / f.1; BASELINE config 4).

Hyper-parameters are the SAC branch of ``PBDroneSimulator.setup_agent`` (Sol/Model/PBDroneSimulator.py:290-331:
qf [256, 256, 128], pi [256, 256], ReLU, batch 1024, buffer 1 048 576, learning_starts 8192, train_freq 3,
gradient_steps 5, tau 0.005, lr 2.5e-4, gamma 0.99, ent_coef "auto", target_entropy "auto"); the update is the
maths of SB3's ``SAC.train`` that the reference relies on (squashed diagonal Gaussian actor with log-std clamped to
[-20, 2], twin critics, entropy-coefficient auto-tuning towards -|A|, Polyak targets every gradient step, time-limit
truncations not treated as terminal, next observation of a finished episode = its terminal observation).
What changes is where the data lives: the replay buffer is a set of device tensors filled straight from the fused
step kernel's outputs (no numpy hop, no per-env Python), and under ``torchrun`` every gradient step all-reduces two
flat buckets (critics + log-alpha, actor) over NCCL -- the environment shards need no collective.
With ``rollout_impl="fused"`` the collection phase samples the actor with the library's kernels (``dn_sac_act``,
include/dnsac.h: Philox noise keyed by the global env id) and is replayed from one CUDA graph per phase; the gradient
step is the same torch code either way.
"""
from __future__ import annotations

import ctypes as C
import math
import time
from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.distributed as dist
from torch import nn

from ._fused import Handle, PhaseGraph, capture_graphs, flat_views, offsets, sm100, widths_ok
from ._fused import world as _world

LOG_STD_MIN, LOG_STD_MAX = -20.0, 2.0      # SB3 sac/policies.py


@dataclass
class SACConfig:
    """Defaults = PBDroneSimulator.setup_agent's SAC branch (PBDroneSimulator.py:304-327)."""
    learning_starts: int = 8192
    train_freq: int = 3            # env.step calls (x num_envs transitions) between update phases
    gradient_steps: int = 5
    batch_size: int = 1024
    tau: float = 0.005
    target_update_interval: int = 1
    buffer_size: int = 1_048_576   # transitions in total (SB3 divides by n_envs)
    learning_rate: float = 2.5e-4
    gamma: float = 0.99
    pi_arch: tuple = (256, 256)
    qf_arch: tuple = (256, 256, 128)
    n_critics: int = 2
    ent_coef_init: float = 1.0     # ent_coef="auto" -> log_ent_coef = log(1.0)
    target_entropy: Optional[float] = None   # "auto" -> -|A|
    seed: int = 42
    matmul_precision: str = "tf32"
    cuda_graph: bool = True        # replay each gradient step from three captured CUDA graphs (CUDA devices only)
    rollout_impl: str = "torch"    # "torch": torch.Generator noise, one launch at a time; "fused": dn_sac_act (Philox noise keyed
                                   # by the global env id), every collection phase after learning_starts replayed from a CUDA graph

    def __post_init__(self):
        if self.rollout_impl not in ("torch", "fused"):
            raise ValueError(f"rollout_impl={self.rollout_impl!r}: 'torch' or 'fused'")


def _relu_mlp(sizes, out_dim=None):
    layers = []
    for a, b in zip(sizes[:-1], sizes[1:]):
        layers += [nn.Linear(a, b), nn.ReLU()]
    if out_dim is not None:
        layers.append(nn.Linear(sizes[-1], out_dim))
    return nn.Sequential(*layers)


class Actor(nn.Module):
    """SB3 sac.policies.Actor: latent MLP -> (mu, log_std) heads, tanh-squashed Gaussian."""

    def __init__(self, obs_dim, act_dim, arch):
        super().__init__()
        self.latent = _relu_mlp((obs_dim,) + tuple(arch))
        self.mu = nn.Linear(arch[-1], act_dim)
        self.log_std = nn.Linear(arch[-1], act_dim)

    def forward(self, obs, generator=None, deterministic=False, eps=None):
        h = self.latent(obs)
        mu, log_std = self.mu(h), self.log_std(h).clamp(LOG_STD_MIN, LOG_STD_MAX)
        if deterministic:
            return torch.tanh(mu), None
        std = log_std.exp()
        if eps is None:            # (the graph-replayed update passes pre-drawn noise: no RNG inside a captured graph)
            eps = torch.randn(mu.shape, device=mu.device, dtype=mu.dtype, generator=generator)
        g = mu + std * eps
        a = torch.tanh(g)
        # Normal(mu, std).log_prob(g).sum - sum log(1 - tanh(g)^2 + eps)   (SquashedDiagGaussianDistribution, epsilon 1e-6)
        logp = (-0.5 * eps.pow(2) - log_std - 0.5 * math.log(2 * math.pi)).sum(-1) - torch.log(1 - a.pow(2) + 1e-6).sum(-1)
        return a, logp


class Critics(nn.Module):
    """n_critics independent Q(s, a) MLPs (SB3 ContinuousCritic, share_features_extractor=False)."""

    def __init__(self, obs_dim, act_dim, arch, n):
        super().__init__()
        self.qs = nn.ModuleList([_relu_mlp((obs_dim + act_dim,) + tuple(arch), 1) for _ in range(n)])

    def forward(self, obs, act):
        x = torch.cat([obs, act], dim=-1)
        return [q(x).squeeze(-1) for q in self.qs]


class _FlatGrads:
    """All gradients of a parameter list as views into ONE tensor (one all-reduce per optimiser step)."""

    def __init__(self, params, device):
        self.params = list(params)
        self.flat = torch.zeros(sum(p.numel() for p in self.params), device=device)
        for p, g in zip(self.params, flat_views(self.flat, self.params)):
            p.grad = g
        self.calls = 0

    def zero(self):
        self.flat.zero_()

    def allreduce(self):
        w = _world()
        if w > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.flat.div_(w)
            self.calls += 1


class ReplayBuffer:
    """Device-resident circular buffer, [capacity_steps, N, ...] (SB3 ReplayBuffer with n_envs = N,
    handle_timeout_termination=True, optimize_memory_usage=False)."""

    def __init__(self, capacity_transitions: int, num_envs: int, obs_dim: int, act_dim: int, device):
        self.cap = max(capacity_transitions // num_envs, 1)
        self.N, self.pos, self.full = num_envs, 0, False
        f = dict(dtype=torch.float32, device=device)
        self.obs = torch.empty(self.cap, num_envs, obs_dim, **f)
        self.next_obs = torch.empty(self.cap, num_envs, obs_dim, **f)
        self.act = torch.empty(self.cap, num_envs, act_dim, **f)
        self.rew = torch.empty(self.cap, num_envs, **f)
        self.done = torch.empty(self.cap, num_envs, **f)        # 1 only for true terminations (timeouts excluded)

    def add(self, obs, next_obs, act, rew, done_bits, terminal_obs):
        self.write(self.pos, obs, next_obs, act, rew, done_bits, terminal_obs)
        self.pos = (self.pos + 1) % self.cap
        self.full = self.full or self.pos == 0

    def write(self, row, obs, next_obs, act, rew, done_bits, terminal_obs):
        """One step of transitions into `row`: a host integer, or a one-element int64 device tensor (a CUDA graph can replay
        the write at a slot that moves).  Leaves ``pos`` / ``full`` alone."""
        def put(t, v):
            # index_copy_, not t[row] = v: the advanced-index assignment made fused collection phases 3-5 % longer (B200, 1000 W)
            if torch.is_tensor(row):
                t.index_copy_(0, row, v.unsqueeze(0))
            else:
                t[row].copy_(v)
        put(self.obs, obs)
        # the VecEnv returns the RESET observation on done; the transition's successor is the terminal observation
        put(self.next_obs, torch.where((done_bits != 0).unsqueeze(-1), terminal_obs, next_obs))
        put(self.act, act)
        put(self.rew, rew)
        put(self.done, ((done_bits & 1) != 0).to(torch.float32))          # DN_DONE_TERMINATED; truncated-only -> bootstrap

    def __len__(self):
        return (self.cap if self.full else self.pos) * self.N

    # ---- SaveReplayBufferCallback / load_replay_buffer (Sol/Utilities/Callbacks.py:13-39; PBDroneSimulator.py:357,998-1017) ----
    def save(self, path: str) -> str:
        """``model.save_replay_buffer(path)``: SB3 pickles its ReplayBuffer object; here a dict with that object's attribute
        names and array layouts ([buffer_size, n_envs, ...]) is pickled, which :meth:`load` -- and anything that reads the
        attributes of an SB3 buffer -- understands."""
        import pickle
        n = self.cap if self.full else self.pos
        arr = lambda t: t[:n].detach().cpu().numpy() if not self.full else t.detach().cpu().numpy()
        with open(path, "wb") as f:
            pickle.dump({"observations": arr(self.obs), "next_observations": arr(self.next_obs), "actions": arr(self.act),
                         "rewards": arr(self.rew), "dones": arr(self.done), "pos": self.pos, "full": self.full,
                         "buffer_size": self.cap, "n_envs": self.N, "written_by": "drl_dronenavigation_b200"}, f, protocol=4)
        return path

    def load(self, path: str) -> int:
        """``model.load_replay_buffer(path)``: accepts the dict written by :meth:`save` or a pickled SB3 ``ReplayBuffer`` (when
        SB3 is importable); returns the number of transitions restored.  n_envs must match; a larger saved buffer is truncated
        to the most recent ``capacity`` steps."""
        import pickle
        with open(path, "rb") as f:
            obj = pickle.load(f)
        get = (lambda k: obj[k]) if isinstance(obj, dict) else (lambda k: getattr(obj, k))
        n_envs, pos, full = int(get("n_envs")), int(get("pos")), bool(get("full"))
        if n_envs != self.N:
            raise ValueError(f"replay buffer was saved with n_envs={n_envs}, this trainer has {self.N}")
        def ordered(a):                      # oldest -> newest
            a = torch.as_tensor(a, dtype=torch.float32)
            if full and a.shape[0] > pos:
                a = torch.cat([a[pos:], a[:pos]])
            elif not full:
                a = a[:pos]
            return a[-self.cap:]
        fields = {"obs": "observations", "next_obs": "next_observations", "act": "actions", "rew": "rewards", "done": "dones"}
        # SB3 samples dones * (1 - timeouts) (ReplayBuffer._get_samples with handle_timeout_termination): a time-limit truncation is
        # not a terminal state and must keep its bootstrap.  This buffer stores terminated-only flags in `done`, so an SB3 object
        # that carries `timeouts` is converted on the way in.
        timeouts = None
        try:
            timeouts = get("timeouts")
        except (KeyError, AttributeError):
            pass
        n = 0
        for ours, theirs in fields.items():
            a = ordered(get(theirs))
            if ours == "done" and timeouts is not None:
                a = a * (1.0 - ordered(timeouts).reshape(a.shape))
            dst = getattr(self, ours)
            a = a.reshape((a.shape[0],) + tuple(dst.shape[1:]))
            n = a.shape[0]
            dst[:n].copy_(a.to(dst.device))
        self.full = n == self.cap
        self.pos = 0 if self.full else n
        return n * self.N

    def sample(self, batch_size: int, generator=None):
        n = len(self)
        idx = torch.randint(0, n, (batch_size,), device=self.obs.device, generator=generator)
        flat = lambda t: t.reshape(self.cap * self.N, *t.shape[2:])
        return flat(self.obs)[idx], flat(self.act)[idx], flat(self.rew)[idx], flat(self.next_obs)[idx], flat(self.done)[idx]


class FusedSACActor(Handle):
    """ctypes face of the dn_sac_actor handle (include/dnsac.h): SB3's Actor.forward with sampling as sm_100a kernels (the
    latent ReLU layers on the tcgen05 contraction, heads and sampler in one CUDA-core kernel) on ONE flat FP32 parameter
    vector.  The actor's ``Parameter`` s are views into that vector (:meth:`flatten`, before the optimisers are built), so
    the torch gradient step, state dicts and checkpoints all see the memory the kernels read."""

    ABI = "dn_sac_actor"

    @staticmethod
    def shapes_ok(arch, obs_dim: int, act_dim: int) -> bool:
        """The shapes dn_sac_actor_create accepts: 1..4 hidden layers, every width a multiple of 128 between 128 and 512,
        1 <= obs_dim <= 64, 1 <= act_dim <= 4."""
        return widths_ok(arch, obs_dim) and 1 <= act_dim <= 4

    @staticmethod
    def check_supported(arch, obs_dim: int, act_dim: int, device) -> None:
        if not sm100(device):
            raise RuntimeError(f"rollout_impl='fused' runs the SAC actor on sm_100a kernels: needs a compute-capability-10 CUDA device, "
                               f"got {torch.device(device)}")
        if not FusedSACActor.shapes_ok(arch, obs_dim, act_dim):
            raise RuntimeError(f"rollout_impl='fused': pi_arch={tuple(arch)}, obs_dim={obs_dim}, act_dim={act_dim} is not a shape "
                               "dn_sac_actor_create accepts (1..4 hidden layers, widths multiples of 128 between 128 and 512, "
                               "1 <= obs_dim <= 64, 1 <= act_dim <= 4)")

    @staticmethod
    def flatten(actor: "Actor") -> torch.Tensor:
        """Re-seats the actor's parameters (latent layers, mu, log_std, SB3's order) as views of one new flat vector, values unchanged."""
        ps = list(actor.parameters())
        flat = torch.cat([p.detach().reshape(-1) for p in ps])
        for p, v in zip(ps, flat_views(flat, ps)):
            p.data = v
        return flat

    def __init__(self, actor: "Actor", flat: torch.Tensor, max_rows: int):
        super().__init__(flat.device)
        L, self.flat = self.L, flat
        self.max_rows = int(-(-max_rows // 128) * 128)
        offs = offsets(actor.named_parameters())
        for name, p in actor.named_parameters():
            if p.data_ptr() != flat.data_ptr() + 4 * offs[name]:
                raise RuntimeError(f"FusedSACActor: {name} is not a view of the flat parameter vector (FusedSACActor.flatten first)")
        arch = [m.out_features for m in actor.latent if isinstance(m, nn.Linear)]
        c = L.dn_sac_actor_config()
        c.abi_version = L.DN_ABI_VERSION
        c.obs_dim, c.act_dim, c.max_rows = actor.latent[0].in_features, actor.mu.out_features, self.max_rows
        c.n_hidden = len(arch)
        for l, w in enumerate(arch):            # nn.Sequential indices: Linear at 0, 2, 4, ... (ReLU in between)
            c.hidden[l] = w
            c.w_off[l], c.b_off[l] = offs[f"latent.{2 * l}.weight"], offs[f"latent.{2 * l}.bias"]
        c.precision = L.DN_MLP_BF16X3
        c.mu_w_off, c.mu_b_off = offs["mu.weight"], offs["mu.bias"]
        c.log_std_w_off, c.log_std_b_off = offs["log_std.weight"], offs["log_std.bias"]
        c.n_params = flat.numel()
        self._create(c, flat.data_ptr())

    def act(self, obs: torch.Tensor, sample, action: torch.Tensor = None, log_prob: torch.Tensor = None):
        """dn_sac_act on `obs` [n, obs_dim]: action [n, act_dim] (and log_prob [n] when given).  `sample` is an
        ``_lib.dn_sac_sample`` (seed, global id of row 0, device int64 draw counter, mode).  The BF16 planes are NOT refreshed
        here: call :meth:`sync_weights` after the parameters change."""
        n, A = obs.shape[0], self.cfg_c.act_dim
        action = torch.empty(n, A, dtype=torch.float32, device=self.device) if action is None else action
        for t, shape in ((obs, (n, self.cfg_c.obs_dim)), (action, (n, A))) + (((log_prob, (n,)),) if log_prob is not None else ()):
            if t.dtype != torch.float32 or t.device != self.device or not t.is_contiguous() or tuple(t.shape) != shape:
                raise ValueError(f"dn_sac_act: expected a contiguous float32 tensor of shape {shape} on {self.device}")
        self.call("dn_sac_act", obs.data_ptr(), n, C.byref(sample), action.data_ptr(), None if log_prob is None else log_prob.data_ptr())
        return action

    def buffer(self, name: str, rows: int) -> torch.Tensor:
        """Test hook: the first `rows` rows of an internal buffer in FP32: "h1".."h4" (hi + lo of the BF16 planes of that
        hidden layer), "mu", "log_std" (as the last non-uniform dn_sac_act left them)."""
        planes = name not in ("mu", "log_std")
        raw = self._raw_buffer(name, "<i2" if planes else "<f4")
        if not planes:
            return raw.view(self.max_rows, -1)[:rows].clone()
        p = raw.view(torch.bfloat16).view(2, self.max_rows, -1)[:, :rows]
        return p[0].float() + p[1].float()


class SACLearner:
    """Actor, twin critics + targets, log-alpha and the SAC update; independent of the environment."""

    def __init__(self, obs_dim: int, act_dim: int, cfg: SACConfig = SACConfig(), device="cpu"):
        self.cfg, self.device = cfg, torch.device(device)
        torch.manual_seed(cfg.seed)                         # same seed on every rank -> identical initial parameters
        self.actor = Actor(obs_dim, act_dim, cfg.pi_arch).to(self.device)
        self.actor_flat, self.fused_actor = None, None
        if cfg.rollout_impl == "fused":                     # before the optimisers: they hold the re-seated Parameters
            FusedSACActor.check_supported(cfg.pi_arch, obs_dim, act_dim, self.device)
            self.actor_flat = FusedSACActor.flatten(self.actor)
        self.critic = Critics(obs_dim, act_dim, cfg.qf_arch, cfg.n_critics).to(self.device)
        self.critic_target = Critics(obs_dim, act_dim, cfg.qf_arch, cfg.n_critics).to(self.device)
        self.critic_target.load_state_dict(self.critic.state_dict())
        for p in self.critic_target.parameters():
            p.requires_grad_(False)
        self.log_ent_coef = torch.log(torch.ones(1, device=self.device) * cfg.ent_coef_init).requires_grad_(True)
        self.target_entropy = float(-act_dim) if cfg.target_entropy is None else float(cfg.target_entropy)
        lr = cfg.learning_rate
        # (the Polyak decision is baked into the captured graph, so replay is only used with target_update_interval == 1)
        self.use_graph = bool(cfg.cuda_graph) and self.device.type == "cuda" and cfg.target_update_interval == 1
        self._graphs = None                                 # (key, graphs, static tensors, stage outputs); built lazily
        self.actor_opt = torch.optim.Adam(self.actor.parameters(), lr=lr, capturable=self.use_graph)
        self.critic_opt = torch.optim.Adam(self.critic.parameters(), lr=lr, capturable=self.use_graph)
        self.ent_opt = torch.optim.Adam([self.log_ent_coef], lr=lr, capturable=self.use_graph)
        # bucket 1: critics + log-alpha (their losses do not depend on each other's step); bucket 2: actor
        self.g_critic = _FlatGrads(list(self.critic.parameters()) + [self.log_ent_coef], self.device)
        self.g_actor = _FlatGrads(self.actor.parameters(), self.device)
        self.n_updates = 0
        if self.device.type == "cuda":
            torch.backends.cuda.matmul.allow_tf32 = (cfg.matmul_precision == "tf32")

    @torch.no_grad()
    def act(self, obs, generator=None, deterministic=False):
        return self.actor(obs, generator=generator, deterministic=deterministic)[0]

    def ensure_fused_actor(self, max_rows: int) -> FusedSACActor:
        """The dn_sac_actor handle on this learner's actor (rollout_impl="fused"), created for at least `max_rows` rows."""
        if self.actor_flat is None:
            raise RuntimeError("ensure_fused_actor needs SACConfig(rollout_impl='fused')")
        if self.fused_actor is None or self.fused_actor.max_rows < max_rows:
            if self.fused_actor is not None:
                self.fused_actor.close()
            self.fused_actor = FusedSACActor(self.actor, self.actor_flat, max_rows)
        return self.fused_actor

    def drop_graphs(self) -> None:
        """Forgets the captured gradient-step graphs (the next update captures again).  Called by everything that replaces a
        tensor the graphs point to."""
        self._graphs = None

    def load_optimizer_state(self, state: Dict[str, dict]) -> None:
        """Adam states by optimiser: "actor", "critic" and "ent_coef" map to torch optimiser state dicts such as SB3's
        ``actor.optimizer.pth``, ``critic.optimizer.pth`` and ``ent_coef_optimizer.pth``.  An optimiser that is not named keeps
        its own state, and so does one whose given state covers some but not all of its parameters."""
        for name, opt in (("actor", self.actor_opt), ("critic", self.critic_opt), ("ent_coef", self.ent_opt)):
            if name in state:
                own, st = opt.state_dict(), state[name].get("state", {})
                if len(st) in (0, len(own["param_groups"][0]["params"])):
                    own["state"] = st
                    opt.load_state_dict(own)
        self.drop_graphs()      # load_state_dict re-creates the state tensors

    # ---- one gradient step of SB3's SAC.train, in three stages around the two gradient all-reduces -----------------
    def _stage_critic(self, obs, act, rew, next_obs, done, eps_pi, eps_next, out):
        """actor forward, entropy-coefficient loss, TD target, critic loss; backward into the critics + log-alpha bucket."""
        cfg = self.cfg
        actions_pi, log_prob = self.actor(obs, eps=eps_pi)
        ent_coef = self.log_ent_coef.detach().exp()
        ent_loss = -(self.log_ent_coef * (log_prob + self.target_entropy).detach()).mean()
        with torch.no_grad():
            next_a, next_logp = self.actor(next_obs, eps=eps_next)
            next_q = torch.stack(self.critic_target(next_obs, next_a), 0).min(0).values - ent_coef * next_logp
            target_q = rew + (1.0 - done) * cfg.gamma * next_q
        cur_q = self.critic(obs, act)
        critic_loss = 0.5 * sum(torch.nn.functional.mse_loss(q, target_q) for q in cur_q)
        self.g_critic.zero()
        (critic_loss + ent_loss).backward(inputs=self.g_critic.params)
        out[0].copy_(critic_loss.detach()); out[2].copy_(ent_coef.squeeze(0)); out[3].copy_(ent_loss.detach())
        return actions_pi, log_prob, ent_coef

    def _stage_actor(self, obs, actions_pi, log_prob, ent_coef, out):
        """optimiser steps of log-alpha and the critics, then the actor loss against the UPDATED critics (as in SB3)."""
        self.ent_opt.step()
        self.critic_opt.step()
        q_pi = torch.stack(self.critic(obs, actions_pi), 0).min(0).values
        actor_loss = (ent_coef * log_prob - q_pi).mean()
        self.g_actor.zero()
        actor_loss.backward(inputs=self.g_actor.params)
        out[1].copy_(actor_loss.detach())

    def _stage_finish(self):
        self.actor_opt.step()
        if (self.n_updates + 1) % self.cfg.target_update_interval == 0:
            with torch.no_grad():                            # polyak_update(critic, critic_target, tau)
                tp, sp = list(self.critic_target.parameters()), list(self.critic.parameters())
                torch._foreach_mul_(tp, 1.0 - self.cfg.tau)
                torch._foreach_add_(tp, sp, alpha=self.cfg.tau)

    def _capture(self, B, D, A):
        """Three CUDA graphs per gradient step ([actor fwd + critic losses + backward] | all-reduce | [alpha / critic
        steps + actor loss + backward] | all-reduce | [actor step + Polyak]): a 1024-sample SAC step is ~300 small
        kernels, i.e. launch-bound when issued eagerly."""
        dev = self.device
        f = dict(dtype=torch.float32, device=dev)
        st = dict(obs=torch.zeros(B, D, **f), act=torch.zeros(B, A, **f), rew=torch.zeros(B, **f), next_obs=torch.zeros(B, D, **f),
                  done=torch.zeros(B, **f), eps_pi=torch.zeros(B, A, **f), eps_next=torch.zeros(B, A, **f), out=torch.zeros(4, **f))
        keep = {}                                            # stage 1's outputs, stage 2's inputs

        def critic():
            keep["a"], keep["l"], keep["e"] = self._stage_critic(st["obs"], st["act"], st["rew"], st["next_obs"], st["done"],
                                                                 st["eps_pi"], st["eps_next"], st["out"])

        def actor():
            self._stage_actor(st["obs"], keep["a"], keep["l"], keep["e"], st["out"])
        stages = (critic, actor, self._stage_finish)

        def warmup():
            st["obs"].normal_(); st["next_obs"].normal_(); st["act"].uniform_(-1, 1); st["eps_pi"].normal_(); st["eps_next"].normal_()
            for _ in range(3):
                for stage in stages:
                    stage()
        nets = list(self.actor.parameters()) + list(self.critic.parameters()) + list(self.critic_target.parameters()) + [self.log_ent_coef]
        graphs = capture_graphs(stages, warmup, nets, (self.actor_opt, self.critic_opt, self.ent_opt), dev)
        self._graphs = ((B, D, A), graphs, st, keep)

    def update(self, batch, generator=None) -> Dict[str, torch.Tensor]:
        """One gradient step of SB3's SAC.train on a sampled batch (obs, act, rew, next_obs, done)."""
        obs, act, rew, next_obs, done = batch
        B, D, A = obs.shape[0], obs.shape[1], act.shape[1]
        if self.use_graph and obs.is_cuda:
            if self._graphs is None or self._graphs[0] != (B, D, A):
                self._capture(B, D, A)
            _, (g1, g2, g3), st, _ = self._graphs
            st["obs"].copy_(obs); st["act"].copy_(act); st["rew"].copy_(rew); st["next_obs"].copy_(next_obs); st["done"].copy_(done)
            st["eps_pi"].normal_(generator=generator); st["eps_next"].normal_(generator=generator)
            g1.replay()
            self.g_critic.allreduce()
            g2.replay()
            self.g_actor.allreduce()
            g3.replay()
            out = st["out"].clone()
        else:
            out = torch.zeros(4, device=self.device)
            eps_pi = torch.randn(B, A, device=self.device, generator=generator)
            eps_next = torch.randn(B, A, device=self.device, generator=generator)
            actions_pi, log_prob, ent_coef = self._stage_critic(obs, act, rew, next_obs, done, eps_pi, eps_next, out)
            self.g_critic.allreduce()
            self._stage_actor(obs, actions_pi, log_prob, ent_coef, out)
            self.g_actor.allreduce()
            self._stage_finish()
        self.n_updates += 1
        return {"critic_loss": out[0], "actor_loss": out[1], "ent_coef": out[2], "ent_coef_loss": out[3]}

    def flat_parameters(self) -> torch.Tensor:
        ps = list(self.actor.parameters()) + list(self.critic.parameters()) + [self.log_ent_coef]
        return torch.cat([p.detach().reshape(-1) for p in ps])


class SACTrainer:
    """Off-policy loop on a BatchedDroneEnv shard: train_freq env steps, then gradient_steps updates."""

    def __init__(self, env, cfg: SACConfig = SACConfig()):
        self.env, self.cfg, self.dev = env, cfg, env.device
        self.learner = SACLearner(env.obs_dim, 4, cfg, device=self.dev)
        rank = dist.get_rank() if _world() > 1 else 0
        self.gen = torch.Generator(device=self.dev).manual_seed(cfg.seed + 1000 * (rank + 1))
        self.buffer = ReplayBuffer(cfg.buffer_size, env.num_envs, env.obs_dim, 4, self.dev)
        self.obs = env.reset().clone()
        self.total_steps = 0
        self.collect_graph = bool(cfg.cuda_graph)           # replay the sampled phases of the fused collection from a CUDA graph
        self._collect_phase = PhaseGraph()                  # that graph, keyed by the phase length
        if cfg.rollout_impl == "fused":
            from . import _lib as L
            self.fused = self.learner.ensure_fused_actor(env.num_envs)
            # Philox draw counter on the device (advanced by every drawing dn_sac_act call, also inside graph replays); the key is
            # the seed shared by all ranks and the subsequence the GLOBAL env id, so the noise does not depend on the sharding
            self.draw_counter = torch.zeros(1, dtype=torch.int64, device=self.dev)
            self.samplers = {}
            for mode in (L.DN_SAC_SAMPLE, L.DN_SAC_UNIFORM):
                s = L.dn_sac_sample()
                s.seed, s.row_id_offset, s.counter, s.mode = int(cfg.seed), int(getattr(env, "env_id_offset", 0)), self.draw_counter.data_ptr(), mode
                self.samplers[mode] = s
            self.slot = torch.zeros(1, dtype=torch.int64, device=self.dev)     # replay-buffer row the next step writes (= buffer.pos)
            self.action = torch.empty(env.num_envs, 4, dtype=torch.float32, device=self.dev)

    @torch.no_grad()
    def collect(self, n_steps: int):
        if self.cfg.rollout_impl == "fused":
            return self._collect_fused(n_steps)
        env, N = self.env, self.env.num_envs
        for _ in range(n_steps):
            if self.total_steps < self.cfg.learning_starts:      # SB3: uniform random actions before learning_starts
                a = torch.rand(N, 4, device=self.dev, generator=self.gen) * 2 - 1
            else:
                a = self.learner.act(self.obs, generator=self.gen)
            a = a.contiguous()
            obs, rew, done, _ = env.step(a)
            self.buffer.add(self.obs, obs, a, rew, done, env.terminal_obs)
            self.obs = obs.clone()
            self.total_steps += N * _world()

    def _collect_step(self, mode: int):
        """One env step of a fused phase: dn_sac_act on the current observation, env.step, the replay write at the device-side
        slot, slot + 1.  Nothing here waits for the host."""
        env, buf = self.env, self.buffer
        self.fused.act(self.obs, self.samplers[mode], self.action)
        env.step(self.action)
        buf.write(self.slot, self.obs, env.obs, self.action, env.reward, env.done, env.terminal_obs)
        self.slot.add_(1).remainder_(buf.cap)
        self.obs.copy_(env.obs)

    @property
    def _collect_graph(self) -> Optional[torch.cuda.CUDAGraph]:
        """The captured graph of the fused collection (None until one was captured)."""
        return self._collect_phase.graph

    def _collect_fused(self, n_steps: int):
        """collect() on dn_sac_act.  A phase with a step before learning_starts runs launch by launch (uniform actions for those
        steps, as SB3's action_space.sample()).  Every later phase is ONE CUDA graph -- weight refresh, then n_steps x (act,
        env.step, replay write) -- captured at the second such phase (the first, launched, loads every kernel) and replayed from
        then on.  The host keeps ReplayBuffer.pos / full by arithmetic; the slot tensor is set from pos before every phase."""
        from . import _lib as L
        cfg, buf = self.cfg, self.buffer
        per_step = self.env.num_envs * _world()
        self.slot.fill_(buf.pos)
        if self.total_steps < cfg.learning_starts:
            self.fused.sync_weights()
            for k in range(n_steps):
                self._collect_step(L.DN_SAC_UNIFORM if self.total_steps + k * per_step < cfg.learning_starts else L.DN_SAC_SAMPLE)
        else:
            def phase():
                self.fused.sync_weights()
                for _ in range(n_steps):
                    self._collect_step(L.DN_SAC_SAMPLE)
            self._collect_phase.run(self.collect_graph, n_steps, phase)
        for _ in range(n_steps):
            buf.pos = (buf.pos + 1) % buf.cap
            buf.full = buf.full or buf.pos == 0
        self.total_steps += n_steps * per_step

    def train_iteration(self) -> Dict[str, float]:
        cfg = self.cfg
        t0 = time.perf_counter()
        cuda = self.dev.type == "cuda"
        if cuda:                     # device events: timing the collection needs no host synchronisation inside the iteration
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        self.collect(cfg.train_freq)
        if cuda:
            ev[1].record()
        t_collect = time.perf_counter()
        out = {}
        grad_steps = 0
        if self.total_steps >= cfg.learning_starts and len(self.buffer) >= cfg.batch_size:
            for _ in range(cfg.gradient_steps):
                out = self.learner.update(self.buffer.sample(cfg.batch_size, generator=self.gen), generator=self.gen)
                grad_steps += 1
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)
        dt = time.perf_counter() - t0
        res = {k: float(v) for k, v in out.items()}
        res.update(samples=cfg.train_freq * self.env.num_envs * _world(), gradient_steps=grad_steps, seconds=dt,
                   sps=cfg.train_freq * self.env.num_envs * _world() / dt,
                   collect_s=ev[0].elapsed_time(ev[1]) / 1000.0 if cuda else t_collect - t0)
        return res
