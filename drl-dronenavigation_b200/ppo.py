"""Torch-native PPO on the device-resident environment (SURVEY.md section 8 f.1).

The update is the maths of the reference's ``PPO.train`` (Sol/Model/Algorithms/sb3_ppo.py:190-316:
per-minibatch advantage normalisation, clipped surrogate, clipped value loss, entropy bonus,
approx-KL early stop at 1.5 x target_kl, grad-norm clipping) with the hyper-parameters of
``PBDroneSimulator.setup_agent`` (Sol/Model/PBDroneSimulator.py:251-286) and SB3's
``ActorCriticPolicy`` defaults the reference relies on (separate pi / vf MLPs [512, 512, 256] with
Tanh, diagonal Gaussian with a state-independent log-std initialised at 0, orthogonal init,
Adam(eps=1e-5)).  What changes is where the data lives: observations, actions, rewards and dones
never leave the GPU (no SB3 numpy hop), GAE is a CUDA kernel (``dn_gae``), and under ``torchrun``
every optimiser step all-reduces ONE flat gradient bucket (~0.8 M parameters, 3.2 MB) over NCCL --
the only collective in the system (the environment shards need none).
"""
from __future__ import annotations

import ctypes as C
import math
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import torch
import torch.distributed as dist
from torch import nn

from ._fused import Handle, PhaseGraph, capture_graphs, flat_views, offsets, sm100, widths_ok
from ._fused import world as _world


@dataclass
class PPOConfig:
    """Defaults = PBDroneSimulator.setup_agent's PPO branch (PBDroneSimulator.py:251-286)."""
    n_steps: int = 4096
    batch_size: int = 512
    n_epochs: int = 10
    gamma: float = 0.99
    gae_lambda: float = 0.95
    ent_coef: float = 0.02
    vf_coef: float = 0.5
    clip_range: float = 0.2
    clip_range_vf: Optional[float] = 0.3
    normalize_advantage: bool = True
    max_grad_norm: float = 0.5
    target_kl: Optional[float] = 0.05
    learning_rate: float = 2.5e-4
    pi_arch: tuple = (512, 512, 256)
    vf_arch: tuple = (512, 512, 256)
    log_std_init: float = 0.0
    adam_eps: float = 1e-5
    seed: int = 42                      # model.set_random_seed(42), PBDroneSimulator.py:690
    matmul_precision: str = "tf32"      # "fp32" | "tf32": precision of the MLP GEMMs of the torch path (cuBLAS)
    cuda_graph: bool = True             # torch path: replay each minibatch step from two captured CUDA graphs (CUDA devices only)
    update_impl: str = "auto"           # "fused": hand-written sm_100a kernels (include/dnppo.h); "torch": eager PyTorch;
                                        # "auto": fused on a compute-capability-10 device when the shapes allow it
    mlp_precision: str = "bf16x3"       # fused path: "bf16x3" (FP32-faithful hi/lo split, default) | "bf16" (labelled option)
    rollout_impl: str = "torch"         # "torch": per-step host loop, torch.Generator noise; "fused": dn_ppo_act (Philox noise keyed by
                                        # the global env id) and the T-step loop replayed from a CUDA graph (needs the fused handle)


_ONES: Dict[tuple, torch.Tensor] = {}


def _ones_row(n, device, dtype):
    key = (n, str(device), dtype)
    t = _ONES.get(key)
    if t is None:
        t = _ONES[key] = torch.ones(1, n, device=device, dtype=dtype)
    return t


class _LinearFn(torch.autograd.Function):
    """y = x W^T + b with the backward pass spelled out for the shapes of this learner (tens of thousands of rows,
    13..512 features), measured on B200 with cuBLAS TF32 (tools/micro/gemm_probe.py, 32768 rows):
      * bias gradient as a GEMV  ones[1,B] @ dy  (23 us) instead of autograd's column-sum reduction (46 us);
      * input width padded to a multiple of 8 (13 -> 16 zero columns): forward 35 -> 20 us, weight gradient
        80 -> 48 us -- unpadded K = 13 makes cuBLAS fall back to an sm_80 64x64 kernel."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        k = x.shape[1]
        pad = (-k) % 8
        if pad:
            x = torch.nn.functional.pad(x, (0, pad))
            w = torch.nn.functional.pad(weight, (0, pad))
        else:
            w = weight
        ctx.save_for_backward(x, w)
        ctx.k = k
        return torch.addmm(bias, x, w.t())

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = (dy @ w)[:, :ctx.k]
        if ctx.needs_input_grad[1]:
            dw = (dy.t() @ x)[:, :ctx.k]
        if ctx.needs_input_grad[2]:
            db = (_ones_row(dy.shape[0], dy.device, dy.dtype) @ dy).squeeze(0)
        return dx, dw, db


class FastLinear(nn.Linear):
    """nn.Linear (same parameters, same state_dict keys) whose CUDA training path goes through _LinearFn."""

    def forward(self, x):
        if x.is_cuda and x.dim() == 2 and torch.is_grad_enabled() and self.weight.requires_grad:
            return _LinearFn.apply(x, self.weight, self.bias)
        return super().forward(x)


def _mlp(sizes, out_dim, out_gain):
    layers: List[nn.Module] = []
    for a, b in zip(sizes[:-1], sizes[1:]):
        lin = FastLinear(a, b)
        nn.init.orthogonal_(lin.weight, gain=math.sqrt(2))
        nn.init.zeros_(lin.bias)
        layers += [lin, nn.Tanh()]
    head = FastLinear(sizes[-1], out_dim)
    nn.init.orthogonal_(head.weight, gain=out_gain)
    nn.init.zeros_(head.bias)
    layers.append(head)
    return nn.Sequential(*layers)


class ActorCritic(nn.Module):
    """SB3 ActorCriticPolicy with share_features_extractor=False and net_arch=dict(pi=..., vf=...)."""

    def __init__(self, obs_dim: int, act_dim: int, cfg: PPOConfig):
        super().__init__()
        self.pi = _mlp((obs_dim,) + tuple(cfg.pi_arch), act_dim, 0.01)
        self.vf = _mlp((obs_dim,) + tuple(cfg.vf_arch), 1, 1.0)
        self.log_std = nn.Parameter(torch.full((act_dim,), float(cfg.log_std_init)))

    def value(self, obs):
        return self.vf(obs).squeeze(-1)

    def act(self, obs, generator=None, deterministic=False):
        mean = self.pi(obs)
        if deterministic:
            action = mean
        else:
            noise = torch.randn(mean.shape, device=mean.device, dtype=mean.dtype, generator=generator)
            action = mean + noise * self.log_std.exp()
        return action, self._log_prob(mean, action), self.value(obs)

    def _log_prob(self, mean, action):
        var = (2 * self.log_std).exp()
        return (-((action - mean) ** 2) / (2 * var) - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)

    def evaluate(self, obs, actions):
        mean = self.pi(obs)
        entropy = (0.5 + 0.5 * math.log(2 * math.pi) + self.log_std).sum().expand(obs.shape[0])
        return self.value(obs), self._log_prob(mean, actions), entropy


def compute_gae_torch(rewards, values, dones, last_values, gamma, lam):
    """Reference recursion (SB3 RolloutBuffer.compute_returns_and_advantage) as plain torch ops; used on
    CPU tensors (gloo tests) and as the FP32 reference of the dn_gae kernel's numerics test."""
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    gae = torch.zeros_like(last_values)
    next_v = last_values
    for t in range(T - 1, -1, -1):
        nnt = 1.0 - (dones[t] != 0).to(rewards.dtype)
        delta = rewards[t] + gamma * next_v * nnt - values[t]
        gae = delta + gamma * lam * nnt * gae
        adv[t] = gae
        next_v = values[t]
    return adv, adv + values


def compute_gae(rewards, values, dones, last_values, gamma, lam):
    """[T, N] tensors -> (advantages, returns).  CUDA tensors go through libdronenav's dn_gae kernel."""
    if not rewards.is_cuda:
        return compute_gae_torch(rewards, values, dones, last_values, gamma, lam)
    from . import _lib as L
    rewards, values, last_values = rewards.contiguous(), values.contiguous(), last_values.contiguous()
    dones = dones.to(torch.uint8).contiguous()
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    T, N = rewards.shape
    stream = C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream)
    with torch.cuda.device(rewards.device):
        L.check(L.lib().dn_gae(rewards.data_ptr(), values.data_ptr(), dones.data_ptr(), last_values.data_ptr(),
                               float(gamma), float(lam), adv.data_ptr(), ret.data_ptr(), T, N, stream), "dn_gae")
    return adv, ret


class FusedUpdate(Handle):
    """ctypes face of the dn_ppo handle (include/dnppo.h): the body of PPO.train's minibatch loop and the policy forward
    as hand-written sm_100a kernels on ONE flat FP32 parameter vector.  The torch ``Parameter`` s of the policy, their
    ``.grad`` s and the Adam moments are views into the flat buffers this object hands to the library, so checkpoints,
    the eager torch path and the kernels all see the same memory."""

    ABI = "dn_ppo"

    @staticmethod
    def shapes_ok(pi_arch, vf_arch, obs_dim: int, act_dim: int) -> bool:
        """The shapes dn_ppo_create accepts: 1..4 hidden layers per network, every hidden width a multiple of 128 between 128
        and 512 (the column-sum accumulator of the bias gradients holds 512 columns), 1 <= obs_dim <= 64, act_dim in (1, 3, 4)."""
        return widths_ok(pi_arch, obs_dim) and widths_ok(vf_arch, obs_dim) and act_dim in (1, 3, 4)

    @staticmethod
    def supported(cfg: "PPOConfig", obs_dim: int, act_dim: int, device) -> bool:
        return sm100(device) and FusedUpdate.shapes_ok(cfg.pi_arch, cfg.vf_arch, obs_dim, act_dim)

    def __init__(self, learner: "PPOLearner", max_rows: int):
        super().__init__(learner.device)
        L = self.L
        self.learner = learner
        cfg, dev = learner.cfg, learner.device
        pol = learner.policy
        self.max_rows = int(-(-max_rows // 128) * 128)
        n = learner.n_params
        f = dict(dtype=torch.float32, device=dev)
        self.params = torch.empty(n, **f)
        self.exp_avg, self.exp_avg_sq = torch.zeros(n, **f), torch.zeros(n, **f)
        self.step = torch.zeros((), **f)
        # re-seat parameters (and the Adam state) as views of the flat vectors
        ps, offs = list(pol.parameters()), offsets(pol.named_parameters())
        with torch.no_grad():
            for p, v, m, m2 in zip(ps, flat_views(self.params, ps), flat_views(self.exp_avg, ps), flat_views(self.exp_avg_sq, ps)):
                v.copy_(p.detach())
                p.data = v
                old = learner.opt.state.get(p)
                if old:                                  # keep the moments of an optimiser that has already stepped / was loaded
                    m.copy_(old["exp_avg"])
                    m2.copy_(old["exp_avg_sq"])
                    self.step.copy_(torch.as_tensor(old["step"], dtype=torch.float32).reshape(()))
                learner.opt.state[p] = {"step": self.step, "exp_avg": m, "exp_avg_sq": m2}
        c = L.dn_ppo_config()
        c.abi_version = L.DN_ABI_VERSION
        c.obs_dim, c.act_dim, c.max_rows = pol.pi[0].in_features, pol.log_std.numel(), self.max_rows
        c.n_pi, c.n_vf = len(cfg.pi_arch), len(cfg.vf_arch)
        for i, w in enumerate(cfg.pi_arch):
            c.pi_hidden[i] = w
        for i, w in enumerate(cfg.vf_arch):
            c.vf_hidden[i] = w
        c.precision = {"bf16x3": L.DN_MLP_BF16X3, "bf16": L.DN_MLP_BF16}[cfg.mlp_precision]
        c.normalize_advantage = int(cfg.normalize_advantage)
        c.world_size = _world()
        c.clip_range = cfg.clip_range
        c.clip_range_vf = -1.0 if cfg.clip_range_vf is None else cfg.clip_range_vf
        c.ent_coef, c.vf_coef, c.max_grad_norm = cfg.ent_coef, cfg.vf_coef, cfg.max_grad_norm
        c.target_kl = -1.0 if cfg.target_kl is None else cfg.target_kl
        c.learning_rate, c.beta1, c.beta2, c.adam_eps = cfg.learning_rate, 0.9, 0.999, cfg.adam_eps
        for l in range(c.n_pi + 1):          # nn.Sequential indices: Linear at 0, 2, 4, ... (Tanh in between)
            c.pi_w_off[l], c.pi_b_off[l] = offs[f"pi.{2 * l}.weight"], offs[f"pi.{2 * l}.bias"]
        for l in range(c.n_vf + 1):
            c.vf_w_off[l], c.vf_b_off[l] = offs[f"vf.{2 * l}.weight"], offs[f"vf.{2 * l}.bias"]
        c.log_std_off, c.n_params = offs["log_std"], n
        self._create(c, self.params.data_ptr(), learner._flat.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                     self.step.data_ptr())
        self.launches = 0

    def forward(self, obs: torch.Tensor):
        """(mean [n, act_dim], value [n]) with the kernels and arithmetic of the update."""
        obs = obs.contiguous().float()
        n = obs.shape[0]
        mean = torch.empty(n, self.cfg_c.act_dim, dtype=torch.float32, device=self.device)
        value = torch.empty(n, dtype=torch.float32, device=self.device)
        self.sync_weights()
        self.call("dn_ppo_forward", obs.data_ptr(), n, mean.data_ptr(), value.data_ptr())
        return mean, value

    def act(self, obs: torch.Tensor, sample, action: torch.Tensor = None, clipped_action: torch.Tensor = None,
            log_prob: torch.Tensor = None, value: torch.Tensor = None, sync: bool = True):
        """ActorCriticPolicy.forward with the sampler of the library (dn_ppo_act): (action, clipped_action, log_prob, value).
        `sample` is an ``_lib.dn_ppo_sample`` (seed, global id of row 0, device int64 draw counter, deterministic, Box bounds).
        Outputs may be passed in (graph capture: fixed pointers); `clipped_action` is only written when given or allocated here.
        ``sync=False`` skips the FP32 -> BF16 weight refresh (the caller knows the parameters did not change)."""
        n = obs.shape[0]
        A = self.cfg_c.act_dim
        f = dict(dtype=torch.float32, device=self.device)
        action = torch.empty(n, A, **f) if action is None else action
        clipped_action = torch.empty(n, A, **f) if clipped_action is None else clipped_action
        log_prob = torch.empty(n, **f) if log_prob is None else log_prob
        value = torch.empty(n, **f) if value is None else value
        dev = torch.device("cuda", torch.cuda.current_device() if self.device.index is None else self.device.index)
        for t, shape in ((obs, (n, self.cfg_c.obs_dim)), (action, (n, A)), (clipped_action, (n, A)), (log_prob, (n,)), (value, (n,))):
            if t.dtype != torch.float32 or t.device != dev or not t.is_contiguous() or tuple(t.shape) != shape:
                raise ValueError(f"dn_ppo_act: expected a contiguous float32 tensor of shape {shape} on {self.device}")
        if sync:
            self.sync_weights()
        self.call("dn_ppo_act", obs.data_ptr(), n, C.byref(sample), action.data_ptr(), clipped_action.data_ptr(), log_prob.data_ptr(),
                  value.data_ptr())
        return action, clipped_action, log_prob, value

    def begin_update(self):
        self.sync_weights()
        self.call("dn_ppo_begin_update")

    def minibatch_grad(self, ro, idx: torch.Tensor):
        self.call("dn_ppo_minibatch_grad", C.byref(ro), idx.data_ptr(), idx.numel())

    def minibatch_apply(self):
        self.call("dn_ppo_minibatch_apply")

    comm_ready = False

    def comm_setup(self) -> bool:
        """Gradient all-reduce over NVLink peer memory (dn_ppo_comm_create / _connect): every rank allocates its exchange region,
        the 64-byte CUDA IPC handles are all-gathered through torch.distributed, every rank maps its peers' regions.  Collective:
        all ranks call it at the same point.  Returns False -- on EVERY rank -- when the job spans several nodes, when
        DN_PPO_ALLREDUCE=nccl, or when any rank could not map a peer (the caller then keeps ncclAllReduce)."""
        import os
        world, rank = dist.get_world_size(), dist.get_rank()
        on_cuda = dist.get_backend() == "nccl"
        dev = self.device if on_cuda else torch.device("cpu")
        ok = (os.environ.get("DN_PPO_ALLREDUCE", "peer") != "nccl" and 2 <= world <= 16
              and int(os.environ.get("LOCAL_WORLD_SIZE", world)) == world)
        hb = (C.c_ubyte * 64)()
        if ok:
            with torch.cuda.device(self.device):
                ok = self.lib.dn_ppo_comm_create(self.handle, rank, world, hb) == 0
        mine = torch.tensor(list(hb) + [1 if ok else 0], dtype=torch.uint8, device=dev)
        allh = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allh, mine)
        allh = torch.stack(allh).cpu()
        ok = bool(allh[:, 64].min().item())
        if ok:
            buf = (C.c_ubyte * (64 * world))(*allh[:, :64].reshape(-1).tolist())
            with torch.cuda.device(self.device):
                ok = self.lib.dn_ppo_comm_connect(self.handle, buf) == 0
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        self.comm_ready = bool(flag.item())
        return self.comm_ready

    def allreduce(self):
        self.call("dn_ppo_allreduce")

    def poll(self):
        a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
        self.lib.dn_ppo_poll(self.handle, C.byref(a), C.byref(b), C.byref(c))
        return bool(a.value), b.value, c.value

    def stats(self):
        st = self.L.dn_ppo_stats()
        self.call("dn_ppo_get_stats", C.byref(st))
        return st

    def buffer(self, name: str, rows: int, cols: int):
        """Test hook: FP32 reconstruction (hi + lo) of the first `rows` rows of an internal BF16 plane pair."""
        planes = self._raw_buffer(name, "<i2").view(torch.bfloat16).view(2, -1, cols)[:, :rows]
        return planes[0].float() + (planes[1].float() if self.learner.cfg.mlp_precision == "bf16x3" else 0.0)


class PPOLearner:
    """Policy + optimiser + the PPO update; independent of the environment (works on any device, which
    is what the world_size-2 gloo tests use)."""

    def __init__(self, obs_dim: int, act_dim: int, cfg: PPOConfig = PPOConfig(), device="cpu"):
        self.cfg, self.device = cfg, torch.device(device)
        torch.manual_seed(cfg.seed)                     # same seed on every rank -> identical initial parameters
        self.policy = ActorCritic(obs_dim, act_dim, cfg).to(self.device)
        self._graphs = None                             # (key, graphs, static tensors) of the update in use; built lazily
        self.use_graph = bool(cfg.cuda_graph) and self.device.type == "cuda"
        self.opt = torch.optim.Adam(self.policy.parameters(), lr=cfg.learning_rate, eps=cfg.adam_eps,
                                    capturable=self.use_graph)
        self.params = [p for p in self.policy.parameters()]
        self.n_params = sum(p.numel() for p in self.params)
        # the one gradient bucket: every parameter's .grad is a view into it, so backward() writes the
        # bucket in place and the all-reduce / norm clip are single operations on one contiguous tensor
        # (one extra element: the fused update carries this rank's KL early-stop vote through the same all-reduce)
        self._bucket = torch.zeros(self.n_params + 1, device=self.device)
        self._flat = self._bucket[:self.n_params]
        for p, g in zip(self.params, flat_views(self._flat, self.params)):
            p.grad = g
        self.n_updates = 0
        self.allreduce_calls = 0
        self.obs_dim, self.act_dim = obs_dim, act_dim
        impl = cfg.update_impl
        if impl not in ("auto", "fused", "torch"):
            raise ValueError(f"update_impl={impl!r}")
        can = FusedUpdate.supported(cfg, obs_dim, act_dim, self.device)
        if impl == "fused" and not can:
            raise RuntimeError("update_impl='fused' needs a compute-capability-10 CUDA device, 1..4 hidden layers per network whose "
                               "widths are multiples of 128 between 128 and 512, 1 <= obs_dim <= 64 and act_dim in (1, 3, 4)")
        self.want_fused = can and impl in ("auto", "fused")
        self.fused: Optional[FusedUpdate] = None
        if self.device.type == "cuda":                  # process-wide switches: set both ways so "fp32" means FP32
            torch.backends.cuda.matmul.allow_tf32 = (cfg.matmul_precision == "tf32")
            torch.backends.cudnn.allow_tf32 = (cfg.matmul_precision == "tf32")

    # ---- fused path (include/dnppo.h) ------------------------------------------------------------------------
    def ensure_fused(self, rows: int) -> Optional[FusedUpdate]:
        """The fused handle with workspaces for at least `rows` rows (re-created when a larger batch shows up)."""
        if not self.want_fused:
            return None
        if self.fused is None or rows > self.fused.max_rows:
            if self.fused is not None:
                torch.cuda.synchronize(self.device)
                self.fused.close()
            self.fused = FusedUpdate(self, rows)
            self.drop_graphs()             # parameters and Adam state were re-seated
        return self.fused

    def drop_graphs(self) -> None:
        """Forgets the captured update graphs (the next update captures again).  Called by everything that replaces a tensor
        the graphs point to."""
        self._graphs = None

    def forward(self, obs):
        """(mean, value) of the policy: fused kernels when available, else the torch modules."""
        fu = self.ensure_fused(obs.shape[0])
        if fu is not None:
            return fu.forward(obs)
        return self.policy.pi(obs), self.policy.value(obs)

    @torch.no_grad()
    def act(self, obs, generator=None, deterministic=False):
        """ActorCriticPolicy.forward: (action, log_prob, value)."""
        if not self.want_fused:
            return self.policy.act(obs, generator=generator, deterministic=deterministic)
        mean, value = self.forward(obs)
        if deterministic:
            action = mean
        else:
            noise = torch.randn(mean.shape, device=mean.device, dtype=mean.dtype, generator=generator)
            action = mean + noise * self.policy.log_std.exp()
        return action, self.policy._log_prob(mean, action), value

    @torch.no_grad()
    def value(self, obs):
        if not self.want_fused:
            return self.policy.value(obs)
        return self.forward(obs)[1]

    def _update_fused(self, obs, actions, old_logp, old_values, advantages, returns, generator) -> Dict[str, float]:
        """PPO.train (sb3_ppo.py:190-316) with the minibatch body in the library: per minibatch ONE gradient half
        (gather .. backward), the flat-bucket all-reduce when there are several ranks, ONE apply half (clip, Adam).  The KL
        early stop (:283-287) is decided on the device (each rank's vote rides in the bucket's extra element, so ranks stop
        together without a second collective or a host synchronisation); the host learns about it from a pinned mirror and
        stops launching -- minibatches launched in between are no-ops on the device."""
        cfg = self.cfg
        B = obs.shape[0]
        mb = min(cfg.batch_size, B)
        if mb % 128 or B % mb:
            raise ValueError(f"fused PPO update: minibatch {mb} must be a multiple of 128 and divide the rollout ({B} samples); "
                             "use update_impl='torch' for ragged batches")
        n_mb = B // mb
        fu = self.ensure_fused(mb)
        world = _world()
        # several ranks: the flat-bucket sum runs over NVLink peer memory inside the library (and inside the minibatch graph) when
        # all ranks share a node, through ncclAllReduce between two graphs otherwise
        peer = world > 1 and (fu.comm_ready or (not getattr(fu, "comm_tried", False) and fu.comm_setup()))
        fu.comm_tried = True
        self.allreduce_impl = "peer" if peer else ("nccl" if world > 1 else "none")
        if peer:
            # the exchange kernels wait for their peers on the device with a bounded spin: ranks enter the update together (one
            # host barrier per update, not per minibatch; rank-0-only work between updates -- logging, checkpoints -- may take long)
            dist.barrier()
        ro = fu.L.dn_ppo_rollout()
        graphs = None
        if cfg.cuda_graph:
            # the ~25 kernels of a minibatch step replayed from CUDA graphs (one for the gradient half, one for the apply half; a
            # single one when there is no all-reduce in between): removes the launch gaps between the short dependent kernels.
            # Graphs bake pointers in, so the rollout is staged in static tensors and the minibatch indices in a static buffer.
            key = ("fused", B, mb, obs.shape[1], actions.shape[1], world, peer)
            if self._graphs is None or self._graphs[0] != key:
                self._capture_fused(fu, key)
            _, graphs, (static, idx) = self._graphs
            for dst, src in zip(static, (obs, actions, old_logp, old_values, advantages, returns)):
                dst.copy_(src)
            keep = list(static)
        else:
            keep = [t.contiguous().float() for t in (obs, actions, old_logp, old_values, advantages, returns)]
        ro.obs, ro.actions, ro.old_log_prob, ro.old_values, ro.advantages, ro.returns = [t.data_ptr() for t in keep]
        fu.begin_update()
        launched = 0
        stop = False
        # When does the host learn that the device stopped?  One rank: a non-blocking look at the pinned mirror after every
        # minibatch (it may lag by a few launches; those are no-ops on the device).  Several ranks: every rank must issue the
        # SAME number of all-reduces, so the decision has to be taken at the same loop positions from a value that is the same
        # everywhere -- the device-side `stopped` state (derived from the all-reduced vote), read with a stream synchronisation
        # every `check_every` minibatches and at the end of every epoch.
        check_every = 4
        for epoch in range(cfg.n_epochs):
            perm = torch.randperm(B, device=self.device, generator=generator)
            keep.append(perm)
            for k in range(n_mb):
                if graphs is not None:
                    idx.copy_(perm[k * mb:(k + 1) * mb])
                    graphs[0].replay()                   # one rank, or peer all-reduce: the whole step
                    if world > 1:
                        self.allreduce_calls += 1
                        if not peer:
                            dist.all_reduce(self._bucket, op=dist.ReduceOp.SUM)
                            graphs[1].replay()
                else:
                    fu.minibatch_grad(ro, perm[k * mb:(k + 1) * mb])
                    if world > 1:
                        if peer:
                            fu.allreduce()
                        else:
                            dist.all_reduce(self._bucket, op=dist.ReduceOp.SUM)
                        self.allreduce_calls += 1
                    fu.minibatch_apply()
                launched += 1
                if cfg.target_kl is None:
                    continue
                if world == 1:
                    stop = fu.poll()[0]
                elif (k + 1) % check_every == 0 or k == n_mb - 1:
                    stop = bool(fu.stats().early_stop)
                if stop:
                    break
            if stop:
                break
        st = fu.stats()                       # synchronises the stream
        epochs_run = -(-st.minibatches // n_mb) if st.minibatches else 0
        self.n_updates += epochs_run
        return {"policy_gradient_loss": st.policy_gradient_loss, "value_loss": st.value_loss,
                "entropy_loss": float(-(0.5 + 0.5 * math.log(2 * math.pi) + self.policy.log_std.detach()).sum()),
                "approx_kl": st.approx_kl, "clip_fraction": st.clip_fraction, "epochs": epochs_run, "minibatches": st.minibatches,
                "optimizer_steps": st.optimizer_steps, "early_stop": bool(st.early_stop), "launched_minibatches": launched,
                "grad_norm": st.last_grad_norm, "std": float(self.policy.log_std.detach().exp().mean()), "impl": "fused/" + cfg.mlp_precision}

    def _capture_fused(self, fu: FusedUpdate, key):
        """CUDA graphs of the fused minibatch step for rollouts of `key` = ("fused", B, mb, D, A, world, peer).  One graph for the
        whole step with one rank or with the peer-memory all-reduce (three kernels of the library between the halves); with
        ncclAllReduce the collective sits between two graphs."""
        _, B, mb, D, A, world, peer = key
        dev = self.device
        f = dict(dtype=torch.float32, device=dev)
        static = [torch.zeros(B, D, **f), torch.zeros(B, A, **f), torch.zeros(B, **f), torch.zeros(B, **f), torch.zeros(B, **f), torch.zeros(B, **f)]
        idx = torch.arange(mb, dtype=torch.long, device=dev)
        ro = fu.L.dn_ppo_rollout()
        ro.obs, ro.actions, ro.old_log_prob, ro.old_values, ro.advantages, ro.returns = [t.data_ptr() for t in static]

        def step():
            fu.minibatch_grad(ro, idx)
            if world > 1 and peer:
                fu.allreduce()                 # (every rank warms up and captures at the same point of the program: the peers answer)
            if world == 1 or peer:
                fu.minibatch_apply()
        stages = (step,) if world == 1 or peer else (step, fu.minibatch_apply)

        def warmup():                          # lazy kernel loading, launch attributes, plans for `mb` rows: one step on zeros
            fu.begin_update()
            for stage in stages:
                stage()
        graphs = capture_graphs(stages, warmup, (fu.params, fu.exp_avg, fu.exp_avg_sq, fu.step), (), dev)
        self._graphs = (key, graphs, (static, idx))

    # ---- the only collective: one flat bucket per optimiser step (between backward and clip, sb3_ppo.py:291-293)
    def _allreduce_grads(self, approx_kl=None) -> bool:
        """ONE collective per minibatch: the flat gradient bucket, whose extra last element carries this rank's KL early-stop
        vote (sb3_ppo.py:283-287) -- a sum > 0 is the MAX over ranks, so ranks leave the epoch loop together without a second
        all-reduce.  Returns the joint stop decision (one host read per minibatch, as in SB3)."""
        cfg, w = self.cfg, _world()
        vote = None
        if cfg.target_kl is not None and approx_kl is not None:
            vote = (approx_kl > 1.5 * cfg.target_kl).to(self._bucket.dtype)
        if w == 1:
            return bool(vote.item() > 0) if vote is not None else False
        self._bucket[-1] = vote if vote is not None else 0.0
        dist.all_reduce(self._bucket, op=dist.ReduceOp.SUM)
        self._flat.div_(w)
        self.allreduce_calls += 1
        return bool(self._bucket[-1].item() > 0) if vote is not None else False

    # ---- one minibatch, in two halves around the gradient all-reduce --------------------------------------
    def _forward_backward(self, obs, actions, old_logp, old_values, advantages, returns, acc):
        """losses of sb3_ppo.py:225-281 + backward into the flat bucket; returns approx_kl (0-d tensor)."""
        cfg = self.cfg
        values, logp, entropy = self.policy.evaluate(obs, actions)
        adv = advantages
        if cfg.normalize_advantage and adv.numel() > 1:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        ratio = torch.exp(logp - old_logp)
        pg_loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 1 - cfg.clip_range, 1 + cfg.clip_range)).mean()
        if cfg.clip_range_vf is None:
            v_pred = values
        else:
            v_pred = old_values + torch.clamp(values - old_values, -cfg.clip_range_vf, cfg.clip_range_vf)
        v_loss = torch.nn.functional.mse_loss(returns, v_pred)
        ent_loss = -entropy.mean()
        loss = pg_loss + cfg.ent_coef * ent_loss + cfg.vf_coef * v_loss
        with torch.no_grad():
            log_ratio = logp - old_logp
            approx_kl = ((torch.exp(log_ratio) - 1) - log_ratio).mean()
            clip_frac = ((ratio - 1).abs() > cfg.clip_range).float().mean()
            acc += torch.stack([pg_loss.detach(), v_loss.detach(), ent_loss.detach(), approx_kl, clip_frac])
        self._flat.zero_()
        loss.backward()
        return approx_kl

    def _clip_and_step(self):
        assert self.fused is None, "the torch optimiser step must not run once the fused update owns the Adam state"
        # th.nn.utils.clip_grad_norm_(parameters, max_grad_norm) on the flat bucket, then Adam
        norm = torch.linalg.vector_norm(self._flat)
        self._flat.mul_(torch.clamp(self.cfg.max_grad_norm / (norm + 1e-6), max=1.0))
        self.opt.step()

    def _capture(self, key):
        """Two CUDA graphs per minibatch step for rollouts of `key` = ("torch", B, mb, D, A): [gather -> forward -> losses ->
        backward] and [clip -> Adam], split where the gradient all-reduce (and the KL early-stop decision of sb3_ppo.py:283-287)
        sits.  The eager loop is CPU-bound (~200 small kernels per minibatch); replay makes it one launch per half."""
        _, B, mb, D, A = key
        dev = self.device
        f = dict(dtype=torch.float32, device=dev)
        st = dict(obs=torch.zeros(B, D, **f), act=torch.zeros(B, A, **f), logp=torch.zeros(B, **f), val=torch.zeros(B, **f),
                  adv=torch.zeros(B, **f), ret=torch.zeros(B, **f), idx=torch.zeros(mb, dtype=torch.long, device=dev),
                  acc=torch.zeros(5, **f), kl=torch.zeros((), **f))

        def half_a():
            i = st["idx"]
            kl = self._forward_backward(st["obs"][i], st["act"][i], st["logp"][i], st["val"][i], st["adv"][i], st["ret"][i], st["acc"])
            st["kl"].copy_(kl)

        def warmup():                          # allocator, cuBLAS workspaces, Adam state
            st["idx"].copy_(torch.arange(mb, device=dev) % B)
            st["obs"].normal_(); st["act"].uniform_(-1, 1); st["adv"].normal_(); st["ret"].normal_()
            for _ in range(3):
                half_a()
                self._clip_and_step()
        graphs = capture_graphs((half_a, self._clip_and_step), warmup, self.params, (self.opt,), dev)
        self._graphs = (key, graphs, st)

    def update(self, obs, actions, old_logp, old_values, advantages, returns, generator=None) -> Dict[str, float]:
        """PPO.train (sb3_ppo.py:190-316) on flat [B, ...] tensors of this rank's rollout."""
        cfg = self.cfg
        B = obs.shape[0]
        mb = min(cfg.batch_size, B)
        if self.want_fused and obs.is_cuda and (mb % 128 or B % mb) and self.fused is None and cfg.update_impl == "auto":
            self.want_fused = False          # ragged / tiny minibatches: this learner stays on the torch path
        if self.want_fused and obs.is_cuda:
            return self._update_fused(obs, actions, old_logp, old_values, advantages, returns, generator)
        if B % mb:
            # SB3's RolloutBuffer.get yields the trailing partial minibatch; neither the graph replay nor the fixed-shape
            # buffers here can, so refuse instead of silently dropping up to mb - 1 samples per epoch
            raise ValueError(f"rollout of {B} samples is not a multiple of the minibatch size {mb}")
        n_mb = B // mb
        graphed = self.use_graph and obs.is_cuda
        if graphed:
            key = ("torch", B, mb, obs.shape[1], actions.shape[1])
            if self._graphs is None or self._graphs[0] != key:
                self._capture(key)
            _, (ga, gb), st = self._graphs
            st["obs"].copy_(obs); st["act"].copy_(actions); st["logp"].copy_(old_logp); st["val"].copy_(old_values)
            st["adv"].copy_(advantages); st["ret"].copy_(returns)
            acc = st["acc"].zero_()
        else:
            acc = torch.zeros(5, device=self.device)
        n_done = 0
        stop = False
        epochs_run = 0
        for epoch in range(cfg.n_epochs):
            perm = torch.randperm(B, device=self.device, generator=generator)
            for k in range(n_mb):
                idx = perm[k * mb:(k + 1) * mb]
                if graphed:
                    st["idx"].copy_(idx)
                    ga.replay()
                    approx_kl = st["kl"]
                else:
                    approx_kl = self._forward_backward(obs[idx], actions[idx], old_logp[idx], old_values[idx],
                                                       advantages[idx], returns[idx], acc)
                n_done += 1
                stop = self._allreduce_grads(approx_kl)      # gradients + the early-stop vote in one collective
                if stop:
                    break                                    # the reduced gradients of this minibatch are discarded, as in SB3
                if graphed:
                    gb.replay()
                else:
                    self._clip_and_step()
            self.n_updates += 1
            epochs_run += 1
            if stop:
                break
        a = (acc / max(n_done, 1)).tolist()
        return {"policy_gradient_loss": a[0], "value_loss": a[1], "entropy_loss": a[2], "approx_kl": a[3],
                "clip_fraction": a[4], "epochs": epochs_run, "minibatches": n_done, "early_stop": bool(stop),
                "std": float(self.policy.log_std.detach().exp().mean())}

    def load_optimizer_state(self, state: Dict[int, dict]) -> None:
        """Adam state by position in ``self.policy.parameters()`` ({"step", "exp_avg", "exp_avg_sq"} per entry), e.g. from an
        SB3 ``policy.optimizer.pth`` re-indexed by checkpoint.load_sb3_zip.  Written into whatever owns the moments: the flat
        vectors of the fused update, or torch.optim.Adam's own tensors."""
        if self.fused is not None:
            with torch.no_grad():
                for i, p in enumerate(self.params):
                    if i in state:
                        st = self.opt.state[p]
                        st["exp_avg"].copy_(state[i]["exp_avg"].to(self.device))
                        st["exp_avg_sq"].copy_(state[i]["exp_avg_sq"].to(self.device))
                        self.fused.step.copy_(torch.as_tensor(state[i]["step"], dtype=torch.float32).reshape(()))
            return
        own = self.opt.state_dict()
        own["state"] = state
        self.opt.load_state_dict(own)
        self.drop_graphs()       # load_state_dict re-creates the state tensors

    def flat_parameters(self) -> torch.Tensor:
        return torch.cat([p.detach().reshape(-1) for p in self.params])


class PPOTrainer:
    """collect_rollouts + train on a BatchedDroneEnv shard (one process per GPU)."""

    def __init__(self, env, cfg: PPOConfig = PPOConfig(), rollout_steps: Optional[int] = None):
        self.env, self.cfg = env, cfg
        self.dev = env.device
        self.T = int(rollout_steps or cfg.n_steps)
        self.learner = PPOLearner(env.obs_dim, 4, cfg, device=self.dev)
        B, mb = self.T * env.num_envs, min(cfg.batch_size, self.T * env.num_envs)
        if cfg.update_impl == "auto" and (mb % 128 or B % mb):
            self.learner.want_fused = False  # the fused kernels need minibatches that are multiples of 128 and divide the rollout
        self.learner.ensure_fused(max(env.num_envs, mb))
        rank = dist.get_rank() if _world() > 1 else 0
        self.gen = torch.Generator(device=self.dev).manual_seed(cfg.seed + 1000 * (rank + 1))   # exploration noise differs per shard
        N, D, T = env.num_envs, env.obs_dim, self.T
        f = dict(dtype=torch.float32, device=self.dev)
        self.b_obs, self.b_act = torch.empty(T, N, D, **f), torch.empty(T, N, 4, **f)
        self.b_logp, self.b_val, self.b_rew = torch.empty(T, N, **f), torch.empty(T, N, **f), torch.empty(T, N, **f)
        self.b_done = torch.empty(T, N, dtype=torch.uint8, device=self.dev)
        self.obs = env.reset().clone()
        self.total_steps = 0
        self.low, self.high = -1.0, 1.0           # Box(-1, 1) with normalize_actions (PBDroneEnv.py:230-236)
        if cfg.rollout_impl not in ("torch", "fused"):
            raise ValueError(f"rollout_impl={cfg.rollout_impl!r}")
        self.rollout_graph = bool(cfg.cuda_graph)           # replay the T-step loop of the fused rollout from a CUDA graph
        self._rollout_phase = PhaseGraph()                  # that graph, keyed by the handle the loop calls
        if cfg.rollout_impl == "fused":
            if self.learner.fused is None:
                raise RuntimeError("rollout_impl='fused' needs the fused PPO handle (update_impl 'fused' or 'auto' on a compute-capability-10 "
                                   "CUDA device, 1..4 hidden layers per network whose widths are multiples of 128 between 128 and 512, "
                                   "1 <= obs_dim <= 64, act_dim in (1, 3, 4), minibatches that are multiples of 128 and divide the rollout)")
            from . import _lib as L
            # Philox draw counter on the device (advanced by every dn_ppo_act call, also inside graph replays); the key is the
            # seed shared by all ranks and the subsequence the GLOBAL env id, so the noise does not depend on the sharding
            self.draw_counter = torch.zeros(1, dtype=torch.int64, device=self.dev)
            self.sample = L.dn_ppo_sample()
            self.sample.seed, self.sample.row_id_offset = int(cfg.seed), int(getattr(env, "env_id_offset", 0))
            self.sample.counter, self.sample.deterministic = self.draw_counter.data_ptr(), 0
            self.sample.low, self.sample.high = self.low, self.high
            self.b_clip = torch.empty(T, N, 4, **f)       # what env.step received
            self.b_term = torch.zeros(T, N, D, **f)       # terminal observations (meaningful where b_done == truncated)

    @torch.no_grad()
    def collect_rollouts(self):
        if self.cfg.rollout_impl == "fused":
            return self._collect_rollouts_fused()
        env, pol = self.env, self.learner
        for t in range(self.T):
            action, logp, value = pol.act(self.obs, generator=self.gen)
            self.b_obs[t], self.b_act[t], self.b_logp[t], self.b_val[t] = self.obs, action, logp, value
            obs, rew, done, _ = env.step(action.clamp(self.low, self.high).contiguous())   # SB3 clips to the Box before env.step
            self.b_rew[t], self.b_done[t] = rew, done
            # bootstrap truncated episodes from the terminal observation (SB3 OnPolicyAlgorithm.collect_rollouts)
            trunc_only = done == 2
            if bool(trunc_only.any()):
                tv = pol.value(env.terminal_obs[trunc_only])
                self.b_rew[t][trunc_only] += self.cfg.gamma * tv
            self.obs = obs.clone()
        last_values = pol.value(self.obs)
        adv, ret = compute_gae(self.b_rew, self.b_val, self.b_done, last_values, self.cfg.gamma, self.cfg.gae_lambda)
        self.total_steps += self.T * env.num_envs * _world()      # global count: every rank collects its own shard
        return adv, ret

    def _rollout_step(self, fu, t: int):
        """Control step t of a fused rollout: act on the current observation, record, step the env (nothing here waits for the host)."""
        env = self.env
        self.b_obs[t].copy_(self.obs)
        fu.act(self.b_obs[t], self.sample, self.b_act[t], self.b_clip[t], self.b_logp[t], self.b_val[t], sync=False)
        env.step(self.b_clip[t])
        self.b_rew[t].copy_(env.reward)
        self.b_done[t].copy_(env.done)
        self.b_term[t].copy_(env.terminal_obs)
        self.obs.copy_(env.obs)

    @property
    def _rollout_graph(self) -> Optional[torch.cuda.CUDAGraph]:
        """The captured graph of the fused rollout (None until one was captured)."""
        return self._rollout_phase.graph

    def _collect_rollouts_fused(self):
        """collect_rollouts on dn_ppo_act.  The T-step loop is one CUDA graph, captured at the second rollout (the first one, launched
        step by step, loads every kernel) and replayed from then on; between its first and last step the host does not wait.  The
        policy is fixed during a rollout, so the truncation bootstrap of SB3's collect_rollouts (V(terminal_obs) of episodes that
        were truncated, not terminated) is deferred to one pass after the loop: the recorded terminal rows are compacted (the one
        host synchronisation of the rollout), their values computed by dn_ppo_forward in chunks of at most max_rows, and
        b_rew[t, i] += gamma V added as the per-step path adds it."""
        from . import _lib as L
        env, pol, cfg = self.env, self.learner, self.cfg
        fu = pol.fused
        fu.sync_weights()                       # the planes the loop reads (the loop itself does not refresh them)

        def rollout():
            for t in range(self.T):
                self._rollout_step(fu, t)
        self._rollout_phase.run(self.rollout_graph, fu, rollout)
        # deferred bootstrap of truncated episodes
        D = env.obs_dim
        idx = (self.b_done.reshape(-1) == L.DN_DONE_TRUNCATED).nonzero().squeeze(1)
        if idx.numel():
            rows = self.b_term.reshape(-1, D).index_select(0, idx)
            tv = torch.cat([fu.forward(rows[i:i + fu.max_rows])[1] for i in range(0, rows.shape[0], fu.max_rows)])
            rew = self.b_rew.view(-1)
            rew[idx] += cfg.gamma * tv
        self.truncated_steps = int(idx.numel())
        last_values = fu.forward(self.obs)[1]
        adv, ret = compute_gae(self.b_rew, self.b_val, self.b_done, last_values, cfg.gamma, cfg.gae_lambda)
        self.total_steps += self.T * env.num_envs * _world()
        return adv, ret

    def train_iteration(self) -> Dict[str, float]:
        t0 = time.perf_counter()
        sync = (lambda: torch.cuda.synchronize(self.dev)) if torch.device(self.dev).type == "cuda" else (lambda: None)
        adv, ret = self.collect_rollouts()
        sync()
        t1 = time.perf_counter()
        N, D = self.env.num_envs, self.env.obs_dim
        out = self.learner.update(self.b_obs.reshape(-1, D), self.b_act.reshape(-1, 4), self.b_logp.reshape(-1),
                                  self.b_val.reshape(-1), adv.reshape(-1), ret.reshape(-1), generator=self.gen)
        sync()
        t2 = time.perf_counter()
        out.update(rollout_s=t1 - t0, update_s=t2 - t1, samples=self.T * N * _world(),
                   sps=self.T * N * _world() / (t2 - t0))
        return out
