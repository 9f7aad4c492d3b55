"""FP64 reference of one PPO minibatch and of one clip_grad_norm_ + Adam step, for the tests of the fused update.

Restates SB3's ``PPO.train`` minibatch body (sb3_ppo.py:213-294) from the flat parameter vector alone, in float64, with plain
torch ops and autograd: the two tanh MLPs of ``ActorCriticPolicy`` (separate pi / vf networks), the diagonal Gaussian
log-prob and entropy, advantage normalisation (unbiased std, + 1e-8), the clipped surrogate, the clipped (or unclipped) value
loss, approx-KL and the clip fraction.  It shares no code with ``PPOLearner`` / ``ActorCritic``: a reference that reused them
would share their mistakes.  ``tests/test_ppo_fp64_reference_cpu.py`` pins it against the FP32 torch learner without a GPU.

It also builds rollouts with branch margins: every sample's probability ratio lies more than ``delta`` (relative) away from
``1 +- clip_range`` and its value change more than ``delta`` away from ``+- clip_range_vf``, so an implementation whose error is
far below ``delta`` takes every clipping branch the reference takes, and the comparisons need no slack for flipped samples.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

HALF_LOG_2PI = 0.5 * math.log(2.0 * math.pi)


@dataclass
class Spec:
    """The shapes of the policy: observation / action widths and the hidden widths of both networks."""
    obs_dim: int
    act_dim: int
    pi_arch: Tuple[int, ...]
    vf_arch: Tuple[int, ...]


def layout(spec: Spec) -> List[Tuple[str, Tuple[int, ...]]]:
    """(name, shape) of every parameter tensor in the order of the flat vector (the policy module's named_parameters order):
    log_std, then the Linear layers of pi, then of vf, under their nn.Sequential indices (0, 2, 4, ... with Tanh in between)."""
    out = [("log_std", (spec.act_dim,))]
    for net, arch, out_dim in (("pi", spec.pi_arch, spec.act_dim), ("vf", spec.vf_arch, 1)):
        sizes = (spec.obs_dim,) + tuple(arch) + (out_dim,)
        for l in range(len(sizes) - 1):
            out += [(f"{net}.{2 * l}.weight", (sizes[l + 1], sizes[l])), (f"{net}.{2 * l}.bias", (sizes[l + 1],))]
    return out


def split(flat: torch.Tensor, spec: Spec) -> Dict[str, torch.Tensor]:
    """name -> view of `flat` (same order as layout())."""
    out, off = {}, 0
    for name, shape in layout(spec):
        k = math.prod(shape)
        out[name] = flat[off:off + k].view(shape)
        off += k
    assert off == flat.numel(), (off, flat.numel())
    return out


def _mlp(x, p, net, depth):
    """tanh MLP; returns (output, hidden activations h_1..h_L, pre-activations z_1..z_L and the output)."""
    hs, zs = [], []
    h = x
    for l in range(depth + 1):
        z = h @ p[f"{net}.{2 * l}.weight"].t() + p[f"{net}.{2 * l}.bias"]
        if z.requires_grad:
            z.retain_grad()
        zs.append(z)
        if l < depth:
            h = torch.tanh(z)
            hs.append(h)
    return zs[-1], hs, zs


def _log_prob(mean, log_std, actions):
    return (-(actions - mean) ** 2 / (2.0 * torch.exp(2.0 * log_std)) - log_std - HALF_LOG_2PI).sum(-1)


@torch.no_grad()
def policy(flat: torch.Tensor, spec: Spec, obs: torch.Tensor):
    """(mean [n, act_dim], value [n]) in FP64."""
    p = split(flat.double(), spec)
    x = obs.double()
    mean, _, _ = _mlp(x, p, "pi", len(spec.pi_arch))
    value, _, _ = _mlp(x, p, "vf", len(spec.vf_arch))
    return mean, value.squeeze(-1)


def minibatch(flat: torch.Tensor, spec: Spec, batch: Sequence[torch.Tensor], clip_range: float, clip_range_vf: Optional[float],
              normalize_advantage: bool, ent_coef: float, vf_coef: float) -> dict:
    """One minibatch of PPO.train in FP64.  `batch` = (obs, actions, old_log_prob, old_values, advantages, returns) rows.
    Returns the hidden activations and pre-activation gradients of both networks (lists over layers 1..L), the flat gradient,
    the loss statistics with their per-sample terms, and the per-sample branch margins."""
    obs, actions, old_logp, old_values, adv, returns = [t.double() for t in batch]
    leaf = flat.detach().double().clone().requires_grad_(True)
    p = split(leaf, spec)
    mean, h_pi, z_pi = _mlp(obs, p, "pi", len(spec.pi_arch))
    value, h_vf, z_vf = _mlp(obs, p, "vf", len(spec.vf_arch))
    value = value.squeeze(-1)
    log_std = p["log_std"]
    logp = _log_prob(mean, log_std, actions)
    entropy = (0.5 + HALF_LOG_2PI + log_std).sum().expand(obs.shape[0])
    if normalize_advantage and adv.numel() > 1:
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    log_ratio = logp - old_logp
    ratio = torch.exp(log_ratio)
    pg_terms = -torch.min(adv * ratio, adv * torch.clamp(ratio, 1.0 - clip_range, 1.0 + clip_range))
    dv = value - old_values
    v_pred = value if clip_range_vf is None else old_values + torch.clamp(dv, -clip_range_vf, clip_range_vf)
    v_terms = (returns - v_pred) ** 2
    pg_loss, v_loss, ent_loss = pg_terms.mean(), v_terms.mean(), -entropy.mean()
    loss = pg_loss + ent_coef * ent_loss + vf_coef * v_loss
    loss.backward()
    with torch.no_grad():
        kl_terms = (ratio - 1.0) - log_ratio
        clipped = ((ratio - 1.0).abs() > clip_range)
        r_margin = torch.minimum((ratio / (1.0 - clip_range) - 1.0).abs(), (ratio / (1.0 + clip_range) - 1.0).abs())
        v_margin = (torch.full_like(dv, math.inf) if clip_range_vf is None
                    else torch.minimum((dv - clip_range_vf).abs(), (dv + clip_range_vf).abs()))
        # sum over the samples of the magnitudes of the per-sample contributions to every weight / bias gradient
        # (|dZ|^T |H| and sum |dZ|): the scale of the rounding error of a gradient that is a cancelling sum over the rows
        mag = split(torch.zeros_like(leaf.grad), spec)
        mag["log_std"].copy_(leaf.grad[:spec.act_dim].abs())
        for net, hs, zs in (("pi", h_pi, z_pi), ("vf", h_vf, z_vf)):
            for l, z in enumerate(zs):
                gz, a = z.grad.abs(), (obs if l == 0 else hs[l - 1]).abs()
                mag[f"{net}.{2 * l}.weight"].copy_(gz.t() @ a)
                mag[f"{net}.{2 * l}.bias"].copy_(gz.sum(0))
    L_pi, L_vf = len(spec.pi_arch), len(spec.vf_arch)
    return {
        "h_pi": [h.detach() for h in h_pi], "h_vf": [h.detach() for h in h_vf],
        "dz_pi": [z.grad for z in z_pi[:L_pi]], "dz_vf": [z.grad for z in z_vf[:L_vf]],
        "grad": leaf.grad.detach(), "grad_magnitude": torch.cat([t.reshape(-1) for t in mag.values()]),
        "stats": {"policy_gradient_loss": float(pg_loss.detach()), "value_loss": float(v_loss.detach()),
                  "approx_kl": float(kl_terms.mean()), "clip_fraction": float(clipped.double().mean())},
        # natural scale of each statistic: the mean magnitude of its per-sample terms (the policy-gradient loss is a mean of
        # terms of both signs and can be far smaller than they are)
        "stat_scale": {"policy_gradient_loss": float(pg_terms.detach().abs().mean()), "value_loss": float(v_terms.detach().mean()),
                       "approx_kl": float(kl_terms.abs().mean()), "clip_fraction": 1.0},
        "n_clipped": int(clipped.sum()),
        "ratio": ratio.detach(), "dv": dv.detach(), "ratio_margin": r_margin, "value_margin": v_margin,
        "mean": mean.detach(), "value": value.detach(),
    }


def clip_adam(grad_sum: torch.Tensor, params: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, step: float, *,
              lr: float, max_grad_norm: float, world_size: int = 1, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-5):
    """clip_grad_norm_ + one torch.optim.Adam step in FP64 from a GIVEN gradient and Adam state.  `grad_sum` is the bucket as the
    all-reduce leaves it (the sum over `world_size` ranks); the step sees the average.  `step` = optimiser steps taken before
    this one.  Returns (params, exp_avg, exp_avg_sq, norm of the averaged gradient)."""
    g = grad_sum.double() / world_size
    norm = float(torch.linalg.vector_norm(g))
    g = g * min(max_grad_norm / (norm + 1e-6), 1.0)
    t = step + 1.0
    m = exp_avg.double() + (1.0 - beta1) * (g - exp_avg.double())          # exp_avg.lerp_(grad, 1 - beta1)
    v = beta2 * exp_avg_sq.double() + (1.0 - beta2) * g * g
    bc1, bc2 = 1.0 - beta1 ** t, 1.0 - beta2 ** t
    p = params.double() - (lr / bc1) * m / (torch.sqrt(v) / math.sqrt(bc2) + eps)
    return p, m, v, norm


# ---- rollouts with branch margins ------------------------------------------------------------------------------------------
def make_rollout(flat: torch.Tensor, spec: Spec, n: int, seed: int, device) -> List[torch.Tensor]:
    """FP32 rollout (obs, actions, old_log_prob, old_values, advantages, returns) whose old log-probs and values are those of
    the current policy plus noise (as if they came from an earlier policy), so that both clipping branches fire."""
    g = torch.Generator(device=device).manual_seed(seed)
    obs = torch.randn(n, spec.obs_dim, device=device, generator=g)
    mean, value = policy(flat, spec, obs)
    log_std = split(flat.double(), spec)["log_std"]
    act = mean + torch.randn(n, spec.act_dim, device=device, generator=g, dtype=torch.float64)
    logp = _log_prob(mean, log_std, act) + 0.3 * torch.randn(n, device=device, generator=g, dtype=torch.float64)
    v = value + 0.5 * torch.randn(n, device=device, generator=g, dtype=torch.float64)
    adv = torch.randn(n, device=device, generator=g) * 2 + 0.3
    ret = v + torch.randn(n, device=device, generator=g, dtype=torch.float64)
    return [obs, act.float(), logp.float(), v.float(), adv, ret.float()]


def _push(x, boundary, delta):
    """x moved to boundary * (1 +- 2 delta) on its own side of the boundary (ratios: relative distance)."""
    side = torch.where(x >= boundary, 1.0, -1.0).to(x.dtype)
    return boundary * (1.0 + 2.0 * delta * side)


@torch.no_grad()
def enforce_margins(flat: torch.Tensor, spec: Spec, rollout: List[torch.Tensor], idx: torch.Tensor, clip_range: float,
                    clip_range_vf: Optional[float], delta: float, min_side: float = 0.1) -> dict:
    """Moves, in place, the old_log_prob / old_value of every sample of rows `idx` whose margin under the parameters `flat` is
    below `delta`: the ratio within `delta` (relative) of 1 +- clip_range, or value - old_value within `delta` of
    +- clip_range_vf.  Asserts afterwards (with the stored FP32 values) that every margin exceeds `delta` and that at least
    `min_side` of the samples lie on each side of each clip boundary.  Returns counts for the test log."""
    obs, act, old_logp, old_v = rollout[0][idx], rollout[1][idx], rollout[2][idx].double(), rollout[3][idx].double()
    mean, value = policy(flat, spec, obs)
    logp = _log_prob(mean, split(flat.double(), spec)["log_std"], act.double())
    ratio = torch.exp(logp - old_logp)
    moved = 0
    for b in (1.0 - clip_range, 1.0 + clip_range):
        near = (ratio / b - 1.0).abs() <= delta
        moved += int(near.sum())
        ratio = torch.where(near, _push(ratio, b, delta), ratio)
    rollout[2][idx] = (logp - torch.log(ratio)).float()
    dv = value - old_v
    if clip_range_vf is not None:
        for b in (-clip_range_vf, clip_range_vf):
            near = (dv - b).abs() <= delta
            moved += int(near.sum())
            dv = torch.where(near, b + 2.0 * delta * torch.where(dv >= b, 1.0, -1.0).to(dv.dtype), dv)
        rollout[3][idx] = (value - dv).float()
    # re-check from the stored FP32 values
    ratio = torch.exp(logp - rollout[2][idx].double())
    r_margin = torch.minimum((ratio / (1.0 - clip_range) - 1.0).abs(), (ratio / (1.0 + clip_range) - 1.0).abs())
    assert float(r_margin.min()) > delta, float(r_margin.min())
    fr = {"ratio<lo": float((ratio < 1.0 - clip_range).double().mean()), "ratio>hi": float((ratio > 1.0 + clip_range).double().mean())}
    fr["ratio inside"] = 1.0 - fr["ratio<lo"] - fr["ratio>hi"]
    if clip_range_vf is not None:
        dv = value - rollout[3][idx].double()
        v_margin = torch.minimum((dv - clip_range_vf).abs(), (dv + clip_range_vf).abs())
        assert float(v_margin.min()) > delta, float(v_margin.min())
        fr["dv<-c"] = float((dv < -clip_range_vf).double().mean())
        fr["dv>c"] = float((dv > clip_range_vf).double().mean())
        fr["dv inside"] = 1.0 - fr["dv<-c"] - fr["dv>c"]
    assert min(fr.values()) >= min_side, fr        # otherwise a clipped branch would go untested
    return {"moved": moved, **fr}


# ---- comparisons ---------------------------------------------------------------------------------------------------------
def net_of(name: str) -> str:
    """log_std belongs to the policy network."""
    return "vf" if name.startswith("vf.") else "pi"


def per_tensor_errors(got: torch.Tensor, ref: torch.Tensor, spec: Spec, scale: Optional[torch.Tensor] = None, floor: float = 1e-3):
    """max |got - ref| / denominator, per parameter tensor of the flat vectors.  The denominator is max |ref| of the tensor, or,
    with `scale` (a flat vector of the same layout), max |scale| of the tensor -- e.g. the sum of the magnitudes of the
    per-sample contributions, the natural scale of the rounding error of a cancelling sum.  Either is floored at `floor` x the
    largest |ref| entry of the tensor's network, so that small or cancelling tensors (the log_std gradient = data term - ent_coef,
    the action-head bias) do not turn an error that is tiny on the network's scale into a large relative one.  Returns
    ({name: error}, [names whose denominator was the floor])."""
    got, ref = got.double(), ref.double()
    sg, sr = split(got, spec), split(ref, spec)
    ss = sr if scale is None else split(scale.double(), spec)
    net_max = {"pi": 0.0, "vf": 0.0}
    for name in sr:
        net_max[net_of(name)] = max(net_max[net_of(name)], float(sr[name].abs().max()))
    errs, floored = {}, []
    for name in sr:
        own, fl = float(ss[name].abs().max()), floor * net_max[net_of(name)]
        if own < fl:
            floored.append(name)
        errs[name] = float((sg[name] - sr[name]).abs().max()) / max(own, fl, 1e-300)
    return errs, floored


def max_rel(got: torch.Tensor, ref: torch.Tensor) -> float:
    """max-norm relative error max |got - ref| / max |ref|."""
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max()) / max(float(ref.abs().max()), 1e-300)


def half_ulp(x: torch.Tensor) -> torch.Tensor:
    """half a unit in the last place of every FP32 value of x (as float64)."""
    a = x.float().abs()
    return 0.5 * (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()
