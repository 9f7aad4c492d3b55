"""The FP64 reference of the PPO minibatch (tests/ppo_fp64_reference.py) against the FP32 torch learner on the CPU, so that the
GPU tests of the fused update rest on a reference that has been checked without a GPU.

Rollouts carry branch margins (every ratio more than 1e-3 relative from 1 +- clip_range, every value change more than 1e-3 from
+- clip_range_vf), so FP32 and FP64 take the same clipping branches and the bounds need no slack for flipped samples:
  * loss statistics and every gradient tensor within 1e-5 (relative; FP32 rounding over sums of <= 512 terms is ~1e-6);
  * one clip_grad_norm_ + Adam step fed the torch learner's OWN gradient and state, in two parts: the clipped gradient within
    1e-5 (the learner's FP32 norm of the bucket, accumulated sequentially on the CPU, is good to ~2e-6 and scales every
    element), then Adam from the learner's clipped gradient: parameters within 1e-6 lr + half an ulp (the FP32 step is a
    few roundings of a quantity of size <= lr, the result is rounded to FP32 once), moments within 1e-6.
"""
import math

import pytest
import torch

from tests import ppo_fp64_reference as R

CASES = {
    "base": dict(obs=13, act=4, pi=(256, 128), vf=(256, 128), kw=dict(max_grad_norm=0.2)),
    "obs12": dict(obs=12, act=4, pi=(128, 128), vf=(128, 128), kw={}),
    "act1": dict(obs=13, act=1, pi=(128, 64), vf=(128, 64), kw={}),
    "act3": dict(obs=13, act=3, pi=(64, 64), vf=(64, 64), kw={}),
    "unequal": dict(obs=13, act=4, pi=(128, 64), vf=(256, 128, 64), kw={}),
    "options": dict(obs=13, act=4, pi=(128, 64), vf=(128, 64),
                    kw=dict(clip_range_vf=None, normalize_advantage=False, ent_coef=0.0, max_grad_norm=1e9)),
}
B, N, DELTA = 512, 2048, 1e-3


def _state(L, key):
    """Adam state `key` of every parameter, flat, in parameter order (zeros before the first step)."""
    return torch.cat([L.opt.state[p][key].reshape(-1) if p in L.opt.state else torch.zeros(p.numel()) for p in L.params])


@pytest.mark.parametrize("case", list(CASES))
def test_fp64_reference_matches_the_fp32_torch_learner(case):
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    c = CASES[case]
    cfg = PPOConfig(pi_arch=c["pi"], vf_arch=c["vf"], batch_size=B, target_kl=None, update_impl="torch", cuda_graph=False, **c["kw"])
    L = PPOLearner(c["obs"], c["act"], cfg, device="cpu")
    spec = R.Spec(c["obs"], c["act"], c["pi"], c["vf"])
    assert [(n, tuple(p.shape)) for n, p in L.policy.named_parameters()] == R.layout(spec)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():                         # non-zero biases and log_std (the initial ones are all zero)
        for p in L.params:
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    ro = R.make_rollout(L.flat_parameters(), spec, N, seed=7, device="cpu")
    for k in range(3):                            # t = 1, 2, 3: the bias corrections of Adam's first steps
        flat = L.flat_parameters()
        idx = torch.randperm(N, generator=g)[:B]
        info = R.enforce_margins(flat, spec, ro, idx, cfg.clip_range, cfg.clip_range_vf, DELTA)
        ref = R.minibatch(flat, spec, [t[idx] for t in ro], cfg.clip_range, cfg.clip_range_vf, cfg.normalize_advantage,
                          cfg.ent_coef, cfg.vf_coef)
        acc = torch.zeros(5)
        L._forward_backward(*[t[idx] for t in ro], acc)
        got = dict(zip(("policy_gradient_loss", "value_loss", "entropy_loss", "approx_kl", "clip_fraction"), acc.tolist()))
        stat_err = {s: abs(got[s] - ref["stats"][s]) / max(abs(ref["stats"][s]), ref["stat_scale"][s]) for s in ref["stats"]}
        errs, floored = R.per_tensor_errors(L._flat, ref["grad"], spec)
        print(case, k, info, "stats", {s: f"{e:.1e}" for s, e in stat_err.items()}, "grad", f"{max(errs.values()):.1e}",
              "floored", floored)
        assert max(stat_err.values()) <= 1e-5, stat_err
        assert got["clip_fraction"] * B == ref["n_clipped"]
        assert max(errs.values()) <= 1e-5, errs
        # one clip + Adam step from the learner's own gradient and state
        grad, p0 = L._flat.clone(), L.flat_parameters()
        m0, v0 = _state(L, "exp_avg"), _state(L, "exp_avg_sq")
        step = float(L.opt.state[L.params[0]]["step"]) if L.params[0] in L.opt.state else 0.0
        assert step == k
        _, _, _, norm = R.clip_adam(grad, p0, m0, v0, step, lr=cfg.learning_rate, max_grad_norm=cfg.max_grad_norm, eps=cfg.adam_eps)
        if case in ("base", "options"):          # clip_grad_norm_ active in "base", inactive in "options"
            assert (norm > cfg.max_grad_norm) == (case == "base"), norm
        L._clip_and_step()
        # (a) the clip (torch scales the bucket in place): the learner's FP32 norm of ~1e5 squares is good to ~2e-6
        clipped = L._flat.clone()
        clip_err = R.max_rel(clipped, grad.double() * min(cfg.max_grad_norm / (norm + 1e-6), 1.0))
        assert clip_err <= 1e-5, clip_err
        # (b) Adam on the learner's clipped gradient
        p_ref, m_ref, v_ref, _ = R.clip_adam(clipped, p0, m0, v0, step, lr=cfg.learning_rate, max_grad_norm=math.inf,
                                             eps=cfg.adam_eps)
        p1 = L.flat_parameters()
        excess = float(((p1.double() - p_ref).abs() - R.half_ulp(p1)).max())
        m_err, v_err = R.max_rel(_state(L, "exp_avg"), m_ref), R.max_rel(_state(L, "exp_avg_sq"), v_ref)
        print(f"   clip {clip_err:.1e} (norm {norm:.3f}), adam: max |dp| - ulp/2 = {excess / cfg.learning_rate:.1e} lr, "
              f"moments {m_err:.1e} {v_err:.1e}")
        assert excess <= 1e-6 * cfg.learning_rate
        assert m_err <= 1e-6 and v_err <= 1e-6


def test_margins_hold_and_both_branches_fire():
    """The rollout helper moves near-boundary samples off the boundaries and leaves >= 10 % on each side of each boundary."""
    spec = R.Spec(13, 4, (64,), (64,))
    g = torch.Generator().manual_seed(1)
    flat = 0.1 * torch.randn(sum(torch.Size(s).numel() for _, s in R.layout(spec)), generator=g)
    ro = R.make_rollout(flat, spec, 4096, seed=3, device="cpu")
    idx = torch.arange(4096)
    info = R.enforce_margins(flat, spec, ro, idx, 0.2, 0.3, 1e-2)
    assert info["moved"] > 0, info              # delta = 1e-2 catches samples near the boundaries: they were moved
    ref = R.minibatch(flat, spec, [t[idx] for t in ro], 0.2, 0.3, True, 0.02, 0.5)
    assert float(ref["ratio_margin"].min()) > 1e-2 and float(ref["value_margin"].min()) > 1e-2
