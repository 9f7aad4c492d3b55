"""The fused PPO minibatch update (include/dnppo.h: tcgen05 contractions + hand-written head / loss / Adam kernels)
against the plain PyTorch FP32 path of the same learner (autograd + torch.optim.Adam, cuBLAS FP32, no TF32): loss
statistics, every gradient, the post-Adam parameters, the KL early stop and whole multi-epoch updates."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _cc10():
    return torch.cuda.is_available() and torch.cuda.get_device_capability()[0] == 10


def make_rollout(L, B, seed):
    """A rollout whose old log-probs / values come from a perturbed copy of the policy, so ratios differ from 1, both
    clipping branches of the surrogate and of the value loss fire, and the gradients are not degenerate."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.randn(B, L.obs_dim, device="cuda", generator=g)
    with torch.no_grad():
        mean = L.policy.pi(obs)
        act = mean + torch.randn(B, L.act_dim, device="cuda", generator=g)
        v, logp, _ = L.policy.evaluate(obs, act)
        logp = logp + 0.3 * torch.randn(B, device="cuda", generator=g)
        v = v + 0.5 * torch.randn(B, device="cuda", generator=g)
    adv = torch.randn(B, device="cuda", generator=g) * 2 + 0.3
    ret = v + torch.randn(B, device="cuda", generator=g)
    return obs, act, logp, v, adv, ret


def pair(arch, batch, **kw):
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    base = dict(pi_arch=arch, vf_arch=arch, batch_size=batch, cuda_graph=False, matmul_precision="fp32")
    base.update(kw)
    ref = PPOLearner(13, 4, PPOConfig(update_impl="torch", **base), device="cuda")
    fus = PPOLearner(13, 4, PPOConfig(update_impl="fused", **base), device="cuda")
    # non-trivial biases and log_std (the initial ones are all zero), identical in both
    g = torch.Generator(device="cuda").manual_seed(5)
    with torch.no_grad():
        for pr, pf in zip(ref.policy.parameters(), fus.policy.parameters()):
            if pr.dim() == 1:
                pr.add_(0.1 * torch.randn(pr.shape, device="cuda", generator=g))
            pf.copy_(pr)
    return ref, fus


def per_tensor_rel(L, a, b):
    """max |a - b| / max |b| for every parameter tensor of the flat vectors a, b."""
    out, off = {}, 0
    for name, p in L.policy.named_parameters():
        k = p.numel()
        out[name] = float((a[off:off + k] - b[off:off + k]).abs().max() / b[off:off + k].abs().max().clamp_min(1e-30))
        off += k
    return out


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
@pytest.mark.parametrize("arch,B", [((128,), 256), ((256, 128), 1024), ((512, 512, 256), 4096), ((512, 512, 256), 32768),
                                     ((512, 512, 256, 128), 2048)])
def test_one_minibatch_matches_fp32_torch(arch, B):
    """loss terms, every gradient and the post-Adam parameters within 1e-4 (relative, per tensor) of the FP32 path."""
    ref, fus = pair(arch, B)
    ro = make_rollout(ref, B, seed=B)
    idx = torch.randperm(B, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    # reference: forward + losses + backward
    acc = torch.zeros(5, device="cuda")
    kl = ref._forward_backward(*[t[idx] for t in ro], acc)
    g_ref = ref._flat.clone()
    # fused: same rows
    fu = fus.ensure_fused(B)
    # (a) forward activations, layer by layer
    from drl_dronenavigation_b200 import _lib as Lm
    r = Lm.dn_ppo_rollout()
    keep = [t.contiguous() for t in ro]
    r.obs, r.actions, r.old_log_prob, r.old_values, r.advantages, r.returns = [t.data_ptr() for t in keep]
    fu.begin_update()
    fu.minibatch_grad(r, idx)
    torch.cuda.synchronize()
    with torch.no_grad():
        h = ro[0][idx]
        for l, w in enumerate(arch):
            h = torch.tanh(torch.nn.functional.linear(h, ref.policy.pi[2 * l].weight, ref.policy.pi[2 * l].bias))
            got = fu.buffer(f"pi.h{l + 1}", B, w)
            assert float((got - h).abs().max()) < 5e-5, (l, float((got - h).abs().max()))     # |h| <= 1
    g_fus = fus._flat.clone()
    rel = per_tensor_rel(ref, g_fus, g_ref)
    print("gradient rel errors:", {k: f"{v:.1e}" for k, v in rel.items()})
    assert max(rel.values()) < 1e-4, rel
    st = fu.stats()
    a = acc.tolist()
    assert abs(st.policy_gradient_loss - a[0]) < 1e-4 * max(1.0, abs(a[0])) and abs(st.value_loss - a[1]) < 1e-4 * max(1.0, abs(a[1]))
    assert abs(st.approx_kl - a[3]) < 1e-4 * max(1.0, abs(a[3])) and abs(st.clip_fraction - a[4]) < 2e-3
    assert abs(st.last_approx_kl - float(kl)) < 1e-4 * max(1.0, abs(float(kl)))
    # optimiser step
    p0 = ref.flat_parameters().clone()
    ref.cfg.target_kl = None
    ref._clip_and_step()
    fus.cfg.target_kl = None
    fu.cfg_c.target_kl = -1.0
    # the vote was computed with the configured target_kl; force "continue" for this comparison
    fus._bucket[-1] = 0.0
    fu.minibatch_apply()
    torch.cuda.synchronize()
    p_ref, p_fus = ref.flat_parameters(), fus.flat_parameters()
    moved = (p_ref - p0).abs()
    rel_p = per_tensor_rel(ref, p_fus, p_ref)
    print("parameter rel errors:", {k: f"{v:.1e}" for k, v in rel_p.items()}, "mean step", float(moved.mean()))
    # Post-Adam parameters: within 1e-4 of the tensor's largest entry, plus half a percent of ONE learning-rate step.  Adam turns
    # a gradient g into a step lr * g / (|g| + eps) (first step); where |g| ~ eps = 1e-5 that map has a slope of lr / (4 eps), so
    # an absolute gradient error of 7e-8 (7e-6 of the tensor's largest gradient, the accuracy of the BF16 hi/lo products) moves
    # such a coordinate by ~0.2 % of lr = 4e-7 -- visible only in the action head, whose weights are ~1e-3 (orthogonal gain 0.01).
    lr = ref.cfg.learning_rate
    off = 0
    for name, p in ref.policy.named_parameters():
        k = p.numel()
        d = float((p_fus[off:off + k] - p_ref[off:off + k]).abs().max())
        assert d <= 1e-4 * float(p_ref[off:off + k].abs().max()) + 5e-3 * lr, (name, d, rel_p[name])
        off += k
    assert sum(v < 1e-4 for v in rel_p.values()) >= len(rel_p) - 1, rel_p
    # and the step itself (not just the parameter) agrees: the update of a coordinate is ~lr in size
    dstep = ((p_fus - p0) - (p_ref - p0)).abs()
    assert float(dstep.mean()) < 2e-2 * float(moved.mean()), (float(dstep.mean()), float(moved.mean()))
    # BF16 planes of the weights were refreshed from the new parameters
    w1 = fu.buffer("pi.w1", arch[0], 64)[:, :13]
    assert float((w1 - fus.policy.pi[0].weight.detach()).abs().max()) < 1e-5      # hi + lo planes carry ~17 mantissa bits


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
def test_forward_matches_torch_policy():
    ref, fus = pair((512, 512, 256), 1024)
    g = torch.Generator(device="cuda").manual_seed(11)
    for n in (1, 100, 128, 1000, 4096):
        obs = torch.randn(n, 13, device="cuda", generator=g)
        mean, value = fus.forward(obs)
        with torch.no_grad():
            m_ref, v_ref = ref.policy.pi(obs), ref.policy.value(obs)
        assert float((mean - m_ref).abs().max()) < 2e-5 and float((value - v_ref).abs().max()) < 5e-5, n
    a, logp, v = fus.act(obs, deterministic=True)
    assert torch.equal(a, mean) and logp.shape == (4096,) and torch.equal(v, value)


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
def test_kl_early_stop_leaves_parameters_untouched():
    """sb3_ppo.py:283-287: the minibatch whose approx_kl exceeds 1.5 target_kl is evaluated but not applied, and nothing after it."""
    ref, fus = pair((256, 128), 1024, n_epochs=4, target_kl=1e-6)
    ro = make_rollout(ref, 4096, seed=1)
    p0 = fus.flat_parameters().clone()
    out = fus.update(*ro, generator=torch.Generator(device="cuda").manual_seed(1))
    out_ref = ref.update(*ro, generator=torch.Generator(device="cuda").manual_seed(1))
    assert out["early_stop"] and out["minibatches"] == 1 and out["optimizer_steps"] == 0 and out["epochs"] == 1
    assert out_ref["early_stop"] and out_ref["minibatches"] == 1
    assert torch.equal(p0, fus.flat_parameters())
    assert abs(out["approx_kl"] - out_ref["approx_kl"]) < 1e-4 * max(1.0, abs(out_ref["approx_kl"]))
    # the next update starts clean
    fus.cfg.target_kl = None
    fus.fused.close(); fus.fused = None
    out2 = fus.update(*ro, generator=torch.Generator(device="cuda").manual_seed(2))
    assert not out2["early_stop"] and out2["minibatches"] == 16 and out2["optimizer_steps"] == 16
    assert not torch.equal(p0, fus.flat_parameters())


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
@pytest.mark.parametrize("precision,tol", [("bf16x3", 0.05), ("bf16", 0.6)])
def test_whole_update_tracks_fp32_torch(precision, tol):
    """Two updates of 3 epochs x 8 minibatches with the same minibatch order: the fused learner follows the FP32 torch learner
    (Adam amplifies rounding noise on near-zero-gradient coordinates to +-lr per step, so the comparison is in aggregate)."""
    ref, fus = pair((512, 512, 256), 1024, n_epochs=3, target_kl=None, mlp_precision=precision)
    ro = make_rollout(ref, 8192, seed=2)
    p0 = ref.flat_parameters().clone()
    for seed in (1, 2):
        o_ref = ref.update(*ro, generator=torch.Generator(device="cuda").manual_seed(seed))
        o_fus = fus.update(*ro, generator=torch.Generator(device="cuda").manual_seed(seed))
        assert o_fus["minibatches"] == o_ref["minibatches"] == 24 and o_fus["optimizer_steps"] == 24
        for k in ("policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction"):
            assert abs(o_fus[k] - o_ref[k]) < (2e-3 if precision == "bf16x3" else 5e-2) * max(1.0, abs(o_ref[k])), (k, o_fus[k], o_ref[k])
    d = (fus.flat_parameters() - ref.flat_parameters()).abs()
    moved = (ref.flat_parameters() - p0).abs()
    print(precision, "mean |diff|", float(d.mean()), "mean movement", float(moved.mean()), "max diff", float(d.max()))
    assert float(d.mean()) < tol * float(moved.mean())
    assert float(fus.fused.step) == 48.0


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
def test_trainer_uses_the_fused_update_and_learns_to_reduce_value_loss():
    import bench
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    targets, init, dim, is_circle = bench.track_setup("circle")
    env = BatchedDroneEnv(2048, targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                          include_distance=True, normalize_actions=True)
    tr = PPOTrainer(env, PPOConfig(batch_size=4096, n_epochs=4), rollout_steps=16)
    assert tr.learner.fused is not None
    outs = [tr.train_iteration() for _ in range(4)]
    assert all(o["impl"].startswith("fused") for o in outs)
    assert np.isfinite([o["value_loss"] for o in outs]).all() and outs[-1]["value_loss"] < outs[0]["value_loss"]
    env.close()


def _graph_replay_outputs(batch, rollout, presize):
    """Final parameters and the statistics of two updates, launch by launch and replayed from CUDA graphs, each followed by an
    update that stops at once.  `presize` > 0: the handle is first sized by a forward of that many rows."""
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    outs = {}
    for graph in (False, True):
        L = PPOLearner(13, 4, PPOConfig(batch_size=batch, n_epochs=3, target_kl=None, cuda_graph=graph, update_impl="fused"), device="cuda")
        ro = make_rollout(L, rollout, seed=4)
        if presize:
            L.forward(ro[0][:presize])
            assert L.fused.max_rows == presize
        r1 = L.update(*ro, generator=torch.Generator(device="cuda").manual_seed(1))
        if presize:
            assert L.fused.max_rows == presize                # the minibatches ran on the handle the forward sized
        ro2 = make_rollout(L, rollout, seed=5)
        r2 = L.update(*ro2, generator=torch.Generator(device="cuda").manual_seed(2))
        L.cfg.target_kl = 1e-7                       # third update: stops at once, nothing applied
        L.fused.close(); L.fused = None
        p_before = L.flat_parameters().clone()
        r3 = L.update(*ro2, generator=torch.Generator(device="cuda").manual_seed(3))
        assert r3["early_stop"] and r3["optimizer_steps"] == 0 and torch.equal(p_before, L.flat_parameters())
        outs[graph] = (L.flat_parameters().clone(), r1, r2)
    return outs


def _assert_bit_identical(outs):
    assert torch.equal(outs[False][0], outs[True][0])
    for k in ("policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction", "minibatches", "optimizer_steps"):
        assert outs[False][1][k] == outs[True][1][k] and outs[False][2][k] == outs[True][2][k], k


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
def test_graph_replay_of_the_fused_step_is_bit_identical():
    """The fused minibatch step replayed from CUDA graphs (static rollout / index buffers) is the same computation as the
    launch-by-launch path: every kernel reduces in an order fixed by its geometry, so the parameters agree BIT FOR BIT, over two
    updates (Adam state carried across replays) and through a KL early stop."""
    _assert_bit_identical(_graph_replay_outputs(1024, 8192, 0))


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
def test_graph_replay_is_bit_identical_at_the_bench_line_shape():
    """As above on the handle the trainer builds for the bench line: sized by the rollout forward over 65 536 envs, then used for
    32 768-row minibatches (plans re-made for the smaller row count, tensor maps over the larger workspaces)."""
    _assert_bit_identical(_graph_replay_outputs(32768, 65536, 65536))
