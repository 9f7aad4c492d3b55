"""dn_ppo_act (include/dnppo.h) and the fused rollout of PPOTrainer on the GPU: the sampler against its FP64 restatement
(tests/ppo_act_reference.py), shard invariance, the ratio of a fresh rollout, the rollout against a launch-by-launch replay
with the per-step truncation bootstrap, graph replay against launch by launch, and training."""
import numpy as np
import pytest
import torch

from tests import ppo_act_reference as R

pytestmark = pytest.mark.gpu

LOG_STD = [-0.7, 0.4, 0.0, -1.6]


def _learner(act_dim, arch=(256, 128)):
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    L = PPOLearner(13, act_dim, PPOConfig(pi_arch=arch, vf_arch=arch, update_impl="fused"), device="cuda")
    fu = L.ensure_fused(4096)
    with torch.no_grad():
        L.policy.log_std.copy_(torch.tensor(LOG_STD[:act_dim]))
        for p in L.policy.pi[-1].parameters():        # means of order 1 (the initial head gives ~0.01)
            p.mul_(60.0)
    fu.sync_weights()
    return L, fu


def _sample(counter, seed=77, offset=0, deterministic=0, low=-1.0, high=1.0):
    from drl_dronenavigation_b200 import _lib
    s = _lib.dn_ppo_sample()
    s.seed, s.row_id_offset, s.counter, s.deterministic, s.low, s.high = seed, offset, counter.data_ptr() if counter is not None else None, \
        deterministic, low, high
    return s


@pytest.mark.parametrize("act_dim", [1, 3, 4])
@pytest.mark.parametrize("rows", [1000, 4096])
def test_sampler_matches_the_fp64_restatement(act_dim, rows):
    L, fu = _learner(act_dim)
    g = torch.Generator(device="cuda").manual_seed(act_dim)
    obs = torch.randn(rows, 13, device="cuda", generator=g) * 2
    mean, value = fu.forward(obs)
    ls = np.array(LOG_STD[:act_dim], dtype=np.float32)
    seed, offset = 0x1234_5678_9ABC, 3 * 10 ** 9                       # row ids above 2^32
    counter = torch.full((1,), 5, dtype=torch.int64, device="cuda")
    # deterministic: action = mean, value, both bit-identical to dn_ppo_forward; the counter is not touched
    a, c, lp, v = fu.act(obs, _sample(None, seed, offset, deterministic=1))
    assert torch.equal(a, mean) and torch.equal(v, value)
    assert torch.equal(c, mean.clamp(-1.0, 1.0))
    np.testing.assert_allclose(lp.cpu().numpy(), R.log_prob(mean.cpu().numpy(), mean.cpu().numpy(), ls), rtol=0, atol=1e-5)
    assert int(counter.item()) == 5
    worst_z = worst_lp = 0.0
    m64 = mean.double().cpu().numpy()
    for k in range(4):
        a, c, lp, v = fu.act(obs, _sample(counter, seed, offset))
        assert int(counter.item()) == 6 + k                           # exactly one draw per stochastic call
        assert torch.equal(v, value)
        assert torch.equal(c, a.clamp(-1.0, 1.0))                      # clipped action = clamp(action), exactly
        a64 = a.double().cpu().numpy()
        z_ref = R.normals(seed, 5 + k, offset + np.arange(rows), act_dim)
        std = np.exp(ls.astype(np.float64))
        z_dev = (a64 - m64) / std
        # FP32 logf / sqrtf / sincospif / fmaf: a few ulp of |z|, plus the rounding of the stored action (ulp(|action|) / std)
        err = np.abs(z_dev - z_ref)
        bound = 4e-6 * np.maximum(1.0, np.abs(z_ref)) + np.abs(a64) * 2.0 ** -23 / std
        assert (err <= bound).all(), float((err / bound).max())
        worst_z = max(worst_z, float((err / np.maximum(1.0, np.abs(z_ref))).max()))
        # log-prob: FP64 of the kernel's own action and mean; FP32 sums of act_dim terms
        terms = 0.5 * (a64 - m64) ** 2 * np.exp(-2.0 * ls.astype(np.float64)) + np.abs(ls) + 0.92
        lp_ref = R.log_prob(a64, m64, ls)
        lerr = np.abs(lp.double().cpu().numpy() - lp_ref)
        assert (lerr <= 8 * 2.0 ** -23 * terms.sum(-1) + 1e-7).all(), float(lerr.max())
        worst_lp = max(worst_lp, float(lerr.max()))
        assert (a.abs() > 1).any()                                     # the clamp was exercised
    print(f"act_dim {act_dim}, {rows} rows: max |z - z_fp64| / max(1, |z|) = {worst_z:.2e}, max |log_prob - fp64| = {worst_lp:.2e}")


def test_two_shards_draw_what_one_call_draws():
    L, fu = _learner(4)
    N = 512
    obs = torch.randn(2 * N, 13, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    c1 = torch.full((1,), 11, dtype=torch.int64, device="cuda")
    whole = fu.act(obs, _sample(c1, offset=0))
    c2 = torch.full((1,), 11, dtype=torch.int64, device="cuda")
    lo = fu.act(obs[:N].contiguous(), _sample(c2, offset=0))
    c2.fill_(11)
    hi = fu.act(obs[N:].contiguous(), _sample(c2, offset=N))
    for w, p, q in zip(whole, lo, hi):
        assert torch.equal(w, torch.cat([p, q]))
    assert int(c1.item()) == int(c2.item()) == 12


def test_a_rollout_drawn_by_the_sampler_starts_the_update_at_ratio_one():
    L, fu = _learner(4, arch=(512, 512, 256))
    B, mb = 4096, 1024
    g = torch.Generator(device="cuda").manual_seed(8)
    obs = torch.randn(B, 13, device="cuda", generator=g)
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    act, _, logp, val = fu.act(obs, _sample(counter))
    adv = torch.randn(B, device="cuda", generator=g)
    ret = val + torch.randn(B, device="cuda", generator=g)
    keep = [t.contiguous() for t in (obs, act, logp, val, adv, ret)]
    ro = fu.L.dn_ppo_rollout()
    ro.obs, ro.actions, ro.old_log_prob, ro.old_values, ro.advantages, ro.returns = [t.data_ptr() for t in keep]
    fu.begin_update()
    fu.minibatch_grad(ro, torch.randperm(B, device="cuda", generator=g)[:mb].contiguous())
    st = fu.stats()
    print(f"first minibatch on a sampled rollout: approx_kl = {st.approx_kl:.2e}, clip_fraction = {st.clip_fraction}")
    assert st.clip_fraction == 0.0 and abs(st.approx_kl) <= 1e-7


def _env(N, max_steps):
    import bench
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    targets, init, dim, is_circle = bench.track_setup("circle")
    return BatchedDroneEnv(N, targets, max_steps=max_steps, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                           include_distance=True, normalize_actions=True, normalize_obs=True, device="cuda:0")


def _trainer(N, T, max_steps, **kw):
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    cfg = PPOConfig(n_steps=T, batch_size=2048, n_epochs=2, rollout_impl="fused", update_impl="fused", **kw)
    return PPOTrainer(_env(N, max_steps), cfg, rollout_steps=T)


def _rollout_state(tr, adv, ret):
    return {k: getattr(tr, k).clone() for k in ("b_obs", "b_act", "b_clip", "b_logp", "b_val", "b_rew", "b_done", "draw_counter", "obs")} | \
        {"adv": adv.clone(), "ret": ret.clone()}


def test_fused_rollout_equals_a_launch_by_launch_replay_with_the_per_step_bootstrap():
    """Rollout 1 is launched step by step, rollout 2 is the captured graph's first replay.  A fresh env of the same configuration
    is stepped with their recorded clipped actions, one launch at a time, and bootstrapped the old way: dn_ppo_forward on the
    truncated rows' terminal observations after every step.  Everything the trainer recorded must match bit for bit."""
    from drl_dronenavigation_b200 import _lib as L
    from drl_dronenavigation_b200.ppo import compute_gae
    N, T, max_steps = 1024, 40, 8
    tr = _trainer(N, T, max_steps)
    fu, gamma = tr.learner.fused, tr.cfg.gamma
    runs = [_rollout_state(tr, *tr.collect_rollouts())]
    assert tr._rollout_graph is None
    runs.append(_rollout_state(tr, *tr.collect_rollouts()))
    assert tr._rollout_graph is not None
    env = _env(N, max_steps)
    obs = env.reset().clone()
    for k, run in enumerate(runs):
        n_trunc = int((run["b_done"] == L.DN_DONE_TRUNCATED).sum())
        print(f"rollout {k + 1}: {n_trunc} truncated env-steps of {T * N} ({100.0 * n_trunc / (T * N):.1f} %)")
        assert n_trunc >= 0.01 * T * N
        assert int(run["draw_counter"].item()) == (k + 1) * T
        rew = torch.empty(T, N, device="cuda")
        val = torch.empty(T, N, device="cuda")
        for t in range(T):
            assert torch.equal(run["b_obs"][t], obs), (k, t)
            assert torch.equal(run["b_clip"][t], run["b_act"][t].clamp(-1.0, 1.0))
            val[t] = fu.forward(obs)[1]
            o, r, d, _ = env.step(run["b_clip"][t].contiguous())
            rew[t] = r
            trunc = d == L.DN_DONE_TRUNCATED
            if bool(trunc.any()):
                tv = fu.forward(env.terminal_obs[trunc])[1]
                rew[t][trunc] += gamma * tv
            assert torch.equal(run["b_done"][t], d), (k, t)
            obs = o.clone()
        assert torch.equal(run["b_val"], val)
        assert torch.equal(run["b_rew"], rew)
        assert torch.equal(run["obs"], obs)
        adv, ret = compute_gae(rew, val, run["b_done"], fu.forward(obs)[1], gamma, tr.cfg.gae_lambda)
        assert torch.equal(run["adv"], adv) and torch.equal(run["ret"], ret)
    env.close()
    tr.env.close()


def test_graph_replay_equals_launch_by_launch():
    """Three rollouts each: the first launched step by step in both trainers, then graph capture + replays against launches."""
    N, T = 512, 24
    out = {}
    for graph in (False, True):
        tr = _trainer(N, T, 8)
        tr.rollout_graph = graph
        out[graph] = [_rollout_state(tr, *tr.collect_rollouts()) for _ in range(3)]
        assert (tr._rollout_graph is not None) == graph
        tr.env.close()
    for a, b in zip(out[False], out[True]):
        for k in a:
            assert torch.equal(a[k], b[k]), k
    assert int(out[True][-1]["draw_counter"].item()) == 3 * T


def test_trainer_with_the_fused_rollout_learns_to_reduce_value_loss():
    import bench
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    targets, init, dim, is_circle = bench.track_setup("circle")
    env = BatchedDroneEnv(2048, targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                          include_distance=True, normalize_actions=True)
    tr = PPOTrainer(env, PPOConfig(batch_size=4096, n_epochs=4, rollout_impl="fused"), rollout_steps=16)
    assert tr.learner.fused is not None
    outs = [tr.train_iteration() for _ in range(4)]
    assert all(o["impl"].startswith("fused") for o in outs)
    assert tr._rollout_graph is not None and int(tr.draw_counter.item()) == 4 * 16
    assert np.isfinite([o["value_loss"] for o in outs]).all() and outs[-1]["value_loss"] < outs[0]["value_loss"]
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible GPUs")
def test_handles_on_two_devices_of_one_process_compute_the_same():
    """A PPO handle and a SAC actor on device 1, then on device 0, from the same parameters; dn_ppo_forward and dn_sac_act
    (deterministic) run on device 1 first.  What a handle sets up for its kernels (the contraction's shared-memory limit, the
    SM count that sizes its grids) belongs to its own device, so device 0 runs too and gives the same bits."""
    from drl_dronenavigation_b200 import _lib
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    from drl_dronenavigation_b200.sac import SACConfig, SACLearner
    learners = {}
    for d in (1, 0):
        ppo = PPOLearner(13, 4, PPOConfig(pi_arch=(256, 128), vf_arch=(256, 128), update_impl="fused"), device=f"cuda:{d}")
        sac = SACLearner(13, 4, SACConfig(pi_arch=(256, 256), rollout_impl="fused"), device=f"cuda:{d}")
        if d == 0:
            with torch.no_grad():
                for a, b in zip(list(ppo.policy.parameters()) + list(sac.actor.parameters()),
                                list(learners[1][0].policy.parameters()) + list(learners[1][1].actor.parameters())):
                    a.copy_(b.to(a.device))
        learners[d] = (ppo, sac, ppo.ensure_fused(4096), sac.ensure_fused_actor(4096))
    obs = torch.randn(1000, 13, generator=torch.Generator().manual_seed(5)) * 2
    s = _lib.dn_sac_sample()
    s.seed, s.row_id_offset, s.counter, s.mode = 77, 0, None, _lib.DN_SAC_DETERMINISTIC
    out = {}
    for d in (1, 0):
        _, _, fu, fa = learners[d]
        o = obs.to(f"cuda:{d}")
        mean, value = fu.forward(o)
        out[d] = [t.cpu() for t in (mean, value, fa.act(o, s))]
    for a, b in zip(out[1], out[0]):
        assert torch.equal(a, b)
    assert out[0][2].abs().max() > 0
