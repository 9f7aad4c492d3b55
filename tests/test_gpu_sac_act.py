"""dn_sac_act (include/dnsac.h) and the fused collection of SACTrainer on the GPU: the ReLU forward contraction against
FP64, the actor's hidden layers / heads / sampler against an FP64 actor on the same parameters (tests/sac_act_reference.py),
uniform mode bit for bit, the draw counter, shard invariance, the fused collection against a launch-by-launch replay and
against itself launched, a checkpoint load between phases, and a short training run."""
import copy

import numpy as np
import pytest
import torch

from tests import sac_act_reference as R
from tests.test_gpu_mlp import join_planes, rel, run_gemm, split_planes

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24          # unit roundoff of FP32


@pytest.mark.parametrize("passes", [3, 1])
@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (256, 128, 64), (384, 256, 128), (1024, 512, 512), (4096, 256, 64), (2048, 512, 256)])
def test_relu_forward_contraction_matches_fp64(passes, M, N, K):
    """dn_mlp_gemm(kind 0, act 2): max(A W^T + b, 0), hi / lo planes, against FP64 on the same planes and (bf16x3) on the
    un-split FP32 operands -- the bounds of the tanh forward in test_gpu_mlp.py."""
    tol = {3: 3e-5, 1: 2e-2}
    g = torch.Generator(device="cuda").manual_seed(7 * M + N + K)
    x = torch.randn(M, K, device="cuda", generator=g)
    w = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    a, b = split_planes(x), split_planes(w)
    out = torch.zeros(2, M, N, dtype=torch.bfloat16, device="cuda")
    run_gemm(0, passes, M, N, K, 1, a, b, bias=bias, act=2, out=out)
    ref = (join_planes(a, passes) @ join_planes(b, passes).t() + bias.double()).clamp_min(0.0)
    got = join_planes(out, passes)
    assert (got >= 0).all() and ((ref == 0) == (got == 0)).float().mean() > 0.99
    assert rel(got, ref) < tol[passes], rel(got, ref)
    if passes == 3:
        ref32 = (x.double() @ w.double().t() + bias.double()).clamp_min(0.0)
        assert rel(got, ref32) < 3e-5, rel(got, ref32)
    print(f"relu fwd passes={passes} {M}x{N}x{K}: rel err {rel(got, ref):.2e}")


MAX_ROWS = 16384 + 128
ROWS = (1, 127, 129, 4096, 16384, MAX_ROWS)


def _learner(arch, act_dim, max_rows=MAX_ROWS, seed=3):
    """A fused-collection SACLearner whose heads give |mu| up to ~4 (tanh saturation) and log_std spread over [-3, 1]."""
    from drl_dronenavigation_b200.sac import SACConfig, SACLearner
    L = SACLearner(13, act_dim, SACConfig(pi_arch=arch, rollout_impl="fused", seed=seed), device="cuda")
    with torch.no_grad():
        L.actor.mu.weight.mul_(8.0)
        L.actor.mu.bias.copy_(torch.linspace(-1.0, 1.0, act_dim))
        L.actor.log_std.weight.mul_(2.0)
        L.actor.log_std.bias.copy_(torch.linspace(-2.0, 0.3, act_dim))
    fa = L.ensure_fused_actor(max_rows)
    fa.sync_weights()
    return L, fa


def _sample(counter, mode, seed=77, offset=0):
    from drl_dronenavigation_b200 import _lib
    s = _lib.dn_sac_sample()
    s.seed, s.row_id_offset, s.mode = seed, offset, mode
    s.counter = counter.data_ptr() if counter is not None else None
    return s


def _params(L):
    return {k: v.detach().double().cpu().numpy() for k, v in L.actor.state_dict().items()}


def _obs(rows, seed):
    return torch.randn(rows, 13, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)) * 2


# Bounds (deterministic mode).  Hidden layers: BF16x3 products carry ~2^-16 relative to |a||b| per term and the stored
# activation ~2^-17 relative (test_gpu_ppo_fp64.py's h bound, 5e-5 absolute for activations of order 1): 5e-5 max(1, |h|).
# Heads: FP32 dot products of the kernel's own activations, |mu - mu64(h_dev)| <= 2e-5 max(1, sum_j |w_j h_j|); end to end the
# hidden-layer error propagates through the head weights: + sum_j |w_j| hbound_j.
@pytest.mark.parametrize("act_dim", [1, 3, 4])
@pytest.mark.parametrize("arch", [(256, 256), (128,), (128, 256, 512, 384)])
def test_deterministic_actor_matches_fp64(arch, act_dim):
    from drl_dronenavigation_b200 import _lib
    L, fa = _learner(arch, act_dim)
    P = _params(L)
    worst = {"h": 0.0, "mu": 0.0, "ls": 0.0}
    for rows in ROWS:
        obs = _obs(rows, rows)
        act = fa.act(obs, _sample(None, _lib.DN_SAC_DETERMINISTIC), log_prob=(lp := torch.empty(rows, device="cuda")))
        hs, mu64, ls64, a64, lp64 = R.actor_forward(P, obs.double().cpu().numpy())
        for l, h64 in enumerate(hs, 1):
            hd = fa.buffer(f"h{l}", rows).double().cpu().numpy()
            err = np.abs(hd - h64)
            assert (err <= 5e-5 * np.maximum(1.0, np.abs(h64).max())).all(), (l, float(err.max()))
            worst["h"] = max(worst["h"], float(err.max() / max(1.0, np.abs(h64).max())))
        h_last = fa.buffer(f"h{len(arch)}", rows).double().cpu().numpy()
        mu_d = fa.buffer("mu", rows).double().cpu().numpy()
        ls_d = fa.buffer("log_std", rows).double().cpu().numpy()
        hb = 5e-5 * max(1.0, np.abs(hs[-1]).max())
        for name, dev, ref, w, b in (("mu", mu_d, mu64, P["mu.weight"], P["mu.bias"]), ("ls", ls_d, ls64, P["log_std.weight"], P["log_std.bias"])):
            own = h_last @ w.T + b
            if name == "ls":
                own = np.clip(own, -20.0, 2.0)
            mag = np.abs(h_last) @ np.abs(w).T
            assert (np.abs(dev - own) <= 2e-5 * np.maximum(1.0, mag)).all(), (name, float(np.abs(dev - own).max()))
            bound = 2e-5 * np.maximum(1.0, mag) + hb * np.abs(w).sum(1)
            assert (np.abs(dev - ref) <= bound).all(), (name, float(np.abs(dev - ref).max()))
            worst[name] = max(worst[name], float(np.abs(dev - ref).max()))
        # action = tanhf(mu): the mu error (tanh is 1-Lipschitz, slope 1 - a^2) plus two ulp of tanhf
        a = act.double().cpu().numpy()
        mu_bound = 2e-5 * np.maximum(1.0, np.abs(h_last) @ np.abs(P["mu.weight"]).T) + hb * np.abs(P["mu.weight"]).sum(1)
        assert (np.abs(a - a64) <= (1 - a64 ** 2) * mu_bound * 1.01 + 2.5e-7).all(), float(np.abs(a - a64).max())
        assert np.isfinite(lp.cpu().numpy()).all()
    print(f"arch {arch}, act_dim {act_dim}: max |h - fp64| / max(1, |h|) = {worst['h']:.2e}, max |mu - fp64| = {worst['mu']:.2e}, "
          f"max |log_std - fp64| = {worst['ls']:.2e}")


@pytest.mark.parametrize("act_dim", [1, 3, 4])
def test_sampler_matches_fp64_with_the_restated_noise(act_dim):
    """Sample mode against the FP64 squashed Gaussian on the FP64 actor, eps from the restatement.
    Action: the pre-activation g = mu + std eps is off by mu_err + |eps| std ls_err (the deterministic test's bounds) plus the
    sampler's FP32 arithmetic (eps from logf / sqrtf / sincospif: 4e-6 max(1, |eps|) as in test_gpu_ppo_act.py; expf, fmaf:
    4 ulp of |std eps| + |mu|); tanh maps that with slope 1 - a^2, and tanhf adds 2 ulp of 1.
    log_prob: per component the Gaussian term is off by |eps| deps + ls_err, the squash term by c(a) da with
    c = 2|a| / (1 - a^2 + 1e-6) plus the rounding of 1 - a^2 + 1e-6 (2.4e-7 absolute) over (1 - a^2 + 1e-6); FP32 sums: 8 ulp
    of the sum of magnitudes."""
    from drl_dronenavigation_b200 import _lib
    L, fa = _learner((256, 256), act_dim)
    P = _params(L)
    rows, seed, offset = 16384, 0x1234_5678_9ABC, 3 * 10 ** 9
    counter = torch.full((1,), 5, dtype=torch.int64, device="cuda")
    obs = _obs(rows, 11)
    hs, mu64, ls64, _, _ = R.actor_forward(P, obs.double().cpu().numpy())
    h_last = hs[-1]
    hb = 5e-5 * max(1.0, np.abs(h_last).max())
    mag = lambda w: 2e-5 * np.maximum(1.0, np.abs(h_last) @ np.abs(w).T) + hb * np.abs(w).sum(1)
    mu_b, ls_b = mag(P["mu.weight"]), mag(P["log_std.weight"])
    worst_a = worst_lp = 0.0
    lp = torch.empty(rows, device="cuda")
    for k in range(3):
        a = fa.act(obs, _sample(counter, _lib.DN_SAC_SAMPLE, seed, offset), log_prob=lp).double().cpu().numpy()
        assert int(counter.item()) == 6 + k
        eps = R.normals(seed, 5 + k, offset + np.arange(rows), act_dim)
        a64, lp64 = R.squash(mu64, ls64, eps)
        std = np.exp(ls64)
        dg = mu_b + np.abs(eps) * std * ls_b * 1.01 + std * 4e-6 * np.maximum(1.0, np.abs(eps)) + 4 * EPS32 * (np.abs(std * eps) + np.abs(mu64))
        da = (1 - a64 ** 2) * dg * 1.01 + 2.5e-7
        assert (np.abs(a - a64) <= da).all(), float((np.abs(a - a64) / da).max())
        worst_a = max(worst_a, float(np.abs(a - a64).max()))
        q = 1 - a64 ** 2 + 1e-6
        deps = 4e-6 * np.maximum(1.0, np.abs(eps))
        terms = 0.5 * eps ** 2 + np.abs(ls64) + 0.92 + np.abs(np.log(q))
        lb = (np.abs(eps) * deps + ls_b + 2 * np.abs(a64) / q * da + 2.4e-7 / q).sum(-1) + 8 * EPS32 * terms.sum(-1) + 1e-6
        lerr = np.abs(lp.double().cpu().numpy() - lp64)
        assert (lerr <= lb).all(), float((lerr / lb).max())
        worst_lp = max(worst_lp, float(lerr.max()))
    sat = float((np.abs(a64) > 0.999).mean())
    print(f"act_dim {act_dim}: max |a - fp64| = {worst_a:.2e}, max |log_prob - fp64| = {worst_lp:.2e}, |a| > 0.999 in {100 * sat:.1f} %")
    assert sat > 0.01                                         # the saturated regime, where the squash term is ill-conditioned, is exercised


def test_uniform_mode_is_bit_exact_and_the_counter_advances_per_drawing_call():
    from drl_dronenavigation_b200 import _lib
    L, fa = _learner((256, 256), 4, max_rows=4096)
    rows, seed, offset = 4000, 99, (1 << 32) - 7
    obs = _obs(rows, 1)
    counter = torch.full((1,), 2 ** 32 - 2, dtype=torch.int64, device="cuda")    # crosses the mod 2^32 wrap
    lp = torch.empty(rows, device="cuda")
    for k in range(3):
        a = fa.act(obs, _sample(counter, _lib.DN_SAC_UNIFORM, seed, offset), log_prob=lp)
        np.testing.assert_array_equal(a.cpu().numpy(), R.uniform_actions(seed, 2 ** 32 - 2 + k, offset + np.arange(rows), 4))
        assert torch.equal(lp, torch.full_like(lp, float(np.float32(-4 * np.log(2.0)))))
    assert int(counter.item()) == 2 ** 32 + 1
    # inside a graph: sample + uniform advance it, deterministic does not
    counter.zero_()
    out = torch.empty(rows, 4, device="cuda")
    fa.act(obs, _sample(counter, _lib.DN_SAC_SAMPLE), out)
    fa.act(obs, _sample(None, _lib.DN_SAC_DETERMINISTIC), out)
    assert int(counter.item()) == 1
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fa.act(obs, _sample(counter, _lib.DN_SAC_SAMPLE), out)
        fa.act(obs, _sample(counter, _lib.DN_SAC_UNIFORM), out)
        fa.act(obs, _sample(counter, _lib.DN_SAC_DETERMINISTIC), out)
    for r in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert int(counter.item()) == 1 + 3 * 2


def test_two_shards_draw_what_one_call_draws():
    from drl_dronenavigation_b200 import _lib
    L, fa = _learner((256, 256), 4, max_rows=1024)
    N = 512
    obs = _obs(2 * N, 3)
    for mode in (_lib.DN_SAC_SAMPLE, _lib.DN_SAC_UNIFORM):
        c1 = torch.full((1,), 11, dtype=torch.int64, device="cuda")
        l1 = torch.empty(2 * N, device="cuda")
        whole = fa.act(obs, _sample(c1, mode), log_prob=l1).clone()
        c2 = torch.full((1,), 11, dtype=torch.int64, device="cuda")
        la, lb = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
        lo = fa.act(obs[:N].contiguous(), _sample(c2, mode, offset=0), log_prob=la).clone()
        c2.fill_(11)
        hi = fa.act(obs[N:].contiguous(), _sample(c2, mode, offset=N), log_prob=lb).clone()
        assert torch.equal(whole, torch.cat([lo, hi])) and torch.equal(l1, torch.cat([la, lb]))
        assert int(c1.item()) == int(c2.item()) == 12


def _env(N, max_steps=8):
    import bench
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    targets, init, dim, is_circle = bench.track_setup("circle")
    return BatchedDroneEnv(N, targets, max_steps=max_steps, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                           include_distance=True, normalize_actions=True, normalize_obs=True, device="cuda:0")


def _trainer(N, learning_starts, slots=7, **kw):
    from drl_dronenavigation_b200.sac import SACConfig, SACTrainer
    cfg = SACConfig(rollout_impl="fused", learning_starts=learning_starts, buffer_size=N * slots, **kw)    # 7 slots: the ring wraps
    return SACTrainer(_env(N), cfg)


def _state(tr):
    b = tr.buffer
    n = b.cap if b.full else b.pos            # rows written so far (the rest is uninitialised memory)
    return {"obs_buf": b.obs[:n].clone(), "next_obs": b.next_obs[:n].clone(), "act": b.act[:n].clone(), "rew": b.rew[:n].clone(),
            "done": b.done[:n].clone(),
            "obs": tr.obs.clone(), "counter": tr.draw_counter.clone(), "slot": tr.slot.clone(), "pos": b.pos, "full": b.full}


def test_fused_collection_equals_a_launch_by_launch_replay():
    """Five phases of train_freq = 3 steps with learning_starts = 4 N: phase 1 uniform, phase 2 mixed (uniform, uniform...
    then sampled), phase 3 launched, phase 4 captured, phase 5 replayed.  A fresh env of the same configuration is stepped
    with the recorded actions one launch at a time; every action is recomputed by dn_sac_act from the recorded observation
    with the counter value of its step.  Buffer rows, observations, counter and slot must match bit for bit."""
    from drl_dronenavigation_b200 import _lib as L
    N = 1024
    tr = _trainer(N, 4 * N)
    fa, cap = tr.fused, tr.buffer.cap
    states = []
    for phase in range(5):
        tr.collect(3)
        torch.cuda.synchronize()
        states.append(_state(tr))
        assert int(tr.slot.item()) == tr.buffer.pos
        assert (tr._collect_graph is not None) == (phase >= 3)
    assert int(tr.draw_counter.item()) == 15 and tr.buffer.full and tr.buffer.pos == 15 % cap
    env = _env(N)
    obs = env.reset().clone()
    final = states[-1]
    n_done = 0
    for t in range(15):
        s, row = states[t // 3], t % cap          # (a phase writes 3 < cap rows: its snapshot still holds all of them)
        assert torch.equal(s["obs_buf"][row], obs), t
        mode = L.DN_SAC_UNIFORM if t * N < 4 * N else L.DN_SAC_SAMPLE
        ctr = torch.full((1,), t, dtype=torch.int64, device="cuda")
        a = fa.act(obs, _sample_tr(tr, ctr, mode)).clone()
        assert torch.equal(a, s["act"][row]), t
        o, r, d, _ = env.step(a)
        nxt = torch.where((d != 0).unsqueeze(-1), env.terminal_obs, o)
        assert torch.equal(s["next_obs"][row], nxt) and torch.equal(s["rew"][row], r), t
        assert torch.equal(s["done"][row], ((d & 1) != 0).float()), t
        n_done += int((d != 0).sum())
        obs = o.clone()
    assert torch.equal(final["obs"], obs)
    assert n_done > 0
    env.close()
    tr.env.close()


def _sample_tr(tr, counter, mode):
    from drl_dronenavigation_b200 import _lib
    s = _lib.dn_sac_sample()
    s.seed, s.row_id_offset, s.counter, s.mode = tr.cfg.seed, tr.env.env_id_offset, counter.data_ptr(), mode
    return s


def test_graph_replay_equals_launching():
    N = 512
    out = {}
    for graph in (False, True):
        tr = _trainer(N, 3 * N)
        tr.collect_graph = graph
        out[graph] = []
        for _ in range(5):
            tr.collect(3)
            out[graph].append(_state(tr))
        assert (tr._collect_graph is not None) == graph
        tr.env.close()
    for a, b in zip(out[False], out[True]):
        for k in a:
            assert (a[k] == b[k]) if not torch.is_tensor(a[k]) else torch.equal(a[k], b[k]), k


def test_a_checkpoint_load_between_phases_is_sampled_with(tmp_path):
    """Trainer B replays its captured graph; then B's learner loads A's (different) weights from an SB3 archive.  The next
    phase's actions must be A's actor on the recorded observations with the restated noise."""
    from drl_dronenavigation_b200.checkpoint import load_sb3_zip, save_sb3_sac_zip
    N = 512
    A = _trainer(N, 0, seed=5)
    with torch.no_grad():
        A.learner.actor.mu.weight.mul_(-3.0)
    path = save_sb3_sac_zip(str(tmp_path / "a.zip"), A.learner)
    B = _trainer(N, 0, seed=6)
    for _ in range(3):
        B.collect(3)
    assert B._collect_graph is not None
    load_sb3_zip(path, B.learner)
    for pa, pb in zip(A.learner.actor.parameters(), B.learner.actor.parameters()):
        assert torch.equal(pa, pb)
    pos, ctr = B.buffer.pos, int(B.draw_counter.item())
    B.collect(3)
    torch.cuda.synchronize()
    ref = copy.deepcopy(A.learner.actor).double()
    for k in range(3):
        row = (pos + k) % B.buffer.cap
        eps = torch.from_numpy(R.normals(B.cfg.seed, ctr + k, np.arange(N), 4)).cuda()
        with torch.no_grad():
            want, _ = ref(B.buffer.obs[row].double(), eps=eps)
        err = float((B.buffer.act[row].double() - want).abs().max())
        assert err < 1e-4, (k, err)
    A.env.close()
    B.env.close()


def test_short_fused_training_run_keeps_finite_losses_and_a_consistent_buffer():
    N = 2048
    tr = _trainer(N, 2 * 3 * N, slots=64)
    outs = [tr.train_iteration() for _ in range(8)]
    assert outs[0]["gradient_steps"] == 0 and all(o["gradient_steps"] == 5 for o in outs[1:])
    assert all(o["collect_s"] > 0 for o in outs)
    for k in ("critic_loss", "actor_loss", "ent_coef", "ent_coef_loss"):
        assert np.isfinite([o[k] for o in outs[1:]]).all(), k
    assert tr._collect_graph is not None
    assert int(tr.slot.item()) == tr.buffer.pos == 24 and len(tr.buffer) == 24 * N
    assert int(tr.draw_counter.item()) == 24
    assert bool((tr.buffer.act[:24].abs() <= 1).all()) and bool(torch.isfinite(tr.buffer.next_obs[:24]).all())
    print("collect_s per iteration:", [round(o["collect_s"] * 1e3, 3) for o in outs], "ms")
    tr.env.close()
