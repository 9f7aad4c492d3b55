"""GPU tests of the learner side: the dn_gae kernel against the plain-torch FP32 recursion, and a short
PPO run on the device-resident environment."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_gae_kernel_matches_torch_reference():
    from drl_dronenavigation_b200.ppo import compute_gae, compute_gae_torch
    g = torch.Generator().manual_seed(0)
    for T, N in ((1, 1), (17, 33), (128, 4099)):
        rew, val = torch.randn(T, N, generator=g), torch.randn(T, N, generator=g)
        done = (torch.rand(T, N, generator=g) < 0.05).to(torch.uint8) * 3
        last = torch.randn(N, generator=g)
        a_ref, r_ref = compute_gae_torch(rew, val, done, last, 0.99, 0.95)
        a, r = compute_gae(rew.cuda(), val.cuda(), done.cuda(), last.cuda(), 0.99, 0.95)
        torch.testing.assert_close(a.cpu(), a_ref, rtol=1e-5, atol=1e-5)      # FP32, same operation order up to FMA contraction
        torch.testing.assert_close(r.cpu(), r_ref, rtol=1e-5, atol=1e-5)


def test_ppo_trainer_runs_on_device():
    import bench
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    targets, init, dim, is_circle = bench.track_setup("circle")
    env = BatchedDroneEnv(2048, targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                          include_distance=True, normalize_actions=True)
    tr = PPOTrainer(env, PPOConfig(batch_size=4096, n_epochs=2), rollout_steps=16)
    p0 = tr.learner.flat_parameters().clone()
    for _ in range(2):
        out = tr.train_iteration()
        assert np.isfinite([out["policy_gradient_loss"], out["value_loss"], out["approx_kl"]]).all()
        assert out["sps"] > 0 and out["samples"] == 16 * 2048
    assert not torch.equal(p0, tr.learner.flat_parameters())
    assert env.launch_count >= 2 * 16
    st = env.episode_stats()
    assert st["episodes"] > 0          # random policy crashes within a few control steps
    env.close()


def test_simulator_manager_short_training_and_test_run():
    """PBDroneSimulator-compatible manager: reference flags -> GPU env -> a few PPO iterations -> evaluation;
    and --run_type test (constant action on the `up` track until termination)."""
    from drl_dronenavigation_b200 import Track, Waypoints
    from drl_dronenavigation_b200.argparser import parse_args
    from drl_dronenavigation_b200.simulator import PBDroneSimulator
    args = parse_args(["--num_envs", "1024", "--total_timesteps", "65536", "--savemodel", "f", "--rollout_steps", "16"])
    sim = PBDroneSimulator(args, Track(Waypoints.circle(radius=1, num_points=6, height=1), circle=True), target_factor=0)
    assert len(sim.targets) == 6
    logs = []
    trainer, ev = sim.run_full_training(log=logs.append)
    assert trainer.total_steps >= 65536 and ev["episodes"] >= 100 and 0.0 <= ev["success_rate"] <= 1.0
    venv = sim.make_env(multi=True, aviary_dim=sim.aviary_dim, initial_xyzs=sim.initial_xyzs, num_envs=3)()
    assert venv.reset().shape == (3, 13)
    venv.close()
    rewards = sim.run_test(log=lambda *_: None)
    assert len(rewards) >= 1 and rewards[-1] in (-10.0,) or len(rewards) > 1


def test_sac_trainer_runs_on_device_with_drag_and_ground_effect():
    """BASELINE config 4 at test size: SAC on the circle track with the drag + ground-effect physics extension."""
    import bench
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.sac import SACConfig, SACTrainer
    targets, init, dim, is_circle = bench.track_setup("circle")
    env = BatchedDroneEnv(1024, targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                          include_distance=True, normalize_actions=True, physics=Physics.PYB_GND_DRAG_DW)
    tr = SACTrainer(env, SACConfig(learning_starts=4096, buffer_size=65536))
    p0 = tr.learner.flat_parameters().clone()
    outs = [tr.train_iteration() for _ in range(6)]
    assert outs[0]["gradient_steps"] == 0 and outs[-1]["gradient_steps"] == 5      # learning_starts respected
    assert np.isfinite([outs[-1]["critic_loss"], outs[-1]["actor_loss"], outs[-1]["ent_coef"]]).all()
    assert len(tr.buffer) == 6 * 3 * 1024 and tr.total_steps == 6 * 3 * 1024
    assert not torch.equal(p0, tr.learner.flat_parameters())
    # time-limit handling: only true terminations are stored as done
    assert float(tr.buffer.done[:tr.buffer.pos].max()) <= 1.0
    assert env.launch_count >= 18
    env.close()


def test_ppo_update_cuda_graph_equals_eager():
    """The two-graph replay of the minibatch step must be the same computation as the eager loop (same seeds ->
    same minibatch order; same kernels -> same parameters up to FP32 reduction-order noise), including the
    KL early stop and a second update (Adam state carried across replays)."""
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    g = torch.Generator(device="cuda").manual_seed(0)
    B = 8192
    obs, act = torch.randn(B, 13, device="cuda", generator=g), torch.rand(B, 4, device="cuda", generator=g) * 2 - 1
    adv, ret = torch.randn(B, device="cuda", generator=g), torch.randn(B, device="cuda", generator=g)
    outs = {}
    for graph in (False, True):
        L = PPOLearner(13, 4, PPOConfig(batch_size=1024, n_epochs=3, target_kl=None, cuda_graph=graph, matmul_precision="fp32", update_impl="torch"), device="cuda")
        assert L.use_graph == graph
        with torch.no_grad():
            v, logp, _ = L.policy.evaluate(obs, act)
        p0 = L.flat_parameters().clone()
        r1 = L.update(obs, act, logp, v, adv, ret, generator=torch.Generator(device="cuda").manual_seed(1))
        r2 = L.update(obs, act, logp, v, adv, ret, generator=torch.Generator(device="cuda").manual_seed(2))
        outs[graph] = (p0, L.flat_parameters().clone(), r1, r2)
    assert torch.equal(outs[False][0], outs[True][0])                 # capture warm-up left the parameters untouched
    # Adam normalises every coordinate's step to ~lr, so coordinates whose gradient is rounding noise may move by up to
    # lr per step in either direction; compare in aggregate (48 steps of lr 2.5e-4 = 1.2e-2 worst case)
    d = (outs[True][1] - outs[False][1]).abs()
    moved = (outs[False][1] - outs[False][0]).abs()
    print("graph-vs-eager: max", float(d.max()), "mean", float(d.mean()), "mean movement", float(moved.mean()))
    assert float(d.mean()) < 0.02 * float(moved.mean()) and float(d.max()) < 2e-3
    for k in ("policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction"):
        assert abs(outs[True][2][k] - outs[False][2][k]) < 1e-4 and abs(outs[True][3][k] - outs[False][3][k]) < 1e-3
    assert outs[True][2]["minibatches"] == outs[False][2]["minibatches"] == 24
    # early stop path under replay
    L = PPOLearner(13, 4, PPOConfig(batch_size=1024, n_epochs=30, target_kl=1e-4, learning_rate=1e-2, cuda_graph=True, update_impl="torch"), device="cuda")
    with torch.no_grad():
        v, logp, _ = L.policy.evaluate(obs, act)
    out = L.update(obs, act, logp, v, adv, ret, generator=torch.Generator(device="cuda").manual_seed(1))
    assert out["early_stop"] and out["epochs"] < 30


def test_manager_saved_cont_and_learning_run_types(tmp_path):
    """--run_type learning (500-step smoke run with the deeper policy), a checkpoint written as an SB3 archive,
    --run_type saved on it, and --run_type cont resuming from it (PBDroneSimulator.py:438-612,701-712)."""
    from drl_dronenavigation_b200 import Track, Waypoints
    from drl_dronenavigation_b200.argparser import parse_args
    from drl_dronenavigation_b200.checkpoint import save_sb3_zip
    from drl_dronenavigation_b200.simulator import PBDroneSimulator
    track = Track(Waypoints.circle(radius=1, num_points=6, height=1), circle=True)
    args = parse_args(["--num_envs", "256", "--total_timesteps", "8192", "--savemodel", "f", "--rollout_steps", "16",
                       "--max_env_steps", "64", "--batch_size", "32"])
    sim = PBDroneSimulator(args, track)
    trainer, out = sim.test_learning(log=lambda *_: None)
    assert trainer.total_steps >= 500 and np.isfinite(out["value_loss"])
    # the deeper architecture: 13-512-512-256-128-4
    assert sum(p.numel() for p in trainer.learner.policy.pi.parameters()) == 13 * 512 + 512 + 512 * 512 + 512 + 512 * 256 + 256 + 256 * 128 + 128 + 128 * 4 + 4
    tr, _ = sim.run_full_training(log=lambda *_: None)
    path = save_sb3_zip(str(tmp_path / "best_model.zip"), tr.learner)
    ev = sim.test_saved(path, episodes=20)
    assert ev["episodes"] >= 20
    args2 = parse_args(["--num_envs", "256", "--total_timesteps", "8192", "--savemodel", "f", "--rollout_steps", "16",
                        "--run_type", "cont", "--model_path", path])
    sim2 = PBDroneSimulator(args2, track)
    tr2, _ = sim2.run_full_training(log=lambda *_: None)
    assert tr2.total_steps >= 8192


def test_sac_update_cuda_graph_equals_eager():
    """The three-graph replay of the SAC gradient step is the same computation as the eager path: same batches and
    noise -> same losses and (up to FP32 reduction-order noise amplified by Adam) the same parameters and targets."""
    from drl_dronenavigation_b200.sac import SACConfig, SACLearner
    g = torch.Generator(device="cuda").manual_seed(0)
    B = 1024
    batches = [(torch.randn(B, 13, device="cuda", generator=g), torch.rand(B, 4, device="cuda", generator=g) * 2 - 1,
                torch.randn(B, device="cuda", generator=g), torch.randn(B, 13, device="cuda", generator=g),
                (torch.rand(B, device="cuda", generator=g) < 0.1).float()) for _ in range(6)]
    res = {}
    for graph in (False, True):
        L = SACLearner(13, 4, SACConfig(cuda_graph=graph, matmul_precision="fp32"), device="cuda")
        assert L.use_graph == graph
        p0 = L.flat_parameters().clone()
        outs = [L.update(b, generator=torch.Generator(device="cuda").manual_seed(10 + k)) for k, b in enumerate(batches)]
        tgt = torch.cat([p.reshape(-1) for p in L.critic_target.parameters()])
        res[graph] = (p0, L.flat_parameters().clone(), tgt.clone(), [{k: float(v) for k, v in o.items()} for o in outs])
    assert torch.equal(res[False][0], res[True][0])                  # capture warm-up left parameters and Adam state untouched
    for a, b in zip(res[True][3], res[False][3]):
        for k in ("critic_loss", "actor_loss", "ent_coef", "ent_coef_loss"):
            assert abs(a[k] - b[k]) <= 1e-3 * max(1.0, abs(b[k])), (k, a[k], b[k])
    moved = (res[False][1] - res[False][0]).abs().mean()
    d = (res[True][1] - res[False][1]).abs()
    print("sac graph-vs-eager: max", float(d.max()), "mean", float(d.mean()), "mean movement", float(moved))
    assert float(d.mean()) < 0.02 * float(moved) and float(d.max()) < 2e-3
    torch.testing.assert_close(res[True][2], res[False][2], rtol=1e-3, atol=1e-5)


def test_ppo_update_graphs_follow_an_optimizer_load():
    """A graphed learner that has already captured its minibatch step loads another learner's parameters and Adam state:
    load_state_dict re-creates the state tensors the graphs pointed to, so the next update must capture again and take the
    steps an eager learner takes from the same state (the tolerances of the graph-vs-eager test above)."""
    import copy
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    g = torch.Generator(device="cuda").manual_seed(0)
    B = 8192
    obs, act = torch.randn(B, 13, device="cuda", generator=g), torch.rand(B, 4, device="cuda", generator=g) * 2 - 1
    adv, ret = torch.randn(B, device="cuda", generator=g), torch.randn(B, device="cuda", generator=g)
    cfg = lambda graph: PPOConfig(batch_size=1024, n_epochs=3, target_kl=None, cuda_graph=graph, matmul_precision="fp32", update_impl="torch")
    src = PPOLearner(13, 4, cfg(False), device="cuda")
    with torch.no_grad():
        v, logp, _ = src.policy.evaluate(obs, act)
    src.update(obs, act, logp, v, adv, ret, generator=torch.Generator(device="cuda").manual_seed(1))
    state = src.opt.state_dict()["state"]
    res = {}
    for graph in (False, True):
        L = PPOLearner(13, 4, cfg(graph), device="cuda")
        if graph:
            L.update(obs, act, logp, v, adv, ret, generator=torch.Generator(device="cuda").manual_seed(2))     # captured
        L.policy.load_state_dict(src.policy.state_dict())
        L.load_optimizer_state(copy.deepcopy(state))
        p0 = L.flat_parameters().clone()
        r = L.update(obs, act, logp, v, adv, ret, generator=torch.Generator(device="cuda").manual_seed(3))
        res[graph] = (p0, L.flat_parameters().clone(), r, float(L.opt.state[L.params[0]]["step"]))
    assert torch.equal(res[False][0], res[True][0])
    assert res[True][3] == res[False][3] == 48.0                      # 24 loaded steps + 24 taken on the loaded state
    d = (res[True][1] - res[False][1]).abs()
    moved = (res[False][1] - res[False][0]).abs()
    print("graph-vs-eager after a load: max", float(d.max()), "mean", float(d.mean()), "mean movement", float(moved.mean()))
    assert float(d.mean()) < 0.02 * float(moved.mean()) and float(d.max()) < 2e-3
    for k in ("policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction"):
        assert abs(res[True][2][k] - res[False][2][k]) < 1e-3, k


def test_sac_update_graphs_follow_an_archive_load(tmp_path):
    """A graphed SAC learner that has already captured its gradient step loads an SB3 archive with its optimisers; its next steps
    must be those of an eager learner loaded from the same archive (the tolerances of the graph-vs-eager test above)."""
    from drl_dronenavigation_b200.checkpoint import load_sb3_zip, save_sb3_sac_zip
    from drl_dronenavigation_b200.sac import SACConfig, SACLearner
    g = torch.Generator(device="cuda").manual_seed(0)
    B = 1024
    batches = [(torch.randn(B, 13, device="cuda", generator=g), torch.rand(B, 4, device="cuda", generator=g) * 2 - 1,
                torch.randn(B, device="cuda", generator=g), torch.randn(B, 13, device="cuda", generator=g),
                (torch.rand(B, device="cuda", generator=g) < 0.1).float()) for _ in range(6)]
    gen = lambda k: torch.Generator(device="cuda").manual_seed(10 + k)
    src = SACLearner(13, 4, SACConfig(cuda_graph=False, matmul_precision="fp32", seed=7), device="cuda")
    for k, b in enumerate(batches[:5]):
        src.update(b, generator=gen(k))
    path = save_sb3_sac_zip(str(tmp_path / "src.zip"), src)
    res = {}
    for graph in (False, True):
        L = SACLearner(13, 4, SACConfig(cuda_graph=graph, matmul_precision="fp32"), device="cuda")
        if graph:
            for k, b in enumerate(batches[:2]):                      # captured
                L.update(b, generator=gen(20 + k))
        load_sb3_zip(path, L, load_optimizer=True)
        p0 = L.flat_parameters().clone()
        outs = [L.update(b, generator=gen(30 + k)) for k, b in enumerate(batches[2:])]
        tgt = torch.cat([p.reshape(-1) for p in L.critic_target.parameters()])
        steps = [float(o.state[p]["step"]) for o in (L.actor_opt, L.critic_opt, L.ent_opt) for p in o.state]
        res[graph] = (p0, L.flat_parameters().clone(), tgt.clone(), [{k: float(v) for k, v in o.items()} for o in outs], steps)
    assert torch.equal(res[False][0], res[True][0])
    assert res[True][4] == res[False][4] == [9.0] * len(res[False][4])    # 5 loaded steps + 4 taken on the loaded state
    for a, b in zip(res[True][3], res[False][3]):
        for k in ("critic_loss", "actor_loss", "ent_coef", "ent_coef_loss"):
            assert abs(a[k] - b[k]) <= 1e-3 * max(1.0, abs(b[k])), (k, a[k], b[k])
    moved = (res[False][1] - res[False][0]).abs().mean()
    d = (res[True][1] - res[False][1]).abs()
    print("sac graph-vs-eager after a load: max", float(d.max()), "mean", float(d.mean()), "mean movement", float(moved))
    assert float(d.mean()) < 0.02 * float(moved) and float(d.max()) < 2e-3
    torch.testing.assert_close(res[True][2], res[False][2], rtol=1e-3, atol=1e-5)


def test_fast_linear_matches_nn_linear():
    """FastLinear (GEMV bias gradient, input width padded to a multiple of 8) against plain nn.Linear in FP32: same
    outputs and the same gradients for input, weight and bias, for the first-layer (13 -> 512) and a square layer."""
    from drl_dronenavigation_b200.ppo import FastLinear
    torch.backends.cuda.matmul.allow_tf32 = False
    for k, n in ((13, 512), (512, 256), (256, 1)):
        torch.manual_seed(k)
        ref = torch.nn.Linear(k, n).cuda()
        fast = FastLinear(k, n).cuda()
        fast.load_state_dict(ref.state_dict())
        x = torch.randn(4096, k, device="cuda")
        xr, xf = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        g = torch.randn(4096, n, device="cuda")
        yr, yf = ref(xr), fast(xf)
        torch.testing.assert_close(yf, yr, rtol=1e-5, atol=1e-5)
        yr.backward(g); yf.backward(g)
        torch.testing.assert_close(xf.grad, xr.grad, rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(fast.weight.grad, ref.weight.grad, rtol=1e-4, atol=1e-3)
        torch.testing.assert_close(fast.bias.grad, ref.bias.grad, rtol=1e-4, atol=1e-3)
    with torch.no_grad():
        assert torch.equal(fast(x), torch.nn.functional.linear(x, fast.weight, fast.bias))      # inference path: plain nn.Linear
