"""Parity of the CUDA path (called through the C ABI) against the CPU oracle.  GPU only."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU

pytestmark = pytest.mark.gpu

HOVER = 0.092227


def _make(track, N, S, normalize_obs=False, max_steps=4096, **kw):
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    ctrl = 240 // S
    ref = make_reference_env(track, pyb_freq=240, ctrl_freq=ctrl, max_steps=max_steps)
    env = BatchedDroneEnv(N, ref._target_points, threshold=0.3, discount=0.999, max_steps=max_steps,
                          aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS, pyb_freq=240, ctrl_freq=ctrl,
                          cylinder=True, circle=(track == "circle"), include_distance=True,
                          normalize_actions=True, normalize_obs=normalize_obs, **kw)
    workers = [OracleWorker(make_reference_env(track, pyb_freq=240, ctrl_freq=ctrl, max_steps=max_steps),
                            normalize_obs=normalize_obs) for _ in range(N)]
    return env, workers


def _actions(mode, T, N, seed):
    rng = np.random.default_rng(seed)
    u = rng.uniform(-1, 1, size=(T, N, 4))
    if mode == "saturating":          # config 2(A): U(-1,1) -> near bang-bang, reset-heavy
        a = u
    elif mode == "hover_band":        # config 2(B): long episodes
        a = HOVER + 0.002 * u
    elif mode == "mixed":             # wider band: tumbles, leaves the tube within ~1 s
        a = HOVER + 0.006 * u
    else:
        raise ValueError(mode)
    return a.astype(np.float32)


def _reset_both(env, workers):
    obs = env.reset().cpu().numpy()
    for i, w in enumerate(workers):
        o, _ = w.reset()
        np.testing.assert_allclose(obs[i], o, atol=1e-6)


@pytest.mark.parametrize("track,S,mode,N,T", [
    ("circle", 1, "saturating", 24, 400),
    ("circle", 1, "hover_band", 16, 480),
    ("circle", 8, "saturating", 24, 120),
    ("circle", 8, "mixed", 24, 150),
    ("reaching", 1, "mixed", 16, 480),
    ("reaching", 8, "saturating", 16, 120),
    ("reaching", 8, "hover_band", 16, 90),
])
def test_lockstep_parity(track, S, mode, N, T):
    env, workers = _make(track, N, S)
    _reset_both(env, workers)
    rep = PU.run_lockstep(env, workers, _actions(mode, T, N, seed=len(track) * 100 + S * 10 + len(mode)), resync_every=240 // S)
    print(f"\n[{track} S={S} {mode}] {rep}")
    assert rep.near_ties <= max(2, rep.env_steps // 200)
    env.close()


def test_action_map_bit_exact():
    """The THRUST action map (rescale_action -> clip -> cmd2pwm -> pwm2rpm) is float32 end to end in the
    reference; the kernel's restatement (constant-divisor divisions via FMA residuals) must give the
    same BITS as numpy for every float32 action: dense sweep of the pass-through band plus random."""
    from oracle.dyn_oracle import physical_action_bounds, rescale_action_batch, thrust_to_rpm_batch, rpm_action_to_rpm
    env, _ = _make("circle", 4, 1)
    b = physical_action_bounds()
    lo = np.float32(0.0895).view(np.int32)
    hi = np.float32(0.0975).view(np.int32)
    band = np.arange(lo, hi + 1, dtype=np.int32).view(np.float32)              # every float32 in [0.0895, 0.0975]
    rnd = np.random.default_rng(0).uniform(-1.2, 1.2, size=1 << 20).astype(np.float32)
    a = np.concatenate([band, rnd, np.array([-1, 1, 0, 0.092227, np.float32(b[0][0]), np.float32(b[1][0])], np.float32)])
    a = a[: (a.size // 4) * 4]
    ref = thrust_to_rpm_batch(rescale_action_batch(a, b), b).reshape(-1)
    got = env.action_to_rpm(torch.from_numpy(a)).cpu().numpy()
    assert ref.dtype == np.float32
    np.testing.assert_array_equal(got.view(np.int32), ref.view(np.int32))
    assert band.size > 800_000
    env.close()
    # RPM action type (BaseSingleAgentAviary.py:176-179), numpy-1.26 float32 semantics
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200 import ActionType
    from oracle.dyn_oracle import make_reference_env
    r0 = make_reference_env("circle")
    env = BatchedDroneEnv(4, r0._target_points, aviary_dim=r0._aviary_dim, initial_xyzs=r0.INIT_XYZS, circle=True, act=ActionType.RPM)
    got = env.action_to_rpm(torch.from_numpy(rnd)).cpu().numpy()
    np.testing.assert_array_equal(got.view(np.int32), rpm_action_to_rpm(rnd).view(np.int32))
    env.close()


def test_reset_after_crash_uses_stale_position():
    """SURVEY 8(c) scenario: max thrust -> -10 at step 53; the returned (reset) obs carries the stale
    distance 0.26039 and the new distance is measured from the stale position."""
    env, workers = _make("circle", 4, 1)
    env.reset()
    a = torch.ones(4, 4, device=env.device)
    for k in range(1, 60):
        o, r, d, f = env.step(a)
        if int(d[0]):
            break
    assert k == 53 and float(r[0]) == -10.0 and int(d[0]) == 1
    assert float(o[0, 12]) == pytest.approx(0.26039, abs=1e-5)
    np.testing.assert_allclose(o[0, :3].cpu().numpy(), [0.5, 0, 0.5])
    st = env.get_state()
    assert float(st["dist"][0]) == pytest.approx(1.04157, abs=1e-5)
    assert int(st["steps"][0]) == 0 and int(st["episode_count"][0]) == 1
    stats = env.episode_stats()
    assert stats["episodes"] == 4 and stats["crashes"] == 4 and stats["length_sum"] == 4 * 53
    env.close()


def test_truncation_step_and_time_limit_bit():
    env, workers = _make("circle", 4, 1, max_steps=7)
    env.reset()
    a = torch.full((4, 4), HOVER, device=env.device)
    bits = [int(env.step(a)[2][0]) for _ in range(8)]
    assert bits == [0] * 7 + [2]
    assert env.episode_stats()["truncations"] == 4
    env.close()


def test_single_step_random_states_all_branches():
    """Differential single-step test from randomised mid-episode states placed near targets, tube walls,
    box walls and the step limit, so that every branch of the reward / termination state machine fires."""
    from oracle.dyn_oracle import bullet_quaternion_from_euler
    N = 768
    rng = np.random.default_rng(7)
    total = PU.ParityReport()
    for track, S in (("circle", 1), ("reaching", 8)):
        env, workers = _make(track, N, S, max_steps=64)
        _reset_both(env, workers)
        T = len(workers[0].env._target_points)
        for i, w in enumerate(workers):
            e = w.env
            steps = int(rng.choice([0, 1, 30, 63, 64]))
            # steps == 0 means "no post-step since the last reset": target 0 and a distance that was
            # measured from the (stale) current position -- the only such states the reference can be in
            idx = 0 if steps == 0 else int(rng.integers(0, T))
            tgt = e._target_points[idx]
            kind = i % 4
            if kind == 0:      # near the current target -> capture / final target
                pos = tgt + rng.normal(0, 0.2, 3)
            elif kind == 1:    # near the tube wall
                prev = e.INIT_XYZS[0] if idx == 0 else e._target_points[idx - 1]
                lam = rng.uniform(0, 1)
                pos = prev + lam * (tgt - prev) + rng.normal(0, 0.25, 3)
            elif kind == 2:    # near the box / ceiling
                pos = np.array([rng.choice([-1, 1]) * (e._x_high - abs(rng.normal(0, 0.01))), rng.uniform(-1, 1),
                                e._z_high - abs(rng.normal(0, 0.01))])
            else:
                pos = e.INIT_XYZS[0] + rng.normal(0, 0.05, 3)
            rpy = rng.normal(0, 0.4, 3)
            st = dict(pos=pos, quat=bullet_quaternion_from_euler(rpy), vel=rng.normal(0, 1.0, 3),
                      rpy_rates=rng.normal(0, 2.0, 3), ang_v=rng.normal(0, 2.0, 3), prev_vel=rng.normal(0, 1.0, 3),
                      prev_ang_v=rng.normal(0, 2.0, 3), dist=float(np.linalg.norm(tgt - pos) + rng.normal(0, 0.01)),
                      prev_dist=float(np.linalg.norm(tgt - pos) + rng.normal(0, 0.02)), target_idx=idx,
                      steps=steps, just_found=bool(rng.integers(0, 2)))
            st["dist"] = abs(st["dist"])
            if steps == 0:
                st["dist"] = st["prev_dist"] = float(np.linalg.norm(pos - tgt))
                st["just_found"] = False
            e.set_state(st)
        PU.upload_oracle_state(env, workers)
        acts = _actions("mixed", 2, N, seed=3)
        rep = PU.run_lockstep(env, workers, acts, resync_every=1, report=None)
        print(f"\n[single-step {track} S={S}] {rep}")
        assert rep.dones > N // 8 and rep.captures > N // 20
        total.near_ties += rep.near_ties
        env.close()
    assert total.near_ties <= 8


STEP_MANY_CONFIGS = [
    ("default", {}), ("wrappers", {"normalize_obs": True, "normalize_reward": True, "clip_reward": 10.0}),
    ("reaching_midpoint", {"reward_id": 4, "random_spawn": "midpoint", "seed": 77}),
    ("progress_line", {"reward_id": 5, "random_spawn": "line", "seed": 78}), ("her_drag_gnd", {"reward_id": 3, "physics": "PYB_GND_DRAG_DW"}),
    ("vel", {"act": "VEL"}), ("cf2p_pid_gnd", {"act": "PID", "drone_model": "CF2P", "physics": "PYB_GND"}),
    ("race_rpm", {"act": "RPM", "drone_model": "RACE"}), ("bootstrapped_line", {"reward_id": 8, "random_spawn": "line", "seed": 79}),
    ("champ_normrew", {"reward_id": 9, "normalize_reward": True}),
]
# N = 1000: every step's observation rows start 16-byte aligned (bulk TMA store); N = 777 with obs_dim 13: three steps in
# four start misaligned, and every warp of such a step takes the per-element store.  The first id of each configuration
# (N = 1000, per-step outputs) keeps its plain name.
STEP_MANY_CASES = [pytest.param(kw, N, per_step, id=name if (N, per_step) == (1000, True) else
                                f"{name}-n{N}-{'per_step' if per_step else 'last_step'}")
                   for name, kw in STEP_MANY_CONFIGS for N in (1000, 777) for per_step in (True, False)]
def bits_equal(a, b):
    """Bit-for-bit equality of two tensors (NaN payloads included)."""
    if a.dtype.is_floating_point:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return torch.equal(a, b)


@pytest.mark.parametrize("kw,N,per_step", STEP_MANY_CASES)
def test_step_many_matches_repeated_step(kw, N, per_step):
    """dn_step_many (T steps, state in registers) is bit-identical to T dn_step launches -- also with the fused
    wrappers, the optional planes (aux / spawn / reward statistics) and the physics add-ons in play, all eight outputs passed.
    per_step_outputs = 1: every output [T, N, ...], the terminal observation and the episode outputs on the finished rows.
    per_step_outputs = 0: only the last step's outputs, the episode outputs only on the rows finished at that step, sentinels
    everywhere else.  The Monitor counts are equal; the return sums are within parity_utils.return_sum_bound of the FP64
    sum of the returns dn_step emitted (k = 1 for dn_step, k = the most episodes of one env for the one flush of dn_step_many)."""
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200.enums import ActionType, DroneModel
    kw = dict(kw)
    if "physics" in kw:
        kw["physics"] = getattr(Physics, kw["physics"])
    if "act" in kw:
        kw["act"] = getattr(ActionType, kw["act"])
    if "drone_model" in kw:
        kw["drone_model"] = getattr(DroneModel, kw["drone_model"])
    norm = kw.pop("normalize_obs", False)
    track = "reaching" if "random_spawn" in kw else "circle"
    envA, _ = _make(track, N, 8, normalize_obs=norm, **kw)
    envB, _ = _make(track, N, 8, normalize_obs=norm, **kw)
    envA.reset(); envB.reset()
    T, D, dev = 40, envA.obs_dim, envA.device
    acts = torch.from_numpy(_actions("saturating", T, N, seed=11)).to(dev)
    lead = (T,) if per_step else ()
    nan = float("nan")
    outs = dict(obs=torch.full((*lead, N, D), nan, device=dev), terminal_obs=torch.full((*lead, N, D), nan, device=dev),
                reward=torch.full((*lead, N), nan, device=dev), done=torch.full((*lead, N), 255, dtype=torch.uint8, device=dev),
                found_targets=torch.full((*lead, N), -1, dtype=torch.int32, device=dev),
                episode_return=torch.full((*lead, N), nan, device=dev),
                episode_length=torch.full((*lead, N), -1, dtype=torch.int32, device=dev))
    envB.step_many(acts, per_step_outputs=per_step, out=outs)
    ep_ret, ep_count = [], torch.zeros(N, dtype=torch.int64, device=dev)
    for t in range(T):
        o, r, d, f = envA.step(acts[t])
        done = d != 0
        ep_ret.append(envA.episode_return[done].double())
        ep_count += done
        if per_step:
            got = {k: v[t] for k, v in outs.items()}
        elif t == T - 1:
            got = outs
        else:
            continue
        assert bits_equal(o, got["obs"]) and bits_equal(r, got["reward"]), t
        assert torch.equal(d, got["done"]) and torch.equal(f, got["found_targets"]), t
        assert bits_equal(envA.terminal_obs[done], got["terminal_obs"][done]), t
        assert bits_equal(envA.episode_return[done], got["episode_return"][done]), t
        assert torch.equal(envA.episode_length[done], got["episode_length"][done]), t
        if not per_step:                                     # rows not finished at the last step keep the sentinels
            assert bool(torch.isnan(got["terminal_obs"][~done]).all()) and bool(torch.isnan(got["episode_return"][~done]).all())
            assert bool((got["episode_length"][~done] == -1).all())
    sa, sb = envA.get_state(), envB.get_state()
    for k in sa:
        assert bits_equal(sa[k], sb[k]), k
    stA, stB = envA.episode_stats(), envB.episode_stats()
    for k in ("episodes", "length_sum", "found_targets", "successes", "crashes", "truncations"):
        assert stA[k] == stB[k], (k, stA, stB)
    assert stA["episodes"] == int(ep_count.sum()) > 0
    ep_ret = torch.cat(ep_ret)
    ref, abs_sum, n = float(ep_ret.sum()), float(ep_ret.abs().sum()), ep_ret.numel()
    assert abs(stA["return_sum"] - ref) <= PU.return_sum_bound(abs_sum, n, 1), (stA["return_sum"], ref)
    assert abs(stB["return_sum"] - ref) <= PU.return_sum_bound(abs_sum, n, int(ep_count.max())), (stB["return_sum"], ref)
    envA.close(); envB.close()


def test_step_host_zero_copy_and_staged_paths_equal_device_step():
    """dn_step_host with pinned (zero-copy) and pageable (staged) host buffers == dn_step on device buffers."""
    envs = [_make("circle", 777, 8)[0] for _ in range(3)]
    for e in envs:
        e.reset()
    N, D = 777, 13
    acts = _actions("saturating", 12, N, seed=4)
    pin = lambda *s, dtype: torch.empty(*s, dtype=dtype).pin_memory()
    h = dict(a=pin(N, 4, dtype=torch.float32), o=pin(N, D, dtype=torch.float32), r=pin(N, dtype=torch.float32),
             d=pin(N, dtype=torch.uint8), t=pin(N, D, dtype=torch.float32), f=pin(N, dtype=torch.int32),
             er=pin(N, dtype=torch.float32), el=pin(N, dtype=torch.int32))
    io_pin = envs[1]._make_io(h["a"], h["o"], h["r"], h["d"], h["t"], h["f"], h["er"], h["el"])
    p = dict(a=np.zeros((N, 4), np.float32), o=np.zeros((N, D), np.float32), r=np.zeros(N, np.float32), d=np.zeros(N, np.uint8),
             f=np.zeros(N, np.int32))
    from drl_dronenavigation_b200 import _lib as L
    io_pg = L.dn_step_io()
    io_pg.actions, io_pg.obs, io_pg.reward, io_pg.done, io_pg.found_targets = (p["a"].ctypes.data, p["o"].ctypes.data, p["r"].ctypes.data,
                                                                               p["d"].ctypes.data, p["f"].ctypes.data)
    n_done = 0
    for t in range(12):
        o, r, d, f = envs[0].step(torch.from_numpy(acts[t]).cuda())
        h["a"].copy_(torch.from_numpy(acts[t]))
        envs[1].step_host(io_pin)
        p["a"][...] = acts[t]
        envs[2].step_host(io_pg)
        for name, dev_t in (("o", o), ("r", r), ("d", d), ("f", f)):
            ref = dev_t.cpu().numpy()
            np.testing.assert_array_equal(h[name].numpy(), ref)
            np.testing.assert_array_equal(p[name], ref)
        done = d.cpu().numpy() != 0
        n_done += int(done.sum())
        np.testing.assert_array_equal(h["t"].numpy()[done], envs[0].terminal_obs.cpu().numpy()[done])
        np.testing.assert_array_equal(h["el"].numpy()[done], envs[0].episode_length.cpu().numpy()[done])
    assert n_done > 100
    for e in envs:
        e.close()


@pytest.mark.parametrize("N,with_info", [(777, True), (4096, False), (1, True)])
def test_step_host_slab_graph_path_equals_device_step(N, with_info):
    """dn_host_buffers + dn_step_host / dn_step_host_async + dn_step_host_wait (the handle's pinned slab, one captured graph per
    step: H2D DMA, fused kernel, D2H DMA) == dn_step on device buffers, including the optional episode outputs."""
    from drl_dronenavigation_b200 import _lib as L
    envs = [_make("circle", N, 8)[0] for _ in range(2)]
    for e in envs:
        e.reset()
    acts = _actions("saturating", 14, N, seed=6)
    io, b = envs[1].host_buffers(with_episode_info=with_info)
    assert (b["terminal_obs"] is not None) == with_info and b["actions"].shape == (N, 4) and b["obs"].shape == (N, 13)
    l0 = envs[1].launch_count
    n_done = 0
    for t in range(14):
        o, r, d, f = envs[0].step(torch.from_numpy(acts[t]).cuda())
        b["actions"][...] = acts[t]
        if t % 2:
            envs[1].step_host(io)
        else:
            envs[1].step_host_async(io)
            with pytest.raises(L.DroneNavError, match="not been waited"):
                envs[1].step_host_async(io)                       # one step in flight at a time
            envs[1].step_host_wait()
        for name, dev_t in (("obs", o), ("reward", r), ("done", d), ("found_targets", f)):
            np.testing.assert_array_equal(b[name], dev_t.cpu().numpy(), err_msg=f"{name} t={t}")
        done = d.cpu().numpy() != 0
        n_done += int(done.sum())
        if with_info:
            np.testing.assert_array_equal(b["terminal_obs"][done], envs[0].terminal_obs.cpu().numpy()[done])
            np.testing.assert_array_equal(b["episode_length"][done], envs[0].episode_length.cpu().numpy()[done])
            np.testing.assert_array_equal(b["episode_return"][done], envs[0].episode_return.cpu().numpy()[done])
    assert envs[1].launch_count - l0 == 14                        # every graph replay counts as one launch of the step kernel
    assert n_done > 0 or N == 1
    # any other pointer set still takes the zero-copy / staged paths
    other = L.dn_step_io()
    pa, po, pr, pd = np.zeros((N, 4), np.float32), np.zeros((N, 13), np.float32), np.zeros(N, np.float32), np.zeros(N, np.uint8)
    other.actions, other.obs, other.reward, other.done = pa.ctypes.data, po.ctypes.data, pr.ctypes.data, pd.ctypes.data
    with pytest.raises(L.DroneNavError, match="dn_host_buffers"):
        envs[1].step_host_async(other)
    envs[1].step_host(other)
    for e in envs:
        e.close()


@pytest.mark.parametrize("form", ["zero_copy", "slab"])
def test_step_host_async_in_flight_refuses_other_calls(form):
    """While a dn_step_host_async step has not been waited for, it still runs against the handle's state: every other call that
    touches that state refuses -- the resident server path of dn_step_host included -- and after dn_step_host_wait the handle
    equals one stepped with dn_step on the same actions."""
    from drl_dronenavigation_b200 import _lib as L
    N, D, T = 777, 13, 6
    envs = [_make("circle", N, 8)[0] for _ in range(2)]
    for e in envs:
        e.reset()
    pin = lambda *s, dtype: torch.empty(*s, dtype=dtype).pin_memory()
    h = dict(actions=pin(N, 4, dtype=torch.float32), obs=pin(N, D, dtype=torch.float32), reward=pin(N, dtype=torch.float32),
             done=pin(N, dtype=torch.uint8), found_targets=pin(N, dtype=torch.int32))
    io_pin = envs[1]._make_io(h["actions"], h["obs"], h["reward"], h["done"], found=h["found_targets"])
    if form == "slab":
        io, b = envs[1].host_buffers()
    else:
        io, b = io_pin, {k: v.numpy() for k, v in h.items()}
    envs[1].host_server(2000)
    acts = _actions("saturating", T, N, seed=8)
    a_dev = torch.from_numpy(acts[0]).cuda()
    for t in range(T):
        o, r, d, f = envs[0].step(torch.from_numpy(acts[t]).cuda())
        b["actions"][...] = acts[t]
        envs[1].step_host_async(io)
        for call in (lambda: envs[1].step_host(io_pin), lambda: envs[1].step(a_dev), envs[1].reset, envs[1].get_state,
                     envs[1].episode_stats):
            with pytest.raises(L.DroneNavError, match="not been waited"):
                call()
        envs[1].step_host_wait()
        for name, dev_t in (("obs", o), ("reward", r), ("done", d), ("found_targets", f)):
            np.testing.assert_array_equal(b[name], dev_t.cpu().numpy(), err_msg=f"{name} t={t}")
    sa, sb = envs[0].get_state(), envs[1].get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert envs[1].episode_stats() == envs[0].episode_stats()
    assert envs[1].host_server_stats()["steps"] == 0
    for e in envs:
        e.close()


@pytest.mark.parametrize("N,norm,idle_us", [(777, False, 2000), (4096, True, 2000), (12, True, 50), (1, False, 2000)])
def test_step_host_resident_server_equals_device_step(N, norm, idle_us):
    """dn_host_server: the RESIDENT step kernel (dn_step_many variant, one host doorbell per step) == dn_step launch by launch --
    every output bit for bit, with rotating action buffers, across idle exits and re-launches of the resident kernel, and with
    other calls on the handle (episode statistics, get_state, a plain device step) in between."""
    import time
    envs = [_make("circle", N, 8, normalize_obs=norm)[0] for _ in range(2)]
    for e in envs:
        e.reset()
    D, T = 13, 40
    acts = _actions("saturating", T, N, seed=9)
    pin = lambda *s, dtype: torch.empty(*s, dtype=dtype).pin_memory()
    h_act = pin(4, N, 4, dtype=torch.float32)
    h = dict(o=pin(N, D, dtype=torch.float32), r=pin(N, dtype=torch.float32), d=pin(N, dtype=torch.uint8), t=pin(N, D, dtype=torch.float32),
             f=pin(N, dtype=torch.int32), er=pin(N, dtype=torch.float32), el=pin(N, dtype=torch.int32))
    ios = [envs[1]._make_io(h_act[k], h["o"], h["r"], h["d"], h["t"], h["f"], h["er"], h["el"]) for k in range(4)]
    envs[1].host_server(idle_us)
    n_done = 0
    for t in range(T):
        a_dev = torch.from_numpy(acts[t]).cuda()
        o, r, d, f = envs[0].step(a_dev)
        if t == 25:                                               # a plain device step in between stops the server first
            o1, r1, d1, f1 = envs[1].step(a_dev)
            torch.cuda.synchronize()
            for x, y in ((o, o1), (r, r1), (d, d1), (f, f1)):
                assert torch.equal(x, y)
            continue
        h_act[t % 4].copy_(torch.from_numpy(acts[t]))
        envs[1].step_host(ios[t % 4])
        for name, dev_t in (("o", o), ("r", r), ("d", d), ("f", f)):
            np.testing.assert_array_equal(h[name].numpy(), dev_t.cpu().numpy(), err_msg=f"{name} t={t}")
        done = d.cpu().numpy() != 0
        n_done += int(done.sum())
        np.testing.assert_array_equal(h["t"].numpy()[done], envs[0].terminal_obs.cpu().numpy()[done])
        np.testing.assert_array_equal(h["el"].numpy()[done], envs[0].episode_length.cpu().numpy()[done])
        np.testing.assert_array_equal(h["er"].numpy()[done], envs[0].episode_return.cpu().numpy()[done])
        if t == 10:
            time.sleep(0.02)                                      # longer than idle_us: the kernel has left, the next step re-launches it
        if t == 18:                                               # statistics are flushed per step and readable at any time
            assert envs[1].episode_stats(clear=False) == envs[0].episode_stats(clear=False)
        if t == 30:
            sa, sb = envs[0].get_state(), envs[1].get_state()
            for k in sa:
                assert torch.equal(sa[k], sb[k]), k
    st = envs[1].host_server_stats()
    assert st["steps"] == T - 1 and 3 <= st["residencies"] <= T - 1, st    # first launch, after the sleep, after each interleaved call
    envs[1].host_server(0)
    sa, sb = envs[0].get_state(), envs[1].get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert envs[1].episode_stats() == envs[0].episode_stats()
    assert n_done > 0 or N <= 12
    for e in envs:
        e.close()


def test_step_host_resident_server_limits():
    from drl_dronenavigation_b200 import _lib as L
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.dyn_oracle import make_reference_env
    ref = make_reference_env("circle")
    env = BatchedDroneEnv(1 << 18, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS, circle=True)
    with pytest.raises(L.DroneNavError, match="resident grid"):
        env.host_server(1000)
    env.close()


def test_ragged_sizes_and_obs12():
    """N not a multiple of the CTA size (tail CTA takes the non-TMA store path), N = 1, 12-dim obs."""
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.dyn_oracle import make_reference_env
    ref = make_reference_env("circle")
    outs = {}
    for N in (1, 3, 127, 130, 1027):
        for inc in (True, False):
            env = BatchedDroneEnv(N, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS,
                                  circle=True, include_distance=inc, normalize_actions=True)
            env.reset()
            a = torch.full((N, 4), HOVER, device=env.device)
            for _ in range(3):
                o, r, d, f = env.step(a)
            assert o.shape == (N, 13 if inc else 12)
            outs[(N, inc)] = o.cpu().numpy()
            env.close()
    for (N, inc), o in outs.items():      # every env got the same actions -> identical rows, equal to N=1
        np.testing.assert_array_equal(o, np.repeat(outs[(1, inc)], N, axis=0))


def test_vec_env_protocol_against_oracle_workers():
    """GpuDroneVecEnv (numpy, pinned host buffers) reproduces the SubprocVecEnv worker contract,
    NormalizeObservation included (the normalised rows amplify FP32 state differences by 1 / sqrt(var): looser obs tolerance)."""
    from drl_dronenavigation_b200.vec_env import GpuDroneVecEnv
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    N, T = 12, 200
    ref = make_reference_env("circle")
    venv = GpuDroneVecEnv(N, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS,
                          circle=True, include_distance=True, normalize_actions=True, normalize_obs=True)
    workers = [OracleWorker(make_reference_env("circle"), normalize_obs=True) for _ in range(N)]
    obs = venv.reset()
    assert obs.shape == (N, 13) and obs.dtype == np.float32
    for i, w in enumerate(workers):
        np.testing.assert_allclose(obs[i], w.reset()[0], atol=2e-4)
    acts = _actions("saturating", T, N, seed=5)
    n_done = 0
    for t in range(T):
        o, r, d, infos = venv.step(acts[t])
        assert d.dtype == np.bool_ and len(infos) == N
        for i, w in enumerate(workers):
            oo, rr, dd, info = w.step(acts[t, i])
            assert bool(d[i]) == dd and infos[i]["found_targets"] == info["found_targets"]
            # FP32 running statistics + normalisation amplify the ill-conditioned ang_v direction entries (9..11)
            np.testing.assert_allclose(o[i][:9], oo[:9], atol=2e-3, rtol=2e-3)
            np.testing.assert_allclose(o[i][12], oo[12], atol=2e-3, rtol=2e-3)
            if w.last_step_ang_v_norm > 0.5 and not dd:      # direction of a non-negligible angular velocity
                np.testing.assert_allclose(o[i][9:12], oo[9:12], atol=5e-2, rtol=5e-2)
            assert abs(r[i] - rr) < 1e-3
            if dd:
                n_done += 1
                assert infos[i]["episode"]["l"] == info["episode"]["l"]
                assert infos[i]["TimeLimit.truncated"] == info["TimeLimit.truncated"]
                np.testing.assert_allclose(infos[i]["terminal_observation"], info["terminal_observation"], atol=2e-3, rtol=2e-3)
    assert n_done > 10
    assert venv.env_is_wrapped(type("Monitor", (), {}))[0]
    venv.close()


def test_vec_env_host_paths_agree():
    """GpuDroneVecEnv with the three host paths (zero copy, slab + graph, resident server): the same SB3 protocol outputs bit for bit,
    per-env NormalizeObservation and Monitor included."""
    from drl_dronenavigation_b200.vec_env import GpuDroneVecEnv
    from oracle.dyn_oracle import make_reference_env
    N, T = 12, 120
    ref = make_reference_env("circle")
    venvs = {p: GpuDroneVecEnv(N, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS, circle=True,
                               include_distance=True, normalize_actions=True, normalize_obs=True, host_path=p)
             for p in ("zero_copy", "slab", "server")}
    obs0 = {p: v.reset() for p, v in venvs.items()}
    acts = _actions("saturating", T, N, seed=21)
    n_done = 0
    for t in range(T):
        outs = {p: v.step(acts[t]) for p, v in venvs.items()}
        o, r, d, infos = outs["zero_copy"]
        n_done += int(d.sum())
        for p in ("slab", "server"):
            o2, r2, d2, infos2 = outs[p]
            np.testing.assert_array_equal(o, o2, err_msg=f"{p} t={t}")
            np.testing.assert_array_equal(r, r2)
            np.testing.assert_array_equal(d, d2)
            for a, b in zip(infos, infos2):
                assert a["found_targets"] == b["found_targets"] and ("episode" in a) == ("episode" in b)
                if "episode" in a:
                    assert a["episode"]["l"] == b["episode"]["l"] and a["episode"]["r"] == b["episode"]["r"]
                    np.testing.assert_array_equal(a["terminal_observation"], b["terminal_observation"])
    for p in ("slab", "server"):
        np.testing.assert_array_equal(obs0["zero_copy"], obs0[p])
    assert n_done > 5
    assert venvs["server"].core.host_server_stats()["steps"] == T
    for v in venvs.values():
        v.close()


FULL_SIZE = [
    # BASELINE.json configs at their full per-GPU sizes (SURVEY 8d): (id, envs, track, env kwargs)
    ("cfg2_4096_circle", 4096, "circle", {}),
    ("cfg3_65536_reaching", 65536, "reaching", {}),
    ("cfg4_16384_drag_gnd", 16384, "circle", {"physics": "PYB_GND_DRAG_DW"}),
    ("cfg5_131072_reward_her", 131072, "circle", {"reward_id": 3}),
    ("cfg5_131072_reward_progress", 131072, "circle", {"reward_id": 5}),
    ("cfg5_131072_reward_reaching", 131072, "circle", {"reward_id": 4}),
    ("cfg5_131072_reward_flythru_normrew", 131072, "circle", {"reward_id": 7, "normalize_reward": True, "clip_reward": 10.0}),
    ("cfg5_131072_reward_bootstrapped", 131072, "circle", {"reward_id": 8}),
    ("cfg5_131072_reward_champ", 131072, "circle", {"reward_id": 9}),
]


@pytest.mark.parametrize("name,N,track,kw", FULL_SIZE, ids=[c[0] for c in FULL_SIZE])
def test_full_size_properties(name, N, track, kw):
    """BASELINE config sizes (S = 8): size-independent properties -- identical action rows give identical env rows
    (bit for bit), unit quaternions, finite outputs, done <=> state reset, Monitor statistics consistent with the
    done bits, and a seeded sample of 16 envs agrees with the oracle stepped on the same actions."""
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    kw = dict(kw)
    okw = {}
    if "physics" in kw:
        kw["physics"] = getattr(Physics, kw["physics"])
        okw["physics"] = "dyn_gnd_drag"
    rid = {0: "default", 3: "her", 4: "reaching", 5: "progress", 7: "flythrugate", 8: "bootstrapped", 9: "champ"}[kw.get("reward_id", 0)]
    ref = make_reference_env(track, pyb_freq=240, ctrl_freq=30)
    env = BatchedDroneEnv(N, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS,
                          pyb_freq=240, ctrl_freq=30, circle=(track == "circle"), include_distance=True, normalize_actions=True, **kw)
    sample = np.linspace(0, N // 2 - 1, 16).astype(int)
    workers = [OracleWorker(make_reference_env(track, pyb_freq=240, ctrl_freq=30, reward_id=rid, **okw), normalize_obs=False,
                            normalize_reward=kw.get("normalize_reward", False), clip_reward=kw.get("clip_reward", 0.0)) for _ in sample]
    env.reset()
    for w in workers:
        w.reset()
    g = torch.Generator(device="cpu").manual_seed(N)
    n_done = 0
    for t in range(24):
        half = (torch.rand(N // 2, 4, generator=g) * 2 - 1)
        if t % 3:
            half = HOVER + 0.006 * half                                 # mix of saturating and near-hover steps
        a = torch.cat([half, half]).to(env.device)                      # env i and i + N/2 see the same actions
        o, r, d, f = env.step(a)
        assert torch.isfinite(o).all() and torch.isfinite(r).all()
        assert torch.equal(o[: N // 2], o[N // 2:]) and torch.equal(r[: N // 2], r[N // 2:]) and torch.equal(d[: N // 2], d[N // 2:])
        st = env.get_state()
        qn = (st["quat"] ** 2).sum(dim=1)
        assert float((qn - 1).abs().max()) < 1e-5
        done = d != 0
        n_done += int(done.sum())
        assert bool((st["steps"][done] == 0).all()) and bool((st["target_idx"][done] == 0).all())
        assert bool((st["steps"][~done] > 0).all())
        on, rn, dn, an = o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy(), half.numpy()
        for j, w in zip(sample, workers):
            oo, rr, dd, info = w.step(an[j])
            bits = (1 if w.last_terminated else 0) | (2 if w.last_truncated else 0)
            if int(dn[j]) != bits:
                assert PU.min_margin(w.env) < 10 * PU.MARGIN_TOL, (name, t, j)   # open loop over 24 steps: near-tie only
                pytest.skip("near-tie between FP32 and FP64 on a sampled env (open loop)")
            assert PU.obs_error(on[j], oo, w.last_step_ang_v_norm) < 1e-3, (name, t, j)
            assert abs(float(rn[j]) - float(rr)) <= 1e-2 + 2e-3 * abs(float(rr)), (name, t, j, rn[j], rr)
    stats = env.episode_stats()
    assert stats["episodes"] == n_done and n_done > 0
    if rid in ("default", "her", "progress"):
        assert stats["crashes"] + stats["truncations"] + stats["successes"] == n_done
    env.close()


@pytest.mark.parametrize("mode", ["line", "midpoint"])
@pytest.mark.parametrize("track", ["circle", "reaching"])
def test_random_spawn_philox_matches_oracle_and_is_shard_invariant(track, mode):
    """DN_SPAWN_LINE (Philox-seeded auto-reset): the CUDA path against the oracle's restatement of the same draws,
    and invariance to sharding -- env g of a shard with env_id_offset = k behaves exactly like env k + g of one big
    handle (Philox subsequence = GLOBAL env id, SURVEY 8e)."""
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    from tests.test_host_emulation import _open_loop
    N, T, S, seed = 8, 120, 8, 0x1234ABCD5678
    ref = make_reference_env(track, pyb_freq=240, ctrl_freq=240 // S)
    mk = lambda n, off: BatchedDroneEnv(n, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS,
                                        pyb_freq=240, ctrl_freq=240 // S, circle=(track == "circle"), include_distance=True,
                                        normalize_actions=True, random_spawn=mode, seed=seed, env_id_offset=off)
    big, shard = mk(N, 100), mk(N // 2, 100 + N // 2)
    workers = [OracleWorker(make_reference_env(track, pyb_freq=240, ctrl_freq=240 // S, random_spawn=mode, seed=seed,
                                               global_env_id=100 + i), normalize_obs=False) for i in range(N)]
    o_big, o_sh = big.reset().cpu().numpy(), shard.reset().cpu().numpy()
    np.testing.assert_array_equal(o_big[N // 2:], o_sh)
    for i, w in enumerate(workers):
        np.testing.assert_allclose(o_big[i], w.reset()[0], atol=2e-6)
    acts = _actions("saturating", T, N, seed=5)

    def step(a):
        o, r, d, f = [x.cpu().numpy().copy() for x in big.step(torch.from_numpy(a).cuda())]
        o2, r2, d2, f2 = [x.cpu().numpy() for x in shard.step(torch.from_numpy(np.ascontiguousarray(a[N // 2:])).cuda())]
        np.testing.assert_array_equal(o[N // 2:], o2)
        np.testing.assert_array_equal(r[N // 2:], r2)
        np.testing.assert_array_equal(d[N // 2:], d2)
        return o, r, d, f
    resets = _open_loop(step, workers, acts)
    assert resets >= 10
    sp = big.get_state()["spawn"].cpu().numpy()[:, :3]
    want = np.stack([w.env.INIT_XYZS[0] for w in workers])
    np.testing.assert_allclose(sp, want, atol=2e-6)
    big.close(); shard.close()


def test_vec_env_collect_rollouts_text_format(tmp_path):
    """collect_rollouts=True (PBDroneEnv.py:152-157,811-821): one text file per env, each line the 13 raw observation
    floats formatted with np.format_float_positional(np.float32(x), unique=False, precision=32) then the reward; the
    NormalizeObservation wrapper then runs on the host with the reference's float64 per-env statistics."""
    from drl_dronenavigation_b200.vec_env import GpuDroneVecEnv
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    N, T = 3, 40
    ref = make_reference_env("circle")
    venv = GpuDroneVecEnv(N, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS, circle=True,
                          include_distance=True, normalize_actions=True, normalize_obs=True, collect_rollouts=True,
                          rollout_dir=str(tmp_path / "rollouts"))
    workers = [OracleWorker(make_reference_env("circle"), normalize_obs=True) for _ in range(N)]
    raw_workers = [OracleWorker(make_reference_env("circle"), normalize_obs=False) for _ in range(N)]
    obs = venv.reset()
    for i, w in enumerate(workers):
        np.testing.assert_allclose(obs[i], w.reset()[0], atol=2e-5)
        raw_workers[i].reset()
    acts = _actions("saturating", T, N, seed=3)
    want_lines = [[] for _ in range(N)]
    for t in range(T):
        o, r, d, infos = venv.step(acts[t])
        for i, w in enumerate(workers):
            oo, rr, dd, info = w.step(acts[t, i])
            ro, _, rd, rinfo = raw_workers[i].step(acts[t, i])
            want_lines[i].append((rinfo["terminal_observation"] if rd else ro, rr))
            assert bool(d[i]) == bool(dd)
            np.testing.assert_allclose(o[i][:9], oo[:9], atol=2e-3, rtol=2e-3)
            if dd:
                np.testing.assert_allclose(infos[i]["terminal_observation"][:9], info["terminal_observation"][:9], atol=2e-3, rtol=2e-3)
    venv.close()
    assert [p.split("rollout_")[-1] for p in venv.rollout_paths] == ["1.txt", "2.txt", "3.txt"]
    for i, path in enumerate(venv.rollout_paths):
        lines = open(path).read().strip().split("\n")
        assert len(lines) == T
        for line, (wo, wr) in zip(lines, want_lines[i]):
            cells = line.split(",")
            assert len(cells) == 14                                   # 13 observation floats + reward
            got = np.array([float(c) for c in cells])
            e = np.abs(got[:13] - wo)
            e[3:6] = np.minimum(e[3:6], np.abs(2 - e[3:6]))
            assert max(e[:9].max(), e[12]) < 2e-4 and abs(got[13] - float(wr)) < 2e-3
            assert all("e" not in c.lower() for c in cells[:13])      # positional notation, as the reference writes it


def test_vec_env_save_and_load_running_stats(tmp_path):
    """eval_env.save(path) (PBDroneSimulator.py:746) and its counterpart: the per-env obs / reward statistics survive a
    round trip, so a restored env normalises the next observation exactly like the one that was saved."""
    from drl_dronenavigation_b200.vec_env import GpuDroneVecEnv
    from oracle.dyn_oracle import make_reference_env
    ref = make_reference_env("circle")
    mk = lambda: GpuDroneVecEnv(5, ref._target_points, aviary_dim=ref._aviary_dim, initial_xyzs=ref.INIT_XYZS, circle=True,
                                include_distance=True, normalize_actions=True, normalize_obs=True, normalize_reward=True)
    a, b = mk(), mk()
    a.reset(); b.reset()
    acts = _actions("mixed", 30, 5, seed=2)
    for t in range(20):
        a.step(acts[t])
    path = str(tmp_path / "vec_normalize.pkl")
    a.save(path)
    b.load_running_stats(path)
    sa, sb = a.core.get_state(), b.core.get_state()
    assert torch.equal(sa["obs_rms"], sb["obs_rms"]) and torch.equal(sa["rew_rms"], sb["rew_rms"])
    assert float(sa["obs_rms"][:, -1].min()) > 20          # counts advanced
    a.close(); b.close()


def test_gymnasium_facade_against_oracle_env():
    """PBDroneEnv facade (single env, gymnasium 5-tuple): reset / step / terminal step / reset again against the oracle
    env, including the attributes the manager pokes (pos, rpy, INIT_XYZS, CTRL_FREQ) and _getDroneStateVector."""
    from drl_dronenavigation_b200.env import PBDroneEnv
    from oracle.dyn_oracle import make_reference_env
    ref = make_reference_env("circle", pyb_freq=240, ctrl_freq=30)
    env = PBDroneEnv(target_points=ref._target_points, threshold=0.3, discount=0.999, max_steps=4096, aviary_dim=ref._aviary_dim,
                     initial_xyzs=ref.INIT_XYZS, pyb_freq=240, ctrl_freq=30, cylinder=True, circle=True, include_distance=True,
                     normalize_actions=True)
    assert env.action_space.shape == (4,) and env.observation_space.shape == (13,) and env.CTRL_FREQ == 30
    obs, info = env.reset(seed=3)
    o_ref, _ = ref.reset()
    np.testing.assert_allclose(obs, o_ref, atol=1e-6)
    assert info == {"found_targets": 0}
    acts = _actions("mixed", 80, 1, seed=9)[:, 0]
    episodes = 0
    for t in range(80):
        o, r, term, trunc, info = env.step(acts[t])
        oo, rr, tt, tr, ii = ref.step(acts[t])
        assert (term, trunc) == (bool(tt), bool(tr)) and info["found_targets"] == ii["found_targets"]
        assert PU.obs_error(o, oo, float(np.linalg.norm(ref.ang_v))) < 1e-3 and abs(r - float(rr)) < 1e-2
        if not (term or trunc):
            sv = env._getDroneStateVector(0)
            assert sv.shape == (20,)
            np.testing.assert_allclose(sv[0:3], ref.pos, atol=1e-4)
            np.testing.assert_allclose(sv[10:13], ref.vel, atol=1e-3)
            np.testing.assert_allclose(sv[16:20], np.float64(ref.last_clipped_action), rtol=1e-6)
            np.testing.assert_allclose(env.rpy[0], ref.rpy, atol=1e-4)
        else:
            episodes += 1
            obs, _ = env.reset()
            o_ref, _ = ref.reset()
            np.testing.assert_allclose(obs, o_ref, atol=1e-5)
            assert np.all(env._getDroneStateVector(0)[16:20] == 0)
    assert episodes >= 1
    env.close()



@pytest.mark.parametrize("model,act,track,S,T,resync", PU.CONTROLLER_CASES)
def test_airframes_and_controller_action_types_lockstep(model, act, track, S, T, resync):
    """DroneModel.CF2P / RACE (BaseAviary.py:927-935) and BaseSingleAgentAviary's action types incl. the fused
    DSLPIDControl: the CUDA path against the oracle in lock-step over 24 envs (see parity_utils.controller_lockstep_case)."""
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.enums import ActionType, DroneModel

    def make(N, targets, init, dim):
        return BatchedDroneEnv(N, targets, threshold=0.3, discount=0.999, max_steps=4096, aviary_dim=dim, initial_xyzs=init,
                               pyb_freq=240, ctrl_freq=240 // S, cylinder=True, circle=(track == "circle"), include_distance=True,
                               act=ActionType(act), drone_model=DroneModel(model))
    env, workers = PU.controller_lockstep_case(make, 24, model, act, track, S, T, resync,
                                               get_pid=lambda e: e.get_state()["pid"].cpu().numpy())
    if act in ("pid", "vel", "one_d_pid"):
        with pytest.raises(Exception, match="not elementwise"):
            env.action_to_rpm(torch.zeros(4, device=env.device))
    env.close()


@pytest.mark.parametrize("track,S,mode,N,T,kw", [
    ("circle", 8, "saturating", 4096, 240, {}),          # BASELINE config 2 at its full size, 8 s of flight per environment
    ("circle", 8, "hover_band", 4096, 120, {}),
    ("reaching", 8, "mixed", 65536, 45, {}),             # BASELINE config 3's per-GPU shard (segment tube)
    ("circle", 1, "saturating", 4096, 480, {"reward_id": "dummy"}),
    ("reaching", 8, "saturating", 16384, 60, {"reward_id": "thrustenv"}),
    ("circle", 8, "mixed", 16384, 60, {"physics": "dyn_gnd_drag"}),              # BASELINE config 4: drag + ground effect, every env
    ("circle", 8, "saturating", 16384, 40, {"physics": "dyn_gnd_drag"}),
    ("circle", 8, "saturating", 131072, 30, {"reward_id": "thrustenv"}),         # BASELINE config 5's per-GPU shard, one reward of the sweep
    ("circle", 8, "saturating", 4096, 60, {"ground_contact": True}),             # analytic ground-plane contact
    ("reaching", 8, "mixed", 4096, 60, {"ground_contact": True, "physics": "dyn_gnd_drag"}),
], ids=["config2_saturating", "config2_hover_band", "config3_65536", "circle_s1_dummy", "reaching_thrustenv", "config4_16384_mixed",
        "config4_16384_saturating", "config5_131072_thrustenv", "ground_contact_circle", "ground_contact_reaching_gnd_drag"])
def test_full_size_lockstep_against_batched_oracle(track, S, mode, N, T, kw):
    """EVERY environment of the BASELINE shapes compared with the FP64 oracle at EVERY step (oracle/batched_oracle.py,
    itself checked against the per-environment oracle and the reference fixtures in tests/test_batched_oracle.py)."""
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.batched_oracle import BatchedOracle
    from oracle.dyn_oracle import circle_track, reaching_track
    from drl_dronenavigation_b200 import Physics
    rid = {"default": 0, "dummy": 1, "thrustenv": 2}[kw.get("reward_id", "default")]
    phys = {"dyn": Physics.DYN, "dyn_gnd_drag": Physics.PYB_GND_DRAG_DW}[kw.get("physics", "dyn")]
    targets, init, dim = circle_track() if track == "circle" else reaching_track()
    env = BatchedDroneEnv(N, targets, threshold=0.3, discount=0.999, max_steps=4096, aviary_dim=dim, initial_xyzs=init,
                          pyb_freq=240, ctrl_freq=240 // S, cylinder=True, circle=(track == "circle"), include_distance=True,
                          normalize_actions=True, reward_id=rid, physics=phys, ground_contact=kw.get("ground_contact", False))
    B = BatchedOracle(N, track, pyb_freq=240, ctrl_freq=240 // S, **kw)
    np.testing.assert_allclose(env.reset().cpu().numpy(), B.reset_obs(), atol=1e-6)
    rep = PU.run_lockstep_batched(env, B, _actions(mode, T, N, seed=N % 97 + S), resync_every=240 // S)
    print(f"\n[full size {track} S={S} {mode} N={N} T={T}] {rep}")
    assert rep.env_steps == N * T and rep.near_ties <= max(2, rep.env_steps // 20000), str(rep)
    assert rep.dones > 0 or mode == "hover_band"
    env.close()
