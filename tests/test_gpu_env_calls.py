"""The environment calls around the step itself: the Monitor totals of dn_episode_stats (also past 2^15 / 2^16 episodes per
dn_step_many launch), dn_reset with a mask against the FP64 oracle, and a dn_get_state / dn_set_state clone with every optional
plane.  GPU only.

Return-sum bound (parity_utils.return_sum_bound, u = 2^-24): dn_step sums at most 32 FP32 returns per warp in a 5-level shuffle
tree and adds those as FP64, so |return_sum - FP64 sum| <= 5 u sum|r| (plus 2^-53 sum|r| per FP64 addition).  dn_step_many first
adds the k episodes of a lane one after another: (k - 1 + 5) u sum|r|, k the most episodes of one lane between two flushes.
All counts are exact."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU

pytestmark = pytest.mark.gpu

HOVER = 0.092227
COUNTS = ("episodes", "length_sum", "found_targets", "successes", "crashes", "truncations")


def _env(N, track="circle", S=8, max_steps=4096, **kw):
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from oracle.dyn_oracle import circle_track, reaching_track
    targets, init, dim = circle_track() if track == "circle" else reaching_track()
    return BatchedDroneEnv(N, targets, threshold=0.3, discount=0.999, max_steps=max_steps, aviary_dim=dim, initial_xyzs=init,
                           pyb_freq=240, ctrl_freq=240 // S, cylinder=True, circle=(track == "circle"), include_distance=True,
                           normalize_actions=True, **kw)


def _saturating(T, N, seed):
    return np.random.default_rng(seed).uniform(-1, 1, size=(T, N, 4)).astype(np.float32)


def _bits_equal(a, b):
    if a.dtype.is_floating_point:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return torch.equal(a, b)


def _outputs(N, D, dev, lead=()):
    """All eight dn_step_io outputs, filled with sentinels (NaN / -1)."""
    nan = float("nan")
    return dict(obs=torch.full((*lead, N, D), nan, device=dev), terminal_obs=torch.full((*lead, N, D), nan, device=dev),
                reward=torch.full((*lead, N), nan, device=dev), done=torch.full((*lead, N), 255, dtype=torch.uint8, device=dev),
                found_targets=torch.full((*lead, N), -1, dtype=torch.int32, device=dev),
                episode_return=torch.full((*lead, N), nan, device=dev),
                episode_length=torch.full((*lead, N), -1, dtype=torch.int32, device=dev))


# --------------------------------------------------------------------------------------------------------------------------
# a. Monitor counters of one dn_step_many launch past 2^15 and 2^16 episodes per lane
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [32769, 65537, 3 * 32767 + 5])
def test_step_many_monitor_counters_past_2_15_and_2_16_episodes_per_launch(T):
    """max_steps = 0: every step of every env truncates, so one launch ends T episodes per lane.  The counts are exact and the
    return sum is within the dn_step_many bound (k <= 32767 between two flushes) of the FP64 sum of the returns a twin env
    emits when it runs the same actions in launches of at most 1000 steps; the final states are bit-identical."""
    N = 100                                                   # the second warp of the last CTA is partial
    X, Y = _env(N, S=1, max_steps=0), _env(N, S=1, max_steps=0)
    X.reset(); Y.reset()
    dev, D = X.device, X.obs_dim
    acts = torch.full((T, N, 4), HOVER, device=dev)
    outX = _outputs(N, D, dev)
    X.step_many(acts, per_step_outputs=False, out=outX)
    ret_sum = torch.zeros((), dtype=torch.float64, device=dev)
    abs_sum = torch.zeros((), dtype=torch.float64, device=dev)
    for t0 in range(0, T, 1000):
        t1 = min(T, t0 + 1000)
        o = _outputs(N, D, dev, lead=(t1 - t0,))
        Y.step_many(acts[t0:t1], per_step_outputs=True, out=o)
        assert bool((o["done"] == 2).all()) and bool((o["episode_length"] == 1).all())
        ret_sum += o["episode_return"].double().sum()
        abs_sum += o["episode_return"].double().abs().sum()
    for k in ("obs", "reward", "done", "found_targets", "terminal_obs", "episode_return", "episode_length"):
        assert _bits_equal(outX[k], o[k][-1]), k
    sx, sy = X.get_state(), Y.get_state()
    for k in sx:
        assert _bits_equal(sx[k], sy[k]), k
    NT = N * T
    for name, env, k in (("one launch", X, 32767), ("launches of 1000 steps", Y, 1000)):
        st = env.episode_stats()
        assert st["episodes"] == st["truncations"] == st["length_sum"] == NT, (name, st)
        assert st["crashes"] == st["successes"] == st["found_targets"] == 0, (name, st)
        ref, a = float(ret_sum), float(abs_sum)
        assert abs(st["return_sum"] - ref) <= PU.return_sum_bound(a, NT, k), (name, st["return_sum"], ref)
    X.close(); Y.close()


# --------------------------------------------------------------------------------------------------------------------------
# b. Monitor totals of dn_step against the per-episode outputs the kernel emits
# --------------------------------------------------------------------------------------------------------------------------
def test_step_monitor_totals_match_emitted_episode_outputs():
    """4096 envs, 240 dn_step launches on the circle track (S = 8, default reward, max_steps = 60): even envs fly saturating
    actions (crashes), odd envs hover, and every 40 steps an eighth of the envs is placed next to the final target (successes)
    and another eighth at the step limit (truncations).  Every count of dn_episode_stats equals the one recounted from done /
    found / episode_length of every step; return_sum is within 5 u sum|r| of the FP64 sum of episode_return.  clear = False is idempotent, clear = True returns the
    totals once and zeroes them."""
    N, T, n_targets = 4096, 240, 6
    env = _env(N, S=8, max_steps=60)
    env.reset()
    dev = env.device
    acts = _saturating(T, N, seed=31)
    rng = np.random.default_rng(32)
    acts[:, 1::2] = HOVER + 0.002 * rng.uniform(-1, 1, size=acts[:, 1::2].shape)
    acts = torch.from_numpy(acts).to(dev)
    final = torch.tensor(env.target_points[-1], dtype=torch.float32, device=dev)
    done_all, found_all, len_all, ret_all = [], [], [], []
    for t in range(T):
        if t % 40 == 5:
            sel = torch.arange(N, device=dev) % 8 == (t // 40) % 8
            at_limit = torch.arange(N, device=dev) % 8 == (t // 40 + 4) % 8
            st = env.get_state()
            pos = st["pos"].clone()
            pos[sel] = final + 0.05 * torch.from_numpy(rng.uniform(-1, 1, size=(int(sel.sum()), 3)).astype(np.float32)).to(dev)
            dist = (pos - final).norm(dim=1)
            new = {k: st[k].clone() for k in ("quat", "vel", "rpy_rates", "ang_v", "target_idx", "steps", "just_found", "dist", "prev_dist")}
            new["quat"][sel] = torch.tensor([0.0, 0.0, 0.0, 1.0], device=dev)
            for k in ("vel", "rpy_rates", "ang_v"):
                new[k][sel] = 0.0
            new["target_idx"][sel] = n_targets - 1
            new["steps"][sel] = 10
            new["steps"][at_limit] = 60
            new["just_found"][sel] = 0
            new["dist"][sel] = dist[sel]
            new["prev_dist"][sel] = dist[sel]
            env.set_state(dict(pos=pos, **new))
        o, r, d, f = env.step(acts[t])
        done = d != 0
        done_all.append(d.clone()); found_all.append(f[done].clone())
        len_all.append(env.episode_length[done].clone()); ret_all.append(env.episode_return[done].double())
    d = torch.stack(done_all)
    found, lens, rets = torch.cat(found_all), torch.cat(len_all), torch.cat(ret_all)
    dd = d[d != 0]
    term = (dd & 1) != 0
    succ = term & (found == n_targets)
    want = dict(episodes=int((d != 0).sum()), length_sum=int(lens.long().sum()), found_targets=int(found.long().sum()),
                truncations=int((dd == 2).sum()), successes=int(succ.sum()), crashes=int((term & ~succ).sum()))
    s1 = env.episode_stats(clear=False)
    s2 = env.episode_stats(clear=False)
    assert s1 == s2
    assert {k: s1[k] for k in COUNTS} == want, (s1, want)
    assert want["successes"] > 0 and want["crashes"] > 0 and want["truncations"] > 0, want
    ref, a = float(rets.sum()), float(rets.abs().sum())
    assert abs(s1["return_sum"] - ref) <= PU.return_sum_bound(a, rets.numel(), 1), (s1["return_sum"], ref)
    assert env.episode_stats(clear=True) == s1
    assert all(v == 0 for v in env.episode_stats().values())
    env.close()


# --------------------------------------------------------------------------------------------------------------------------
# c. dn_reset with a mask against the oracle
# --------------------------------------------------------------------------------------------------------------------------
SEED, OFFSET = 0x5EED1234, 1000
RESET_CASES = [
    # (id, track, env keywords, oracle keywords, normalize_obs)
    ("circle_normobs", "circle", {}, {}, True),
    ("reaching_line_rw4", "reaching", {"random_spawn": "line", "reward_id": 4, "seed": SEED, "env_id_offset": OFFSET},
     {"random_spawn": "line", "reward_id": "reaching", "seed": SEED}, False),
    ("reaching_midpoint_rw4", "reaching", {"random_spawn": "midpoint", "reward_id": 4, "seed": SEED, "env_id_offset": OFFSET},
     {"random_spawn": "midpoint", "reward_id": "reaching", "seed": SEED}, False),
    ("circle_drag_gnd", "circle", {"physics": "PYB_GND_DRAG_DW"}, {"physics": "dyn_gnd_drag"}, False),
]


def _reset_pair(N, track, kw, okw, norm, S=8):
    from drl_dronenavigation_b200 import Physics
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    kw = dict(kw)
    if "physics" in kw:
        kw["physics"] = getattr(Physics, kw["physics"])
    env = _env(N, track, S=S, normalize_obs=norm, **kw)
    gid = (lambda i: {"global_env_id": OFFSET + i}) if "random_spawn" in okw else (lambda i: {})
    workers = [OracleWorker(make_reference_env(track, pyb_freq=240, ctrl_freq=240 // S, **okw, **gid(i)), normalize_obs=norm)
               for i in range(N)]
    return env, workers


@pytest.mark.parametrize("track,kw,okw,norm", [c[1:] for c in RESET_CASES], ids=[c[0] for c in RESET_CASES])
def test_masked_reset_against_oracle(track, kw, okw, norm):
    """20 lock-step control steps with the oracle workers, then dn_reset on a seeded ~40 % mask (one env with steps == 0, the
    stale-distance branch, forced in; one env forced out): the masked rows get the oracle's reset observation and a zeroed
    episode (with a random spawn: the next Philox draw and the oracle's spawn point); the other rows, obs and every state
    field, are bit-identical to before; the Monitor statistics do not move.  Then one more horizon in lock-step.
    NormalizeObservation amplifies FP32 state differences by 1 / sqrt(var) of a few samples (the direction entries of a
    near-zero angular velocity most): there the lock-step phases compare the discrete outputs, rewards and states but not the
    observations, and the oracle workers take the kernel's FP64 running statistics before the reset, so the normalised
    reset observations are compared with the vec-env tolerance."""
    N, S = 300, 8                                             # 300 = one full and one partial 256-thread block of reset_kernel
    env, workers = _reset_pair(N, track, kw, okw, norm, S)
    obs_tol = np.inf if norm else PU.OBS_TOL
    reset_tol = 2e-3 if norm else 2e-6
    o0 = env.reset().cpu().numpy()
    for i, w in enumerate(workers):
        np.testing.assert_allclose(o0[i], w.reset()[0], atol=reset_tol)
    acts = _saturating(50, N, seed=41)
    PU.run_lockstep(env, workers, acts[:20], resync_every=240 // S, obs_tol=obs_tol)   # ends with the oracle state uploaded
    before = {k: v.clone() for k, v in env.get_state().items()}
    obs_before = env.obs.clone()
    stats_before = env.episode_stats()
    rng = np.random.default_rng(42)
    mask = rng.random(N) < 0.4
    zero = np.nonzero(before["steps"].cpu().numpy() == 0)[0]
    assert zero.size > 0
    mask[zero[0]] = True
    out = int(np.nonzero(mask)[0][np.nonzero(mask)[0] != zero[0]][0])
    mask[out] = False
    if norm:
        rms = before["obs_rms"].cpu().numpy()
        D = env.obs_dim
        for i, w in enumerate(workers):
            w.obs_rms.mean, w.obs_rms.var, w.obs_rms.count = rms[i, :D].copy(), rms[i, D:2 * D].copy(), float(rms[i, 2 * D])
    obs = env.reset(torch.from_numpy(mask.astype(np.uint8))).cpu().numpy()
    after = env.get_state()
    m = torch.from_numpy(mask).to(env.device)
    for i in np.nonzero(mask)[0]:
        np.testing.assert_allclose(obs[i], workers[i].reset()[0], atol=reset_tol, err_msg=f"env {i}")
    for k in ("steps", "target_idx", "ep_length"):
        assert bool((after[k][m] == 0).all()), k
    assert bool((after["ep_return"][m] == 0).all())
    if "random_spawn" in kw:
        assert torch.equal(after["episode_count"][m], before["episode_count"][m] + 1)
        want = np.stack([workers[i].env.INIT_XYZS[0] for i in np.nonzero(mask)[0]])
        np.testing.assert_allclose(after["spawn"][m][:, :3].cpu().numpy(), want, atol=2e-6)
    else:
        assert torch.equal(after["episode_count"], before["episode_count"])
    assert _bits_equal(env.obs[~m], obs_before[~m])
    for k in before:
        assert _bits_equal(after[k][~m], before[k][~m]), k
    assert env.episode_stats() == stats_before
    rep = PU.run_lockstep(env, workers, acts[20:], resync_every=240 // S, obs_tol=obs_tol)
    assert rep.near_ties <= 2, str(rep)
    env.close()


def test_reset_edge_masks():
    """An all-zero mask changes nothing; mask = None is bit-identical to an all-ones mask (on a twin env)."""
    N = 300
    _, track, kw, _, _ = RESET_CASES[1]
    A, B = _env(N, track, **kw), _env(N, track, **kw)
    acts = torch.from_numpy(_saturating(20, N, seed=43)).to(A.device)
    for e in (A, B):
        e.reset()
        for t in range(20):
            e.step(acts[t])
    sa, oa = A.get_state(), A.obs.clone()
    A.reset(torch.zeros(N, dtype=torch.uint8))
    assert _bits_equal(A.obs, oa)
    for k, v in A.get_state().items():
        assert _bits_equal(v, sa[k]), k
    A.reset(None)
    B.reset(torch.ones(N, dtype=torch.uint8))
    assert _bits_equal(A.obs, B.obs)
    sa, sb = A.get_state(), B.get_state()
    for k in sa:
        assert _bits_equal(sa[k], sb[k]), k
    A.close(); B.close()


# --------------------------------------------------------------------------------------------------------------------------
# d. dn_get_state / dn_set_state clone
# --------------------------------------------------------------------------------------------------------------------------
CLONE_CASES = [
    ("drag_gnd", "circle", {"physics": "PYB_GND_DRAG_DW"}),
    ("normobs_normrew_clip", "circle", {"normalize_obs": True, "normalize_reward": True, "clip_reward": 10.0}),
    ("midpoint_rw4", "reaching", {"random_spawn": "midpoint", "reward_id": 4, "seed": 91}),
    ("rw8", "circle", {"reward_id": 8}),
    ("cf2p_pid", "circle", {"act": "PID", "drone_model": "CF2P"}),
    ("vel", "circle", {"act": "VEL"}),
]


@pytest.mark.parametrize("track,kw", [c[1:] for c in CLONE_CASES], ids=[c[0] for c in CLONE_CASES])
def test_state_clone_continues_bit_identically(track, kw):
    """Env A steps 30 steps; a fresh env B takes A.get_state() through set_state; both step 30 more on the same actions: every
    output (terminal and episode outputs included), the final states and the statistics are identical -- so dn_state_view
    carries every per-env state.  Then a subset of fields is uploaded and the others stay unchanged."""
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200.enums import ActionType, DroneModel
    kw = dict(kw)
    for key, enum in (("physics", Physics), ("act", ActionType), ("drone_model", DroneModel)):
        if key in kw:
            kw[key] = getattr(enum, kw[key])
    N = 1000
    A = _env(N, track, **kw)
    A.reset()
    acts = torch.from_numpy(_saturating(60, N, seed=51)).to(A.device)
    for t in range(30):
        A.step(acts[t])
    A.episode_stats(clear=True)
    B = _env(N, track, **kw)
    B.set_state(A.get_state())
    n_done = 0
    for t in range(30, 60):
        oa, ra, da, fa = [x.clone() for x in A.step(acts[t])]
        ob, rb, db, fb = B.step(acts[t])
        assert _bits_equal(oa, ob) and _bits_equal(ra, rb) and torch.equal(da, db) and torch.equal(fa, fb), t
        done = da != 0
        n_done += int(done.sum())
        assert _bits_equal(A.terminal_obs[done], B.terminal_obs[done]), t
        assert _bits_equal(A.episode_return[done], B.episode_return[done]), t
        assert torch.equal(A.episode_length[done], B.episode_length[done]), t
    assert n_done > 0
    sa, sb = A.get_state(), B.get_state()
    for k in sa:
        assert _bits_equal(sa[k], sb[k]), k
    ta, tb = A.episode_stats(), B.episode_stats()
    assert {k: ta[k] for k in COUNTS} == {k: tb[k] for k in COUNTS}
    assert ta["return_sum"] == pytest.approx(tb["return_sum"], rel=1e-12, abs=1e-12)   # FP64 slot additions in arrival order
    # a subset upload leaves every other field alone
    part = {"pos": sa["pos"] + 0.125, "ep_length": sa["ep_length"] + 7}
    B.set_state(part)
    sb = B.get_state()
    for k in sa:
        assert _bits_equal(sb[k], part[k] if k in part else sa[k]), k
    A.close(); B.close()
